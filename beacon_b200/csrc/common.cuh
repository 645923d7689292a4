// Shared device/host helpers for the beacon_b200 kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/beacon_b200.h"

namespace beacon {

// ---------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

#define BEACON_CUDA_CHECK(expr)                                                                  \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            throw ::beacon::Error(BEACON_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

#define BEACON_REQUIRE(cond, msg)                                        \
    do {                                                                 \
        if (!(cond)) throw ::beacon::Error(BEACON_ERR_INVALID, (msg));   \
    } while (0)

// ---------------------------------------------------------------------------------------
// device math helpers
// ---------------------------------------------------------------------------------------
template <typename R> struct real_traits;
template <> struct real_traits<double> { static constexpr int dtype = BEACON_F64; };
template <> struct real_traits<float> { static constexpr int dtype = BEACON_F32; };

// numpy maximum/minimum: NaN from either argument propagates (CUDA fmin/fmax drop it).
template <typename R> __device__ __forceinline__ R np_max(R a, R b) { return (a != a) ? a : (a > b ? a : b); }
template <typename R> __device__ __forceinline__ R np_min(R a, R b) { return (a != a) ? a : (a < b ? a : b); }

template <typename R> __device__ __forceinline__ R rabs(R x);
template <> __device__ __forceinline__ double rabs(double x) { return fabs(x); }
template <> __device__ __forceinline__ float rabs(float x) { return fabsf(x); }
template <typename R> __device__ __forceinline__ R rsqrt_(R x);
template <> __device__ __forceinline__ double rsqrt_(double x) { return sqrt(x); }
template <> __device__ __forceinline__ float rsqrt_(float x) { return sqrtf(x); }

template <typename R> __device__ __forceinline__ bool finite_(R x) { return isfinite(x); }

// Branch-free division for the hot loops.  nvcc's IEEE fp64 division is a ~25-instruction
// sequence with a range test and a call to a slow path per division: the branches stop the
// scheduler from interleaving independent divisions and the kernels become latency bound.
// fdiv: MUFU.RCP64H seed y0 (measured max relative error 2^-19.9 on B200), ONE cubic step
// a/b = a y0 (1 + e + e^2), e = 1 - b y0 (error e^3 = 2^-60): two roundings on top of it, i.e. a
// quotient within 2 ulp (tools/micro/rcpacc.cu measures the variants); the parity contract is
// 1e-10.  A zero / denormal / non-finite divisor or an overflowing quotient gives NaN or inf like
// the IEEE sequence up to the case b = +-0 with a != 0 (NaN instead of +-inf); none of the divisors
// on these paths can be exactly zero (they are sums with a positive epsilon) and non-finite states
// are flagged in `status`.
__device__ __forceinline__ double fdiv(double a, double b)
{
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(b));
    const double e = fma(-b, y, 1.0);
    // a/b = (a y0)(1 + e + e^2): the product a y0 does not wait for the refinement (dependent chain
    // MUFU -> FMA -> FMA -> FMA instead of MUFU -> FMA -> FMA -> FMA -> MUL), same four fp64 instructions
    const double q0 = a * y;
    return fma(q0, fma(e, e, e), q0);
}
// 0.5 a / b with the halving done on the exponent of the reciprocal seed by the integer pipe (the
// seed is 1/b to 20 bits: never zero or denormal for the finite divisors of these paths).
__device__ __forceinline__ double fdiv_half(double a, double b)
{
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(b));
    const double e = fma(-b, y, 1.0);
    const double hy = __hiloint2double(__double2hiint(y) - 0x00100000, 0);
    const double q0 = a * hy;
    return fma(q0, fma(e, e, e), q0);
}
__device__ __forceinline__ float fdiv_half(float a, float b) { return 0.5f * (a / b); }
// clamp(r, 0, 1) = max(0, min(r, 1)) decided on the high word with integer compares (the fp64
// pipe is the bottleneck of these kernels): sign bit -> 0, exponent >= 0 -> 1, else r.
// -0.0 -> 0.  A NaN ratio gives 0 or 1 instead of NaN (numpy's maximum/minimum would propagate
// it): the NaN lattice value that caused it persists and spreads through the other stencil
// terms, and the env is flagged BEACON_STATUS_NONFINITE, so nothing is hidden.
__device__ __forceinline__ double clamp01(double r)
{
    const int hi = __double2hiint(r);
    return hi < 0 ? 0.0 : (hi >= 0x3ff00000 ? 1.0 : r);
}
__device__ __forceinline__ float clamp01(float r) { return r < 0.0f ? 0.0f : (r > 1.0f ? 1.0f : r); }
// 0.5 * clamp(r, 0, 1) (half of the minmod limiter; the halving is exact) with the clamp done on the
// words of 0.5 r by the integer pipe: high word = max(min(hi, hi(0.5)), 0), low word cleared when
// either bound is active (one unsigned compare covers the sign bit and hi >= hi(0.5)).
// Same NaN / -0.0 behaviour as clamp01.
__device__ __forceinline__ double half_clamp01(double r)
{
    const double hr = 0.5 * r;
    int hi = __double2hiint(hr), lo = __double2loint(hr);
    lo = ((unsigned)hi >= 0x3fe00000u) ? 0 : lo;
    hi = max(min(hi, 0x3fe00000), 0);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ float half_clamp01(float r) { return 0.5f * clamp01(r); }
// clamp(hr, 0, 0.5) for an already halved ratio
__device__ __forceinline__ double clamp0h(double hr)
{
    int hi = __double2hiint(hr), lo = __double2loint(hr);
    lo = ((unsigned)hi >= 0x3fe00000u) ? 0 : lo;
    hi = max(min(hi, 0x3fe00000), 0);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ float clamp0h(float hr) { return hr < 0.0f ? 0.0f : (hr > 0.5f ? 0.5f : hr); }
__device__ __forceinline__ float fdiv(float a, float b) { return a / b; }

// x / 3 without the reciprocal seed: q = x (1/3), one residual correction q += (x - 3 q)(1/3) — three dependent
// fp64 instructions instead of MUFU + four (the quotient is within 1 ulp of the correctly rounded one)
__device__ __forceinline__ double div3(double x)
{
    const double c = 1.0 / 3.0, q = x * c;
    return fma(fma(-3.0, q, x), c, q);
}
__device__ __forceinline__ float div3(float x) { return x / 3.0f; }
// sign / zero tests of floating-point values on the integer pipe (the fp64 pipe is the scarce resource)
__device__ __forceinline__ bool same_sign(double a, double b) { return (__double2hiint(a) ^ __double2hiint(b)) >= 0; }
__device__ __forceinline__ bool same_sign(float a, float b) { return (__float_as_int(a) ^ __float_as_int(b)) >= 0; }
__device__ __forceinline__ bool is_zero(double a) { return ((__double2hiint(a) & 0x7fffffff) | __double2loint(a)) == 0; }
__device__ __forceinline__ bool is_zero(float a) { return (__float_as_int(a) & 0x7fffffff) == 0; }
template <typename R> __device__ __forceinline__ R qnan();
template <> __device__ __forceinline__ double qnan<double>() { return __longlong_as_double(0x7ff8000000000000LL); }
template <> __device__ __forceinline__ float qnan<float>() { return __int_as_float(0x7fc00000); }

// Branch-free square root, same idea: MUFU.RSQ64H seed, two Newton steps on 1/sqrt(x), one
// residual correction of sqrt(x); x = 0 is mapped to 0 by a select; negative / non-finite -> NaN.
__device__ __forceinline__ double fsqrt(double x)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-(x * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-(x * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    double s = x * y;
    s = fma(0.5 * y, fma(-s, s, x), s);
    return x == 0.0 ? 0.0 : s;
}
__device__ __forceinline__ float fsqrt(float x) { return sqrtf(x); }

template <typename T> __device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block-wide sum: warp shuffles, then the warp partials are added in warp order
// by every thread (same order everywhere -> identical result in all threads).
// `scratch` needs blockDim.x/32 entries; contains two barriers.
template <typename T> __device__ __forceinline__ T block_sum(T v, T *scratch)
{
    v = warp_sum(v);
    const int nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    T r = scratch[0];
    for (int w = 1; w < nw; w++) r += scratch[w];
    return r;
}

// ---------------------------------------------------------------------------------------
// Bulk asynchronous copies (TMA engine, 1-D: cp.async.bulk -> SASS UBLKCP) between global memory
// and shared memory.  Per-env field planes are contiguous and 16-byte multiples (SURVEY.md
// appendix A), so a whole plane moves with one instruction issued by one thread, without
// passing through registers; completion of loads is signalled on an mbarrier (transaction
// bytes), stores are tracked by bulk groups.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.release.cta.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_all()
{
    asm volatile("cp.async.bulk.commit_group;\n\tcp.async.bulk.wait_group 0;" ::: "memory");
}
// generic-proxy accesses before <-> async-proxy (bulk copy) accesses after
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_async_gmem() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// ---------------------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG (Salmon et al. 2011).  One call -> 4 x 32 random bits.
// Counter = (draw index lo/hi, global env index lo/hi), key = seed: the noise an env sees
// depends only on (seed, global env index, draw index), never on batch size or sharding.
// ---------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)M0 * c[0], p1 = (uint64_t)M1 * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += W0; k1 += W1;
    }
}

// U(-sigma, sigma) from (seed, env, draw): 53-bit mantissa uniform in [0,1).
__host__ __device__ __forceinline__ double philox_uniform_pm(uint64_t seed, uint64_t env, uint64_t draw, double sigma)
{
    uint32_t c[4] = {(uint32_t)draw, (uint32_t)(draw >> 32), (uint32_t)env, (uint32_t)(env >> 32)};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    uint64_t bits = (((uint64_t)c[0] << 32) | c[1]) >> 11;
    double u = (double)bits * (1.0 / 9007199254740992.0);
    return -sigma + 2.0 * sigma * u;
}

// ---------------------------------------------------------------------------------------
// host-side env base: owns device buffers, exposes named state fields
// ---------------------------------------------------------------------------------------
struct DeviceBuffer {
    void *ptr = nullptr;
    size_t bytes = 0;
    DeviceBuffer() = default;
    DeviceBuffer(const DeviceBuffer &) = delete;
    DeviceBuffer &operator=(const DeviceBuffer &) = delete;
    ~DeviceBuffer() { if (ptr) cudaFree(ptr); }
    void alloc(size_t n)
    {
        if (ptr) { cudaFree(ptr); ptr = nullptr; }
        bytes = n;
        if (n) {
            BEACON_CUDA_CHECK(cudaMalloc(&ptr, n));
            BEACON_CUDA_CHECK(cudaMemset(ptr, 0, n));
        }
    }
    template <typename T> T *as() const { return static_cast<T *>(ptr); }
};

struct Field {
    std::string name;
    void *ptr;          // device pointer, [batch, count] contiguous
    int64_t count;      // elements per env
    int elem_bytes;     // 8/4 real, 4 int32
    bool is_int;
};

struct StepArgs {
    const void *actions; const void *noise; void *obs; void *rwd; uint8_t *done; uint8_t *trunc;
    int32_t *status; int64_t *iters; int32_t n_fused; cudaStream_t stream;
};
struct ResetArgs {
    const uint8_t *mask; const int32_t *n_warm; const void *noise; int32_t max_warm; void *obs; cudaStream_t stream;
};

class Env {
public:
    beacon_common common{};
    beacon_env_info_t info{};
    std::vector<Field> fields;
    int64_t launches = 0;
    // step_host: hand page-locked caller buffers to the kernel itself (one CTA per env streams its rows
    // over PCIe while the others compute).  Off for the thread-per-env ODE kernels, whose small
    // scattered accesses are faster through staged bulk copies (measured: lorenz 0.50 G vs 0.21 G env-actions/s).
    bool host_zero_copy = true;
    // host staging buffers for step_host
    DeviceBuffer d_act, d_noise, d_obs, d_rwd, d_done, d_trunc, d_status;

    virtual ~Env() {}
    virtual void reset(const ResetArgs &a) = 0;
    virtual void step(const StepArgs &a) = 0;
    // per-env physical parameters (beacon_env_set_physics / get_physics): rayleigh and mixing only
    virtual void set_physics(const char *, const double *, cudaStream_t)
    {
        throw Error(BEACON_ERR_INVALID, "per-env physical parameters apply to rayleigh and mixing only");
    }
    virtual void get_physics(const char *, double *, cudaStream_t)
    {
        throw Error(BEACON_ERR_INVALID, "per-env physical parameters apply to rayleigh and mixing only");
    }

    int real_bytes() const { return info.dtype == BEACON_F64 ? 8 : 4; }
    const Field *find(const char *name) const
    {
        for (auto &f : fields) if (f.name == name) return &f;
        return nullptr;
    }
    void add_field(const char *name, void *ptr, int64_t count, bool is_int = false)
    {
        fields.push_back(Field{name, ptr, count, is_int ? 4 : real_bytes(), is_int});
        info.n_fields = (int32_t)fields.size();
    }
    void step_host(const void *actions, const void *noise, void *obs, void *rwd, uint8_t *done, uint8_t *trunc,
                   int32_t *status, cudaStream_t stream);
};

// Let `kernel` launch with `bytes` of dynamic shared memory.  The limit is an attribute of the kernel
// function, shared by every env of the process on that instance, so it is only ever raised: lowering it
// to a smaller env's size would make the next launch of a larger env fail.
template <typename K> inline void raise_dynamic_smem_limit(K kernel, size_t bytes)
{
    cudaFuncAttributes fa;
    BEACON_CUDA_CHECK(cudaFuncGetAttributes(&fa, (const void *)kernel));
    if ((size_t)fa.maxDynamicSharedSizeBytes < bytes)
        BEACON_CUDA_CHECK(cudaFuncSetAttribute((const void *)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
}

// upload a host float64 array as `R`
template <typename R> inline void upload_as(DeviceBuffer &dst, const double *src, size_t n)
{
    std::vector<R> tmp(n);
    for (size_t i = 0; i < n; i++) tmp[i] = (R)src[i];
    dst.alloc(n * sizeof(R));
    BEACON_CUDA_CHECK(cudaMemcpy(dst.ptr, tmp.data(), n * sizeof(R), cudaMemcpyHostToDevice));
}

// factories implemented in the per-env translation units
Env *make_shkadov(const beacon_common &, const beacon_shkadov_params &, const double *h_init, const double *q_init);
Env *make_burgers(const beacon_common &, const beacon_burgers_params &);
Env *make_sloshing(const beacon_common &, const beacon_sloshing_params &, const double *h_init, const double *q_init);
Env *make_lorenz(const beacon_common &, const beacon_lorenz_params &);
Env *make_vortex(const beacon_common &, const beacon_vortex_params &);
Env *make_mac(const beacon_common &, const beacon_mac_params &, int kind, const double *u0, const double *v0,
              const double *p0, const double *s0);

}  // namespace beacon
