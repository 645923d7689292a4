// C-ABI of libbeacon_b200.so (include/beacon_b200.h): thin exception-free shell over the
// per-env classes.  No torch types, plain pointers and sizes.
#include <cstring>

#include <cstdlib>
#include "common.cuh"

using namespace beacon;

struct beacon_env {
    Env *impl;
};

static thread_local std::string g_last_error;

template <typename F> static int guard(F &&f)
{
    try {
        f();
        return BEACON_OK;
    } catch (const Error &e) {
        g_last_error = e.what();
        return e.code;
    } catch (const std::exception &e) {
        g_last_error = e.what();
        return BEACON_ERR_INVALID;
    } catch (...) {
        g_last_error = "unknown error";
        return BEACON_ERR_INVALID;
    }
}

static void check_common(const beacon_common *c)
{
    BEACON_REQUIRE(c != nullptr, "common options must not be NULL");
    BEACON_REQUIRE(c->batch > 0, "batch must be positive");
    int ndev = 0;
    BEACON_CUDA_CHECK(cudaGetDeviceCount(&ndev));
    BEACON_REQUIRE(c->device >= 0 && c->device < ndev, "no such CUDA device");
    BEACON_CUDA_CHECK(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    BEACON_CUDA_CHECK(cudaGetDeviceProperties(&prop, c->device));
    if (prop.major != 10)
        throw Error(BEACON_ERR_UNSUPPORTED, "libbeacon_b200 is built for sm_100a (B200) only; device is sm_" +
                                                std::to_string(prop.major) + std::to_string(prop.minor));
}

template <typename F> static int create(const beacon_common *c, beacon_env **out, F &&make)
{
    return guard([&] {
        BEACON_REQUIRE(out != nullptr, "out must not be NULL");
        *out = nullptr;
        check_common(c);
        Env *e = make();
        *out = new beacon_env{e};
    });
}

namespace beacon {
// Device-visible alias of a page-locked host buffer (unified addressing maps every cudaHostAlloc /
// cudaHostRegister allocation into the device address space), or NULL for pageable memory.
static void *mapped_alias(const void *host, bool allowed)
{
    static const bool staged_only = getenv("BEACON_STEP_HOST_STAGED") != nullptr;   // A/B switch
    if (!host || staged_only || !allowed) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

// One gym step with HOST buffers.  Page-locked buffers are handed to the kernel as they are: every env's
// CTA reads its action row and writes its observation / reward / flag rows straight over PCIe when it
// starts / finishes, so the transfers of one env overlap the compute of the others and no copy
// is queued behind the kernel.  Pageable buffers go through device staging buffers and
// cudaMemcpyAsync.  Either way the call returns after the stream has drained: the results are in
// the caller's buffers.
void Env::step_host(const void *actions, const void *noise, void *obs, void *rwd, uint8_t *done, uint8_t *trunc,
                    int32_t *status, cudaStream_t stream)
{
    const size_t B = (size_t)info.batch, rb = (size_t)real_bytes();
    const size_t act_bytes = info.act_is_int ? B * 4 : B * (size_t)info.act_dim * rb;
    const size_t noise_bytes = B * (size_t)info.noise_dim * rb;
    const size_t obs_bytes = B * (size_t)info.n_obs * rb, rwd_bytes = B * (size_t)info.rwd_dim * rb;
    if (!d_obs.ptr) {
        d_act.alloc(act_bytes ? act_bytes : 8); d_noise.alloc(noise_bytes ? noise_bytes : 8);
        d_obs.alloc(obs_bytes); d_rwd.alloc(rwd_bytes); d_done.alloc(B); d_trunc.alloc(B); d_status.alloc(B * 4);
    }
    BEACON_REQUIRE(actions && obs && rwd && done && trunc, "step_host: NULL buffer");
    const bool zc = host_zero_copy;
    void *m_act = mapped_alias(actions, zc), *m_noise = mapped_alias(noise, zc), *m_obs = mapped_alias(obs, zc), *m_rwd = mapped_alias(rwd, zc);
    void *m_done = mapped_alias(done, zc), *m_trunc = mapped_alias(trunc, zc), *m_status = mapped_alias(status, zc);
    if (!m_act) BEACON_CUDA_CHECK(cudaMemcpyAsync(d_act.ptr, actions, act_bytes, cudaMemcpyHostToDevice, stream));
    if (noise && !m_noise) BEACON_CUDA_CHECK(cudaMemcpyAsync(d_noise.ptr, noise, noise_bytes, cudaMemcpyHostToDevice, stream));
    StepArgs a{m_act ? m_act : d_act.ptr, noise ? (m_noise ? m_noise : d_noise.ptr) : nullptr, m_obs ? m_obs : d_obs.ptr,
               m_rwd ? m_rwd : d_rwd.ptr, m_done ? (uint8_t *)m_done : d_done.as<uint8_t>(),
               m_trunc ? (uint8_t *)m_trunc : d_trunc.as<uint8_t>(),
               (status && m_status) ? (int32_t *)m_status : d_status.as<int32_t>(), nullptr, 1, stream};
    step(a);
    if (!m_obs) BEACON_CUDA_CHECK(cudaMemcpyAsync(obs, d_obs.ptr, obs_bytes, cudaMemcpyDeviceToHost, stream));
    if (!m_rwd) BEACON_CUDA_CHECK(cudaMemcpyAsync(rwd, d_rwd.ptr, rwd_bytes, cudaMemcpyDeviceToHost, stream));
    if (!m_done) BEACON_CUDA_CHECK(cudaMemcpyAsync(done, d_done.ptr, B, cudaMemcpyDeviceToHost, stream));
    if (!m_trunc) BEACON_CUDA_CHECK(cudaMemcpyAsync(trunc, d_trunc.ptr, B, cudaMemcpyDeviceToHost, stream));
    if (status && !m_status) BEACON_CUDA_CHECK(cudaMemcpyAsync(status, d_status.ptr, B * 4, cudaMemcpyDeviceToHost, stream));
    BEACON_CUDA_CHECK(cudaStreamSynchronize(stream));
}
}  // namespace beacon

extern "C" {

int beacon_shkadov_create(const beacon_common *c, const beacon_shkadov_params *p, const double *h_init,
                          const double *q_init, beacon_env **out)
{
    return create(c, out, [&] { BEACON_REQUIRE(p, "params NULL"); return make_shkadov(*c, *p, h_init, q_init); });
}
int beacon_burgers_create(const beacon_common *c, const beacon_burgers_params *p, beacon_env **out)
{
    return create(c, out, [&] { BEACON_REQUIRE(p, "params NULL"); return make_burgers(*c, *p); });
}
int beacon_sloshing_create(const beacon_common *c, const beacon_sloshing_params *p, const double *h_init,
                           const double *q_init, beacon_env **out)
{
    return create(c, out, [&] { BEACON_REQUIRE(p, "params NULL"); return make_sloshing(*c, *p, h_init, q_init); });
}
int beacon_lorenz_create(const beacon_common *c, const beacon_lorenz_params *p, beacon_env **out)
{
    return create(c, out, [&] { BEACON_REQUIRE(p, "params NULL"); return make_lorenz(*c, *p); });
}
int beacon_vortex_create(const beacon_common *c, const beacon_vortex_params *p, beacon_env **out)
{
    return create(c, out, [&] { BEACON_REQUIRE(p, "params NULL"); return make_vortex(*c, *p); });
}
int beacon_rayleigh_create(const beacon_common *c, const beacon_mac_params *p, const double *u_init,
                           const double *v_init, const double *p_init, const double *T_init, beacon_env **out)
{
    return create(c, out, [&] {
        BEACON_REQUIRE(p, "params NULL");
        return make_mac(*c, *p, BEACON_RAYLEIGH, u_init, v_init, p_init, T_init);
    });
}
int beacon_mixing_create(const beacon_common *c, const beacon_mac_params *p, const double *C_init, beacon_env **out)
{
    return create(c, out, [&] {
        BEACON_REQUIRE(p, "params NULL");
        return make_mac(*c, *p, BEACON_MIXING, nullptr, nullptr, nullptr, C_init);
    });
}

void beacon_env_destroy(beacon_env *env)
{
    if (!env) return;
    cudaSetDevice(env->impl->common.device);
    delete env->impl;
    delete env;
}

int beacon_env_info(const beacon_env *env, beacon_env_info_t *info)
{
    return guard([&] {
        BEACON_REQUIRE(env && info, "NULL argument");
        *info = env->impl->info;
    });
}

int beacon_env_reset(beacon_env *env, const uint8_t *mask, const int32_t *n_warm, const void *noise,
                     int32_t max_warm, void *obs, beacon_stream_t stream)
{
    return guard([&] {
        BEACON_REQUIRE(env, "NULL handle");
        BEACON_REQUIRE(max_warm >= 0, "max_warm must be >= 0");
        BEACON_CUDA_CHECK(cudaSetDevice(env->impl->common.device));
        env->impl->reset(ResetArgs{mask, n_warm, noise, max_warm, obs, (cudaStream_t)stream});
    });
}

int beacon_env_step(beacon_env *env, const void *actions, const void *noise, void *obs, void *rwd, uint8_t *done,
                    uint8_t *trunc, int32_t *status, int64_t *iters, int32_t n_fused, beacon_stream_t stream)
{
    return guard([&] {
        BEACON_REQUIRE(env, "NULL handle");
        BEACON_REQUIRE(n_fused >= 1, "n_fused must be >= 1");
        BEACON_REQUIRE(actions && obs && rwd && done && trunc, "step: actions/obs/rwd/done/trunc must not be NULL");
        BEACON_CUDA_CHECK(cudaSetDevice(env->impl->common.device));
        env->impl->step(StepArgs{actions, noise, obs, rwd, done, trunc, status, iters, n_fused, (cudaStream_t)stream});
    });
}

int beacon_env_step_host(beacon_env *env, const void *actions, const void *noise, void *obs, void *rwd,
                         uint8_t *done, uint8_t *trunc, int32_t *status, beacon_stream_t stream)
{
    return guard([&] {
        BEACON_REQUIRE(env, "NULL handle");
        BEACON_CUDA_CHECK(cudaSetDevice(env->impl->common.device));
        env->impl->step_host(actions, noise, obs, rwd, done, trunc, status, (cudaStream_t)stream);
    });
}

int beacon_env_field(const beacon_env *env, int32_t index, const char **name, int64_t *count, int32_t *is_int)
{
    return guard([&] {
        BEACON_REQUIRE(env, "NULL handle");
        BEACON_REQUIRE(index >= 0 && index < (int32_t)env->impl->fields.size(), "field index out of range");
        const Field &f = env->impl->fields[index];
        if (name) *name = f.name.c_str();
        if (count) *count = f.count;
        if (is_int) *is_int = f.is_int ? 1 : 0;
    });
}

static int copy_state(beacon_env *env, const char *field, void *buf, const void *cbuf, beacon_stream_t stream)
{
    return guard([&] {
        BEACON_REQUIRE(env && field && (buf || cbuf), "NULL argument");
        const Field *f = env->impl->find(field);
        if (!f) throw Error(BEACON_ERR_INVALID, std::string("unknown state field '") + field + "'");
        BEACON_CUDA_CHECK(cudaSetDevice(env->impl->common.device));
        size_t bytes = (size_t)env->impl->info.batch * (size_t)f->count * (size_t)f->elem_bytes;
        if (buf) BEACON_CUDA_CHECK(cudaMemcpyAsync(buf, f->ptr, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        else BEACON_CUDA_CHECK(cudaMemcpyAsync(f->ptr, cbuf, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    });
}

int beacon_env_get_state(beacon_env *env, const char *field, void *buf, beacon_stream_t stream)
{
    return copy_state(env, field, buf, nullptr, stream);
}
int beacon_env_set_state(beacon_env *env, const char *field, const void *buf, beacon_stream_t stream)
{
    return copy_state(env, field, nullptr, buf, stream);
}

int beacon_env_set_physics(beacon_env *env, const char *name, const double *values, beacon_stream_t stream)
{
    return guard([&] {
        BEACON_REQUIRE(env, "NULL handle");
        BEACON_CUDA_CHECK(cudaSetDevice(env->impl->common.device));
        env->impl->set_physics(name, values, (cudaStream_t)stream);
    });
}
int beacon_env_get_physics(beacon_env *env, const char *name, double *values, beacon_stream_t stream)
{
    return guard([&] {
        BEACON_REQUIRE(env, "NULL handle");
        BEACON_CUDA_CHECK(cudaSetDevice(env->impl->common.device));
        env->impl->get_physics(name, values, (cudaStream_t)stream);
    });
}

int beacon_peer_alloc(int32_t device, uint64_t bytes, void **ptr)
{
    return guard([&] {
        BEACON_REQUIRE(ptr && bytes > 0, "peer_alloc: bad argument");
        BEACON_CUDA_CHECK(cudaSetDevice(device));
        BEACON_CUDA_CHECK(cudaMalloc(ptr, (size_t)bytes));
        BEACON_CUDA_CHECK(cudaMemset(*ptr, 0, (size_t)bytes));
    });
}
int beacon_peer_export(void *ptr, uint8_t handle[BEACON_PEER_HANDLE_BYTES])
{
    static_assert(sizeof(cudaIpcMemHandle_t) == BEACON_PEER_HANDLE_BYTES, "IPC handle size");
    return guard([&] {
        BEACON_REQUIRE(ptr && handle, "peer_export: NULL argument");
        cudaIpcMemHandle_t h;
        BEACON_CUDA_CHECK(cudaIpcGetMemHandle(&h, ptr));
        memcpy(handle, &h, sizeof(h));
    });
}
int beacon_peer_open(const uint8_t handle[BEACON_PEER_HANDLE_BYTES], int32_t device, void **ptr)
{
    return guard([&] {
        BEACON_REQUIRE(ptr && handle, "peer_open: NULL argument");
        BEACON_CUDA_CHECK(cudaSetDevice(device));
        cudaIpcMemHandle_t h;
        memcpy(&h, handle, sizeof(h));
        BEACON_CUDA_CHECK(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    });
}
int beacon_peer_close(void *ptr)
{
    return guard([&] {
        BEACON_REQUIRE(ptr, "peer_close: NULL argument");
        BEACON_CUDA_CHECK(cudaIpcCloseMemHandle(ptr));
    });
}
int beacon_peer_free(int32_t device, void *ptr)
{
    return guard([&] {
        BEACON_REQUIRE(ptr, "peer_free: NULL argument");
        BEACON_CUDA_CHECK(cudaSetDevice(device));
        BEACON_CUDA_CHECK(cudaFree(ptr));
    });
}

int64_t beacon_env_launch_count(const beacon_env *env) { return env ? env->impl->launches : 0; }

const char *beacon_last_error(void) { return g_last_error.c_str(); }
const char *beacon_version(void) { return "beacon_b200 0.2 (sm_100a)"; }

}  // extern "C"
