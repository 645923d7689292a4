// rayleigh-v0 and mixing-v0 — 2D incompressible flow on a MAC staggered grid, Chorin projection
// with the reference's own Jacobi pressure iteration, scalar (temperature / concentration)
// transport, probe history and reward.
//
// Reference: /root/reference/beacon/rayleigh/rayleigh.py — solve() :160-240, predictor :371-407,
// poisson :412-456, corrector :461-464, transport :469-487, get_obs :243-262, get_rwd :265-275;
// /root/reference/beacon/mixing/mixing.py — solve() :136-209, get_control :212-234,
// predictor :382-416, poisson :421-465, corrector :470-473, transport :478-495,
// get_obs :237-256, get_rwd :259-264.
//
// B200 design: ONE CTA PER ENVIRONMENT (or one cluster, mac_kernel with ctas_per_env > 1) runs every
// sub-step of every fused action without returning to the host.  Three kernels (DESIGN.md 3.4 - 3.6):
//   * mac_reg_kernel  — rayleigh 50x50: phi and the Poisson right-hand side of a 2x5 tile in
//     REGISTERS, in-place Jacobi sweeps over two strided exchange planes (one barrier per sweep),
//     convergence test two sweeps behind and interleaved with the next sweep (exact sweep counts),
//     u, v, T planes in shared memory (TMA bulk loads / stores), 2 CTAs per SM;
//   * mac_big_kernel  — mixing 100x100: the same register-resident Poisson with 4x5 tiles, field
//     planes in L2/HBM, tile copies of p, us, vs in a thread-interleaved scratch, u / v staged in
//     the exchange planes for the predictor (TMA bulk copies), transport in two row passes;
//   * mac_kernel      — generic kernel for any other grid: one env over G = ctas_per_env CTAs
//     (1 by default, 2..8 as a thread-block cluster, DESIGN.md 3.6), each with its slab of rows of
//     the two phi planes in shared memory, right-hand side in registers, fields in global memory;
//     at G > 1 halo rows and residual partials go through DSMEM, one cluster barrier per sweep, the
//     transport wavefront chained from rank to rank.  At G = 1 the slab is the whole array (grids
//     up to ~100x100 cells) and every barrier is a CTA barrier.
// Common to all:
//   * the residual reproduces the reference's: sum over the whole ghost-inclusive array after
//     the ghost update (ghost copies re-count the wall-adjacent cells; mixing's top ghost is 0);
//     all threads evaluate the same sum in the same order, so `while err > tol` is uniform;
//   * the in-place lexicographic transport sweep (a Gauss-Seidel-like dependence on the new
//     west/south neighbours) is split in two: all threads pre-compute, per cell, the part of the
//     update that only involves OLD values plus the coefficients multiplying the new neighbours;
//     then one warp runs the remaining 2-FMA recurrence as a skewed wavefront, rows across lanes,
//     the new west value travelling by warp shuffle (no barriers).
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <string>
#include <type_traits>

#include "common.cuh"

namespace beacon {

#define MAC_RPL 2   // rows per lane in the transport wavefront

// Row-pair stride (in columns) of the wavefront coefficient planes: at least NY+1 columns and
// stride - 1 = 1 mod 8, so that the 16-byte accesses of 8 consecutive lanes (addresses
// lane * (stride - 1) * 16 B + const) fall into 8 different 16-byte bank groups.
constexpr int wavefront_row_stride(int ny) { return ((ny + 1 - 2 + 7) / 8) * 8 + 2; }

template <typename R> struct MacArgs {
    int nx, ny, ld, n, ndt_act, n_act, kind, n_sgts, nx_sgts, itmax, tiles_i, tiles_j;
    int nx_obs_pts, ny_obs_pts, n_obs_steps, nx_obs, ny_obs, n_obs, tr_pass;
    R dx, dy, dt, inv_dx, inv_dy, inv_dx2, inv_dy2, dx2, dy2, inv_den, pk1, pk2, cscale, dcoef, tcoef, Tc, Th, Cmax, u_max, ref_c, tol;
    int B, mode, n_fused;
    int G, slab_rows;                  // mac_kernel: CTAs per env, rows of a phi slab plane (halos included)
    R *u, *v, *p, *s, *us, *vs, *cc;   // [B, n] planes (s = T or C); us/vs/cc are workspaces
    R *a_cur, *obs_hist;
    int32_t *stp, *a_int;
    const R *u0, *v0, *p0, *s0;
    const void *actions;
    const uint8_t *mask;
    R *obs, *rwd;
    uint8_t *done, *trunc;
    int32_t *status;
    int64_t *iters;
    unsigned long long *dbg;   // optional per-phase cycle counters (BEACON_MAC_DEBUG), block 0 only
    const R *phys;             // per-env instances: [B][3] rows of (dcoef, tcoef, u_max), built by mac_phys_derive
};

// The physical constants of an env inside the kernel bodies (template switch PHYS): the handle's
// (a.dcoef, a.tcoef, a.u_max) in the uniform instances, whose machine code is the same as before the
// switch existed; in the per-env instances the env's row of a.phys, read once per CTA into the static
// shared array s_coef (MAC_LOAD_COEF, before a CTA barrier) and broadcast from there.  Every CTA of a
// cluster belongs to one env and reads the same row.  Names, not locals: a new local captured by the
// bodies' lambdas would change the register allocation of the uniform instances (DESIGN.md 3.7).
#define MAC_DCOEF (PHYS ? s_coef[0] : a.dcoef)
#define MAC_TCOEF (PHYS ? s_coef[1] : a.tcoef)
#define MAC_UMAX (PHYS ? s_coef[2] : a.u_max)
#define MAC_LOAD_COEF(b)                                  \
    __shared__ R s_coef[3];                               \
    if (PHYS && tid < 3) s_coef[tid] = a.phys[3 * (size_t)(b) + tid]

// numpy pairwise sum for n <= 128 (np.mean of the action vector, rayleigh.py:165)
template <typename R> __device__ R np_pairwise_small(const R *a, int n)
{
    if (n < 8) {
        R res = R(0);
        for (int i = 0; i < n; i++) res += a[i];
        return res;
    }
    R r[8];
    int i;
    for (i = 0; i < 8; i++) r[i] = a[i];
    for (i = 8; i < n - (n % 8); i += 8)
        for (int k = 0; k < 8; k++) r[k] += a[i + k];
    R res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
}

// ---------------------------------------------------------------------------------------
// mac_kernel — the generic kernel: one environment over G = a.G CTAs, a thread-block cluster
// when G > 1 (DESIGN.md 3.6).  Rank g owns the interior rows ib..ie of a balanced slab; the left
// wall and ghost row 0 go to rank 0, the right wall and ghost row nx+1 to rank G-1.  Fields stay
// in their global planes; each CTA keeps only its slab of the two phi planes (one halo row on
// each side) in shared memory.  A Jacobi sweep pushes its first and last rows into the
// neighbours' halo rows through DSMEM and ends in one cluster barrier, where every CTA also
// receives the per-warp residual partials of every rank.  Phases that read rows written by
// another CTA follow a cluster barrier (release / acquire).  The transport wavefront of rank
// g + 1 starts on the new values of rank g's last row, handed over through DSMEM in chunks of
// MAC_CLUSTER_CHUNK columns, each published with a cluster-scope release / acquire flag.
// CLUSTER = false is the G = 1 instance (a plain launch): the slab is the whole array, nothing goes
// through DSMEM, every barrier is a CTA barrier (env_barrier) and the neighbour tests of the sweep and
// the wavefront fold away.  With G a run-time value these cost 25 % per sweep at G = 1 (B200).
// ---------------------------------------------------------------------------------------
#define MAC_CLUSTER_MAX 8          // portable cluster size
#define MAC_CLUSTER_MIN_ROWS 4     // rows of the thinnest slab: one tile height
#define MAC_CLUSTER_MAX_LD 512     // columns (ny + 2) of the wavefront hand-off buffers
#define MAC_CLUSTER_CHUNK 8        // columns per hand-off flag: a cluster-scope release per chunk, not per column
#define MAC_CLUSTER_SMEM (200 * 1024)   // phi slabs and transport planes; the hand-off buffers and static arrays take the rest of 227 KB
// bytes of the wavefront hand-off buffers (G > 1 only), after the phi slabs in dynamic shared memory
#define MAC_HANDOFF_BYTES(R) (MAC_CLUSTER_MAX_LD * sizeof(R) + MAC_CLUSTER_MAX_LD / MAC_CLUSTER_CHUNK * sizeof(int))

__device__ __forceinline__ void cluster_barrier()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// barrier of the CTAs of one env
template <bool CLUSTER> __device__ __forceinline__ void env_barrier()
{
    if (CLUSTER) cluster_barrier();
    else __syncthreads();
}
__device__ __forceinline__ unsigned cluster_rank()
{
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// generic address of the same shared-memory object in CTA `rank` of the cluster
template <typename P> __device__ __forceinline__ P *cluster_map(P *p, unsigned rank)
{
    uint64_t r;
    asm volatile("mapa.u64 %0, %1, %2;" : "=l"(r) : "l"(p), "r"(rank));
    return reinterpret_cast<P *>(r);
}
__device__ __forceinline__ void st_release_cluster(int *p, int v)
{
    asm volatile("st.release.cluster.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_cluster(const int *p)
{
    int v;
    asm volatile("ld.acquire.cluster.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// G > 1: the wavefront hand-off buffers, after the phi slabs and transport planes in dynamic shared memory
// (MacEnv sizes both): new values of rank g-1's last row by column, and one flag per chunk of it that holds
// the sub-step sequence number once the chunk is ready
template <typename R> __device__ __forceinline__ R *handoff_west(R *phiA, const MacArgs<R> &a)
{
    return phiA + a.ld * max(2 * a.slab_rows, 3 * ((a.slab_rows - 2 + a.tr_pass - 1) / a.tr_pass));
}
template <typename R> __device__ __forceinline__ int *handoff_flags(R *phiA, const MacArgs<R> &a)
{
    return reinterpret_cast<int *>(handoff_west(phiA, a) + MAC_CLUSTER_MAX_LD);
}

template <typename R, int TI, int TJ, int T, bool CLUSTER, bool PHYS>
__device__ __forceinline__ void mac_body(const MacArgs<R> a, const unsigned thread_x)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ R s_part[2][MAC_CLUSTER_MAX][T / 32];   // residual partials of every rank, by sweep parity
    __shared__ R s_red[T / 32];
    __shared__ R s_rank[MAC_CLUSTER_MAX];             // per-rank reward partials (mixing)
    __shared__ int s_bad[MAC_CLUSTER_MAX];            // per-rank non-finite flags
    __shared__ R s_seg[128];
    __shared__ R s_act[128];
    const int tid = thread_x, G = CLUSTER ? a.G : 1;
    const unsigned rank = CLUSTER ? cluster_rank() : 0;
    const int b = blockIdx.x / G;
    const int nx = a.nx, ny = a.ny, ld = a.ld;
    const bool resetting = a.mode == 1;
    if (resetting && a.mask && !a.mask[b]) return;     // uniform over the cluster: no DSMEM access yet
    MAC_LOAD_COEF(b);                                  // read after the env barrier below
    const bool ray = a.kind == BEACON_RAYLEIGH;
    const bool first = rank == 0, last = rank == (unsigned)G - 1;

    // ---- slab: rows ib..ie (S rows), balanced to within one row --------------------------------
    const int base = nx / G, rem = nx % G;
    const int S = base + ((int)rank < rem), ib = 1 + (int)rank * base + min((int)rank, rem), ie = ib + S - 1;
    const int S_left = rank > 0 ? base + ((int)rank - 1 < rem) : 0;
    const int r0 = first ? 0 : ib, r1 = last ? nx + 1 : ie;   // rows of the whole-array passes (ghost rows included)
    const int e0 = r0 * ld, e1 = (r1 + 1) * ld;

    // ---- planes: phi slabs [S + 2][ld] (local row li = i - ib + 1), fields in global memory --------
    const int slab = a.slab_rows * ld;
    R *phiA = reinterpret_cast<R *>(smem_raw), *phiB = phiA + slab;
    R *lA = nullptr, *lB = nullptr, *rA = nullptr, *rB = nullptr;   // neighbours' halo rows, same planes
    if (!first) { lA = cluster_map(phiA, rank - 1) + (S_left + 1) * ld; lB = cluster_map(phiB, rank - 1) + (S_left + 1) * ld; }
    if (!last) { rA = cluster_map(phiA, rank + 1); rB = cluster_map(phiB, rank + 1); }
    const size_t row = (size_t)b * a.n;
    R *u = a.u + row, *v = a.v + row, *p = a.p + row, *s = a.s + row, *us = a.us + row, *vs = a.vs + row;

    const int tiles_i = (S + TI - 1) / TI;
    const bool has_tile = tid < tiles_i * a.tiles_j;
    const int ti = tid / a.tiles_j, tj = tid - ti * a.tiles_j;
    const int i0 = ib + ti * TI, j0 = 1 + tj * TJ;
#define CELL_LOOP                                       \
    _Pragma("unroll") for (int r = 0; r < TI; r++)      \
    _Pragma("unroll") for (int k = 0; k < TJ; k++)
#define CELL_OK(i, j) (has_tile && (i) <= ie && (j) <= ny)

    if (CLUSTER)
        for (int e = tid; e < MAC_CLUSTER_MAX_LD / MAC_CLUSTER_CHUNK; e += T) handoff_flags(phiA, a)[e] = 0;

    // ---- load / reset (own rows) -----------------------------------------------------------------
    if (resetting) {
        for (int e = e0 + tid; e < e1; e += T) {
            u[e] = ray ? a.u0[e] : R(0); v[e] = ray ? a.v0[e] : R(0); p[e] = ray ? a.p0[e] : R(0); s[e] = a.s0[e];
            us[e] = R(0); vs[e] = R(0);
        }
        if (first) {
            for (int e = tid; e < a.n_obs; e += T) a.obs_hist[(size_t)b * a.n_obs + e] = R(0);
            for (int e = tid; e < (ray ? a.n_sgts : 0); e += T) a.a_cur[(size_t)b * a.n_sgts + e] = R(0);
            if (tid == 0) { a.stp[b] = 0; if (!ray) a.a_int[b] = 1; }
        }
        env_barrier<CLUSTER>();
        if (first) {                                           // history zero, newest slot from the init state
            R *hist = a.obs_hist + (size_t)b * a.n_obs;
            const int per_step = 3 * a.nx_obs_pts * a.ny_obs_pts;
            for (int e = tid; e < a.n_obs; e += T) {
                int st = e / per_step, rm = e - st * per_step;
                R val = R(0);
                if (st == a.n_obs_steps - 1) {
                    int f = rm / (a.nx_obs_pts * a.ny_obs_pts), q = rm - f * (a.nx_obs_pts * a.ny_obs_pts);
                    int pi = q / a.ny_obs_pts, pj = q - pi * a.ny_obs_pts;
                    int x = a.nx_obs / 2 + pi * a.nx_obs, y = a.ny_obs / 2 + pj * a.ny_obs;
                    val = (f == 0) ? s[x * ld + y] : (f == 1 ? u[x * ld + y] : v[x * ld + y]);
                }
                hist[e] = val;
                a.obs[(size_t)b * a.n_obs + e] = val;
            }
        }
        return;                                                // no DSMEM access after the barrier
    }
    int stp = a.stp[b];
    int status = 0, seq = 0;
    env_barrier<CLUSTER>();                                    // s_flag cleared in every rank

    for (int act = 0; act < a.n_fused; act++) {
        const size_t orow = (size_t)act * a.B + b;
        // ---- action conditioning: every rank computes it, rank 0 stores it -------------------------
        if (ray) {
            const R *ain = (const R *)a.actions + orow * a.n_sgts;
            if (tid == 0) {                                        // rayleigh.py:164-171
                const int ns = a.n_sgts;
                for (int j = 0; j < ns; j++) s_act[j] = ain[j];
                R mean = np_pairwise_small(s_act, ns) / R(ns);
                R m = R(1);
                for (int j = 0; j < ns; j++) { s_act[j] = s_act[j] - mean; m = np_max(m, rabs(s_act[j]) / a.Cmax); }
                for (int j = 0; j < ns; j++) {
                    s_act[j] = s_act[j] / m; s_seg[j] = a.Th + s_act[j];
                    if (first) a.a_cur[(size_t)b * ns + j] = s_act[j];
                }
            }
        } else if (tid == 0) {                                     // get_control, mixing.py:212-234
            int ai = ((const int32_t *)a.actions)[orow];
            R ut = 0, ub = 0, vl = 0, vr = 0;
            if (ai == 0) { ub = MAC_UMAX; ut = -MAC_UMAX; }
            if (ai == 1) { ub = -MAC_UMAX; ut = MAC_UMAX; }
            if (ai == 2) { vr = MAC_UMAX; vl = -MAC_UMAX; }
            if (ai == 3) { vr = -MAC_UMAX; vl = MAC_UMAX; }
            s_seg[0] = ut; s_seg[1] = ub; s_seg[2] = vl; s_seg[3] = vr;
            if (first) a.a_int[b] = ai;
        }
        __syncthreads();
        long long it_total = 0;

        for (int it = 0; it < a.ndt_act; it++) {
            seq += 1;
            // ---- boundary conditions: rayleigh.py:180-202, mixing.py:153-171, own walls and own i range ----
            {
                const int nl = first ? ny + 2 : 0, nr = last ? ny + 2 : 0;
                const int ihi = last ? nx + 1 : ie, ni = ihi - ib + 1;
                for (int k = tid; k < nl + nr + 2 * ni; k += T) {
                    if (k < nl) {                                      // left wall (i = 0/1)
                        int j = k;
                        if (j >= 1 && j <= ny) { u[1 * ld + j] = R(0); s[0 * ld + j] = s[1 * ld + j]; }
                        if (j >= 2 && j <= ny) v[0 * ld + j] = ray ? -v[1 * ld + j] : R(2) * s_seg[2] - v[1 * ld + j];
                    } else if (k < nl + nr) {                          // right wall
                        int j = k - nl;
                        if (j >= 1 && j <= ny) { u[(nx + 1) * ld + j] = R(0); s[(nx + 1) * ld + j] = s[nx * ld + j]; }
                        if (j >= 2 && j <= ny) v[(nx + 1) * ld + j] = ray ? -v[nx * ld + j] : R(2) * s_seg[3] - v[nx * ld + j];
                    } else if (k < nl + nr + ni) {                     // top wall (j = ny+1)
                        int i = ib + k - nl - nr;
                        R ui = (i == 1 || i == nx + 1) ? R(0) : u[i * ld + ny];
                        u[i * ld + ny + 1] = ray ? -ui : R(2) * s_seg[0] - ui;
                        if (i <= nx) {
                            v[i * ld + ny + 1] = R(0);
                            s[i * ld + ny + 1] = ray ? R(2) * a.Tc - s[i * ld + ny] : s[i * ld + ny];
                        }
                    } else {                                           // bottom wall (j = 0/1)
                        int i = ib + k - nl - nr - ni;
                        R ui = (i == 1 || i == nx + 1) ? R(0) : u[i * ld + 1];
                        u[i * ld + 0] = ray ? -ui : R(2) * s_seg[1] - ui;
                        if (i <= nx) {
                            v[i * ld + 1] = R(0);
                            if (ray) {
                                int sg = (i - 1) / a.nx_sgts;
                                if (sg < a.n_sgts) s[i * ld + 0] = R(2) * s_seg[sg] - s[i * ld + 1];
                            } else s[i * ld + 0] = s[i * ld + 1];
                        }
                    }
                }
            }
            for (int e = tid; e < 2 * slab; e += T) phiA[e] = R(0);   // both planes: they doubled as transport scratch
            env_barrier<CLUSTER>();                            // walls of the neighbours; zeroed halos before any push

            // ---- predictor (own rows; reads the neighbours' wall rows) ---------------------------------
            CELL_LOOP {
                const int i = i0 + r, j = j0 + k;
                if (CELL_OK(i, j)) {
                    const R uc = u[i * ld + j], vc = v[i * ld + j];
                    if (i >= 2) {
                        R uE = R(0.5) * (u[(i + 1) * ld + j] + uc), uW = R(0.5) * (uc + u[(i - 1) * ld + j]);
                        R uN = R(0.5) * (u[i * ld + j + 1] + uc), uS = R(0.5) * (uc + u[i * ld + j - 1]);
                        R vN = R(0.5) * (v[i * ld + j + 1] + v[(i - 1) * ld + j + 1]), vS = R(0.5) * (vc + v[(i - 1) * ld + j]);
                        R conv = (uE * uE - uW * uW) * a.inv_dx + (uN * vN - uS * vS) * a.inv_dy;
                        R diff = ((u[(i + 1) * ld + j] - R(2) * uc + u[(i - 1) * ld + j]) * a.inv_dx2 +
                                  (u[i * ld + j + 1] - R(2) * uc + u[i * ld + j - 1]) * a.inv_dy2) * MAC_DCOEF;
                        R pres = (p[i * ld + j] - p[(i - 1) * ld + j]) * a.inv_dx;
                        us[i * ld + j] = uc + a.dt * (diff - conv - pres);
                    }
                    if (j >= 2) {
                        R vE = R(0.5) * (v[(i + 1) * ld + j] + vc), vW = R(0.5) * (vc + v[(i - 1) * ld + j]);
                        R uE = R(0.5) * (u[(i + 1) * ld + j] + u[(i + 1) * ld + j - 1]), uW = R(0.5) * (uc + u[i * ld + j - 1]);
                        R vN = R(0.5) * (v[i * ld + j + 1] + vc), vS = R(0.5) * (vc + v[i * ld + j - 1]);
                        R conv = (uE * vE - uW * vW) * a.inv_dx + (vN * vN - vS * vS) * a.inv_dy;
                        R diff = ((v[(i + 1) * ld + j] - R(2) * vc + v[(i - 1) * ld + j]) * a.inv_dx2 +
                                  (v[i * ld + j + 1] - R(2) * vc + v[i * ld + j - 1]) * a.inv_dy2) * MAC_DCOEF;
                        R pres = (p[i * ld + j] - p[i * ld + j - 1]) * a.inv_dy;
                        R rhs = diff - conv - pres;
                        if (ray) rhs += s[i * ld + j];
                        vs[i * ld + j] = vc + a.dt * rhs;
                    }
                }
            }
            env_barrier<CLUSTER>();                            // us of row ie + 1 comes from rank g + 1

            // ---- Poisson right-hand side into registers --------------------------------------------------
            R c[TI][TJ];
            CELL_LOOP {
                const int i = i0 + r, j = j0 + k;
                c[r][k] = R(0);
                if (CELL_OK(i, j))
                    c[r][k] = ((us[(i + 1) * ld + j] - us[i * ld + j]) * a.inv_dx + (vs[i * ld + j + 1] - vs[i * ld + j]) * a.inv_dy) * a.cscale;
            }
            // ---- Jacobi sweeps: halo rows pushed to the neighbours, one cluster barrier per sweep ------
            R *pin = phiA, *pout = phiB;
            R err = R(1.0e10);
            int itp = 0;
            while (err > a.tol) {
                R acc = R(0);
                R *lout = (itp & 1) ? lA : lB, *rout = (itp & 1) ? rA : rB;   // the neighbours' copies of pout
                if (has_tile) {
#pragma unroll
                    for (int r = 0; r < TI; r++) {
                        const int i = i0 + r;
                        if (i <= ie) {
                            const int li = i - ib + 1;
                            const R *rc = pin + li * ld + j0, *rw = rc - ld, *re = rc + ld;
                            R *po = pout + li * ld;
                            R west = rc[-1], cen = rc[0];
#pragma unroll
                            for (int k = 0; k < TJ; k++) {
                                const int j = j0 + k;
                                if (j <= ny) {
                                    const R east = rc[k + 1];
                                    R nv = ((re[k] + rw[k]) * a.dy2 + (east + west) * a.dx2 - c[r][k]) * a.inv_den;
                                    R d = nv - cen;
                                    R w = R(1);
                                    if (i == 1) { w += R(1); po[j - ld] = nv; }
                                    if (i == nx) { w += R(1); po[j + ld] = nv; }
                                    if (j == 1) { w += R(1); po[0] = nv; }
                                    if (j == ny) { if (ray) { w += R(1); po[ny + 1] = nv; } }
                                    if (i == ib && lout) lout[j] = nv;     // halo row S_left + 1 of rank g - 1
                                    if (i == ie && rout) rout[j] = nv;     // halo row 0 of rank g + 1
                                    acc += w * (d * d);
                                    po[j] = nv;
                                    west = cen; cen = east;
                                }
                            }
                        }
                    }
                }
                acc = warp_sum(acc);
                const int lane = tid & 31, warp = tid >> 5;
                if (!CLUSTER) { if (lane == 0) s_part[itp & 1][0][warp] = acc; }
                else if (lane < G) cluster_map(&s_part[itp & 1][rank][warp], lane)[0] = acc;
                env_barrier<CLUSTER>();
                err = R(0);
                for (int g = 0; g < G; g++) {                  // same partials, same order in every thread of the cluster
                    R eg = s_part[itp & 1][g][0];
#pragma unroll
                    for (int w = 1; w < T / 32; w++) eg += s_part[itp & 1][g][w];
                    err += eg;
                }
                R *t = pin; pin = pout; pout = t;
                itp += 1;
                if (itp > a.itmax) { status |= BEACON_STATUS_POISSON_OVERFLOW; break; }
            }
            it_total += itp;
            const R *phi = pin;

            // ---- p += phi (own rows, ghost rows at the ends) and corrector --------------------------------
            for (int e = e0 + tid; e < e1; e += T) p[e] += phi[e - (ib - 1) * ld];
            CELL_LOOP {
                const int i = i0 + r, j = j0 + k;
                if (CELL_OK(i, j)) {
                    const int li = i - ib + 1;
                    if (i >= 2) u[i * ld + j] = us[i * ld + j] - a.dt * (phi[li * ld + j] - phi[(li - 1) * ld + j]) * a.inv_dx;
                    if (j >= 2) v[i * ld + j] = vs[i * ld + j] - a.dt * (phi[li * ld + j] - phi[li * ld + j - 1]) * a.inv_dy;
                }
            }
            env_barrier<CLUSTER>();                            // u of row ie + 1 comes from rank g + 1

            // ---- transport: coefficients per pass in the phi planes, wavefront chained over the ranks -----
            {
                const int passes = a.tr_pass, rows = (S + passes - 1) / passes;
                R *cA = phiA, *cW = phiA + rows * ld, *cS = phiA + 2 * rows * ld;
                const R kx = MAC_TCOEF * a.inv_dx2, ky = MAC_TCOEF * a.inv_dy2;
                R *s_west = handoff_west(phiA, a);
                int *s_flag = handoff_flags(phiA, a);
                int *right_flag = last ? nullptr : cluster_map(s_flag, rank + 1);
                R *right_west = last ? nullptr : cluster_map(s_west, rank + 1);
                for (int ps = 0; ps < passes; ps++) {
                    const int pb = ib + ps * rows, pe = min(ie, pb + rows - 1);
                    // old values of row ie + 1 (rank g + 1) are read here, before this rank's last pass
                    // hands over the columns that rank g + 1 needs before it overwrites that row
                    CELL_LOOP {
                        const int i = i0 + r, j = j0 + k;
                        if (CELL_OK(i, j) && i >= pb && i <= pe) {
                            const R uE = u[(i + 1) * ld + j], uW = u[i * ld + j], vN = v[i * ld + j + 1], vS = v[i * ld + j];
                            const R sc = s[i * ld + j], sE = s[(i + 1) * ld + j], sN = s[i * ld + j + 1];
                            R diff0 = ((sE - R(2) * sc) * a.inv_dx2 + (sN - R(2) * sc) * a.inv_dy2) * MAC_TCOEF;
                            R conv0 = (uE * (R(0.5) * (sE + sc)) - uW * (R(0.5) * sc)) * a.inv_dx +
                                      (vN * (R(0.5) * (sN + sc)) - vS * (R(0.5) * sc)) * a.inv_dy;
                            const int e = (i - pb) * ld + j;
                            cA[e] = sc + a.dt * (diff0 - conv0);
                            cW[e] = a.dt * (kx + R(0.5) * uW * a.inv_dx);
                            cS[e] = a.dt * (ky + R(0.5) * vS * a.inv_dy);
                        }
                    }
                    __syncthreads();
                    if (tid < 32) {
                        constexpr int RPL = MAC_RPL;
                        const int lanes = (pe - pb + 1 + RPL - 1) / RPL;
                        const int lane = tid;
                        const int rb = pb + lane * RPL;
                        const bool from_left = ps == 0 && !first;        // row pb - 1 is rank g - 1's last row
                        const bool to_right = ps == passes - 1 && !last;  // row pe = ie feeds rank g + 1
                        R prev[RPL];
#pragma unroll
                        for (int q = 0; q < RPL; q++) prev[q] = (rb + q <= pe) ? s[(rb + q) * ld + 0] : R(0);
                        R last_new = R(0);
                        const int steps = ny + lanes - 1;
                        for (int t = 0; t < steps; t++) {
                            R wv = __shfl_up_sync(0xffffffffu, last_new, 1);
                            const int j = t - lane + 1;
                            if (lane < lanes && j >= 1 && j <= ny) {
                                if (lane == 0) {
                                    if (from_left) {
                                        if ((j - 1) % MAC_CLUSTER_CHUNK == 0)
                                            while (ld_acquire_cluster(&s_flag[(j - 1) / MAC_CLUSTER_CHUNK]) != seq) {}
                                        wv = s_west[j];
                                    } else wv = s[(pb - 1) * ld + j];
                                }
#pragma unroll
                                for (int q = 0; q < RPL; q++) {
                                    const int i = rb + q;
                                    if (i <= pe) {
                                        const int e = (i - pb) * ld + j;
                                        R nv = (cA[e] + cS[e] * prev[q]) + cW[e] * wv;
                                        s[i * ld + j] = nv;
                                        prev[q] = nv;
                                        wv = nv;
                                        if (to_right && i == pe) {
                                            right_west[j] = nv;
                                            if (j % MAC_CLUSTER_CHUNK == 0 || j == ny) st_release_cluster(&right_flag[(j - 1) / MAC_CLUSTER_CHUNK], seq);
                                        }
                                    }
                                }
                                last_new = wv;
                            }
                        }
                    }
                    __syncthreads();
                }
            }
        }   // sub-steps
        env_barrier<CLUSTER>();                                // every rank's rows done

        // ---- observations and reward: rank 0 writes, every rank contributes its rows -----------------
        R part = R(0);
        if (!ray) for (int e = e0 + tid; e < e1; e += T) part += rabs(s[e] - a.ref_c);
        part = block_sum(part, s_red);
        bool nonfinite = false;
        for (int e = e0 + tid; e < e1; e += T) nonfinite |= !finite_(s[e]) | !finite_(u[e]) | !finite_(v[e]);
        const int bad = __syncthreads_or(nonfinite ? 1 : 0);
        if (!CLUSTER) { if (tid == 0) { s_rank[0] = part; s_bad[0] = bad; } }
        else if (tid < G) { cluster_map(s_rank, tid)[rank] = part; cluster_map(s_bad, tid)[rank] = bad; }
        if (first) {
            R *hist = a.obs_hist + (size_t)b * a.n_obs;
            const int per_step = 3 * a.nx_obs_pts * a.ny_obs_pts;
            R *out = a.obs + orow * a.n_obs;
            for (int e = tid; e < a.n_obs; e += T) {
                int st = e / per_step, rm = e - st * per_step;
                R val;
                if (st < a.n_obs_steps - 1) val = hist[e + per_step];
                else {
                    int f = rm / (a.nx_obs_pts * a.ny_obs_pts), q = rm - f * (a.nx_obs_pts * a.ny_obs_pts);
                    int pi = q / a.ny_obs_pts, pj = q - pi * a.ny_obs_pts;
                    int x = a.nx_obs / 2 + pi * a.nx_obs, y = a.ny_obs / 2 + pj * a.ny_obs;
                    val = (f == 0) ? s[x * ld + y] : (f == 1 ? u[x * ld + y] : v[x * ld + y]);
                }
                out[e] = val;
            }
            __syncthreads();
            for (int e = tid; e < a.n_obs; e += T) hist[e] = out[e];
        }
        R nu = R(0);
        if (first && ray && tid == 0)                          // rayleigh.py:265-275 (sequential sum over i)
            for (int i = 1; i <= nx; i++) nu -= (s[i * ld + 1] - a.Th) / (R(0.5) * a.dy);
        env_barrier<CLUSTER>();                                // partials in place; obs read before the next walls
        int any_bad = 0;
        R total = R(0);
        for (int g = 0; g < G; g++) { any_bad |= s_bad[g]; total += s_rank[g]; }   // rank order
        if (any_bad) status |= BEACON_STATUS_NONFINITE;
        if (first && tid == 0) {
            a.rwd[orow] = ray ? -(nu / R(nx)) : -(total / R(a.n));
            bool horizon = stp == a.n_act - 1;
            a.done[orow] = horizon; a.trunc[orow] = horizon;
            if (a.iters) a.iters[orow] = it_total;
        }
        stp += 1;
    }   // actions

    if (first && tid == 0) { a.stp[b] = stp; if (a.status) a.status[b] = status; }
    env_barrier<CLUSTER>();                                    // no CTA leaves while a neighbour may write its shared memory
#undef CELL_LOOP
#undef CELL_OK
}
// The wrappers read threadIdx.x, where __launch_bounds__ bounds it, and mac_body takes MacArgs by value: otherwise
// the uniform instance compiles to different code (DESIGN.md 3.7).
template <typename R, int TI, int TJ, int T, bool CLUSTER>
__global__ void __launch_bounds__(T) mac_kernel(const MacArgs<R> a) { mac_body<R, TI, TJ, T, CLUSTER, false>(a, threadIdx.x); }
// per-env physical constants (MacArgs::phys)
template <typename R, int TI, int TJ, int T, bool CLUSTER>
__global__ void __launch_bounds__(T) mac_phys_kernel(const MacArgs<R> a) { mac_body<R, TI, TJ, T, CLUSTER, true>(a, threadIdx.x); }


// ---------------------------------------------------------------------------------------
// Transport wavefront (fp64), one warp, software pipelined by hand.
//   new(i,j) = A(i,j) + B_W(i,j) new(i-1,j) + B_S(i,j) new(i,j-1),  B_S = dky + hk v(i,j)
// Lane l owns rows 2l+1, 2l+2 and does column j = t - l + 1 at step t.  AA / WW hold A and B_W
// as [lane][column 0..NY][row in pair] (one LDS.128 per lane and step), V and S are the
// field planes (row stride LD).  Every address is base(lane) + step * const, so the unrolled
// loop uses immediate offsets only; inactive steps (column outside 1..NY) run on harmless
// in-bounds garbage and are masked by one predicate.  Per step the dependent chain is
// SHFL + 2 DFMA; coefficients are fetched two columns ahead.  A separate (noinline) function so
// that its register allocation is independent of the big per-env kernel around it.
// ---------------------------------------------------------------------------------------
template <typename R> struct vec2_of;
template <> struct vec2_of<double> { typedef double2 type; };
template <> struct vec2_of<float> { typedef float2 type; };

__device__ __forceinline__ double2 lds128_f64(uint32_t a)
{
    double2 v;
    asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ double lds64_f64(uint32_t a)
{
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}

template <int NX, int NY, int LDU, int LDT>
__device__ __noinline__ void transport_wavefront_f64(uint32_t sAA, uint32_t sWW, uint32_t sUV, uint32_t sS, double hk, double dky, int lane)
{
    // sUV: plane of (u, v) pairs, row stride LDU pairs (v = second component); sS: scalar plane, row stride LDT
    constexpr int LANES = NX / 2, STEPS = NY + LANES - 1, RS = wavefront_row_stride(NY);
    const bool on = lane < LANES;
    const int l = on ? lane : 0;                       // lanes beyond the last row pair mimic lane 0, predicate off
    const uint32_t rowA = (uint32_t)(l * RS) * 16u, rowV = (uint32_t)((2 * l + 1) * LDU) * 16u + 8u, rowS = (uint32_t)((2 * l + 1) * LDT) * 8u;
    // column 1: partial sums with the south ghost (column 0, untouched by transport)
    const double2 a1 = lds128_f64(sAA + rowA + 16u), w1c = lds128_f64(sWW + rowA + 16u);
    double p0 = fma(fma(hk, lds64_f64(sUV + rowV + 16u), dky), lds64_f64(sS + rowS), a1.x);
    double p1 = fma(fma(hk, lds64_f64(sUV + rowV + LDU * 16u + 16u), dky), lds64_f64(sS + rowS + LDT * 8u), a1.y);
    double w0 = w1c.x, w1 = w1c.y;
    // bases biased by -lane: element [t] is column t - l + 2 (coefficients) / t - l + 1 (store)
    const uint32_t aA = sAA + rowA + (uint32_t)(2 - l) * 16u, aW = sWW + rowA + (uint32_t)(2 - l) * 16u;
    const uint32_t aV = sUV + rowV + (uint32_t)(2 - l) * 16u;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // store pointers: S plane rows 2l+1, 2l+2, biased so that element [t] is column t - l + 1
    double *S0o = reinterpret_cast<double *>(smem_raw + (sS - (uint32_t)__cvta_generic_to_shared(smem_raw)) + rowS) + (1 - l), *S1o = S0o + LDT;
    double2 an = lds128_f64(aA), wn = lds128_f64(aW);
    double v0n = lds64_f64(aV), v1n = lds64_f64(aV + LDU * 16u);
    double last_new = 0.0;
    const int c0 = on ? -lane : -(1 << 20);
    // unrolled by 6 so that the three column records in flight rotate through registers without
    // copies; the trip count is padded to a multiple of 6 (the extra steps are inactive, their
    // reads stay inside the planes)
    constexpr int STEPS_PAD = ((STEPS + 5) / 6) * 6;
    static_assert(((NX / 2 - 1) * RS + 2 - (NX / 2 - 1) + STEPS_PAD + 1) * 2 <= (NX + 1) * (((NY + 2 + 6) / 8) * 8 + 1), "padded reads leave the A/W planes");
    static_assert((NX - 1) * LDU + 2 - (NX / 2 - 1) + STEPS_PAD + 1 + LDU <= (NX + 2) * LDU, "padded reads leave the (u, v) plane");
#pragma unroll 6
    for (int t = 0; t < STEPS_PAD; t++) {
        // fetch two columns ahead
        const double2 an2 = lds128_f64(aA + (uint32_t)(t + 1) * 16u), wn2 = lds128_f64(aW + (uint32_t)(t + 1) * 16u);
        const double v0n2 = lds64_f64(aV + (uint32_t)(t + 1) * 16u), v1n2 = lds64_f64(aV + LDU * 16u + (uint32_t)(t + 1) * 16u);
        const double wv = __shfl_up_sync(0xffffffffu, last_new, 1);
        const int act_ = (unsigned)(c0 + t) < (unsigned)NY;
        const double s0n = fma(hk, v0n, dky), s1n = fma(hk, v1n, dky);
        const double n0 = fma(w0, wv, p0);
        const double n1 = fma(w1, n0, p1);
        last_new = n1;
        // plain C++ stores (the coefficient loads above are plain asm that never aliases them, so the
        // compiler hoists the loads over the stores: with an ordered asm store every load waited for the
        // previous step's store and its latency sat in the dependent chain — 81 -> 48 cycles per step
        // in isolation, tools/micro/wave.cu)
        if (act_) {
            S0o[t] = n0; S1o[t] = n1;
            p0 = fma(s0n, n0, an.x); p1 = fma(s1n, n1, an.y);
        }
        w0 = wn.x; w1 = wn.y;
        an = an2; wn = wn2; v0n = v0n2; v1n = v1n2;
    }
}

// ---------------------------------------------------------------------------------------
// `!(err > tol)` of one Jacobi sweep decided in fp64: the per-thread residuals `mine` are summed by the
// xor butterfly (16, 8, 4, 2, 1) and the warp partials by a pairwise tree, the same order in every thread.
// Called by ALL threads of the CTA (uniform branch), only when the fp32 total of the fast path lies within
// 1e-4 tol of tol; out of line so that the sweep loop stays compact.
// ---------------------------------------------------------------------------------------
template <typename R, int NW>
__device__ __noinline__ bool residual_converged_exact(R mine, R *s_exact, R tol)
{
    R v = mine;
#pragma unroll
    for (int st = 0; st < 5; st++) v += __shfl_xor_sync(0xffffffffu, v, 16 >> st);
    if ((threadIdx.x & 31) == 0) s_exact[threadIdx.x >> 5] = v;
    __syncthreads();
    R q[NW];
#pragma unroll
    for (int w = 0; w < NW; w++) q[w] = s_exact[w];
#pragma unroll
    for (int st = 1; st < NW; st *= 2)
#pragma unroll
        for (int w = 0; w + st < NW; w += 2 * st) q[w] += q[w + st];
    __syncthreads();
    return !(q[0] > tol);
}

// ---------------------------------------------------------------------------------------
// Register-resident variant (rayleigh 50x50: five planes fit twice per SM).
//   * shared memory: two phi exchange planes (row stride LDP = 57 doubles: with 2x5 tiles laid
//     out 10 per tile-row the 64-bit bank index of a lane's tile origin is 5*lane mod 16 ->
//     conflict free) + U, V, S planes (stride NY+2) = 112 KB -> 2 CTAs/SM;
//   * grid size is a template parameter: every plane access of a thread is base register +
//     immediate offset;
//   * each thread keeps phi AND the Poisson right-hand side of its TI x TJ tile in registers for
//     the whole solve; a sweep reads only the 2(TI+TJ) halo values from the exchange plane and
//     writes its tile (+ the ghost copies it owns) to the other plane: one __syncthreads;
//   * predictor output (us, vs) is staged in registers over one barrier and then overwrites U, V
//     in place (old u, v are dead after the predictor; wall entries are 0 in both); the corrector
//     is a pointwise in-place update; p stays in L2-resident global memory, in a thread-interleaved
//     scratch ([cell][thread], coalesced) for the duration of a launch;
//   * the first sweep (phi = 0) needs no halo: the exchange planes are never zeroed;
//   * transport: A and B_W planes are written by all threads into the (then free) phi planes,
//     B_S comes from V on the fly; ONE warp runs the recurrence over all rows in a single
//     software-pipelined pass (coefficients of column j+1 are loaded while column j waits for
//     the shuffle), critical path per column = SHFL + 2 FMA.
// ---------------------------------------------------------------------------------------
// Row stride of the exchange planes: with ten tiles per tile row (TJ = 5, tid = 10 ti + tj) the tile origins of a
// half-warp fall into 16 distinct 8-byte banks iff (TI * LDP) mod 16 == 2 (TI = 2: 57, TI = 5: 58).
constexpr int mac_ldp(int ld, int ti) { int l = ld; while ((ti * l) % 16 != 2) l++; return l; }

#define MAC_REG_NAME mac_reg_kernel
#define MAC_REG_PHYS false
#include "mac_reg_kernel.cuh"
#undef MAC_REG_NAME
#undef MAC_REG_PHYS
#define MAC_REG_NAME mac_reg_phys_kernel
#define MAC_REG_PHYS true
#include "mac_reg_kernel.cuh"
#undef MAC_REG_NAME
#undef MAC_REG_PHYS

// ---------------------------------------------------------------------------------------
// Three-plane transport wavefront, shared memory only (any real type):
//   new(i,j) = A + B_W new(i-1,j) + B_S new(i,j-1)
// AA / WW / SS hold A, B_W, B_S as [lane = row pair][column 0..NY][row in pair] at byte offsets
// offA / offW / offS of the dynamic shared memory; the ghost row west of the first row and the
// ghost column south of column 1 are folded into A by the threads that wrote the planes (B_W = 0
// on the first row, B_S = 0 in column 1), so the loop is uniform: lane l does column t - l + 1
// at step t, steps before its first column run on in-bounds garbage that the zero B_S of column 1
// wipes out, steps after its last column are masked by the store predicate.  New values
// overwrite A in place.  Per step: 3 x 16-byte loads, 2 shuffles, 4 FMAs, one predicated store.
// ---------------------------------------------------------------------------------------

__device__ __forceinline__ double2 lds_pair(const double2 *p)
{
    return lds128_f64((uint32_t)__cvta_generic_to_shared(p));
}
__device__ __forceinline__ float2 lds_pair(const float2 *p)
{
    float2 v;
    asm("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"((uint32_t)__cvta_generic_to_shared(p)));
    return v;
}

template <typename R, int NY>
__device__ __noinline__ void transport_wavefront3(uint32_t offA, uint32_t offW, uint32_t offS, int lanes, int lane)
{
    typedef typename vec2_of<R>::type R2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int RS = wavefront_row_stride(NY);
    const bool on = lane < lanes;
    const int l = on ? lane : 0;                       // lanes beyond the last row pair mimic lane 0, stores off
    R2 *AA = reinterpret_cast<R2 *>(smem_raw + offA) + l * RS;
    const R2 *WW = reinterpret_cast<const R2 *>(smem_raw + offW) + l * RS, *SS = reinterpret_cast<const R2 *>(smem_raw + offS) + l * RS;
    R p0 = AA[1].x, p1 = AA[1].y, w0 = WW[1].x, w1 = WW[1].y;
    // biased by -lane: element [t] is column t - l + 2 (coefficients) / t - l + 1 (store)
    const R2 *An = AA + (2 - l), *Wn = WW + (2 - l), *Sn = SS + (2 - l);
    R2 *Out = AA + (1 - l);
    R2 an = An[0], wn = Wn[0], sn = Sn[0];
    R last_new = R(0);
    const int c0 = on ? -lane : -(1 << 20);
    const int steps = ((NY + lanes - 1 + 5) / 6) * 6;   // padded: the extra steps are masked, their reads stay in shared memory
#pragma unroll 6
    for (int t = 0; t < steps; t++) {
        // two columns ahead.  Plain (non-volatile) asm loads: a lane never reads a slot of its own row pair that it has
        // stored (loads run two columns ahead of the stores), so they may be hoisted over the C++ stores below; as C++
        // loads of the same array they were ordered behind the previous step's store and their latency sat in the
        // dependent chain: 81 -> 48 cycles per step in isolation (tools/micro/wave.cu)
        const R2 an2 = lds_pair(An + t + 1), wn2 = lds_pair(Wn + t + 1), sn2 = lds_pair(Sn + t + 1);
        const R wv = __shfl_up_sync(0xffffffffu, last_new, 1);
        const R n0 = fma(w0, wv, p0);
        const R n1 = fma(w1, n0, p1);
        last_new = n1;
        if ((unsigned)(c0 + t) < (unsigned)NY) { R2 o; o.x = n0; o.y = n1; Out[t] = o; }
        p0 = fma(sn.x, n0, an.x); p1 = fma(sn.y, n1, an.y);
        w0 = wn.x; w1 = wn.y;
        an = an2; wn = wn2; sn = sn2;
    }
}

// ---------------------------------------------------------------------------------------
// Large-grid variant (mixing 100x100): register-resident Poisson exactly as in mac_reg_kernel
// (phi and the right-hand side of a TI x TJ tile in registers, in-place sweeps, strided exchange
// planes, residual reduction two sweeps behind), the velocity / scalar / pressure planes stay in
// L2-resident global memory (Poisson is > 90 % of the work: ~65 sweeps per sub-step), transport in
// row passes through the three-plane wavefront above.  One CTA per SM.
// ---------------------------------------------------------------------------------------
template <typename R, int NX, int NY, int TI, int TJ, int T, int MINB, bool DBG, bool PHYS>
__device__ __forceinline__ void mac_big_body(const MacArgs<R> &a, const unsigned thread_x)
{
    constexpr int LD = NY + 2, N = (NX + 2) * LD;
    constexpr int LDP = ((LD + 6) / 8) * 8 + 1;         // exchange planes: stride = 1 mod 8
    constexpr int NP = ((NX + 2) * LDP + 3) / 4 * 4;    // plane size: a multiple of 16 bytes for fp32 too (PB is a bulk-copy destination)
    constexpr int TILES_J = NY / TJ, TILES = (NX / TI) * TILES_J, NW = T / 32;
    constexpr int RS = wavefront_row_stride(NY);        // wavefront planes: columns 0..NY per row pair, padded
    constexpr int PASS_ROWS = ((NX / 2 + TI - 1) / TI) * TI >= 64 ? 64 / TI * TI : ((NX / 2 + TI - 1) / TI) * TI;   // rows per transport pass
    constexpr int PASSES = (NX + PASS_ROWS - 1) / PASS_ROWS, LANES_MAX = PASS_ROWS / 2;
    static_assert(NX % TI == 0 && NY % TJ == 0 && TILES <= T && TI % 2 == 0, "tiles must cover the grid exactly");
    static_assert((NP * sizeof(R)) % 16 == 0, "bulk copies need 16-byte aligned planes");
    static_assert(LANES_MAX <= 32 && 3 * (LANES_MAX * RS + 8) * 2 <= 2 * NP, "transport planes must fit the exchange planes");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(16) float s_part[2][NW];     // fp32 warp partials of the residual (see mac_reg_kernel)
    __shared__ R s_exact[NW];                         // fp64 warp partials, only when the fp32 total is too close to tol
    __shared__ __align__(8) uint64_t s_mbar;
    __shared__ R s_red[NW];
    __shared__ R s_seg[128];
    __shared__ R s_act[128];
    const int tid = thread_x, b = blockIdx.x;
    const bool resetting = a.mode == 1;
    if (resetting && a.mask && !a.mask[b]) return;
    const bool ray = a.kind == BEACON_RAYLEIGH;

    R *PA = reinterpret_cast<R *>(smem_raw), *PB = PA + NP;
    const size_t row = (size_t)b * N;
    R *u = a.u + row, *v = a.v + row, *p = a.p + row, *s = a.s + row;
    // Thread-private copies of the tile of p, us, vs live in a per-env scratch laid out
    // [field][cell][thread]: a thread's tile rows are 5 doubles at an odd offset in the planes (a warp
    // access would touch 10 cache lines), in the scratch consecutive lanes are contiguous (2 lines),
    // and the neighbour tile's cell is the same slot 1 / TILES_J threads away — equally coalesced.
    constexpr int CELLS = TI * TJ;
    R *sp = a.cc + (size_t)b * (3 * CELLS * T) + tid, *sus = sp + CELLS * T, *svs = sus + CELLS * T;
#define SC(base, r, k) (base)[((r) * TJ + (k)) * T]

    const bool has_tile = tid < TILES;
    const int ti = tid / TILES_J, tj = tid - ti * TILES_J;
    const int i0 = 1 + ti * TI, j0 = 1 + tj * TJ;
    const int o = i0 * LD + j0, op = i0 * LDP + j0;     // tile origin in field / exchange planes
    const int opx = has_tile ? op : LDP + 1;             // threads without a tile shadow tile 0 in the sweeps (weight 0)
    const bool top = has_tile && i0 == 1, bot = has_tile && i0 + TI - 1 == NX;
    const bool lef = has_tile && j0 == 1, rig = has_tile && j0 + TJ - 1 == NY;
    const R w_has = has_tile ? R(1) : R(0);
    // residual weights: ghost copies re-count wall-adjacent cells; mixing's j = NY+1 ghost is Dirichlet 0 (mixing.py:451)
    const R w_top = top ? R(2) : R(1), w_bot = bot ? R(2) : R(1), w_lef = lef ? R(1) : R(0), w_rig = (rig && ray) ? R(1) : R(0);
    // Halo offsets of the Jacobi sweeps: a Neumann ghost is a copy of the wall-adjacent cell, so wall tiles read
    // their own edge row / column instead (no ghost cell of phi is ever stored); mixing's Dirichlet ghost
    // phi(i, NY+1) = 0 (mixing.py:451) is a constant.  Threads without a tile shadow tile 0.
    const int tix = has_tile ? ti : 0, tjx = has_tile ? tj : 0;
    const int o_n = tix == 0 ? 0 : -LDP, o_s = tix == NX / TI - 1 ? (TI - 1) * LDP : TI * LDP;
    const bool lefx = tjx == 0, rigx = tjx == TILES_J - 1;
    const bool dir_e = rig && !ray;
#define TILE_LOOP                                      \
    _Pragma("unroll") for (int r = 0; r < TI; r++)     \
    _Pragma("unroll") for (int k = 0; k < TJ; k++)
    const int per_step = 3 * a.nx_obs_pts * a.ny_obs_pts;

    if (resetting) {                                   // rayleigh.py:89-128, mixing.py:73-111
        for (int e = tid; e < N; e += T) {
            u[e] = ray ? a.u0[e] : R(0); v[e] = ray ? a.v0[e] : R(0); p[e] = ray ? a.p0[e] : R(0); s[e] = a.s0[e];
        }
        for (int e = tid; e < (ray ? a.n_sgts : 0); e += T) a.a_cur[(size_t)b * a.n_sgts + e] = R(0);
        R *hist = a.obs_hist + (size_t)b * a.n_obs;
        for (int e = tid; e < a.n_obs; e += T) {
            int st = e / per_step, rem = e - st * per_step;
            R val = R(0);
            if (st == a.n_obs_steps - 1) {
                int f = rem / (a.nx_obs_pts * a.ny_obs_pts), q = rem - f * (a.nx_obs_pts * a.ny_obs_pts);
                int pi = q / a.ny_obs_pts, pj = q - pi * a.ny_obs_pts;
                int x = a.nx_obs / 2 + pi * a.nx_obs, y = a.ny_obs / 2 + pj * a.ny_obs;
                val = (f == 0) ? a.s0[x * LD + y] : (ray ? (f == 1 ? a.u0[x * LD + y] : a.v0[x * LD + y]) : R(0));
            }
            hist[e] = val;
            a.obs[(size_t)b * a.n_obs + e] = val;
        }
        if (tid == 0) { a.stp[b] = 0; if (!ray) a.a_int[b] = 1; }
        return;
    }
    int stp = a.stp[b];
    int status = 0;
    MAC_LOAD_COEF(b);                                  // read after the barrier that opens each action
    const R dt = a.dt, inv_dx = a.inv_dx, inv_dy = a.inv_dy;
    // The uniform transport wavefront reads a few never-written padding slots of the planes during its
    // masked steps; their values cannot reach a result as long as they are finite (they are multiplied
    // by the zero B_S of column 1), so the planes must not start with stale NaN bit patterns.
    for (int e = tid; e < 2 * NP; e += T) PA[e] = R(0);
    if (tid == 0) { mbar_init(&s_mbar, 1); fence_async_smem(); }
    uint32_t stage_phase = 0;
    // pressure: the scratch copy is authoritative during the launch; the plane keeps the launch-initial
    // values until the end (needed for the ghost cells, see there)
    if (has_tile) { TILE_LOOP { SC(sp, r, k) = p[o + r * LD + k]; } }
    const bool dbg = DBG && a.dbg != nullptr && b == 0 && tid == 0;
    long long tph[DBG ? 8 : 1] = {0}, tlast = dbg ? clock64() : 0;
#define PHASE(n) do { if (DBG && dbg) { long long tn_ = clock64(); tph[n] += tn_ - tlast; tlast = tn_; } } while (0)

    for (int act = 0; act < a.n_fused; act++) {
        const size_t orow = (size_t)act * a.B + b;
        __syncthreads();
        // ---- action conditioning ----------------------------------------------------------------
        if (ray) {
            if (tid == 0) {                                        // rayleigh.py:164-171
                const R *ain = (const R *)a.actions + orow * a.n_sgts;
                const int ns = a.n_sgts;
                for (int j = 0; j < ns; j++) s_act[j] = ain[j];
                R mean = np_pairwise_small(s_act, ns) / R(ns);
                R m = R(1);
                for (int j = 0; j < ns; j++) { s_act[j] = s_act[j] - mean; m = np_max(m, rabs(s_act[j]) / a.Cmax); }
                for (int j = 0; j < ns; j++) { s_act[j] = s_act[j] / m; s_seg[j] = a.Th + s_act[j]; a.a_cur[(size_t)b * ns + j] = s_act[j]; }
            }
        } else if (tid == 0) {                                     // get_control, mixing.py:212-234
            int ai = ((const int32_t *)a.actions)[orow];
            R ut = 0, ub = 0, vl = 0, vr = 0;
            if (ai == 0) { ub = MAC_UMAX; ut = -MAC_UMAX; }
            if (ai == 1) { ub = -MAC_UMAX; ut = MAC_UMAX; }
            if (ai == 2) { vr = MAC_UMAX; vl = -MAC_UMAX; }
            if (ai == 3) { vr = -MAC_UMAX; vl = MAC_UMAX; }
            s_seg[0] = ut; s_seg[1] = ub; s_seg[2] = vl; s_seg[3] = vr;
            a.a_int[b] = ai;
        }
        __syncthreads();
        long long it_total = 0;

        for (int it = 0; it < a.ndt_act; it++) {
            // ---- boundary conditions: rayleigh.py:180-202, mixing.py:153-171 ---------------------
            for (int k = tid; k < 2 * (NX + 2) + 2 * (NY + 2); k += T) {
                if (k < NY + 2) {                                  // left wall (i = 0/1), index j = k
                    int j = k;
                    if (j >= 1 && j <= NY) { u[1 * LD + j] = R(0); s[0 * LD + j] = s[1 * LD + j]; }
                    if (j >= 2 && j <= NY) v[0 * LD + j] = ray ? -v[1 * LD + j] : R(2) * s_seg[2] - v[1 * LD + j];
                } else if (k < 2 * (NY + 2)) {                     // right wall
                    int j = k - (NY + 2);
                    if (j >= 1 && j <= NY) { u[(NX + 1) * LD + j] = R(0); s[(NX + 1) * LD + j] = s[NX * LD + j]; }
                    if (j >= 2 && j <= NY) v[(NX + 1) * LD + j] = ray ? -v[NX * LD + j] : R(2) * s_seg[3] - v[NX * LD + j];
                } else if (k < 2 * (NY + 2) + (NX + 2)) {          // top wall (j = NY+1), index i
                    int i = k - 2 * (NY + 2);
                    if (i >= 1 && i <= NX + 1) {
                        R ui = (i == 1 || i == NX + 1) ? R(0) : u[i * LD + NY];
                        u[i * LD + NY + 1] = ray ? -ui : R(2) * s_seg[0] - ui;
                    }
                    if (i >= 1 && i <= NX) {
                        v[i * LD + NY + 1] = R(0);
                        s[i * LD + NY + 1] = ray ? R(2) * a.Tc - s[i * LD + NY] : s[i * LD + NY];
                    }
                } else {                                           // bottom wall (j = 0/1)
                    int i = k - 2 * (NY + 2) - (NX + 2);
                    if (i >= 1 && i <= NX + 1) {
                        R ui = (i == 1 || i == NX + 1) ? R(0) : u[i * LD + 1];
                        u[i * LD + 0] = ray ? -ui : R(2) * s_seg[1] - ui;
                    }
                    if (i >= 1 && i <= NX) {
                        v[i * LD + 1] = R(0);
                        if (ray) {
                            int sg = (i - 1) / a.nx_sgts;
                            if (sg < a.n_sgts) s[i * LD + 0] = R(2) * s_seg[sg] - s[i * LD + 1];
                        } else s[i * LD + 0] = s[i * LD + 1];
                    }
                }
            }
            // stage u and v (ghosts included) in the exchange planes, free until the Poisson solve: the
            // predictor reads ~15 neighbours per cell, from shared memory instead of L2.  Two bulk copies
            // (TMA engine) issued by one thread; everybody waits on the mbarrier.
            static_assert((N * sizeof(R)) % 16 == 0, "bulk copies need 16-byte multiples");
            fence_async_gmem(); fence_async_smem();    // my boundary writes / earlier plane accesses -> ordered before the bulk engine's
            __syncthreads();
            if (tid == 0) {
                mbar_expect_tx(&s_mbar, 2u * (uint32_t)(N * sizeof(R)));
                bulk_g2s(PA, u, (uint32_t)(N * sizeof(R)), &s_mbar);
                bulk_g2s(PB, v, (uint32_t)(N * sizeof(R)), &s_mbar);
            }
            mbar_wait(&s_mbar, stage_phase);
            stage_phase ^= 1u;
            __syncthreads();
            PHASE(0);

            // ---- predictor: rayleigh.py:371-407, mixing.py:382-416 (us, vs in registers and in global memory) ----
            R cn[TI][TJ], phi[TI][TJ];
            {
            R usr[TI][TJ], vsr[TI][TJ];
            if (has_tile) {
                const R *uu = PA + o, *vv = PB + o, *sc = s + o;
                R pt[TI][TJ], pwh[TJ], psh[TI];    // my pressure tile, the last row of the tile above, the last column of the left tile
                TILE_LOOP { pt[r][k] = SC(sp, r, k); }
#pragma unroll
                for (int k = 0; k < TJ; k++) pwh[k] = top ? R(0) : SC(sp - TILES_J, TI - 1, k);
#pragma unroll
                for (int r = 0; r < TI; r++) psh[r] = lef ? R(0) : SC(sp - 1, r, TJ - 1);
                TILE_LOOP {
                    const int e = r * LD + k;
                    const R uc = uu[e], vc = vv[e], pc = pt[r][k];
                    usr[r][k] = R(0); vsr[r][k] = R(0);
                    if (r > 0 || !top) {               // i >= 2
                        R uE = R(0.5) * (uu[e + LD] + uc), uW = R(0.5) * (uc + uu[e - LD]);
                        R uN = R(0.5) * (uu[e + 1] + uc), uS = R(0.5) * (uc + uu[e - 1]);
                        R vN = R(0.5) * (vv[e + 1] + vv[e - LD + 1]), vS = R(0.5) * (vc + vv[e - LD]);
                        R conv = (uE * uE - uW * uW) * inv_dx + (uN * vN - uS * vS) * inv_dy;
                        R diff = ((uu[e + LD] - R(2) * uc + uu[e - LD]) * a.inv_dx2 + (uu[e + 1] - R(2) * uc + uu[e - 1]) * a.inv_dy2) * MAC_DCOEF;
                        R pres = (pc - ((r > 0) ? pt[r - 1][k] : pwh[k])) * inv_dx;
                        usr[r][k] = uc + dt * (diff - conv - pres);
                    }
                    if (k > 0 || !lef) {               // j >= 2
                        R vE = R(0.5) * (vv[e + LD] + vc), vW = R(0.5) * (vc + vv[e - LD]);
                        R uE = R(0.5) * (uu[e + LD] + uu[e + LD - 1]), uW = R(0.5) * (uc + uu[e - 1]);
                        R vN = R(0.5) * (vv[e + 1] + vc), vS = R(0.5) * (vc + vv[e - 1]);
                        R conv = (uE * vE - uW * vW) * inv_dx + (vN * vN - vS * vS) * inv_dy;
                        R diff = ((vv[e + LD] - R(2) * vc + vv[e - LD]) * a.inv_dx2 + (vv[e + 1] - R(2) * vc + vv[e - 1]) * a.inv_dy2) * MAC_DCOEF;
                        R pres = (pc - ((k > 0) ? pt[r][k - 1] : psh[r])) * inv_dy;
                        R rhs = diff - conv - pres;
                        if (ray) rhs += sc[e];
                        vsr[r][k] = vc + dt * rhs;
                    }
                }
                TILE_LOOP { SC(sus, r, k) = usr[r][k]; SC(svs, r, k) = vsr[r][k]; }   // walls: 0 (i = 1 / j = 1)
            }
            __syncthreads();                       // us, vs of the neighbouring tiles are visible
            // Poisson right-hand side cn = -div(us, vs)/dt dx2 dy2 / (2 (dx2 + dy2)); phi_1 = cn
            TILE_LOOP {
                R cv = R(0);
                if (has_tile) {
                    const R ue = (r < TI - 1) ? usr[r + 1][k] : (bot ? R(0) : SC(sus + TILES_J, 0, k));     // us(NX+1, j) = 0
                    const R vn = (k < TJ - 1) ? vsr[r][k + 1] : (rig ? R(0) : SC(svs + 1, r, 0));           // vs(i, NY+1) = 0
                    cv = -(((ue - usr[r][k]) * inv_dx + (vn - vsr[r][k]) * inv_dy) * a.cscale) * a.inv_den;
                }
                cn[r][k] = cv; phi[r][k] = cv;
            }
            }

            PHASE(1);
            // ---- Poisson (see mac_reg_kernel): rayleigh.py:412-456 / mixing.py:421-465 ----------------
            R *const pa = PA + opx, *const pb = PB + opx;
            auto tile_acc = [&](const R (&rs)[TI], const R (&dl)[TI], const R (&dr)[TI]) -> R {
                R cl = dl[0] * dl[0], cr = dr[0] * dr[0], mid = R(0);
#pragma unroll
                for (int r = 1; r < TI; r++) { cl = fma(dl[r], dl[r], cl); cr = fma(dr[r], dr[r], cr); }
#pragma unroll
                for (int r = 1; r < TI - 1; r++) mid += rs[r];
                R acc = (TI > 1) ? fma(rs[0], w_top, fma(rs[TI - 1], w_bot, mid)) : rs[0] * (w_top + w_bot - R(1));
                return fma(cl, w_lef, fma(cr, w_rig, acc));
            };
            auto sweep = [&](R (&ph)[TI][TJ], const R *pi, float &wsum) -> R {
                // in place, column by column; halo values are fetched where they are used (register budget)
                R rs[TI], po_[TI], cl = R(0), cr = R(0);
                const R *pn = pi + o_n, *ps = pi + o_s;
                // west / east halo at uniform offsets (conflict free); wall tiles use their own edge column (registers)
#pragma unroll
                for (int r = 0; r < TI; r++) { rs[r] = R(0); const R hw = pi[r * LDP - 1]; po_[r] = lefx ? ph[r][0] : hw; }
#pragma unroll
                for (int k = 0; k < TJ; k++) {
                    if (k < 5) wsum += __shfl_xor_sync(0xffffffffu, wsum, 16 >> k);
                    const R hnk = pn[k], hsk = ps[k];
                    R old[TI];
#pragma unroll
                    for (int r = 0; r < TI; r++) old[r] = ph[r][k];
#pragma unroll
                    for (int r = 0; r < TI; r++) {
                        const R xm = (r > 0) ? old[r - 1] : hnk, xp = (r < TI - 1) ? old[r + 1] : hsk;
                        R yp;
                        if (k < TJ - 1) yp = ph[r][k + 1];
                        else { const R he = pi[r * LDP + TJ]; yp = dir_e ? R(0) : (rigx ? old[r] : he); }
                        const R ym = po_[r];
                        const R nv = fma(xp + xm, a.pk1, fma(yp + ym, a.pk2, cn[r][k]));
                        const R d = nv - old[r];
                        rs[r] = fma(d, d, rs[r]);
                        if (k == 0) cl = fma(d, d, cl);
                        if (k == TJ - 1) cr = fma(d, d, cr);
                        ph[r][k] = nv;
                        po_[r] = old[r];
                    }
                }
#pragma unroll
                for (int st = TJ; st < 5; st++) wsum += __shfl_xor_sync(0xffffffffu, wsum, 16 >> st);
                R mid = R(0);
#pragma unroll
                for (int r = 1; r < TI - 1; r++) mid += rs[r];
                const R acc = (TI > 1) ? fma(rs[0], w_top, fma(rs[TI - 1], w_bot, mid)) : rs[0] * (w_top + w_bot - R(1));
                return fma(cl, w_lef, fma(cr, w_rig, acc));
            };
            auto commit = [&](const R (&nw)[TI][TJ], R *po) {
                if (has_tile) { TILE_LOOP { po[r * LDP + k] = nw[r][k]; } }
            };
            auto total32 = [&](const float *part) -> float {   // fixed pairwise order in every thread -> uniform decision
                static_assert(NW % 4 == 0, "warp partials are read as float4");
                float q[NW];
#pragma unroll
                for (int w = 0; w < NW; w += 4) {
                    const float4 v = *reinterpret_cast<const float4 *>(part + w);
                    q[w] = v.x; q[w + 1] = v.y; q[w + 2] = v.z; q[w + 3] = v.w;
                }
#pragma unroll
                for (int st = 1; st < NW; st *= 2)
#pragma unroll
                    for (int w = 0; w + st < NW; w += 2 * st) q[w] += q[w + st];
                return q[0];
            };
            const float tolf = (float)a.tol, tol_band = 1.0e-4f * (float)a.tol;
            auto converged = [&](const float err32, const R mine) -> bool {   // see mac_reg_kernel
                if (fabsf(err32 - tolf) > tol_band) return !(err32 > tolf);
                return residual_converged_exact<R, NW>(mine, s_exact, a.tol);
            };
            R accp, accq = R(0);
            {   // sweep 1 starts from phi = 0: phi_1 = cn, no halo reads
                R rs[TI], dl[TI], dr[TI];
#pragma unroll
                for (int r = 0; r < TI; r++) {
                    rs[r] = R(0);
#pragma unroll
                    for (int k = 0; k < TJ; k++) {
                        const R cv = cn[r][k];
                        rs[r] = fma(cv, cv, rs[r]);
                        if (k == 0) dl[r] = cv;
                        if (k == TJ - 1) dr[r] = cv;
                    }
                }
                accp = tile_acc(rs, dl, dr) * w_has;
                commit(phi, pb);
                __syncthreads();
            }
            {   // sweep 2
                float ws = (float)accp;
                const R acc = sweep(phi, pb, ws) * w_has;
                commit(phi, pa);
                if ((tid & 31) == 0) s_part[1][tid >> 5] = ws;
                __syncthreads();
                accq = accp; accp = acc;
            }
            int itp;
            const R *pf;                                  // plane holding the final iterate (tile-relative)
            // One CTA per SM: nobody fills the gaps of a sweep, so the tile stores must overlap the arithmetic.  The
            // stores of sweep k overwrite phi_{k-2}, which a converged solve returns — hence the decision on sweep k-2
            // (partials published at the previous barrier) is taken FIRST, right after the west halo loads are issued,
            // and every tile column is stored as soon as it is computed.  Compared with deciding after the sweep
            // (mac_reg_kernel, where a second CTA hides the store phase and the exposed decision latency cost more than
            // it won) a converged solve also drops one speculative sweep instead of two.  Same decisions, same sweep
            // counts.  Where exactly the decision sits matters through the register allocation: taken after the first
            // column it left 14 spilled doubles per sweep in the loop (3.81 k env-actions/s), here 5 (4.09 k).
            auto iter = [&](const R *pi, R *po, const float *part_rd, float *part_wr, const int kdec) -> int {
                float wsum = (float)accp;
                R rt = R(0), rb = R(0), rm = R(0), po_[TI], cl = R(0), cr = R(0);   // residual: first / last / middle tile rows
                const R *pn = pi + o_n, *ps = pi + o_s;
#pragma unroll
                for (int r = 0; r < TI; r++) { const R hw = pi[r * LDP - 1]; po_[r] = lefx ? phi[r][0] : hw; }
                {                                 // sweep kdec = k - 2: converged?  (nothing of phi_{k-2} has been overwritten yet)
                    const float err = total32(part_rd);
                    if (kdec > a.itmax) return 2;
                    if (converged(err, accq)) return 1;
                }
#pragma unroll
                for (int k = 0; k < TJ; k++) {
                    if (k < 5) wsum += __shfl_xor_sync(0xffffffffu, wsum, 16 >> k);
                    const R hnk = pn[k], hsk = ps[k];
                    R old[TI];
#pragma unroll
                    for (int r = 0; r < TI; r++) old[r] = phi[r][k];
#pragma unroll
                    for (int r = 0; r < TI; r++) {
                        const R xm = (r > 0) ? old[r - 1] : hnk, xp = (r < TI - 1) ? old[r + 1] : hsk;
                        R yp;
                        if (k < TJ - 1) yp = phi[r][k + 1];
                        else { const R he = pi[r * LDP + TJ]; yp = dir_e ? R(0) : (rigx ? old[r] : he); }
                        const R ym = po_[r];
                        const R nv = fma(xp + xm, a.pk1, fma(yp + ym, a.pk2, cn[r][k]));
                        const R d = nv - old[r];
                        if (r == 0) rt = fma(d, d, rt); else if (r == TI - 1) rb = fma(d, d, rb); else rm = fma(d, d, rm);
                        if (k == 0) cl = fma(d, d, cl);
                        if (k == TJ - 1) cr = fma(d, d, cr);
                        phi[r][k] = nv;
                        po_[r] = old[r];
                    }
                    if (has_tile) {
#pragma unroll
                        for (int r = 0; r < TI; r++) po[r * LDP + k] = phi[r][k];
                    }
                }
#pragma unroll
                for (int st = TJ; st < 5; st++) wsum += __shfl_xor_sync(0xffffffffu, wsum, 16 >> st);
                static_assert(TI > 1, "first and last tile row are distinct");
                const R acc0 = fma(rt, w_top, fma(rb, w_bot, rm));
                const R acc = fma(cl, w_lef, fma(cr, w_rig, acc0)) * w_has;
                if ((tid & 31) == 0) part_wr[tid >> 5] = wsum;
                __syncthreads();
                accq = accp; accp = acc;
                return 0;
            };
            for (int k = 3;; k += 2) {
                // odd k: phi_{k-1} (in PA) -> phi_k (into PB, which holds phi_{k-2} until the decision on it is taken)
                int st = iter(pa, pb, s_part[1], s_part[0], k - 2);
                if (st) { if (st == 2) status |= BEACON_STATUS_POISSON_OVERFLOW; itp = k - 2; pf = pb; break; }
                st = iter(pb, pa, s_part[0], s_part[1], k - 1);
                if (st) { if (st == 2) status |= BEACON_STATUS_POISSON_OVERFLOW; itp = k - 1; pf = pa; break; }
            }
            TILE_LOOP { phi[r][k] = pf[r * LDP + k]; }     // the converged iterate
            it_total += itp;
            PHASE(2);

            // ---- p += phi (rayleigh.py:219 / mixing.py:188; ghost cells: end of the launch) and corrector (:461-464 / :470-473) ----
            if (has_tile) {
                R *uu = u + o, *vv = v + o;
#pragma unroll
                for (int r0 = 0; r0 < TI; r0 += 2) {             // two tile rows at a time: their loads first
                    R pold[2][TJ], uso[2][TJ], vso[2][TJ];
#pragma unroll
                    for (int rr = 0; rr < 2; rr++)
#pragma unroll
                        for (int k = 0; k < TJ; k++) { pold[rr][k] = SC(sp, r0 + rr, k); uso[rr][k] = SC(sus, r0 + rr, k); vso[rr][k] = SC(svs, r0 + rr, k); }
#pragma unroll
                    for (int rr = 0; rr < 2; rr++)
#pragma unroll
                        for (int k = 0; k < TJ; k++) {
                            const int r = r0 + rr, e = r * LD + k;
                            SC(sp, r, k) = pold[rr][k] + phi[r][k];
                            if (r > 0 || !top) { const R pw = (r > 0) ? phi[r - 1][k] : pf[-LDP + k]; uu[e] = uso[rr][k] - dt * (phi[r][k] - pw) * inv_dx; }
                            if (k > 0 || !lef) { const R ps = (k > 0) ? phi[r][k - 1] : pf[r * LDP - 1]; vv[e] = vso[rr][k] - dt * (phi[r][k] - ps) * inv_dy; }
                        }
                }
            }
            __syncthreads();
            PHASE(3);

            // ---- transport: rayleigh.py:469-487 / mixing.py:478-495, in PASSES row blocks -------------
            {
                const R kx = MAC_TCOEF * a.inv_dx2, ky = MAC_TCOEF * a.inv_dy2;
                constexpr uint32_t PLANE_B = (uint32_t)((LANES_MAX * RS + 8) * 2 * sizeof(R));
                R *AA = PA, *WW = reinterpret_cast<R *>(smem_raw + PLANE_B), *SS = reinterpret_cast<R *>(smem_raw + 2 * PLANE_B);
                for (int ps = 0; ps < PASSES; ps++) {
                    const int ib = 1 + ps * PASS_ROWS, ie = min(NX, ib + PASS_ROWS - 1);
                    typedef typename vec2_of<R>::type R2;
                    static_assert(PASS_ROWS % 2 == 0, "a pass is LANES_MAX whole row pairs");
                    // The coefficients are a pointwise function of old values, so for this phase the cells are dealt out
                    // row-contiguous instead of by tile: a thread takes row-pair slots (rows i, i + 1 at column j) with
                    // consecutive j across the lanes — every global load of u, v, C is coalesced (the tile-wise loads touched
                    // ~10 cache lines per warp instruction) and all 512 threads work in both passes.
                    {
                        const int nslots = ((ie - ib + 2) >> 1) * NY;
                        R2 *Ap = reinterpret_cast<R2 *>(AA), *Wp = reinterpret_cast<R2 *>(WW), *Sp = reinterpret_cast<R2 *>(SS);
                        constexpr int TRIPS = ((PASS_ROWS / 2) * NY + T - 1) / T;
#pragma unroll 3
                        for (int n = 0; n < TRIPS; n++) {
                            const int q = tid + n * T;
                            if (q < nslots) {
                                const int rp = q / NY, j = 1 + q - rp * NY, i = ib + 2 * rp;
                                const R *uu = u + i * LD + j, *vv = v + i * LD + j, *sc = s + i * LD + j;
                                const R u0 = uu[0], u1 = uu[LD], u2 = uu[2 * LD];
                                const R v00 = vv[0], v01 = vv[1], v10 = vv[LD], v11 = vv[LD + 1];
                                const R s00 = sc[0], s10 = sc[LD], s20 = sc[2 * LD], s01 = sc[1], s11 = sc[LD + 1];
                                R2 xa, xw, xs;
#pragma unroll
                                for (int h = 0; h < 2; h++) {
                                    const R uE = h ? u2 : u1, uW = h ? u1 : u0, vN = h ? v11 : v01, vS = h ? v10 : v00;
                                    const R s0 = h ? s10 : s00, sE = h ? s20 : s10, sN = h ? s11 : s01;
                                    R diff0 = ((sE - R(2) * s0) * a.inv_dx2 + (sN - R(2) * s0) * a.inv_dy2) * MAC_TCOEF;
                                    R conv0 = (uE * (R(0.5) * (sE + s0)) - uW * (R(0.5) * s0)) * inv_dx + (vN * (R(0.5) * (sN + s0)) - vS * (R(0.5) * s0)) * inv_dy;
                                    R A = s0 + dt * (diff0 - conv0);
                                    R BW = dt * (kx + R(0.5) * uW * inv_dx);
                                    R BS = dt * (ky + R(0.5) * vS * inv_dy);
                                    if (j == 1) { A = fma(BS, sc[h * LD - 1], A); BS = R(0); }                   // south ghost column
                                    if (h == 0 && rp == 0) { A = fma(BW, sc[-LD], A); BW = R(0); }               // row west of the pass
                                    if (h == 0) { xa.x = A; xw.x = BW; xs.x = BS; } else { xa.y = A; xw.y = BW; xs.y = BS; }
                                }
                                Ap[rp * RS + j] = xa; Wp[rp * RS + j] = xw; Sp[rp * RS + j] = xs;
                            }
                        }
                    }
                    __syncthreads();
                    PHASE(4);
                    if (tid < 32) transport_wavefront3<R, NY>(0u, PLANE_B, 2 * PLANE_B, (ie - ib + 2) / 2, tid);
                    __syncthreads();
                    PHASE(5);
                    // the transported rows back to the plane, by ALL threads and row-contiguous (a warp writes 32
                    // consecutive cells of one row: 2-3 cache lines instead of the ~10 a tile-wise store touches)
                    {
                        const R *AAs = AA;
                        const int nrow = ie - ib + 1;
                        for (int q = tid; q < nrow * NY; q += T) {
                            const int ri = q / NY, j = 1 + q - ri * NY;
                            s[(ib + ri) * LD + j] = AAs[(((ri >> 1) * RS + j) << 1) + (ri & 1)];
                        }
                    }
                    __syncthreads();
                    PHASE(6);
                }
            }
        }   // sub-steps

        // ---- observations (probe history) and reward --------------------------------------------------
        {
            R *hist = a.obs_hist + (size_t)b * a.n_obs;
            R *out = a.obs + orow * a.n_obs;
            for (int e = tid; e < a.n_obs; e += T) {              // rayleigh.py:243-262, mixing.py:237-256
                int st = e / per_step, rem = e - st * per_step;
                R val;
                if (st < a.n_obs_steps - 1) val = hist[e + per_step];
                else {
                    int f = rem / (a.nx_obs_pts * a.ny_obs_pts), q = rem - f * (a.nx_obs_pts * a.ny_obs_pts);
                    int pi = q / a.ny_obs_pts, pj = q - pi * a.ny_obs_pts;
                    int x = a.nx_obs / 2 + pi * a.nx_obs, y = a.ny_obs / 2 + pj * a.ny_obs;
                    val = (f == 0) ? s[x * LD + y] : (f == 1 ? u[x * LD + y] : v[x * LD + y]);
                }
                out[e] = val;
            }
            __syncthreads();
            for (int e = tid; e < a.n_obs; e += T) hist[e] = out[e];
            R rwd;
            if (ray) {                                            // rayleigh.py:265-275 (sequential sum)
                rwd = R(0);
                if (tid == 0) {
                    R nu = R(0);
                    for (int i = 1; i <= NX; i++) nu -= (s[i * LD + 1] - a.Th) / (R(0.5) * a.dy);
                    nu /= R(NX);
                    rwd = -nu;
                }
            } else {                                              // mixing.py:259-264 (mean over the whole array)
                R part = R(0);
                for (int e = tid; e < N; e += T) part += rabs(s[e] - a.ref_c);
                rwd = -(block_sum(part, s_red) / R(N));
            }
            bool nonfinite = false;
            for (int e = tid; e < N; e += T) nonfinite |= !finite_(s[e]) | !finite_(u[e]) | !finite_(v[e]);
            if (__syncthreads_or(nonfinite ? 1 : 0)) status |= BEACON_STATUS_NONFINITE;
            if (tid == 0) {
                a.rwd[orow] = rwd;
                bool horizon = stp == a.n_act - 1;
                a.done[orow] = horizon; a.trunc[orow] = horizon;
                if (a.iters) a.iters[orow] = it_total;
            }
            stp += 1;
        }
    }   // actions

    // pressure back to its plane.  Ghost cells of p accumulate the same increments as their wall-
    // adjacent cells (phi ghosts are copies; mixing's j = NY+1 ghost of phi is 0) and never feed back:
    // ghost += adjacent(final) - adjacent(launch start, still in the plane).
    if (has_tile) {
        R *pp = p + o;
        if (top) {
#pragma unroll
            for (int k = 0; k < TJ; k++) pp[-LD + k] += SC(sp, 0, k) - pp[k];
        }
        if (bot) {
#pragma unroll
            for (int k = 0; k < TJ; k++) pp[TI * LD + k] += SC(sp, TI - 1, k) - pp[(TI - 1) * LD + k];
        }
        if (lef) {
#pragma unroll
            for (int r = 0; r < TI; r++) pp[r * LD - 1] += SC(sp, r, 0) - pp[r * LD];
        }
        if (rig && ray) {
#pragma unroll
            for (int r = 0; r < TI; r++) pp[r * LD + TJ] += SC(sp, r, TJ - 1) - pp[r * LD + TJ - 1];
        }
        TILE_LOOP { pp[r * LD + k] = SC(sp, r, k); }
    }
    if (tid == 0) { a.stp[b] = stp; if (a.status) a.status[b] = status; }
    if (DBG && dbg) { for (int n = 0; n < (DBG ? 8 : 1); n++) a.dbg[n] += (unsigned long long)tph[n]; }
#undef PHASE
#undef SC
#undef TILE_LOOP
}
template <typename R, int NX, int NY, int TI, int TJ, int T, int MINB, bool DBG>
__global__ void __launch_bounds__(T, MINB) mac_big_kernel(const MacArgs<R> a) { mac_big_body<R, NX, NY, TI, TJ, T, MINB, DBG, false>(a, threadIdx.x); }
// per-env physical constants (MacArgs::phys); a name that tools/sass_census.py's patterns for mac_big_kernel do not match
template <typename R, int NX, int NY, int TI, int TJ, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) mac_big_phys_kernel(const MacArgs<R> a) { mac_big_body<R, NX, NY, TI, TJ, T, MINB, false, true>(a, threadIdx.x); }

// ---------------------------------------------------------------------------------------
// Capacity of mac_kernel with G > 1 CTAs per env: "" when (nx, ny) fits, else the reason.
// Slabs of at least MAC_CLUSTER_MIN_ROWS rows; 4x5 tiles of the thickest slab within 512 threads; two phi
// slab planes of (rows + 2) x (ny + 2) in the shared-memory budget; ny + 2 within the hand-off buffers.
// The transport coefficients take 3 planes of a pass of at most 32 * MAC_RPL rows (cluster_passes).
template <typename R> static std::string cluster_misfit(int nx, int ny, int G)
{
    const int ld = ny + 2, Smax = (nx + G - 1) / G;
    if (G > MAC_CLUSTER_MAX) return "at most " + std::to_string(MAC_CLUSTER_MAX) + " CTAs per env (portable cluster size)";
    if (nx / G < MAC_CLUSTER_MIN_ROWS)
        return "slabs of " + std::to_string(nx / G) + " rows, fewer than " + std::to_string(MAC_CLUSTER_MIN_ROWS);
    if (ld > MAC_CLUSTER_MAX_LD) return "ny + 2 = " + std::to_string(ld) + " columns, more than " + std::to_string(MAC_CLUSTER_MAX_LD);
    if (((Smax + 3) / 4) * ((ny + 4) / 5) > 512) return "slab of " + std::to_string(Smax) + " rows needs more than 512 tiles of 4x5 cells";
    if (2 * (size_t)(Smax + 2) * ld * sizeof(R) > MAC_CLUSTER_SMEM || 3 * (size_t)ld * sizeof(R) > MAC_CLUSTER_SMEM)
        return "two phi slab planes of " + std::to_string(Smax + 2) + " rows exceed " + std::to_string(MAC_CLUSTER_SMEM / 1024) + " KB";
    return "";
}
// transport passes of a slab: at most 32 * MAC_RPL rows each (one warp), 3 coefficient planes in the budget
template <typename R> static int cluster_passes(int Smax, int ld)
{
    int ps = 1;
    while ((Smax + ps - 1) / ps > 32 * MAC_RPL || 3 * (size_t)((Smax + ps - 1) / ps) * ld * sizeof(R) > MAC_CLUSTER_SMEM) ps++;
    return ps;
}

// Per-env physical constants: row b of `tab` from the raw per-env values of `raw` ([2][B] float64: rayleigh ra;
// mixing re, pe), with the host's expressions of MacEnv's constructor, in double, then cast to R: a row holds
// bitwise the constants of a uniform handle created with that env's values (IEEE division and square root on
// both sides, no fast-math).  Runs when the values change, never on the step path.
template <typename R>
__global__ void mac_phys_derive(const double *raw, R *tab, int B, int ray, double pr, double L, double u_max)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (ray) {
        const double ra = raw[b];
        tab[3 * b] = (R)std::sqrt(pr / ra); tab[3 * b + 1] = (R)(1.0 / std::sqrt(pr * ra)); tab[3 * b + 2] = (R)u_max;
    } else {
        const double re = raw[b], pe = raw[B + b];
        tab[3 * b] = (R)(1.0 / re); tab[3 * b + 1] = (R)(1.0 / pe); tab[3 * b + 2] = (R)(re * 0.01 / L);   // u_max = re nu / L, params.py
    }
}

template <typename R> class MacEnv : public Env {
    beacon_mac_params p;
    int kind, G = 1;
    DeviceBuffer u, v, pp, s, us, vs, cc, a_cur, a_int, obs_hist, stp, u0, v0, p0, s0, dbgbuf;
    DeviceBuffer phys_raw, phys_tab;   // per-env physical parameters, allocated by the first set_physics
    MacArgs<R> base{};
    void (*kernel)(const MacArgs<R>) = nullptr;
    void (*phys_kernel)(const MacArgs<R>) = nullptr;   // the per-env instance of `kernel`
    double mix_L = 0;                                   // mixing: L = nx dx, for u_max = re nu / L
    int T = 0;
    size_t smem = 0;
    bool reg_variant = false, dbg_variant = false, big_variant = false;

public:
    MacEnv(const beacon_common &c, const beacon_mac_params &pp_, int kind_, const double *hu, const double *hv,
           const double *hp, const double *hs)
        : p(pp_), kind(kind_)
    {
        common = c;
        const int B = c.batch, nx = p.nx, ny = p.ny, ld = ny + 2, n = (nx + 2) * ld;
        const bool ray = kind == BEACON_RAYLEIGH;
        BEACON_REQUIRE(nx >= 4 && ny >= 4 && p.ndt_act > 0 && p.itmax > 0, "mac2d: bad sizes");
        BEACON_REQUIRE(hs != nullptr, "mac2d: scalar init field must not be NULL");
        if (ray) {
            BEACON_REQUIRE(hu && hv && hp, "rayleigh: init fields must not be NULL");
            BEACON_REQUIRE(p.n_sgts >= 1 && p.n_sgts <= 128 && p.nx_sgts >= 1 && p.n_sgts * p.nx_sgts <= nx, "rayleigh: bad segment layout");
        }
        const int npts = p.nx_obs_pts * p.ny_obs_pts;
        BEACON_REQUIRE(npts > 0 && p.n_obs_steps > 0, "mac2d: bad probe layout");
        BEACON_REQUIRE(p.nx_obs / 2 + (p.nx_obs_pts - 1) * p.nx_obs <= nx + 1 && p.ny_obs / 2 + (p.ny_obs_pts - 1) * p.ny_obs <= ny + 1,
                       "mac2d: probes outside the domain");
        info.kind = kind; info.batch = B; info.dtype = real_traits<R>::dtype; info.device = c.device;
        info.n_obs = 3 * p.n_obs_steps * npts; info.act_dim = ray ? p.n_sgts : 1; info.act_is_int = ray ? 0 : 1;
        info.rwd_dim = 1; info.n_act = p.n_act; info.noise_dim = 0;

        MacArgs<R> &a = base;
        // kernel: mac_reg_kernel and mac_big_kernel for their grids, else mac_kernel with the whole array in
        // one CTA; ctas_per_env = G > 1 selects mac_kernel over a cluster of G CTAs on any grid
        const size_t plane = (size_t)n * sizeof(R);
        int TI, TJ;
        BEACON_REQUIRE(p.ctas_per_env >= 0, "mac2d: ctas_per_env must be >= 0 (0 and 1: one CTA per env)");
        G = std::max(p.ctas_per_env, 1);
        if (G > 1) {
            const std::string why = cluster_misfit<R>(nx, ny, G);
            if (why.size()) throw Error(BEACON_ERR_UNSUPPORTED, "mac2d: ctas_per_env=" + std::to_string(G) + ": " + why);
        }
        reg_variant = false;
        if (G > 1) {
            // selected below, after the transport passes
        } else if (ray && nx == 50 && ny == 50 && p.n_sgts <= 32 && !getenv("BEACON_MAC_V1")) {
            // five planes fit twice per SM: register-resident phi tiles, 2 CTAs/SM
            if (getenv("BEACON_MAC_DEBUG")) kernel = mac_reg_kernel<R, 50, 50, 2, 5, 256, true>;
            else kernel = mac_reg_kernel<R, 50, 50, 2, 5, 256, false>;
            phys_kernel = mac_reg_phys_kernel<R, 50, 50, 2, 5, 256, false>;
            T = 256; TI = 2; TJ = 5; dbg_variant = true;
            smem = sizeof(R) * (2 * (size_t)((51 * mac_ldp(52, 2) + 3) / 4 * 4) + 2 * 52 * 53 + 52 * mac_ldp(52, 2)); reg_variant = true;
        } else if (nx == 100 && ny == 100 && !getenv("BEACON_MAC_V1")) {
            // register-resident Poisson, fields in L2: one CTA of 500 tile threads per SM
            if (getenv("BEACON_MAC_DEBUG")) kernel = mac_big_kernel<R, 100, 100, 4, 5, 512, 1, true>;
            else kernel = mac_big_kernel<R, 100, 100, 4, 5, 512, 1, false>;
            phys_kernel = mac_big_phys_kernel<R, 100, 100, 4, 5, 512, 1>;
            T = 512; TI = 4; TJ = 5; dbg_variant = true; big_variant = true;
            smem = sizeof(R) * 2 * (size_t)((102 * 105 + 3) / 4 * 4);
        } else if (2 * plane + 1024 <= 220 * 1024 && ((nx + 3) / 4) * ((ny + 4) / 5) <= 512) {
            kernel = mac_kernel<R, 4, 5, 512, false>; T = 512; TI = 4; TJ = 5; smem = 2 * plane;
            phys_kernel = mac_phys_kernel<R, 4, 5, 512, false>;
        } else {
            std::string msg = "mac2d: grid too large for the one-CTA-per-env kernel (max ~100x100 cells)";
            for (int g = 2; g <= MAC_CLUSTER_MAX; g++)
                if (!cluster_misfit<R>(nx, ny, g).size()) { msg += " (ctas_per_env=" + std::to_string(g) + " would fit)"; break; }
            throw Error(BEACON_ERR_UNSUPPORTED, msg);
        }
        // transport scratch = 3 planes of ceil(nx/passes) rows inside the two phi planes
        a.tr_pass = 1;
        while (3 * (size_t)((nx + a.tr_pass - 1) / a.tr_pass) * ld > 2 * (size_t)n || (nx + a.tr_pass - 1) / a.tr_pass > 32 * MAC_RPL)
            a.tr_pass++;
        a.G = G; a.slab_rows = nx + 2;                                  // mac_kernel at G = 1: the slab is the whole array
        if (G > 1) {
            // one cluster of G CTAs per env: slab rows, phi slab planes + transport passes (cluster_misfit), hand-off buffers
            const int Smax = (nx + G - 1) / G;
            a.slab_rows = Smax + 2;
            a.tr_pass = cluster_passes<R>(Smax, ld);
            const int rows = (Smax + a.tr_pass - 1) / a.tr_pass;
            kernel = mac_kernel<R, 4, 5, 512, true>; T = 512; TI = 4; TJ = 5;
            phys_kernel = mac_phys_kernel<R, 4, 5, 512, true>;
            smem = sizeof(R) * (size_t)ld * std::max(2 * a.slab_rows, 3 * rows) + MAC_HANDOFF_BYTES(R);
        }
        raise_dynamic_smem_limit(kernel, smem);
        if (G > 1) {
            cudaLaunchConfig_t cfg = {};
            cudaLaunchAttribute at[1];
            cfg.gridDim = dim3(B * G); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem;
            at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = G; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            int clusters = 0;
            BEACON_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg));
            if (clusters < 1)
                throw Error(BEACON_ERR_UNSUPPORTED, "mac2d: no cluster of " + std::to_string(G) + " CTAs of " + std::to_string(smem) +
                                                        " B shared memory fits this device");
        }

        const size_t nb = (size_t)B * plane;
        u.alloc(nb); v.alloc(nb); pp.alloc(nb); s.alloc(nb); us.alloc(nb); vs.alloc(nb);
        a_cur.alloc((size_t)B * (ray ? p.n_sgts : 1) * sizeof(R)); a_int.alloc((size_t)B * 4);
        obs_hist.alloc((size_t)B * info.n_obs * sizeof(R)); stp.alloc((size_t)B * 4);
        if (ray) { upload_as<R>(u0, hu, n); upload_as<R>(v0, hv, n); upload_as<R>(p0, hp, n); }
        upload_as<R>(s0, hs, n);
        add_field("u", u.ptr, n); add_field("v", v.ptr, n); add_field("p", pp.ptr, n); add_field(ray ? "T" : "C", s.ptr, n);
        if (!reg_variant && !big_variant) { add_field("us", us.ptr, n); add_field("vs", vs.ptr, n); }
        if (big_variant) cc.alloc((size_t)B * 3 * TI * TJ * T * sizeof(R));  // [B][p, us, vs][cell][thread] tile scratch
        if (ray) add_field("a", a_cur.ptr, p.n_sgts); else add_field("a", a_int.ptr, 1, true);
        add_field("obs", obs_hist.ptr, info.n_obs); add_field("stp", stp.ptr, 1, true);

        a.nx = nx; a.ny = ny; a.ld = ld; a.n = n; a.ndt_act = p.ndt_act; a.n_act = p.n_act; a.kind = kind;
        a.n_sgts = p.n_sgts; a.nx_sgts = p.nx_sgts > 0 ? p.nx_sgts : 1; a.itmax = p.itmax;
        a.tiles_i = (nx + TI - 1) / TI; a.tiles_j = (ny + TJ - 1) / TJ;
        a.nx_obs_pts = p.nx_obs_pts; a.ny_obs_pts = p.ny_obs_pts; a.n_obs_steps = p.n_obs_steps; a.nx_obs = p.nx_obs; a.ny_obs = p.ny_obs;
        a.n_obs = info.n_obs;
        const double dx = p.dx, dy = p.dy, dt = p.dt;
        a.dx = (R)dx; a.dy = (R)dy; a.dt = (R)dt; a.inv_dx = (R)(1.0 / dx); a.inv_dy = (R)(1.0 / dy);
        a.inv_dx2 = (R)(1.0 / (dx * dx)); a.inv_dy2 = (R)(1.0 / (dy * dy)); a.dx2 = (R)(dx * dx); a.dy2 = (R)(dy * dy);
        a.inv_den = (R)(0.5 / (dx * dx + dy * dy));
        a.pk1 = (R)(dy * dy * (0.5 / (dx * dx + dy * dy))); a.pk2 = (R)(dx * dx * (0.5 / (dx * dx + dy * dy)));
        a.cscale = (R)(dx * dx * dy * dy / dt);                   // b*dx*dx*dy*dy with b = div/dt
        a.dcoef = (R)(ray ? std::sqrt(p.pr / p.ra) : 1.0 / p.re); // momentum diffusion factor
        a.tcoef = (R)(ray ? 1.0 / std::sqrt(p.pr * p.ra) : 1.0 / p.pe);
        a.Tc = (R)p.Tc; a.Th = (R)p.Th; a.Cmax = (R)p.C; a.u_max = (R)p.u_max; a.ref_c = (R)p.ref_c; a.tol = (R)p.tol;
        a.B = B;
        a.u = u.as<R>(); a.v = v.as<R>(); a.p = pp.as<R>(); a.s = s.as<R>(); a.us = us.as<R>(); a.vs = vs.as<R>(); a.cc = cc.as<R>();
        a.a_cur = a_cur.as<R>(); a.a_int = a_int.as<int32_t>(); a.obs_hist = obs_hist.as<R>(); a.stp = stp.as<int32_t>();
        a.u0 = u0.as<R>(); a.v0 = v0.as<R>(); a.p0 = p0.as<R>(); a.s0 = s0.as<R>();
        mix_L = (double)nx * dx;
    }

    // ---- per-env physical parameters ------------------------------------------------------------
    // slot of `name` in phys_raw: rayleigh "ra"; mixing "re", "pe"
    int phys_slot(const char *name) const
    {
        const bool ray = kind == BEACON_RAYLEIGH;
        const std::string nm = name ? name : "";
        if (ray && nm == "ra") return 0;
        if (!ray && nm == "re") return 0;
        if (!ray && nm == "pe") return 1;
        throw Error(BEACON_ERR_INVALID, std::string(ray ? "rayleigh" : "mixing") + " has no per-env physical parameter '" + nm +
                                            "' (it has " + (ray ? "\"ra\")" : "\"re\", \"pe\")"));
    }
    double phys_uniform(int slot) const { return kind == BEACON_RAYLEIGH ? p.ra : (slot == 0 ? p.re : p.pe); }
    void set_physics(const char *name, const double *values, cudaStream_t st) override
    {
        const int slot = phys_slot(name), B = info.batch;
        BEACON_REQUIRE(values != nullptr, "set_physics: values must not be NULL");
        std::vector<double> h(values, values + B);   // pageable: the copy below has read it when it returns
        for (int b = 0; b < B; b++)
            if (!std::isfinite(h[b]) || !(h[b] > 0))
                throw Error(BEACON_ERR_INVALID, std::string("set_physics: ") + name + "[" + std::to_string(b) + "] = " + std::to_string(h[b]) +
                                                    ": values must be finite and > 0");
        if (kind == BEACON_MIXING && slot == 0 && p.re * 0.01 / mix_L != p.u_max)
            throw Error(BEACON_ERR_UNSUPPORTED, "set_physics: per-env re sets u_max = re * 0.01 / L with L = nx dx; this handle's u_max "
                                                "does not follow that rule");
        if (!base.phys) {
            // first call: the per-env instance takes over every launch of the handle
            raise_dynamic_smem_limit(phys_kernel, smem);
            if (G > 1) {
                cudaLaunchConfig_t cfg = {};
                cudaLaunchAttribute at[1];
                cfg.gridDim = dim3(B * G); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem;
                at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = G; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
                cfg.attrs = at; cfg.numAttrs = 1;
                int clusters = 0;
                BEACON_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&clusters, phys_kernel, &cfg));
                if (clusters < 1) throw Error(BEACON_ERR_UNSUPPORTED, "mac2d: the per-env instance does not fit a cluster of " + std::to_string(G) + " CTAs");
            }
            std::vector<double> init(2 * (size_t)B);
            for (int b = 0; b < B; b++) { init[b] = phys_uniform(0); init[B + b] = phys_uniform(1); }
            phys_raw.alloc(init.size() * sizeof(double));
            phys_tab.alloc(3 * (size_t)B * sizeof(R));
            BEACON_CUDA_CHECK(cudaMemcpy(phys_raw.ptr, init.data(), init.size() * sizeof(double), cudaMemcpyHostToDevice));
            base.phys = phys_tab.as<R>();
        }
        BEACON_CUDA_CHECK(cudaMemcpyAsync(phys_raw.as<double>() + (size_t)slot * B, h.data(), (size_t)B * sizeof(double), cudaMemcpyHostToDevice, st));
        mac_phys_derive<R><<<(B + 127) / 128, 128, 0, st>>>(phys_raw.as<double>(), phys_tab.as<R>(), B, kind == BEACON_RAYLEIGH, p.pr, mix_L, p.u_max);
        BEACON_CUDA_CHECK(cudaGetLastError());
        launches++;
    }
    void get_physics(const char *name, double *values, cudaStream_t st) override
    {
        const int slot = phys_slot(name), B = info.batch;
        BEACON_REQUIRE(values != nullptr, "get_physics: values must not be NULL");
        if (!base.phys) { std::fill(values, values + B, phys_uniform(slot)); return; }
        BEACON_CUDA_CHECK(cudaMemcpyAsync(values, phys_raw.as<double>() + (size_t)slot * B, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
        BEACON_CUDA_CHECK(cudaStreamSynchronize(st));
    }

    void run(const MacArgs<R> &a_, cudaStream_t st)
    {
        MacArgs<R> a = a_;
        auto kernel = a.phys ? phys_kernel : this->kernel;
        static const bool debug = getenv("BEACON_MAC_DEBUG") != nullptr;
        if (debug && dbg_variant && !a.phys && a.mode == 0) {            // tuning aid: cycles per phase of env 0
            if (!dbgbuf.ptr) dbgbuf.alloc(8 * sizeof(unsigned long long));
            BEACON_CUDA_CHECK(cudaMemsetAsync(dbgbuf.ptr, 0, 64, st));
            a.dbg = dbgbuf.as<unsigned long long>();
        }
        if (G > 1) {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(a.B * G); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem; cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = G; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            BEACON_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, a));
        } else
            kernel<<<a.B, T, smem, st>>>(a);
        BEACON_CUDA_CHECK(cudaGetLastError());
        launches++;
        if (debug && dbg_variant && !a.phys && a.mode == 0) {
            unsigned long long h[8];
            BEACON_CUDA_CHECK(cudaMemcpyAsync(h, dbgbuf.ptr, 64, cudaMemcpyDeviceToHost, st));
            BEACON_CUDA_CHECK(cudaStreamSynchronize(st));
            fprintf(stderr, "[mac phases, env 0, cycles] bc %llu predictor %llu poisson %llu corrector %llu trcoef %llu wavefront %llu copyout %llu\n",
                    h[0], h[1], h[2], h[3], h[4], h[5], h[6]);
        }
    }
    void reset(const ResetArgs &r) override
    {
        BEACON_REQUIRE(r.obs != nullptr, "reset: obs must not be NULL");
        MacArgs<R> a = base; a.mode = 1; a.mask = r.mask; a.obs = (R *)r.obs;
        run(a, r.stream);
    }
    void step(const StepArgs &s_) override
    {
        MacArgs<R> a = base; a.mode = 0; a.n_fused = s_.n_fused; a.actions = s_.actions;
        a.obs = (R *)s_.obs; a.rwd = (R *)s_.rwd; a.done = s_.done; a.trunc = s_.trunc; a.status = s_.status; a.iters = s_.iters;
        run(a, s_.stream);
    }
};

Env *make_mac(const beacon_common &c, const beacon_mac_params &p, int kind, const double *u0, const double *v0,
              const double *p0, const double *s0)
{
    if (c.dtype == BEACON_F64) return new MacEnv<double>(c, p, kind, u0, v0, p0, s0);
    if (c.dtype == BEACON_F32) return new MacEnv<float>(c, p, kind, u0, v0, p0, s0);
    throw Error(BEACON_ERR_INVALID, "unknown dtype");
}

}  // namespace beacon
