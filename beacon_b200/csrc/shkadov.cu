// shkadov-v0 / shkadov_separable-v0 — falling-film (Shkadov 2-equation model) with jet forcing.
//
// Reference: /root/reference/beacon/shkadov/shkadov.py — solve() :188-236, d1tvd :494-504,
// d3o2u :485-491, rhsq :507-512, adams :515-518, get_obs :239-250, get_rwd :253-264,
// step :161-185, reset :113-151.
//
// B200 design (one CTA per environment, register-resident state):
//   * each thread owns C consecutive lattice points; h, q and the two Adams-Bashforth
//     right-hand sides of those points live in REGISTERS for the whole launch (all
//     ndt_act sub-steps of all fused actions) — no HBM and no shared-memory traffic for them;
//   * per sub-step only the chunk edges (5 h, 3 q, 3 q^2/h values per thread) go through a
//     double-buffered shared-memory exchange: ONE __syncthreads per sub-step;
//   * every limiter ratio / flux face is evaluated once (the face left of a chunk is the only
//     redundant one);
//   * ALL warps run one compact branch-free loop body: the outlet is aligned to the end of its chunk
//     (host-chosen shift `off`), inlet / outlet special cases are per-thread selects at compile-time
//     positions, the sub-step loop is unrolled by two (see the role table in the kernel);
//   * inlet noise of a whole action is generated up front by Philox (or read from the caller's
//     tensor in parity mode); a chunk meets at most one jet and interpolates its amplitude itself;
//   * observation gather, per-jet reward reductions (warp shuffles) and the blow-up guard run
//     once per action on a shared-memory copy of the final h, q.
// HBM traffic per launch is the F-model floor (state in + out, obs/reward out); the kernel is
// bound by the fp64 pipe (4 true divisions per point per sub-step), see DESIGN.md.
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace beacon {

template <typename R> struct ShkArgs {
    // geometry / numerics
    int nx, ndt_act, n_act, n_interp, n_jets, jet_pos, jet_hw, jet_space, l_obs, n_obs, obs_stride, l_rwd;
    int per_jet_rwd, off, tail_aligned, jets_overlap, jets_simple, jz0, jz_len;
    R inv_dx, inv_2dx3, inv_dx3, hdt, p5d, eps, jet_amp, dx, blow_lo, blow_hi, blowup_rwd;
    R k3[5], kc, kc3, c12;       // d3o2u coefficients / (2 dx^3), closure 1/dx^3 and 3/dx^3, 1.2/dx (fast body)
    double sigma;
    uint64_t seed;
    int64_t env_base;
    // persistent state [B, .]
    R *h, *q, *rhsh, *rhsq, *u_cur, *u_prev;
    int32_t *stp;
    unsigned long long *draws;   // noise draws consumed so far, per env
    const R *h_init, *q_init;
    // per-call
    int mode;                    // 0 = step, 1 = reset
    int n_fused, max_warm, B;
    const R *actions;            // [K,B,n_jets]
    const R *noise;              // nullable [K,B,ndt_act]
    const uint8_t *mask;         // reset only, nullable
    const int32_t *n_warm;       // reset only, nullable
    const int32_t *order;        // reset only, nullable: CTA -> env permutation (longest warm-up first)
    R *obs, *rwd;
    uint8_t *done, *trunc;
    int32_t *status;
};

// shared-memory exchange slots per thread
enum { XH0 = 0, XH1, XH2, XHL2, XHL1, XQ0, XQL2, XQL1, XZ0, XZL2, XZL1, XN };

template <typename R, int C, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) shkadov_kernel(const ShkArgs<R> a)
{
    static_assert(C >= 3, "halo exchange needs at least 3 points per thread");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, b = a.order ? a.order[blockIdx.x] : (int)blockIdx.x;
    const int nx = a.nx, nj = a.n_jets;

    if (a.mode == 1 && a.mask && !a.mask[b]) return;

    // ---- shared memory carve-up ------------------------------------------------------
    R *ex = reinterpret_cast<R *>(smem_raw);            // [2][XN][T]
    R *s_h = ex + 2 * XN * T;                           // [nx] action-end copy of h
    R *s_q = s_h + nx;                                  // [nx]
    R *s_noise = s_q + nx;                              // [ndt_act]
    R *s_jet = s_noise + a.ndt_act;                     // [2][nj] jet_amp * interpolated action
    R *s_ucur = s_jet + 2 * nj;                         // [nj]
    R *s_uprev = s_ucur + nj;                           // [nj]
    R *s_term = s_uprev + nj;                           // [nj] per-jet reward terms
    R *s_alpha = s_term + nj;                           // [ndt_act] min(i / n_interp, 1)
    R *s_jw = s_alpha + a.ndt_act;                              // [C + jz_len + C] parabola weight per point of the jet zone, zero padded
    short *s_jj = reinterpret_cast<short *>(s_jw + a.jz_len + 2 * C);   // [jz_len] jet index or -1

    // ---- static per-thread geometry ---------------------------------------------------
    const int a0 = tid * C - a.off;                     // first point of my chunk
    const bool has_jet = (a0 + C - 1 >= a.jz0) && (a0 < a.jz0 + a.jz_len) && nj > 0;
    const int tl = tid > 0 ? tid - 1 : 0, tr = tid < T - 1 ? tid + 1 : T - 1;
    const bool interior_thread = a0 >= 2 && a0 + C - 1 <= nx - 4;   // full stencil, all points updated
    // Warp roles (warp-uniform: no warp executes two variants of the update and stalls the others at
    // the barrier; and as few distinct loop bodies as possible, each compact: the bodies of all
    // resident warps must stay in the instruction cache — three 40 KB bodies measured 0.7x):
    //   FAST     every chunk of the warp is handled by ONE branch-free body.  The host aligns the
    //            chunks so that the outlet point nx-1 is the LAST point of its chunk: the outlet copy,
    //            the two one-sided closures of d3o2u and the not-updated point sit at compile-time
    //            positions and are selected by `is_last`.  Thread 0 holds `off` phantom points, the
    //            inlet point 0 and the faces with phi = 0: selects on per-thread thresholds (zero for
    //            everybody else), confined to m < 3 when off <= 1 (F_SMALL), or for all m in warp 0
    //            (F_LARGE) while the other warps run the body without them (F_NONE).  Lanes beyond
    //            the domain run the same arithmetic on phantom points (never stored, never read by
    //            a result that is kept);
    //   IDLE     warps entirely beyond the domain only keep the barrier count;
    //   GENERAL  anything else (tiny lattices, overlapping / dense jets): per-point index tests.
    enum { F_NONE = 0, F_SMALL, F_LARGE, ROLE_GENERAL, ROLE_IDLE };
    const int w_lo = (tid & ~31) * C - a.off, w_hi = w_lo + 32 * C - 1;
    const int last_tid = (nx - 1 + a.off) / C;
    int role = ROLE_GENERAL;
    if (w_lo >= nx) role = ROLE_IDLE;
    else if (a.tail_aligned && a.jets_simple && nx - 4 >= C) {
        // (warp 0 must not hold the outlet specials too: first thread's chunk ends before nx-3)
        if (a.off <= 1) role = F_SMALL;
        else role = w_lo <= 0 ? F_LARGE : F_NONE;
        if (w_lo <= 0 && last_tid == 0) role = ROLE_GENERAL;
    }
    const bool is_last = tid == last_tid;
    const int zf = tid == 0 ? a.off + 2 : 0;            // faces m < zf have phi = 0
    const int np = tid == 0 ? a.off + 1 : 0;            // points m < np are not updated
    // jets: when consecutive jet zones are at least C-1 points apart a chunk meets at most one jet
    int myjet = -1;
    if (a.jets_simple && nj > 0) {
        int j = (a0 + C - 1 - a.jz0) / a.jet_space;      // last jet starting at or before my last point
        if (a0 + C - 1 >= a.jz0) {
            if (j >= nj) j = nj - 1;
            if (a0 <= a.jz0 + j * a.jet_space + 2 * a.jet_hw) myjet = j;
        }
    }
    const int kb = a0 - a.jz0 + C;                       // my first point in the zero-padded weight table
    const bool edge_thread = (a0 <= 0) || (a0 <= nx - 1 && a0 + C - 1 >= nx - 1);   // owns point 0 or nx-1

    // jet zone tables (shkadov.py:224-232): weight v = (k-s)(e-k)/(0.25 (e-s)^2)
    for (int k = tid; k < a.jz_len; k += T) {
        int i = a.jz0 + k, jj = -1;
        R w = R(0);
        if (a.jet_space > 0) {
            int j = (i - a.jz0) / a.jet_space;
            if (j >= nj) j = nj - 1;
            int s = a.jz0 + j * a.jet_space, e = s + 2 * a.jet_hw;
            if (i >= s && i <= e) { jj = j; w = R((long long)(i - s) * (long long)(e - i)) / (R(0.25) * R((long long)(e - s) * (long long)(e - s))); }
        }
        s_jw[C + k] = w;
        s_jj[k] = (short)jj;
    }
    for (int k = tid; k < C; k += T) { s_jw[k] = R(0); s_jw[C + a.jz_len + k] = R(0); }
    for (int i = tid; i < a.ndt_act; i += T) s_alpha[i] = (R)fmin((double)i / (double)a.n_interp, 1.0);
    for (int k = tid; k < 2 * XN * T; k += T) ex[k] = R(1);   // slots of threads beyond the domain are read (and discarded): keep them finite

    // ---- load state into registers ----------------------------------------------------
    R hv[C], qv[C], rh[C], rq[C];
    const size_t row = (size_t)b * nx;
    const bool resetting = a.mode == 1;
#pragma unroll
    for (int m = 0; m < C; m++) {
        int i = a0 + m;
        bool real = i >= 0 && i < nx;
        if (resetting) {                                 // reset_fields + load, shkadov.py:113-151
            hv[m] = real ? a.h_init[i] : R(1);
            qv[m] = real ? a.q_init[i] : R(1);
            rh[m] = R(0);
            rq[m] = R(0);
        } else {
            hv[m] = real ? a.h[row + i] : R(1);
            qv[m] = real ? a.q[row + i] : R(1);
            rh[m] = real ? a.rhsh[row + i] : R(0);
            rq[m] = real ? a.rhsq[row + i] : R(0);
        }
    }
    for (int j = tid; j < nj; j += T) {
        s_ucur[j] = resetting ? R(0) : a.u_cur[(size_t)b * nj + j];
        s_uprev[j] = resetting ? R(0) : a.u_prev[(size_t)b * nj + j];
    }
    int stp = resetting ? 0 : a.stp[b];
    unsigned long long draws = a.draws[b];
    int status = 0;
    const int n_actions = resetting ? (a.n_warm ? min(a.n_warm[b], a.max_warm) : 0) : a.n_fused;
    const uint64_t env_gid = (uint64_t)(a.env_base + b);

    for (int act = 0; act < n_actions; act++) {
        __syncthreads();   // previous action's shared-memory readers are done
        // ---- new action: up <- u, u <- a (shkadov.py:193-194); noise for the whole action
        for (int j = tid; j < nj; j += T) {
            s_uprev[j] = s_ucur[j];
            s_ucur[j] = resetting ? R(0) : a.actions[((size_t)act * a.B + b) * nj + j];
        }
        for (int i = tid; i < a.ndt_act; i += T) {
            if (a.noise) s_noise[i] = a.noise[((size_t)act * a.B + b) * a.ndt_act + i];
            else s_noise[i] = (R)philox_uniform_pm(a.seed, env_gid, draws + (unsigned long long)i, a.sigma);
        }
        draws += (unsigned long long)a.ndt_act;
        __syncthreads();

        // One sub-step of a chunk, shkadov.py:199-236.  KIND is the warp role.
        auto substep = [&](const int it, auto kind_tag) {
            constexpr int KIND = decltype(kind_tag)::value;
            constexpr bool FAST = KIND != ROLE_GENERAL;
            const int buf = it & 1;
            R *X = ex + buf * XN * T;
            // ---- boundary conditions, shkadov.py:204-207 -------------------------------
            if (KIND == F_SMALL || KIND == F_LARGE) {
                const R hin = R(1) + s_noise[it];
#pragma unroll
                for (int m = 0; m < (KIND == F_SMALL ? 2 : C); m++)
                    if (m < np) { hv[m] = hin; qv[m] = R(1); }           // point 0 (and the phantom points left of it)
            }
            if (FAST) {
                if (is_last) { hv[C - 1] = hv[C - 2]; qv[C - 1] = qv[C - 2]; }
            } else if (edge_thread) {
#pragma unroll
                for (int m = 0; m < C; m++) {
                    int i = a0 + m;
                    if (i == 0) { hv[m] = R(1) + s_noise[it]; qv[m] = R(1); }
                    if (m > 0 && i == nx - 1) { hv[m] = hv[m - 1]; qv[m] = qv[m - 1]; }   // off guarantees m > 0
                }
            }
            // ---- q2h = q*q/(h+eps), shkadov.py:213 --------------------------------------
            R zv[C];
#pragma unroll
            for (int m = 0; m < C; m++) zv[m] = fdiv(qv[m] * qv[m], hv[m] + a.eps);
            // ---- publish chunk edges ---------------------------------------------------
            X[XH0 * T + tid] = hv[0]; X[XH1 * T + tid] = hv[1]; X[XH2 * T + tid] = hv[2];
            X[XHL2 * T + tid] = hv[C - 2]; X[XHL1 * T + tid] = hv[C - 1];
            X[XQ0 * T + tid] = qv[0]; X[XQL2 * T + tid] = qv[C - 2]; X[XQL1 * T + tid] = qv[C - 1];
            X[XZ0 * T + tid] = zv[0]; X[XZL2 * T + tid] = zv[C - 2]; X[XZL1 * T + tid] = zv[C - 1];
            // jet amplitudes of this sub-step, shkadov.py:224-226
            if (!FAST) {
                if (!a.jets_simple && (tid < nj || nj > T)) {
                    R alpha = s_alpha[it];
                    for (int j = tid; j < nj; j += T)
                        s_jet[buf * nj + j] = a.jet_amp * ((R(1) - alpha) * s_uprev[j] + alpha * s_ucur[j]);
                }
            }
            __syncthreads();

            // The update of a chunk.  UK: F_* as above; ROLE_GENERAL = per-point index tests; -1 =
            // interior chunk of a GENERAL warp (full stencil everywhere, any jet layout).
            auto update = [&](auto upd_tag) {
                constexpr int UK = decltype(upd_tag)::value;
                constexpr bool UFAST = UK == F_NONE || UK == F_SMALL || UK == F_LARGE;
                // ---- extended stencils ---------------------------------------------------
                R uh[C + 5];   // h at a0-2 .. a0+C+2
                uh[0] = X[XHL2 * T + tl]; uh[1] = X[XHL1 * T + tl];
#pragma unroll
                for (int m = 0; m < C; m++) uh[m + 2] = hv[m];
                uh[C + 2] = X[XH0 * T + tr]; uh[C + 3] = X[XH1 * T + tr]; uh[C + 4] = X[XH2 * T + tr];
                R uq[C + 3], uz[C + 3];   // q, q2h at a0-2 .. a0+C
                uq[0] = X[XQL2 * T + tl]; uq[1] = X[XQL1 * T + tl];
                uz[0] = X[XZL2 * T + tl]; uz[1] = X[XZL1 * T + tl];
#pragma unroll
                for (int m = 0; m < C; m++) { uq[m + 2] = qv[m]; uz[m + 2] = zv[m]; }
                uq[C + 2] = X[XQ0 * T + tr]; uz[C + 2] = X[XZ0 * T + tr];

                // ---- TVD faces (d1tvd, shkadov.py:494-504): F_f = u_f + 0.5 phi_f (u_{f+1}-u_f) ----
                R Fq[C + 1], Fz[C + 1];   // faces a0-1 .. a0+C-1
                {
                    R dq[C + 2], dz[C + 2];   // differences u_{k+1}-u_k for k = a0-2 .. a0+C-1
#pragma unroll
                    for (int k = 0; k < C + 2; k++) { dq[k] = uq[k + 1] - uq[k]; dz[k] = uz[k + 1] - uz[k]; }
#pragma unroll
                    for (int m = 0; m < C + 1; m++) {
                        // half of the minmod limiter, 0.5 max(0, min(r, 1))
                        R pq = clamp0h(fdiv_half(dq[m], dq[m + 1] + R(1.0e-8)));
                        R pz = clamp0h(fdiv_half(dz[m], dz[m + 1] + R(1.0e-8)));
                        if (UK == ROLE_GENERAL) { if (a0 - 1 + m <= 0) { pq = R(0); pz = R(0); } }   // phi[0] = 0
                        if (UK == F_LARGE || (UK == F_SMALL && m < 3)) { if (m < zf) { pq = R(0); pz = R(0); } }
                        Fq[m] = uq[m + 1] + pq * dq[m + 1];
                        Fz[m] = uz[m + 1] + pz * dz[m + 1];
                    }
                }
                // ---- rhs, jets, Adams-Bashforth ----------------------------------------
                const R *sj = s_jet + buf * nj;
                R myamp = R(0);                                  // shkadov.py:224-226, my jet only
                if ((UFAST || a.jets_simple) && myjet >= 0) {
                    const R alpha = s_alpha[it];
                    myamp = a.jet_amp * ((R(1) - alpha) * s_uprev[myjet] + alpha * s_ucur[myjet]);
                }
                const R hdt = a.hdt;
#pragma unroll
                for (int m = 0; m < C; m++) {
                    const int i = a0 + m;
                    R nrh = (Fq[m + 1] - Fq[m]) * a.inv_dx;                       // rhsh = d1tvd(q)
                    const R hh = hv[m];
                    R nrq;
                    if (UFAST) {
                        R d3p1 = (-uh[m + 5] + R(6) * uh[m + 4] - R(12) * uh[m + 3] + R(10) * uh[m + 2] - R(3) * uh[m + 1]) * a.inv_2dx3 + R(1);
                        if (m == C - 3) {                         // i = nx-3 / nx-2 of the outlet chunk: one-sided closures
                            R c = fma(a.kc, uh[m + 4], R(1)); c = fma(-a.kc3, uh[m + 3], c); c = fma(a.kc3, uh[m + 2], c); c = fma(-a.kc, uh[m + 1], c);
                            if (is_last) d3p1 = c;
                        }
                        if (m == C - 2) {
                            R c = fma(-a.kc, uh[m], R(1)); c = fma(a.kc3, uh[m + 1], c); c = fma(-a.kc3, uh[m + 2], c); c = fma(a.kc, uh[m + 3], c);
                            if (is_last) d3p1 = c;
                        }
                        const R t1 = fma(hh, d3p1, -fdiv(qv[m], fma(hh, hh, a.eps)));
                        nrq = fma(a.c12, Fz[m + 1] - Fz[m], -(a.p5d * t1));                   // rhsq(), :507-512 (1.2/dx folded)
                    } else {
                        R dq2h = (Fz[m + 1] - Fz[m]) * a.inv_dx;
                        // d3o2u, shkadov.py:485-491 (uh[m+2] is h_i)
                        R d3 = (-uh[m + 5] + R(6) * uh[m + 4] - R(12) * uh[m + 3] + R(10) * uh[m + 2] - R(3) * uh[m + 1]) * a.inv_2dx3;
                        if (UK == ROLE_GENERAL) {
                            if (i == nx - 3) d3 = (uh[m + 4] - R(3) * uh[m + 3] + R(3) * uh[m + 2] - uh[m + 1]) * a.inv_dx3;
                            if (i == nx - 2) d3 = (-uh[m] + R(3) * uh[m + 1] - R(3) * uh[m + 2] + uh[m + 3]) * a.inv_dx3;
                        }
                        nrq = R(1.2) * dq2h - a.p5d * (hh * (d3 + R(1)) - fdiv(qv[m], hh * hh + a.eps));   // rhsq(), :507-512
                    }
                    if (UFAST || a.jets_simple) {
                        if (myjet >= 0) nrq += myamp * s_jw[kb + m];
                    } else if (has_jet) {
                        int k = i - a.jz0;
                        if (k >= 0 && k < a.jz_len) {
                            if (!a.jets_overlap) {
                                int jj = s_jj[k];
                                if (jj >= 0) nrq += sj[jj] * s_jw[C + k];
                            } else {                                             // generic: jets may overlap
                                for (int j = 0; j < nj; j++) {
                                    int s = a.jz0 + j * a.jet_space, e = s + 2 * a.jet_hw;
                                    if (i >= s && i <= e)
                                        nrq += sj[j] * (R((long long)(i - s) * (long long)(e - i)) / (R(0.25) * R((long long)(e - s) * (long long)(e - s))));
                                }
                            }
                        }
                    }
                    bool upd = true;                                              // adams(), :515-518: points 1 .. nx-2
                    if (UK == F_SMALL && m < 2) upd = m >= np;
                    if (UK == F_LARGE) upd = m >= np;
                    if (UFAST && m == C - 1) upd = upd && !is_last;
                    if (UK == ROLE_GENERAL) upd = i >= 1 && i <= nx - 2;
                    if (upd) {
                        hv[m] = hh + hdt * (R(-3) * nrh + rh[m]);
                        qv[m] = qv[m] + hdt * (R(-3) * nrq + rq[m]);
                        rh[m] = nrh;
                        rq[m] = nrq;
                    }
                }
            };
            if (FAST) update(kind_tag);
            else if (interior_thread) update(std::integral_constant<int, -1>{});
            else if (a0 < nx) update(std::integral_constant<int, ROLE_GENERAL>{});
        };

        // The single-body case runs the sub-step loop unrolled by two: the register rotation of the state
        // arrays (old values are still needed while the new ones are formed) then costs no copies
        // (+13 % measured).  With two bodies resident (F_LARGE + F_NONE) the unrolled pair does not pay
        // (instruction-cache footprint), they run one sub-step per trip.
        auto run_fast = [&](auto tag, auto unroll_tag) {
            int it = 0;
            if (decltype(unroll_tag)::value)
                for (; it + 1 < a.ndt_act; it += 2) { substep(it, tag); substep(it + 1, tag); }
            for (; it < a.ndt_act; it++) substep(it, tag);
        };
        if (role == F_SMALL) {
            run_fast(std::integral_constant<int, F_SMALL>{}, std::true_type{});
        } else if (role == F_NONE) {
            run_fast(std::integral_constant<int, F_NONE>{}, std::false_type{});
        } else if (role == F_LARGE) {
            run_fast(std::integral_constant<int, F_LARGE>{}, std::false_type{});
        } else if (role == ROLE_GENERAL) {
            for (int it = 0; it < a.ndt_act; it++) substep(it, std::integral_constant<int, ROLE_GENERAL>{});
        } else {
            for (int it = 0; it < a.ndt_act; it++) {           // beyond the domain: jets table duty, barrier count
                if (!a.jets_simple) {
                    R alpha = s_alpha[it];
                    for (int j = tid; j < nj; j += T)
                        s_jet[(it & 1) * nj + j] = a.jet_amp * ((R(1) - alpha) * s_uprev[j] + alpha * s_ucur[j]);
                }
                __syncthreads();
            }
        }

        // ---- action epilogue: obs, reward, guards -----------------------------------------
        __syncthreads();
        bool bad = false, nonfinite = false;
#pragma unroll
        for (int m = 0; m < C; m++) {
            int i = a0 + m;
            if (i >= 0 && i < nx) {
                s_h[i] = hv[m];
                s_q[i] = qv[m];
                bad |= (hv[m] < a.blow_lo) | (hv[m] > a.blow_hi);              // shkadov.py:176
                nonfinite |= !finite_(hv[m]) | !finite_(qv[m]);
            }
        }
        const int flags = __syncthreads_or((bad ? 1 : 0) | (nonfinite ? 4 : 0));
        const bool blow = flags & 1;
        if (flags & 1) status |= BEACON_STATUS_BLOWUP;
        if (flags & 4) status |= BEACON_STATUS_NONFINITE;

        const bool last = act == n_actions - 1;
        if (!resetting || last) {
            // observations, shkadov.py:239-250
            const size_t orow = resetting ? (size_t)b : ((size_t)act * a.B + b);
            R *obs = a.obs + orow * (size_t)(nj * a.n_obs);
            for (int e = tid; e < nj * a.n_obs; e += T) {
                int j = e / a.n_obs, k = e - j * a.n_obs;
                obs[e] = s_q[a.jet_pos + j * a.jet_space - a.l_obs + k * a.obs_stride];
            }
        }
        if (!resetting) {
            // rewards, shkadov.py:253-264 (joint) / :469-481 (per jet)
            const int warp = tid >> 5, lane = tid & 31;
            for (int j = warp; j < nj; j += T / 32) {
                int s = a.jet_pos + j * a.jet_space;
                R acc = R(0);
                for (int k = lane; k < a.l_rwd; k += 32) { R d = s_h[s + k] - R(1); acc += d * d; }
                acc = warp_sum(acc);
                if (lane == 0) s_term[j] = acc * a.dx;
            }
            __syncthreads();
            const size_t orow = (size_t)act * a.B + b;
            const R denom = R(nj * a.l_rwd);
            if (a.per_jet_rwd) {
                for (int j = tid; j < nj; j += T) a.rwd[orow * nj + j] = blow ? a.blowup_rwd : (R(0) - s_term[j]) / denom;
            } else if (tid == 0) {
                R r = R(0);
                for (int j = 0; j < nj; j++) r -= s_term[j];
                r /= denom;
                a.rwd[orow] = blow ? a.blowup_rwd : r;
            }
            if (tid == 0) {
                bool horizon = stp == a.n_act - 1;                            // shkadov.py:173-180
                a.done[orow] = (horizon || blow) ? 1 : 0;
                a.trunc[orow] = (horizon && !blow) ? 1 : 0;
            }
            stp += 1;
        }
    }   // actions

    if (resetting && n_actions == 0) {
        // plain reset: observation of the init state
        __syncthreads();
#pragma unroll
        for (int m = 0; m < C; m++) { int i = a0 + m; if (i >= 0 && i < nx) s_q[i] = qv[m]; }
        __syncthreads();
        R *obs = a.obs + (size_t)b * (size_t)(nj * a.n_obs);
        for (int e = tid; e < nj * a.n_obs; e += T) {
            int j = e / a.n_obs, k = e - j * a.n_obs;
            obs[e] = s_q[a.jet_pos + j * a.jet_space - a.l_obs + k * a.obs_stride];
        }
    }

    // ---- store state ----------------------------------------------------------------------
#pragma unroll
    for (int m = 0; m < C; m++) {
        int i = a0 + m;
        if (i >= 0 && i < nx) {
            a.h[row + i] = hv[m]; a.q[row + i] = qv[m]; a.rhsh[row + i] = rh[m]; a.rhsq[row + i] = rq[m];
        }
    }
    __syncthreads();
    for (int j = tid; j < nj; j += T) {
        a.u_cur[(size_t)b * nj + j] = s_ucur[j];
        a.u_prev[(size_t)b * nj + j] = s_uprev[j];
    }
    if (tid == 0) {
        a.stp[b] = resetting ? 0 : stp;
        a.draws[b] = draws;
        if (a.status) a.status[b] = status;
    }
}

// Reset order: CTAs are handed to the SMs in blockIdx order, and a reset with random warm steps
// (shkadov.py:118-123, U{0..400} actions per env) finishes when its longest env does.  One small CTA
// sorts the env indices by decreasing n_warm (counting sort over <= 2048 bins; ties in any order —
// only the schedule depends on it, never a result) so that the longest envs start first and the
// short ones fill the tail.
__global__ void __launch_bounds__(1024) shkadov_order_kernel(const int32_t *n_warm, const uint8_t *mask, int B, int max_warm, int32_t *order)
{
    constexpr int NB = 2048;
    __shared__ int hist[NB + 1];
    const int tid = threadIdx.x, T = blockDim.x;
    for (int k = tid; k <= NB; k += T) hist[k] = 0;
    __syncthreads();
    auto bin_of = [&](int b) {
        int w = (mask && !mask[b]) ? 0 : min(max(n_warm[b], 0), max_warm);
        int q = (int)(((long long)w * (NB - 1)) / (long long)(max_warm > 0 ? max_warm : 1));
        return NB - 1 - q;                                  // bin 0 = longest
    };
    for (int b = tid; b < B; b += T) atomicAdd(&hist[bin_of(b)], 1);
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int k = 0; k < NB; k++) { int c = hist[k]; hist[k] = run; run += c; }
    }
    __syncthreads();
    for (int b = tid; b < B; b += T) order[atomicAdd(&hist[bin_of(b)], 1)] = b;
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
template <typename R> class ShkadovEnv : public Env {
    beacon_shkadov_params p;
    DeviceBuffer h, q, rhsh, rhsq, u_cur, u_prev, stp, draws, h_init, q_init, order;
    ShkArgs<R> base{};
    int C = 0, T = 0;
    size_t smem = 0;
    void (*kernel)(const ShkArgs<R>) = nullptr;

    template <int CC, int TT, int MB> void pick()
    {
        C = CC; T = TT;
        kernel = shkadov_kernel<R, CC, TT, MB>;
    }

public:
    ShkadovEnv(const beacon_common &c, const beacon_shkadov_params &pp, const double *h0, const double *q0) : p(pp)
    {
        common = c;
        const int B = c.batch, nx = p.nx, nj = p.n_jets;
        BEACON_REQUIRE(B > 0 && nx >= 8 && nj >= 0 && p.ndt_act > 0 && p.n_interp > 0, "shkadov: bad sizes");
        BEACON_REQUIRE(p.jet_hw > 0 || nj == 0, "shkadov: jet_hw must be positive");
        // every lattice index the path touches must be inside the domain
        if (nj > 0) {
            int last = p.jet_pos + (nj - 1) * p.jet_space;
            BEACON_REQUIRE(p.jet_pos - p.jet_hw >= 1 && last + p.jet_hw <= nx - 2, "shkadov: jets outside the domain");
            BEACON_REQUIRE(p.jet_pos - p.l_obs >= 0 && last - p.l_obs + (p.n_obs - 1) * p.obs_stride < nx,
                           "shkadov: observation probes outside the domain");
            BEACON_REQUIRE(last + p.l_rwd <= nx, "shkadov: reward zone outside the domain");
            BEACON_REQUIRE(nj < 32768, "shkadov: too many jets");
        }
        info.kind = BEACON_SHKADOV; info.batch = B; info.dtype = real_traits<R>::dtype; info.device = c.device;
        info.n_obs = nj * p.n_obs; info.act_dim = nj; info.act_is_int = 0;
        info.rwd_dim = p.per_jet_rwd ? nj : 1; info.n_act = p.n_act; info.noise_dim = p.ndt_act;

        // (points per thread, threads, min CTAs/SM) variants; the first that covers nx is used
        // unless BEACON_SHKADOV_CFG="C,T,MINB" selects one explicitly (tuning).
        int wc = 0, wt = 0, wm = 0;
        if (const char *e = getenv("BEACON_SHKADOV_CFG")) sscanf(e, "%d,%d,%d", &wc, &wt, &wm);
        bool ok = false;
#define BEACON_SHK_TRY(CC, TT, MB)                                                             \
        if (!ok && (wc ? (wc == CC && wt == TT && wm == MB) : true) && (long)CC * TT >= nx + (CC - nx % CC) % CC) { pick<CC, TT, MB>(); ok = true; }
        // measured on B200 (profiles/sweep_shkadov_r1j_*.txt): 10 jets (nx 1350) 6,256,2; 20 jets (nx 1850)
        // 10,192,2; 41 jets (nx 2900) 6,512,1
        BEACON_SHK_TRY(6, 256, 2)
        if (wc) { BEACON_SHK_TRY(9, 160, 3) BEACON_SHK_TRY(9, 160, 2) BEACON_SHK_TRY(11, 128, 3) BEACON_SHK_TRY(11, 128, 2) BEACON_SHK_TRY(5, 640, 1) BEACON_SHK_TRY(10, 320, 1) }   // tuning only
        BEACON_SHK_TRY(10, 192, 2)
        BEACON_SHK_TRY(6, 512, 1)
        BEACON_SHK_TRY(12, 512, 1)
#undef BEACON_SHK_TRY
        if (!ok) throw Error(BEACON_ERR_UNSUPPORTED, "shkadov: no kernel variant covers this nx (max about 6130) or BEACON_SHKADOV_CFG is unknown");

        size_t nb = (size_t)B * nx * sizeof(R);
        h.alloc(nb); q.alloc(nb); rhsh.alloc(nb); rhsq.alloc(nb);
        u_cur.alloc((size_t)B * (nj ? nj : 1) * sizeof(R)); u_prev.alloc((size_t)B * (nj ? nj : 1) * sizeof(R));
        stp.alloc((size_t)B * 4); draws.alloc((size_t)B * 8);
        upload_as<R>(h_init, h0, nx); upload_as<R>(q_init, q0, nx);
        add_field("h", h.ptr, nx); add_field("q", q.ptr, nx); add_field("rhsh", rhsh.ptr, nx); add_field("rhsq", rhsq.ptr, nx);
        add_field("u", u_cur.ptr, nj); add_field("up", u_prev.ptr, nj); add_field("stp", stp.ptr, 1, true);
        add_field("draws", draws.ptr, 2, true);        // uint64 Philox draw counter as two int32 words (checkpoint / resume)

        ShkArgs<R> &a = base;
        a.nx = nx; a.ndt_act = p.ndt_act; a.n_act = p.n_act; a.n_interp = p.n_interp; a.n_jets = nj;
        a.jet_pos = p.jet_pos; a.jet_hw = p.jet_hw; a.jet_space = p.jet_space; a.l_obs = p.l_obs; a.n_obs = p.n_obs;
        a.obs_stride = p.obs_stride; a.l_rwd = p.l_rwd; a.per_jet_rwd = p.per_jet_rwd;
        // Chunks are shifted left by `off` phantom points so that the outlet point nx-1 is the last point
        // of its chunk (the LAST warp role then has its special cases at compile-time positions).
        a.off = (C - nx % C) % C;
        a.tail_aligned = 1;
        if ((size_t)T * C < (size_t)nx + a.off || getenv("BEACON_SHKADOV_NOALIGN")) {   // no room: old layout, general path
            a.off = ((nx - 1) % C == 0) ? 1 : 0;         // keep points nx-2 and nx-1 in one chunk
            a.tail_aligned = 0;
        }
        BEACON_REQUIRE((size_t)T * C - a.off >= (size_t)nx, "shkadov: internal chunking error");
        a.jets_overlap = (nj > 1 && p.jet_space <= 2 * p.jet_hw) ? 1 : 0;
        a.jz0 = p.jet_pos - p.jet_hw;
        a.jets_simple = (nj > 0 && p.jet_space > 0 && (nj == 1 || p.jet_space - 2 * p.jet_hw - 1 >= C - 1) && !a.jets_overlap) ? 1 : 0;
        a.jz_len = nj > 0 ? (nj - 1) * p.jet_space + 2 * p.jet_hw + 1 : 0;
        a.inv_dx = (R)(1.0 / p.dx); a.inv_2dx3 = (R)(1.0 / (2.0 * p.dx * p.dx * p.dx)); a.inv_dx3 = (R)(1.0 / (p.dx * p.dx * p.dx));
        {
            const double i3 = 1.0 / (2.0 * p.dx * p.dx * p.dx), w[5] = {-3.0, 10.0, -12.0, 6.0, -1.0};
            for (int k = 0; k < 5; k++) a.k3[k] = (R)(w[k] * i3);
            a.kc = (R)(2.0 * i3); a.kc3 = (R)(6.0 * i3); a.c12 = (R)(1.2 / p.dx);
        }
        a.hdt = (R)(0.5 * p.dt); a.p5d = (R)(1.0 / (5.0 * p.delta)); a.eps = (R)p.eps; a.jet_amp = (R)p.jet_amp; a.dx = (R)p.dx;
        a.blow_lo = (R)p.blow_lo; a.blow_hi = (R)p.blow_hi; a.blowup_rwd = (R)p.blowup_rwd;
        a.sigma = p.sigma; a.seed = c.seed; a.env_base = c.env_index_base;
        a.h = h.as<R>(); a.q = q.as<R>(); a.rhsh = rhsh.as<R>(); a.rhsq = rhsq.as<R>();
        a.u_cur = u_cur.as<R>(); a.u_prev = u_prev.as<R>(); a.stp = stp.as<int32_t>();
        a.draws = draws.as<unsigned long long>(); a.h_init = h_init.as<R>(); a.q_init = q_init.as<R>();
        a.B = B;

        smem = sizeof(R) * ((size_t)2 * XN * T + 2 * (size_t)nx + 2 * (size_t)p.ndt_act + 6 * (size_t)(nj ? nj : 1) + a.jz_len + 2 * C) +
               sizeof(short) * (size_t)a.jz_len + 16;
        BEACON_REQUIRE(smem <= 227 * 1024, "shkadov: shared-memory budget exceeded");
        raise_dynamic_smem_limit(kernel, smem);
    }

    void launch(const ShkArgs<R> &a, cudaStream_t s)
    {
        kernel<<<a.B, T, smem, s>>>(a);
        BEACON_CUDA_CHECK(cudaGetLastError());
        launches++;
    }

    void reset(const ResetArgs &r) override
    {
        ShkArgs<R> a = base;
        a.mode = 1; a.mask = r.mask; a.n_warm = r.n_warm; a.max_warm = r.n_warm ? r.max_warm : 0;
        a.noise = (const R *)r.noise; a.obs = (R *)r.obs; a.status = nullptr; a.n_fused = 0;
        BEACON_REQUIRE(r.obs != nullptr, "reset: obs must not be NULL");
        static const bool in_order = getenv("BEACON_SHKADOV_RESET_INORDER") != nullptr;   // A/B switch
        if (r.n_warm && a.max_warm > 0 && a.B > 1 && !in_order) {
            if (!order.ptr) order.alloc((size_t)a.B * sizeof(int32_t));
            shkadov_order_kernel<<<1, 1024, 0, r.stream>>>(r.n_warm, r.mask, a.B, a.max_warm, order.as<int32_t>());
            BEACON_CUDA_CHECK(cudaGetLastError());
            launches++;
            a.order = order.as<int32_t>();
        }
        launch(a, r.stream);
    }

    void step(const StepArgs &s) override
    {
        ShkArgs<R> a = base;
        a.mode = 0; a.n_fused = s.n_fused; a.actions = (const R *)s.actions; a.noise = (const R *)s.noise;
        a.obs = (R *)s.obs; a.rwd = (R *)s.rwd; a.done = s.done; a.trunc = s.trunc; a.status = s.status;
        launch(a, s.stream);
    }
};

Env *make_shkadov(const beacon_common &c, const beacon_shkadov_params &p, const double *h0, const double *q0)
{
    BEACON_REQUIRE(h0 && q0, "shkadov: init fields must not be NULL");
    if (c.dtype == BEACON_F64) return new ShkadovEnv<double>(c, p, h0, q0);
    if (c.dtype == BEACON_F32) return new ShkadovEnv<float>(c, p, h0, q0);
    throw Error(BEACON_ERR_INVALID, "unknown dtype");
}

}  // namespace beacon
