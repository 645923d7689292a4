// mac_reg_kernel.cuh: the register-resident MAC kernel (rayleigh 50x50, mac2d.cu), included twice by mac2d.cu:
// MAC_REG_NAME = mac_reg_kernel with MAC_REG_PHYS = false (the uniform instances) and mac_reg_phys_kernel with
// MAC_REG_PHYS = true (per-env physical constants, MacArgs::phys).  The kernel is stamped out twice, not wrapped
// around a shared __device__ body as mac_kernel and mac_big_kernel are: inlined into a wrapper, the body
// compiles to different machine code with more spills (DESIGN.md 3.4), and the uniform instance must stay as it
// was.  The second name is one that tools/sass_census.py's pattern for mac_reg_kernel does not match.
template <typename R, int NX, int NY, int TI, int TJ, int T, bool DBG>
__global__ void __launch_bounds__(T, 2) MAC_REG_NAME(const MacArgs<R> a)
{
    constexpr bool PHYS = MAC_REG_PHYS;
    typedef typename vec2_of<R>::type R2;
    constexpr int LD = NY + 2, N = (NX + 2) * LD;       // field planes in global memory
    constexpr int LDP = mac_ldp(LD, TI);                // exchange planes: conflict-free stride (8-byte elements)
    constexpr int NP = ((NX + 1) * LDP + 3) / 4 * 4;    // rows 0 .. NX (no ghost row NX+1: wall tiles read their own edge)
    // u and v live INTERLEAVED in one plane of (u, v) pairs: the tile origins of a quarter-warp fall into 8 distinct
    // 16-byte bank groups iff 2 LDU = 2 mod 8 (LDU = 53), one LDS.128 fetches both components, and every access is
    // conflict free — two separate planes of stride NY+2 = 52 cannot be (the banks 0, 5, 8, 13 are oversubscribed for
    // 2x5 tiles whatever the thread mapping; a stride of 57 for each does not fit twice per SM).  T uses the stride
    // of the exchange planes.  Measured: shared-memory bank conflicts were 25 % of all wavefronts before.
    constexpr int LDU = ((LD + 2) / 4) * 4 + 1, NU = (NX + 2) * LDU;      // in (u, v) pairs
    constexpr int LDT = LDP, NT = (NX + 2) * LDT;
    static_assert(TI != 2 || (2 * LDU) % 8 == 2, "u/v plane stride");
    constexpr int TILES_J = NY / TJ, TILES = (NX / TI) * TILES_J, NW = T / 32;
    static_assert(NX % TI == 0 && NY % TJ == 0 && TILES <= T, "tiles must cover the grid exactly");
    static_assert(NX <= 64, "transport wavefront: two rows per lane");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(16) float s_part[2][NW];     // fp32 warp partials of the residual (see the Poisson section)
    __shared__ R s_exact[NW];                         // fp64 warp partials, only when the fp32 total is too close to tol
    __shared__ R s_seg[32];
    __shared__ R s_act[32];
    static_assert((NP * sizeof(R)) % 16 == 0, "planes must stay 16-byte aligned");
    const int tid = threadIdx.x, b = blockIdx.x;
    const bool resetting = a.mode == 1;
    if (resetting && a.mask && !a.mask[b]) return;

    R *PA = reinterpret_cast<R *>(smem_raw), *PB = PA + NP;
    R2 *UV = reinterpret_cast<R2 *>(PB + NP);
    R *S = reinterpret_cast<R *>(UV + NU);
    const size_t row = (size_t)b * N;
    R *gu = a.u + row, *gv = a.v + row, *gp = a.p + row, *gs = a.s + row;

    const bool has_tile = tid < TILES;
    const int ti = tid / TILES_J, tj = tid - ti * TILES_J;
    const int i0 = 1 + ti * TI, j0 = 1 + tj * TJ;
    const int o = i0 * LD + j0, op = i0 * LDP + j0;     // tile origin in global field / exchange planes
    const int ou = i0 * LDU + j0, ot = i0 * LDT + j0;   // ... in the (u, v) plane and in the T plane
    const int opx = has_tile ? op : LDP + 1;             // threads without a tile shadow tile 0 in the sweeps (weight 0)
    const bool top = has_tile && i0 == 1, bot = has_tile && i0 + TI - 1 == NX;
    const bool lef = has_tile && j0 == 1, rig = has_tile && j0 + TJ - 1 == NY;
    const R w_has = has_tile ? R(1) : R(0);
    const R w_top = top ? R(2) : R(1), w_bot = bot ? R(2) : R(1), w_lef = lef ? R(1) : R(0), w_rig = rig ? R(1) : R(0);
    // Halo offsets of the Jacobi sweeps.  All ghost cells of phi are Neumann copies of the wall-adjacent cell
    // (rayleigh.py:436-445), so a wall tile reads that cell — its own edge row / column in the exchange plane —
    // instead of a ghost: no ghost cell of phi is ever stored (30 predicated stores per thread and sweep, ~10
    // shared-memory wavefronts per warp and sweep, gone).  Threads without a tile shadow tile 0.
    const int tix = has_tile ? ti : 0, tjx = has_tile ? tj : 0;
    const int o_n = tix == 0 ? 0 : -LDP, o_s = tix == NX / TI - 1 ? (TI - 1) * LDP : TI * LDP;
#define TILE_LOOP                                      \
    _Pragma("unroll") for (int r = 0; r < TI; r++)     \
    _Pragma("unroll") for (int k = 0; k < TJ; k++)

    if (resetting) {                                   // rayleigh.py:89-128
        for (int e = tid; e < N; e += T) { gu[e] = a.u0[e]; gv[e] = a.v0[e]; gp[e] = a.p0[e]; gs[e] = a.s0[e]; }
        for (int e = tid; e < a.n_sgts; e += T) a.a_cur[(size_t)b * a.n_sgts + e] = R(0);
        const int per_step = 3 * a.nx_obs_pts * a.ny_obs_pts;
        R *hist = a.obs_hist + (size_t)b * a.n_obs;
        for (int e = tid; e < a.n_obs; e += T) {
            int st = e / per_step, rem = e - st * per_step;
            R val = R(0);
            if (st == a.n_obs_steps - 1) {
                int f = rem / (a.nx_obs_pts * a.ny_obs_pts), q = rem - f * (a.nx_obs_pts * a.ny_obs_pts);
                int pi = q / a.ny_obs_pts, pj = q - pi * a.ny_obs_pts;
                int x = a.nx_obs / 2 + pi * a.nx_obs, y = a.ny_obs / 2 + pj * a.ny_obs;
                val = (f == 0) ? a.s0[x * LD + y] : (f == 1 ? a.u0[x * LD + y] : a.v0[x * LD + y]);
            }
            hist[e] = val;
            a.obs[(size_t)b * a.n_obs + e] = val;
        }
        if (tid == 0) a.stp[b] = 0;
        return;
    }
    MAC_LOAD_COEF(b);                                  // read after the barrier below
    for (int e = tid; e < 2 * NP; e += T) PA[e] = R(0);   // masked wavefront steps read padding slots: keep them finite
    // state planes global -> shared, into the padded / interleaved layouts (once per launch)
    for (int e = tid; e < N; e += T) {
        const int i = e / LD, j = e - i * LD;
        R2 w; w.x = gu[e]; w.y = gv[e];
        UV[i * LDU + j] = w;
        S[i * LDT + j] = gs[e];
    }
    for (int e = tid; e < NX + 2; e += T) {            // padding columns: read by masked wavefront steps, keep them finite
        for (int j = LD; j < LDU; j++) { R2 z; z.x = R(0); z.y = R(0); UV[e * LDU + j] = z; }
        for (int j = LD; j < LDT; j++) S[e * LDT + j] = R(0);
    }
    __syncthreads();
    // The pressure stays in global memory (L2).  During the launch the authoritative copy of a thread's tile lives in a
    // scratch laid out [cell][thread] (the `vs` workspace plane): a tile row is 5 doubles at an odd offset in the plane,
    // so a tile-wise warp access touches ~13 cache lines, in the scratch consecutive lanes are contiguous (2 lines) and
    // the neighbour tile's cell is the same slot 1 / TILES_J threads away.  The plane keeps the launch-initial values
    // until the end: ghost cells of p only ever accumulate the same increments as their wall-adjacent cells (phi
    // ghosts are copies) and never feed back, so they are brought up to date once, at the end of the launch.
    static_assert(TI * TJ * T <= N, "the pressure scratch must fit the vs plane");
    R *const sp = a.vs + row + tid;
#define PSCR(r, k) sp[((r) * TJ + (k)) * T]
    if (has_tile) { TILE_LOOP { PSCR(r, k) = gp[o + r * LD + k]; } }
    int stp = a.stp[b];
    int status = 0;
    const R dt = a.dt, inv_dx = a.inv_dx, inv_dy = a.inv_dy;
    const bool dbg = DBG && a.dbg != nullptr && b == 0 && tid == 0;
    long long tph[DBG ? 8 : 1] = {0}, tlast = dbg ? clock64() : 0;
#define PHASE(n) do { if (DBG && dbg) { long long tn_ = clock64(); tph[n] += tn_ - tlast; tlast = tn_; } } while (0)

    for (int act = 0; act < a.n_fused; act++) {
        const size_t orow = (size_t)act * a.B + b;
        __syncthreads();
        if (tid == 0) {                                            // rayleigh.py:164-171
            const R *ain = (const R *)a.actions + orow * a.n_sgts;
            const int ns = a.n_sgts;
            for (int j = 0; j < ns; j++) s_act[j] = ain[j];
            R mean = np_pairwise_small(s_act, ns) / R(ns);
            R m = R(1);
            for (int j = 0; j < ns; j++) { s_act[j] = s_act[j] - mean; m = np_max(m, rabs(s_act[j]) / a.Cmax); }
            for (int j = 0; j < ns; j++) { s_act[j] = s_act[j] / m; s_seg[j] = a.Th + s_act[j]; a.a_cur[(size_t)b * ns + j] = s_act[j]; }
        }
        __syncthreads();
        long long it_total = 0;

#define UU(i, j) UV[(i) * LDU + (j)].x
#define VV(i, j) UV[(i) * LDU + (j)].y
#define SS(i, j) S[(i) * LDT + (j)]
        // ---- boundary conditions, rayleigh.py:180-202, split by field: the velocity ghosts do not depend on T, the
        // T ghosts need the transported T.  Executed by the threads t0, t0 + nt, ... of the caller's group.
        auto bc_uv = [&](const int t0, const int nt, const bool walls) {
            for (int k = t0; k < 2 * (NX + 2) + 2 * (NY + 2); k += nt) {
                if (k < NY + 2) {
                    int j = k;
                    if (walls && j >= 1 && j <= NY) UU(1, j) = R(0);
                    if (j >= 2 && j <= NY) VV(0, j) = -VV(1, j);
                } else if (k < 2 * (NY + 2)) {
                    int j = k - (NY + 2);
                    if (walls && j >= 1 && j <= NY) UU(NX + 1, j) = R(0);
                    if (j >= 2 && j <= NY) VV(NX + 1, j) = -VV(NX, j);
                } else if (k < 2 * (NY + 2) + (NX + 2)) {
                    int i = k - 2 * (NY + 2);
                    if (i >= 1 && i <= NX + 1) UU(i, NY + 1) = (i == 1 || i == NX + 1) ? -R(0) : -UU(i, NY);
                    if (walls && i >= 1 && i <= NX) VV(i, NY + 1) = R(0);
                } else {
                    int i = k - 2 * (NY + 2) - (NX + 2);
                    if (i >= 1 && i <= NX + 1) UU(i, 0) = (i == 1 || i == NX + 1) ? -R(0) : -UU(i, 1);
                    if (walls && i >= 1 && i <= NX) VV(i, 1) = R(0);
                }
            }
        };
        auto bc_s = [&](const int t0, const int nt) {
            for (int k = t0; k < 2 * (NX + 2) + 2 * (NY + 2); k += nt) {
                if (k < NY + 2) {
                    int j = k;
                    if (j >= 1 && j <= NY) SS(0, j) = SS(1, j);
                } else if (k < 2 * (NY + 2)) {
                    int j = k - (NY + 2);
                    if (j >= 1 && j <= NY) SS(NX + 1, j) = SS(NX, j);
                } else if (k < 2 * (NY + 2) + (NX + 2)) {
                    int i = k - 2 * (NY + 2);
                    if (i >= 1 && i <= NX) SS(i, NY + 1) = R(2) * a.Tc - SS(i, NY);
                } else {
                    int i = k - 2 * (NY + 2) - (NX + 2);
                    if (i >= 1 && i <= NX) {
                        int sg = (i - 1) / a.nx_sgts;
                        if (sg < a.n_sgts) SS(i, 0) = R(2) * s_seg[sg] - SS(i, 1);
                    }
                }
            }
        };
        // ---- predictor into registers, rayleigh.py:371-407: the right-hand sides of u* and v* (v: WITHOUT the buoyancy
        // term); u* = u + dt rhs_u and v* = v + dt (rhs_v + T) are formed later with the transported T: the same
        // operations in the same order as the reference's expressions
        R us[TI][TJ], vs[TI][TJ];
        auto predictor = [&]() {
            const R2 *uv = UV + ou;
            // Not read (the pressure comes from the scratch).  It keeps gp and o among the lambda's captures, on which
            // nvcc's code for this kernel depends: without it the fp64 instance spills 8 B more.
            [[maybe_unused]] const R *p = gp + o;
            // (u, v) pairs of the tile and its one-cell ring are fetched as 16-byte words where they are used (equal
            // addresses are merged by the compiler)
            TILE_LOOP {
                const R2 *q = uv + r * LDU + k;
                const R2 c = q[0], E = q[LDU], W = q[-LDU], Nn = q[1], Ss = q[-1];
                const R uc = c.x, vc = c.y, pc = PSCR(r, k);
                us[r][k] = R(0); vs[r][k] = R(0);
                if (r > 0 || !top) {               // i >= 2
                    R uE = R(0.5) * (E.x + uc), uW = R(0.5) * (uc + W.x);
                    R uN = R(0.5) * (Nn.x + uc), uS = R(0.5) * (uc + Ss.x);
                    R vN = R(0.5) * (Nn.y + q[-LDU + 1].y), vS = R(0.5) * (vc + W.y);
                    R conv = (uE * uE - uW * uW) * inv_dx + (uN * vN - uS * vS) * inv_dy;
                    R diff = ((E.x - R(2) * uc + W.x) * a.inv_dx2 + (Nn.x - R(2) * uc + Ss.x) * a.inv_dy2) * MAC_DCOEF;
                    const R pw = r > 0 ? PSCR(r - 1, k) : (sp - TILES_J)[((TI - 1) * TJ + k) * T];
                    R pres = (pc - pw) * inv_dx;
                    us[r][k] = diff - conv - pres;
                }
                if (k > 0 || !lef) {               // j >= 2
                    R vE = R(0.5) * (E.y + vc), vW = R(0.5) * (vc + W.y);
                    R uE = R(0.5) * (E.x + q[LDU - 1].x), uW = R(0.5) * (uc + Ss.x);
                    R vN = R(0.5) * (Nn.y + vc), vS = R(0.5) * (vc + Ss.y);
                    R conv = (uE * vE - uW * vW) * inv_dx + (vN * vN - vS * vS) * inv_dy;
                    R diff = ((E.y - R(2) * vc + W.y) * a.inv_dx2 + (Nn.y - R(2) * vc + Ss.y) * a.inv_dy2) * MAC_DCOEF;
                    const R ps = k > 0 ? PSCR(r, k - 1) : (sp - 1)[(r * TJ + TJ - 1) * T];
                    R pres = (pc - ps) * inv_dy;
                    vs[r][k] = diff - conv - pres;
                }
            }
        };
        const R kx = MAC_TCOEF * a.inv_dx2, ky = MAC_TCOEF * a.inv_dy2;
        constexpr int RS = wavefront_row_stride(NY);       // columns 0..NY per row pair (0 unused), padded
        static_assert(NX % 2 == 0 && NX / 2 <= 32, "wavefront layout: one lane per row pair");
        static_assert(2 * (NX / 2) * RS <= NP, "wavefront planes must fit the exchange planes");
        auto wavefront = [&]() {
            const R hk = R(0.5) * dt * inv_dy, dky = dt * ky;
            if constexpr (std::is_same<R, double>::value) {
                transport_wavefront_f64<NX, NY, LDU, LDT>((uint32_t)__cvta_generic_to_shared(PA), (uint32_t)__cvta_generic_to_shared(PB),
                                                          (uint32_t)__cvta_generic_to_shared(UV), (uint32_t)__cvta_generic_to_shared(S), hk, dky, tid);
            } else {
                // Lane l owns rows 2l+1, 2l+2 and does column j = t - l + 1 at step t.  The loop is
                // uniform: inactive steps (j outside 1..NY) compute on harmless in-bounds garbage and
                // are masked by ONE predicate (stores, partial sums); per step the dependent chain is
                // SHFL + 2 DFMA, the coefficients of column j+1 are fetched while it waits.
                constexpr int LANES = NX / 2, STEPS = NY + LANES - 1;
                const int lane = tid;
                const bool on = lane < LANES;
                const int l = on ? lane : 0;
                const R2 *Vr0 = UV + (2 * l + 1) * LDU, *Vr1 = Vr0 + LDU;
                R *Sr0 = S + (2 * l + 1) * LDT, *Sr1 = Sr0 + LDT;
                const R *AAr = PA + (size_t)l * RS * 2, *WWr = PB + (size_t)l * RS * 2;
                // column 1: partial sums with the south ghost (column 0, untouched by transport)
                R p0 = fma(fma(hk, Vr0[1].y, dky), Sr0[0], AAr[2]), p1 = fma(fma(hk, Vr1[1].y, dky), Sr1[0], AAr[3]);
                R w0 = WWr[2], w1 = WWr[3];
                R last_new = R(0);
                // pointers biased by -lane: element [t] is column t - lane + 2 (prefetch) / t - lane + 1 (store)
                // (lanes beyond the last row pair mimic lane 0 with the predicate off)
                const R *An = AAr + 2 * (2 - l), *Wn = WWr + 2 * (2 - l);
                const R2 *V0n = Vr0 + (2 - l), *V1n = Vr1 + (2 - l);
                R *S0o = Sr0 + (1 - l), *S1o = Sr1 + (1 - l);
                const int c0 = on ? -lane : -(1 << 20);
    #pragma unroll 2
                for (int t = 0; t < STEPS; t++) {
                    const R wv = __shfl_up_sync(0xffffffffu, last_new, 1);
                    const bool act_ = (unsigned)(c0 + t) < (unsigned)NY;
                    const R a0n = An[2 * t], a1n = An[2 * t + 1], w0n = Wn[2 * t], w1n = Wn[2 * t + 1];
                    const R s0n = fma(hk, V0n[t].y, dky), s1n = fma(hk, V1n[t].y, dky);
                    const R n0 = fma(w0, wv, p0);
                    const R n1 = fma(w1, n0, p1);
                    last_new = n1;
                    if (act_) {
                        S0o[t] = n0; S1o[t] = n1;
                        p0 = fma(s0n, n0, a0n); p1 = fma(s1n, n1, a1n);
                    }
                    w0 = w0n; w1 = w1n;
                }
            }
        };
        // The sub-steps are software pipelined across the CTA's warps: the transport of sub-step it-1 is a one-warp
        // recurrence (the wavefront, ~9 k cycles) and none of what follows it at the start of sub-step it needs the new
        // T — the velocity ghost cells and the whole predictor up to the buoyancy term.  So while warp 0 runs the
        // wavefront, the other warps apply the velocity boundary conditions (walls are not re-written: they stay zero
        // and the wavefront reads them) and compute the predictor of THEIR tiles; after the barrier warp 0 catches up
        // with the predictor of its tiles while the others set the T ghosts.  Before: 7 of 8 warps idle for 14 % of the
        // kernel's time.
        const int warp = tid >> 5;
        for (int it = 0; it <= a.ndt_act; it++) {
            // stage X: transport of the previous sub-step (warp 0) || velocity BCs + predictor of this one (the others);
            // stage Y: warp 0 catches up with the predictor of its tiles, the others set the T ghost cells.
            // One two-trip loop so that the predictor exists ONCE in the instruction stream.
            bool last = false;
#pragma unroll 1
            for (int stage = 0; stage < 2; stage++) {
                bool pred;
                if (stage == 0) {
                    if (warp == 0) {
                        if (it > 0) wavefront();
                        pred = false;
                    } else {
                        pred = it < a.ndt_act;
                        if (pred) {
                            bc_uv(tid - 32, T - 32, it == 0);
                            asm volatile("bar.sync 1, %0;" ::"r"(T - 32) : "memory");   // warps 1.. only: their ghost cells are in place
                        }
                    }
                } else {
                    pred = warp == 0;
                    if (!pred) bc_s(tid - 32, T - 32);
                }
                if (pred && has_tile) predictor();
                if (stage == 0) {
                    __syncthreads();               // T is final; velocity ghosts final
                    PHASE(0);
                    if (it == a.ndt_act) { last = true; break; }
                }
            }
            if (last) break;
            if (has_tile) {                        // u* = u + dt rhs_u, v* = v + dt (rhs_v + T), rayleigh.py:393,404
                TILE_LOOP {                        // (T of the cell itself, no ghost; the pair is one conflict-free 16-byte load)
                    const R2 c = UV[ou + r * LDU + k];
                    us[r][k] = (r > 0 || !top) ? c.x + dt * us[r][k] : c.x;
                    vs[r][k] = (k > 0 || !lef) ? c.y + dt * (vs[r][k] + S[ot + r * LDT + k]) : c.y;
                }
            }
            __syncthreads();                       // every read of the old u, v is done
            if (has_tile) { TILE_LOOP { R2 w; w.x = us[r][k]; w.y = vs[r][k]; UV[ou + r * LDU + k] = w; } }
            __syncthreads();                       // U, V now hold the starred fields (walls: 0)
            PHASE(1);

            // ---- Poisson: rhs and phi in registers, rayleigh.py:412-456 -------------------------------
            // phi_new = (xp+xm)*k1 + (yp+ym)*k2 + cn with k1 = dy2/(2(dx2+dy2)), k2 = dx2/(2(dx2+dy2)),
            // cn = -b dx2 dy2/(2(dx2+dy2)): 2 DADD + 2 DFMA per cell.  phi is one register tile updated
            // in place; sweep s writes exchange plane P[s&1] (P[1] = PB).
            // The residual reduction is taken off the critical path: while sweep k is computed, the
            // warp reduction of sweep k-1's residual is interleaved with it (one shuffle stage per
            // tile column) and the CTA total of sweep k-2 (warp partials published one barrier ago) is
            // summed; the convergence decision for sweep k-2 is made before sweep k is committed.  A
            // converged solve drops the two speculative sweeps and re-reads its tile of phi_{k-2}
            // from the exchange plane that still holds it, so the sweep count and the result are
            // exactly those of the reference's `while err > tol` loop.
            // The reduction itself runs in fp32 (5 SHFL + 2 LDS.128 + 7 FADD per sweep instead of 10 SHFL +
            // 8 LDS.64 + 12 DADD): its only use is the comparison with tol, and an fp32 sum of 256 positive
            // terms is within ~1e-6 of the fp64 one.  Whenever the fp32 total lies within 1e-4 tol of tol
            // (a few solves in a thousand) the decision is retaken from the per-thread fp64 residuals of
            // that sweep, kept in a register, with the fp64 butterfly + pairwise tree: the stop test is
            // decided by fp64 arithmetic in every case where fp32 could have changed it.
            R cn[TI][TJ], phi[TI][TJ];
            R *const pa = PA + opx, *const pb = PB + opx;
            auto tile_acc = [&](const R (&rs)[TI], const R (&dl)[TI], const R (&dr)[TI]) -> R {
                // residual over the ghost-inclusive array: ghost copies re-count the wall-adjacent cells
                R cl = dl[0] * dl[0], cr = dr[0] * dr[0];
#pragma unroll
                for (int r = 1; r < TI; r++) { cl = fma(dl[r], dl[r], cl); cr = fma(dr[r], dr[r], cr); }
                R mid = R(0);
#pragma unroll
                for (int r = 1; r < TI - 1; r++) mid += rs[r];
                R acc = (TI > 1) ? fma(rs[0], w_top, fma(rs[TI - 1], w_bot, mid)) : rs[0] * (w_top + w_bot - R(1));
                return fma(cl, w_lef, fma(cr, w_rig, acc)) * w_has;
            };
            // one sweep (every thread; threads without a tile work on tile 0's addresses and weigh 0)
            // + the warp reduction of the previous sweep's residual, one stage per column
            auto sweep = [&](R (&ph)[TI][TJ], const R *pi, float &wsum) -> R {
                // in place, column by column: the old values of column k-1 are kept in `po_`, column k+1
                // is still old when column k is computed (one register tile, no copies)
                R hn[TJ], hs[TJ], hw[TI], he[TI];    // halo: rows i0-1 / i0+TI, columns j0-1 / j0+TJ (wall tiles: their own edge)
                const R *pn = pi + o_n, *ps = pi + o_s;
#pragma unroll
                for (int k = 0; k < TJ; k++) { hn[k] = pn[k]; hs[k] = ps[k]; }
                // west / east: every lane loads at the same tile-relative offset (conflict free; clamped offsets would put
                // the lanes of wall tiles one bank off the others: 2-way conflicts in every warp, measured -3.7 %) and
                // wall tiles take their own edge column from registers instead
                const bool lefx = tjx == 0, rigx = tjx == TILES_J - 1;
#pragma unroll
                for (int r = 0; r < TI; r++) { hw[r] = pi[r * LDP - 1]; he[r] = pi[r * LDP + TJ]; }
                R rs[TI], dl[TI], dr[TI], po_[TI];
#pragma unroll
                for (int r = 0; r < TI; r++) { rs[r] = R(0); po_[r] = lefx ? ph[r][0] : hw[r]; he[r] = rigx ? ph[r][TJ - 1] : he[r]; }
#pragma unroll
                for (int k = 0; k < TJ; k++) {
                    if (k < 5) wsum += __shfl_xor_sync(0xffffffffu, wsum, 16 >> k);
                    R old[TI], nv[TI];
#pragma unroll
                    for (int r = 0; r < TI; r++) old[r] = ph[r][k];
#pragma unroll
                    for (int r = 0; r < TI; r++) {
                        const R xm = (r > 0) ? old[r - 1] : hn[k], xp = (r < TI - 1) ? old[r + 1] : hs[k];
                        const R ym = po_[r], yp = (k < TJ - 1) ? ph[r][k + 1] : he[r];
                        nv[r] = fma(xp + xm, a.pk1, fma(yp + ym, a.pk2, cn[r][k]));
                        const R d = nv[r] - old[r];
                        rs[r] = fma(d, d, rs[r]);
                        if (k == 0) dl[r] = d;
                        if (k == TJ - 1) dr[r] = d;
                    }
#pragma unroll
                    for (int r = 0; r < TI; r++) { po_[r] = old[r]; ph[r][k] = nv[r]; }
                }
#pragma unroll
                for (int st = TJ; st < 5; st++) wsum += __shfl_xor_sync(0xffffffffu, wsum, 16 >> st);
                return tile_acc(rs, dl, dr);
            };
            auto commit = [&](const R (&nw)[TI][TJ], R *po) {
                if (has_tile) { TILE_LOOP { po[r * LDP + k] = nw[r][k]; } }
            };
            auto total32 = [&](const float *part) -> float {   // same pairwise order in every thread -> uniform decision
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
            // `while err > tol` for one sweep: fp32 total when it is clearly on one side of tol, else the fp64 total of
            // the per-thread residuals `mine` of that sweep (butterfly + pairwise tree, the order of the fp64-only code).
            // The branch is uniform (every thread holds the same fp32 total); a NaN total takes the fp64 path.
            auto converged = [&](const float err32, const R mine) -> bool {
                if (fabsf(err32 - tolf) > tol_band) return !(err32 > tolf);
                return residual_converged_exact<R, NW>(mine, s_exact, a.tol);      // cold, out of line
            };
            R accp, accq = R(0);                          // residuals (this thread) of the last committed sweep and of the one before
            // sweep 1 starts from phi = 0: phi_1 = cn, no halo reads
            {
                R rs[TI], dl[TI], dr[TI];
#pragma unroll
                for (int r = 0; r < TI; r++) {
                    rs[r] = R(0);
#pragma unroll
                    for (int k = 0; k < TJ; k++) {
                        R cv = R(0);
                        if (has_tile) {
                            const R ue = (r < TI - 1) ? us[r + 1][k] : UV[ou + (r + 1) * LDU + k].x;
                            const R vn = (k < TJ - 1) ? vs[r][k + 1] : UV[ou + r * LDU + k + 1].y;
                            cv = -(((ue - us[r][k]) * inv_dx + (vn - vs[r][k]) * inv_dy) * a.cscale) * a.inv_den;
                        }
                        cn[r][k] = cv; phi[r][k] = cv;
                        rs[r] = fma(cv, cv, rs[r]);
                        if (k == 0) dl[r] = cv;
                        if (k == TJ - 1) dr[r] = cv;
                    }
                }
                accp = tile_acc(rs, dl, dr);
                commit(phi, pb);
                __syncthreads();
            }
            // sweep 2 (speculative until sweep 1's residual is known, two barriers from now)
            {
                float ws = (float)accp;
                const R acc = sweep(phi, pb, ws);
                commit(phi, pa);
                if ((tid & 31) == 0) s_part[1][tid >> 5] = ws;
                __syncthreads();
                accq = accp; accp = acc;
            }
            int itp;
            const R *pf;                                  // plane holding the final iterate (tile-relative)
            for (int k = 3;; k += 2) {
                {   // odd k: phi_{k-1} (in PA) -> phi_k; decide on sweep k-2 (still in PB)
                    float ws = (float)accp;
                    const R acc = sweep(phi, pa, ws);
                    const float err = total32(s_part[1]);
                    if (k - 2 > a.itmax) { status |= BEACON_STATUS_POISSON_OVERFLOW; itp = k - 2; pf = pb; break; }
                    if (converged(err, accq)) { itp = k - 2; pf = pb; break; }
                    commit(phi, pb);
                    if ((tid & 31) == 0) s_part[0][tid >> 5] = ws;
                    __syncthreads();
                    accq = accp; accp = acc;
                }
                {   // even k+1: phi_k (in PB) -> phi_{k+1}; decide on sweep k-1 (still in PA)
                    float ws = (float)accp;
                    const R acc = sweep(phi, pb, ws);
                    const float err = total32(s_part[0]);
                    if (k - 1 > a.itmax) { status |= BEACON_STATUS_POISSON_OVERFLOW; itp = k - 1; pf = pa; break; }
                    if (converged(err, accq)) { itp = k - 1; pf = pa; break; }
                    commit(phi, pa);
                    if ((tid & 31) == 0) s_part[1][tid >> 5] = ws;
                    __syncthreads();
                    accq = accp; accp = acc;
                }
            }
            TILE_LOOP { phi[r][k] = pf[r * LDP + k]; }     // the converged iterate
            it_total += itp;
            PHASE(2);

            // ---- p += phi (rayleigh.py:219; ghost cells: see the end of the launch) and in-place corrector (:461-464)
            if (has_tile) {
                R2 *uv = UV + ou;
                TILE_LOOP {
                    PSCR(r, k) += phi[r][k];
                    R2 w = uv[r * LDU + k];
                    if (r > 0 || !top) { const R pw = (r > 0) ? phi[r - 1][k] : pf[-LDP + k]; w.x = w.x - dt * (phi[r][k] - pw) * inv_dx; }
                    if (k > 0 || !lef) { const R ps = (k > 0) ? phi[r][k - 1] : pf[r * LDP - 1]; w.y = w.y - dt * (phi[r][k] - ps) * inv_dy; }
                    uv[r * LDU + k] = w;
                }
            }
            __syncthreads();

            PHASE(3);
            // ---- transport, rayleigh.py:469-487:  new(i,j) = A + BW*new(i-1,j) + BS*new(i,j-1) ----------
            // All threads write A and B_W of their cells into the (now free) exchange planes in the
            // layout the wavefront warp wants: [lane = row pair][column][row in pair], so that one
            // LDS.128 fetches both rows of a lane and every address is base(lane) + 16*step.  The
            // west ghost row (i = 0, never updated) is folded into A of row 1 (B_W := 0 there).
            {
                if (has_tile) {
                    const R2 *uv = UV + ou;
                    const R *sc = S + ot;
                    R Av[TI][TJ], Wv[TI][TJ];
                    TILE_LOOP {
                        const int e = r * LDT + k;
                        const R2 c = uv[r * LDU + k];
                        const R uE = uv[(r + 1) * LDU + k].x, uW = c.x, vN = uv[r * LDU + k + 1].y, vS = c.y;
                        const R s0 = sc[e], sE = sc[e + LDT], sN = sc[e + 1];
                        R diff0 = ((sE - R(2) * s0) * a.inv_dx2 + (sN - R(2) * s0) * a.inv_dy2) * MAC_TCOEF;
                        R conv0 = (uE * (R(0.5) * (sE + s0)) - uW * (R(0.5) * s0)) * inv_dx + (vN * (R(0.5) * (sN + s0)) - vS * (R(0.5) * s0)) * inv_dy;
                        R A = s0 + dt * (diff0 - conv0);
                        R BW = dt * (kx + R(0.5) * uW * inv_dx);
                        if (r == 0 && top) { A = fma(BW, sc[e - LDT], A); BW = R(0); }
                        Av[r][k] = A; Wv[r][k] = BW;
                    }
                    // [row pair][column][row in pair]: with two-row tiles the two rows of a column are ONE 16-byte slot
                    // (conflict free for a quarter-warp: 58 ti + 5 tj mod 8 is a permutation); other tile heights store
                    // element by element
                    if constexpr (TI == 2) {
                        R2 *A2 = reinterpret_cast<R2 *>(PA) + ti * RS + j0, *W2 = reinterpret_cast<R2 *>(PB) + ti * RS + j0;
#pragma unroll
                        for (int k = 0; k < TJ; k++) {
                            R2 x; x.x = Av[0][k]; x.y = Av[1][k]; A2[k] = x;
                            R2 y; y.x = Wv[0][k]; y.y = Wv[1][k]; W2[k] = y;
                        }
                    } else {
                        TILE_LOOP {
                            const int gi = TI * ti + r, idx = ((gi >> 1) * RS + j0 + k) * 2 + (gi & 1);
                            PA[idx] = Av[r][k];
                            PB[idx] = Wv[r][k];
                        }
                    }
                }
                __syncthreads();
                PHASE(4);
                PHASE(5);
            }
        }   // sub-steps

        // ---- observations and reward, rayleigh.py:243-275 ---------------------------------------------
        {
            R *hist = a.obs_hist + (size_t)b * a.n_obs;
            const int per_step = 3 * a.nx_obs_pts * a.ny_obs_pts;
            R *out = a.obs + orow * a.n_obs;
            for (int e = tid; e < a.n_obs; e += T) {
                int st = e / per_step, rem = e - st * per_step;
                R val;
                if (st < a.n_obs_steps - 1) val = hist[e + per_step];
                else {
                    int f = rem / (a.nx_obs_pts * a.ny_obs_pts), q = rem - f * (a.nx_obs_pts * a.ny_obs_pts);
                    int pi = q / a.ny_obs_pts, pj = q - pi * a.ny_obs_pts;
                    int x = a.nx_obs / 2 + pi * a.nx_obs, y = a.ny_obs / 2 + pj * a.ny_obs;
                    val = (f == 0) ? SS(x, y) : (f == 1 ? UU(x, y) : VV(x, y));
                }
                out[e] = val;
            }
            __syncthreads();
            for (int e = tid; e < a.n_obs; e += T) hist[e] = out[e];
            bool nonfinite = false;
            for (int e = tid; e < N; e += T) {
                const int i = e / LD, j = e - i * LD;
                const R2 w = UV[i * LDU + j];
                nonfinite |= !finite_(SS(i, j)) | !finite_(w.x) | !finite_(w.y);
            }
            if (__syncthreads_or(nonfinite ? 1 : 0)) status |= BEACON_STATUS_NONFINITE;
            if (tid == 0) {
                R nu = R(0);
                for (int i = 1; i <= NX; i++) nu -= (SS(i, 1) - a.Th) / (R(0.5) * a.dy);
                nu /= R(NX);
                a.rwd[orow] = -nu;
                bool horizon = stp == a.n_act - 1;
                a.done[orow] = horizon; a.trunc[orow] = horizon;
                if (a.iters) a.iters[orow] = it_total;
            }
            stp += 1;
        }
    }   // actions

    __syncthreads();
    for (int e = tid; e < N; e += T) {                 // state planes shared -> global
        const int i = e / LD, j = e - i * LD;
        const R2 w = UV[i * LDU + j];
        gu[e] = w.x; gv[e] = w.y; gs[e] = SS(i, j);
    }
    if (has_tile) {                                    // pressure back to its plane; ghost += adjacent(final) - adjacent(launch start)
        R *pp = gp + o;
        if (top) {
#pragma unroll
            for (int k = 0; k < TJ; k++) pp[-LD + k] += PSCR(0, k) - pp[k];
        }
        if (bot) {
#pragma unroll
            for (int k = 0; k < TJ; k++) pp[TI * LD + k] += PSCR(TI - 1, k) - pp[(TI - 1) * LD + k];
        }
        if (lef) {
#pragma unroll
            for (int r = 0; r < TI; r++) pp[r * LD - 1] += PSCR(r, 0) - pp[r * LD];
        }
        if (rig) {
#pragma unroll
            for (int r = 0; r < TI; r++) pp[r * LD + TJ] += PSCR(r, TJ - 1) - pp[r * LD + TJ - 1];
        }
        TILE_LOOP { pp[r * LD + k] = PSCR(r, k); }
    }
    if (tid == 0) { a.stp[b] = stp; if (a.status) a.status[b] = status; }
    if (DBG && dbg) { for (int n = 0; n < (DBG ? 8 : 1); n++) a.dbg[n] += (unsigned long long)tph[n]; }
#undef PHASE
#undef TILE_LOOP
#undef PSCR
#undef UU
#undef VV
#undef SS
}
