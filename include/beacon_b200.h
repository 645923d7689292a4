/*
 * beacon_b200.h — C-ABI of the B200-native batched env dynamics (libbeacon_b200.so).
 *
 * Drop-in boundary for the hot path of jviquerat/beacon: the per-environment solver step
 * behind env.step()/env.reset() (SURVEY.md §8b).  The reference has no FFI layer — its
 * boundary is the gym.Env duck type — so the entry points below are what a ctypes/cffi
 * binding inside the reference's env classes would call in place of `self.solve(...)`,
 * `self.get_obs()`, `self.get_rwd()` (see INTEGRATION.md).  Reference sites replaced:
 *
 *   beacon_shkadov_create   shkadov/shkadov.py:20-110   (__init__: derived ints, load())
 *   beacon_burgers_create   burgers/burgers.py:21-65
 *   beacon_sloshing_create  sloshing/sloshing.py:19-86
 *   beacon_lorenz_create    lorenz/lorenz.py:22-57
 *   beacon_vortex_create    vortex/vortex.py:21-76
 *   beacon_rayleigh_create  rayleigh/rayleigh.py:20-86
 *   beacon_mixing_create    mixing/mixing.py:21-70
 *   beacon_env_reset        <env>.reset()  (shkadov.py:113-151, rayleigh.py:89-128, ...)
 *   beacon_env_step         <env>.step()   = solve() + get_obs() + get_rwd() + done/trunc
 *                           (shkadov.py:161-264, rayleigh.py:138-275, mixing.py:114-264,
 *                            burgers.py:98-166, sloshing.py:141-244, lorenz.py:98-172,
 *                            vortex.py:125-208)
 *   beacon_env_get_state / set_state   the public numpy attributes (env.h, env.q, env.u ...)
 *
 * Conventions
 *   - plain C: pointers + sizes, no exceptions cross the boundary; every call returns 0 on
 *     success or a negative beacon_error, and beacon_last_error() gives the message
 *     (thread-local).
 *   - unless a function name ends in _host, all data pointers are DEVICE pointers owned by the
 *     caller (e.g. torch tensors); calls are asynchronous on `stream`.
 *   - a handle owns the persistent device state of `batch` independent environments;
 *     not thread-safe per handle, re-entrant across handles.
 *   - `dtype` selects the arithmetic type of the whole path (state, actions, obs, rewards).
 *   - all derived integers (lattice indices, sub-step counts) are computed by the host with the
 *     reference's own expressions and passed in the params structs: probe indices and actuator
 *     masks are bit-exact by construction.
 */
#ifndef BEACON_B200_H
#define BEACON_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define BEACON_API
#else
#define BEACON_API __attribute__((visibility("default")))
#endif

typedef struct beacon_env beacon_env;          /* opaque handle */
typedef struct CUstream_st *beacon_stream_t;   /* == cudaStream_t */

enum beacon_dtype { BEACON_F64 = 0, BEACON_F32 = 1 };

enum beacon_error {
    BEACON_OK = 0,
    BEACON_ERR_INVALID = -1,    /* bad argument */
    BEACON_ERR_CUDA = -2,       /* CUDA runtime error (message has the cudaError string) */
    BEACON_ERR_UNSUPPORTED = -3 /* valid request the kernels do not cover (message says why) */
};

/* per-env status bits written by step/reset (reference: print("Blowup") shkadov.py:177,
 * exit(1) rayleigh.py:221-224; NaN never trips the reference guards) */
enum beacon_status {
    BEACON_STATUS_BLOWUP = 1,
    BEACON_STATUS_POISSON_OVERFLOW = 2,
    BEACON_STATUS_NONFINITE = 4
};

enum beacon_env_kind {
    BEACON_SHKADOV = 0, BEACON_BURGERS = 1, BEACON_SLOSHING = 2, BEACON_LORENZ = 3,
    BEACON_VORTEX = 4, BEACON_RAYLEIGH = 5, BEACON_MIXING = 6
};

/* Common creation options. */
typedef struct {
    int32_t batch;            /* number of environments held by the handle */
    int32_t device;           /* CUDA device ordinal */
    int32_t dtype;            /* beacon_dtype */
    int32_t reserved;
    uint64_t seed;            /* Philox key for on-device inlet noise */
    int64_t env_index_base;   /* global index of env 0 (multi-GPU shards: results independent of sharding) */
} beacon_common;

/* shkadov / shkadov_separable: shkadov.py:32-76 (ints by int(x/dx) truncation, host-computed) */
typedef struct {
    int32_t nx, ndt_act, n_act, n_interp, n_jets;
    int32_t jet_pos, jet_hw, jet_space;       /* lattice units */
    int32_t l_obs, n_obs, obs_stride, l_rwd;  /* obs: q[s:s+l_obs:obs_stride][:n_obs] per jet */
    int32_t per_jet_rwd;                      /* 1: rwd is [.., n_jets] (separable, shkadov.py:469-481) */
    int32_t reserved;
    double dx, dt, delta, eps, jet_amp, sigma;
    double blow_lo, blow_hi, blowup_rwd;      /* -5 h_max, 5 h_max, -1 (shkadov.py:176-180) */
} beacon_shkadov_params;

/* burgers.py:25-43 */
typedef struct {
    int32_t nx, ndt_act, n_act, ctrl_pos, n_obs_pts, reserved;
    double dx, dt, amp, sigma, u_target;
} beacon_burgers_params;

/* sloshing.py:23-50 */
typedef struct {
    int32_t nx, ndt_act, n_act, n_interp, obs_smpl, n_obs;
    double dx, dt, g, amp, alpha;
    double blow_lo, blow_hi;                  /* -5 h_max, 2 h_max (sloshing.py:152) */
} beacon_sloshing_params;

/* lorenz.py:26-41 */
typedef struct {
    int32_t ndt_act, n_act;
    double dt, sigma, rho, beta;
    double x0[3];                             /* (10,10,10) lorenz.py:73-75 */
    double forcing[3];                        /* actions table {-1,0,1} lorenz.py:50 */
} beacon_lorenz_params;

/* vortex.py:25-61 */
typedef struct {
    int32_t ndt_act, n_act;
    double dt, lmbda_re, lmbda_cx, mu_re, mu_cx, alpha_re, alpha_cx, ire, omega_s, omega_f,
        domega, gamma, beta_m, weight, mod_min, mod_max, phase_min, phase_max;
    double x0[4];                             /* vortex.py:92-95 */
} beacon_vortex_params;

/* rayleigh.py:24-56 and mixing.py:25-49 share the MAC-grid projection solver */
typedef struct {
    int32_t nx, ny, ndt_act, n_act;
    int32_t n_sgts, nx_sgts;                  /* rayleigh bottom-plate segments (0 for mixing) */
    int32_t nx_obs_pts, ny_obs_pts, n_obs_steps, nx_obs, ny_obs;
    int32_t itmax;                            /* 300000 */
    double dx, dy, dt;
    double pr, ra, Tc, Th, C;                 /* rayleigh */
    double re, pe, u_max, ref_c;              /* mixing; ref_c = side^2/(L*H)*C0 (mixing.py:261) */
    double tol;                               /* 1e-8 rayleigh.py:414 / 1e-4 mixing.py:423 */
    /* How many SMs one environment may occupy.  0 or 1: one CTA per env (grids up to ~100x100
     * cells).  2..8: one thread-block cluster of exactly that many CTAs per env, each owning a slab of
     * >= 4 rows of i, on any grid whose slab fits (DESIGN.md 3.6); anything else is rejected at create. */
    int32_t ctas_per_env;
} beacon_mac_params;

/* What a handle looks like from outside. */
typedef struct {
    int32_t kind, batch, dtype, device;
    int32_t n_obs;          /* observation length per env */
    int32_t act_dim;        /* action entries per env (1 for Discrete) */
    int32_t act_is_int;     /* 1: actions are int32 [batch]; 0: real [batch, act_dim] */
    int32_t rwd_dim;        /* 1, or n_jets when per-jet rewards were requested (shkadov) */
    int32_t n_act;          /* episode horizon */
    int32_t noise_dim;      /* noise entries per env per action accepted by step (0: none) */
    int32_t n_fields;       /* number of named state fields */
    int32_t reserved;
} beacon_env_info_t;

/* ---- creation ----------------------------------------------------------------------- */
/* h_init/q_init etc. are HOST float64 arrays (the parsed init_field.dat columns); they are
 * converted to `dtype` and kept on the device as the reset state. */
BEACON_API int beacon_shkadov_create(const beacon_common *c, const beacon_shkadov_params *p,
                                     const double *h_init, const double *q_init, beacon_env **out);
BEACON_API int beacon_burgers_create(const beacon_common *c, const beacon_burgers_params *p, beacon_env **out);
BEACON_API int beacon_sloshing_create(const beacon_common *c, const beacon_sloshing_params *p,
                                      const double *h_init, const double *q_init, beacon_env **out);
BEACON_API int beacon_lorenz_create(const beacon_common *c, const beacon_lorenz_params *p, beacon_env **out);
BEACON_API int beacon_vortex_create(const beacon_common *c, const beacon_vortex_params *p, beacon_env **out);
/* rayleigh: u/v/p/T_init are HOST [(nx+2),(ny+2)] float64 (rayleigh.py:356-362) */
BEACON_API int beacon_rayleigh_create(const beacon_common *c, const beacon_mac_params *p, const double *u_init,
                                      const double *v_init, const double *p_init, const double *T_init,
                                      beacon_env **out);
/* mixing: C_init is the HOST analytic patch field (mixing.py:90-94) */
BEACON_API int beacon_mixing_create(const beacon_common *c, const beacon_mac_params *p, const double *C_init,
                                    beacon_env **out);
BEACON_API void beacon_env_destroy(beacon_env *env);
BEACON_API int beacon_env_info(const beacon_env *env, beacon_env_info_t *info);

/* ---- the hot path ------------------------------------------------------------------- */
/*
 * reset: envs with mask[b] != 0 (all when mask == NULL) return to the reset state.
 *   n_warm  (shkadov only, nullable) int32 [batch]: number of zero-action warm steps to run
 *           after loading the init state (the reference draws random.randint(0,400),
 *           shkadov.py:120); `noise` (nullable) real [max_warm, batch, noise_dim] supplies the
 *           inlet noise of those steps, otherwise on-device Philox.
 *   obs     real [batch, n_obs] (rows of unmasked envs untouched).
 */
BEACON_API int beacon_env_reset(beacon_env *env, const uint8_t *mask, const int32_t *n_warm, const void *noise,
                                int32_t max_warm, void *obs, beacon_stream_t stream);

/*
 * step: advances every env by n_fused consecutive actions in ONE launch (n_fused = 1 is the
 * gym step).  Shapes (K = n_fused, B = batch):
 *   actions  real [K, B, act_dim] or int32 [K, B]
 *   noise    nullable real [K, B, noise_dim]: shkadov inlet noise per sub-step (noise_dim =
 *            ndt_act, shkadov.py:204), burgers per action (noise_dim = 1, burgers.py:127);
 *            NULL -> on-device Philox U(-sigma, sigma)
 *   obs      real [K, B, n_obs];  rwd real [K, B, rwd_dim]
 *   done, trunc  uint8 [K, B];   status int32 [B] (OR-ed beacon_status bits)
 *   iters    nullable int64 [K, B]: sum of Poisson sweeps of the action (rayleigh/mixing)
 */
BEACON_API int beacon_env_step(beacon_env *env, const void *actions, const void *noise, void *obs, void *rwd,
                               uint8_t *done, uint8_t *trunc, int32_t *status, int64_t *iters,
                               int32_t n_fused, beacon_stream_t stream);

/* Same as beacon_env_step with n_fused = 1 and HOST buffers; returns after the stream has drained,
 * with obs/rwd/done/trunc/status in the caller's buffers.  Pageable buffers are staged (actions and
 * noise copied to the device, results copied back).  Page-locked buffers (cudaHostAlloc /
 * cudaHostRegister, e.g. torch pinned tensors) are read and written by the step kernel itself over
 * PCIe — every env's rows move when its CTA starts / finishes, overlapped with the compute of the
 * others (thread-per-env lorenz / vortex always stage).  BEACON_STEP_HOST_STAGED=1 forces staging. */
BEACON_API int beacon_env_step_host(beacon_env *env, const void *actions, const void *noise, void *obs, void *rwd,
                                    uint8_t *done, uint8_t *trunc, int32_t *status, beacon_stream_t stream);

/* ---- state access (parity from identical states, checkpointing) --------------------- */
/* Field names follow the reference attributes: shkadov "h","q","rhsh","rhsq","u","up","stp";
 * burgers "u","up","upp","a","stp"; sloshing "h","q","rhsh","rhsq","u","up","stp";
 * lorenz/vortex "x","fx","stp" (+ vortex "t","y"); rayleigh "u","v","p","T","a","obs","stp";
 * mixing "u","v","p","C","obs","stp".  Real fields are `dtype`, "stp" is int32; shkadov and burgers
 * also expose "draws": the uint64 Philox draw counter of the inlet noise as two int32 words, so that a
 * state dump restores the noise stream too.
 * beacon_env_field reports the per-env element count and whether the field is integer. */
BEACON_API int beacon_env_field(const beacon_env *env, int32_t index, const char **name, int64_t *count,
                                int32_t *is_int);
BEACON_API int beacon_env_get_state(beacon_env *env, const char *field, void *buf, beacon_stream_t stream);
BEACON_API int beacon_env_set_state(beacon_env *env, const char *field, const void *buf, beacon_stream_t stream);

/* ---- per-env physical parameters (rayleigh, mixing) -------------------------------------
 * Each env of a batch may run at its own Rayleigh (rayleigh "ra"), Reynolds and Péclet number (mixing
 * "re", "pe"); a handle is created with one value for all of them.  values: HOST float64 [batch], each
 * finite and > 0.  A set is stream-ordered with the launches: it takes effect at the next reset or step
 * on `stream`.  From the first set on, the handle's launches use the per-env kernel instances (a
 * handle that is never set runs exactly as before).  mixing "re" also sets the lid / wall speed
 * u_max = re * 0.01 / L (L = nx dx), as the constructor does.  An unknown name, a name of the other
 * environment, any other environment or a bad value return BEACON_ERR_INVALID and change nothing.
 * get_physics returns the current values (the handle's scalar for every env before the first set)
 * after the stream has drained. */
BEACON_API int beacon_env_set_physics(beacon_env *env, const char *name, const double *values, beacon_stream_t stream);
BEACON_API int beacon_env_get_physics(beacon_env *env, const char *name, double *values, beacon_stream_t stream);

/* ---- learner-rank buffers in peer memory (multi-GPU, one process per GPU) -------------
 * The only exchange of the path is the gather of observations / rewards / flags to the learner
 * rank (SURVEY.md §8e; reference call sites whose outputs travel: get_obs / get_rwd,
 * shkadov.py:239-264, rayleigh.py:243-275).  Instead of a collective after the step, the learner
 * exports ONE device allocation over CUDA IPC, every other process maps it, and beacon_env_step is
 * given obs / rwd / done / trunc pointers INSIDE that mapping: each env's CTA then writes its rows
 * straight into the learner GPU's HBM over NVLink when it finishes (the same mechanism as the
 * zero-copy host path of beacon_env_step_host), overlapped with the compute of the other envs.
 * Completion is the caller's business (a stream-ordered barrier after the step).
 *   beacon_peer_alloc   cudaMalloc'ed, zero-filled buffer on `device` (IPC needs an allocation base)
 *   beacon_peer_export  64-byte cudaIpcMemHandle_t of a beacon_peer_alloc'ed buffer
 *   beacon_peer_open    map an exported buffer into this process for use from `device`
 *   beacon_peer_close   unmap (importing processes);  beacon_peer_free: release (exporting process)
 */
#define BEACON_PEER_HANDLE_BYTES 64
BEACON_API int beacon_peer_alloc(int32_t device, uint64_t bytes, void **ptr);
BEACON_API int beacon_peer_export(void *ptr, uint8_t handle[BEACON_PEER_HANDLE_BYTES]);
BEACON_API int beacon_peer_open(const uint8_t handle[BEACON_PEER_HANDLE_BYTES], int32_t device, void **ptr);
BEACON_API int beacon_peer_close(void *ptr);
BEACON_API int beacon_peer_free(int32_t device, void *ptr);

/* number of kernel launches issued by this handle so far (bench.py's gpu_launches claim) */
BEACON_API int64_t beacon_env_launch_count(const beacon_env *env);

BEACON_API const char *beacon_last_error(void);
BEACON_API const char *beacon_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BEACON_B200_H */
