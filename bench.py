#!/usr/bin/env python
"""bench.py — env-actions/sec of the batched env dynamics on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--env shkadov] [--batch B] [--extras all|none|a,b] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the UNMODIFIED reference (numpy + numba) on the host cores

A "step" is one gym step of the whole batch (= batch env-actions) through the C-ABI with all solver
sub-steps fused in one kernel launch.  The headline (`value`, `e2e`, `roofline`) is BASELINE.json
configs[1]: shkadov-v0, 10 jets, 1024 envs per GPU (weak scaling: every rank steps its own envs).
BASELINE.json's metric names TWO workloads and a >= 4096-env target, so the same JSON line carries, under
`workloads`, the other BASELINE configs measured by the same code in the same run: rayleigh-v0 x 4096
(configs[4]), shkadov-v0 x 4096, shkadov_separable-v0 41 jets x 512 per GPU (configs[2]), mixing-v0 x 1024
(configs[3]) and the single-env burgers-v0 episode (configs[0]).  Prints ONE JSON line (rank 0).

Roofline: the kernels keep every solver sub-step on chip, so HBM sees one state load + store per action
(F-model, a few % of peak) and the S-model "algorithmic bytes" of SURVEY.md §8d are not compulsory traffic
(reported as `s_model_effective`, may exceed 1).  `roofline.frac` is the fraction of the unit that really
binds — the fp64 pipe (shkadov) or the shared-memory pipe (rayleigh, mixing) — computed IN THE RUN from
the static SASS census of the shipped kernels (beacon_b200/lib/sass_census.json, tools/sass_census.py)
x the trip counts of this run (sub-steps; Jacobi sweeps counted by the kernel itself) / measured seconds /
(unit throughput x sampled SM clock).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (env, ctor kwargs, default envs per GPU, default timed steps, description)
    "shkadov": ("shkadov", dict(n_jets=10), 1024, 400, "shkadov-v0 n_jets=10 nx=1350, 50 sub-steps/action (BASELINE configs[1])"),
    "shkadov_b4096": ("shkadov", dict(n_jets=10), 4096, 100, "shkadov-v0 n_jets=10 nx=1350, 4096 envs per GPU"),
    "shkadov_separable": ("shkadov", dict(n_jets=41, per_jet_rwd=True), 512, 100, "shkadov_separable-v0 n_jets=41 nx=2900 (BASELINE configs[2]: 4096 envs over 8 GPUs)"),
    "rayleigh": ("rayleigh", dict(), 4096, 10, "rayleigh-v0 50x50, 200 sub-steps/action, Jacobi Poisson (BASELINE configs[4])"),
    "mixing": ("mixing", dict(), 1024, 3, "mixing-v0 100x100, 250 sub-steps/action, Jacobi Poisson (BASELINE configs[3])"),
    "burgers": ("burgers", dict(), 1, 200, "burgers-v0 nx=500, 62 sub-steps/action, single env (BASELINE configs[0])"),
    "sloshing": ("sloshing", dict(), 4096, 200, "sloshing-v0 nx=200, 50 sub-steps/action"),
    "lorenz": ("lorenz", dict(), 65536, 500, "lorenz-v0 LSRK4"),
}
DEFAULT_EXTRAS = ("rayleigh", "shkadov_b4096", "shkadov_separable", "mixing", "burgers")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of the headline workload; the other batched workloads time at most this many "
                         "(the burgers and VectorEnv episodes keep their episode lengths)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--env", default="shkadov", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="envs per GPU of the headline workload")
    ap.add_argument("--extras", default=None, help="'all' (default with the default --env), 'none', or a comma list of workloads")
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="budget of each cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload returned (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path: it needs --impl b200")
    return args


DUMP_LIMIT = 64 * 1024 * 1024


def dump_outputs(path, obs, rwd, done, trunc):
    """obs / reward / done / truncated of one batched step as float64 (flags as float32) .npy files.  A batch whose
    arrays exceed DUMP_LIMIT is written as a fixed sample of env rows, listed in sample_rows.npy."""
    arrs = {"obs": obs.double(), "reward": rwd.double(), "done": done.float(), "truncated": trunc.float()}
    arrs = {k: a.cpu().numpy() for k, a in arrs.items()}
    B = obs.shape[0]
    row_bytes = sum(a[0].nbytes for a in arrs.values())
    os.makedirs(path, exist_ok=True)
    if B * row_bytes > DUMP_LIMIT:
        n = (DUMP_LIMIT - 4096) // (row_bytes + 8)                  # 4096: room for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        np.save(os.path.join(path, "sample_rows.npy"), rows.astype(np.float64))
        arrs = {k: a[rows] for k, a in arrs.items()}
    for k, a in arrs.items():
        np.save(os.path.join(path, k + ".npy"), a)


# --------------------------------------------------------------------------------------------
# models: algorithmic bytes (SURVEY.md §8d S-model / F-model) and the on-chip units that bind
# --------------------------------------------------------------------------------------------
def s_model_bytes(wl, d, sweeps_per_action=0.0):
    """every live field read + written once per solver sub-step / Jacobi sweep (unfused stencil code), fp64"""
    if wl.startswith("shkadov"):
        return 3200.0 * d["nx"]
    if wl == "burgers":
        return 3 * d["nx"] * 8.0 * d["ndt_act"]
    if wl == "sloshing":
        return 8 * (d["nx"] + 2) * 8.0 * d["ndt_act"]
    if wl == "rayleigh":
        return (21 * d["ndt_act"] + 3 * sweeps_per_action) * (d["nx"] + 2) * (d["ny"] + 2) * 8.0
    if wl == "mixing":
        return (20 * d["ndt_act"] + 3 * sweeps_per_action) * (d["nx"] + 2) * (d["ny"] + 2) * 8.0
    return 112.0


def f_model_bytes(wl, d, n_obs, rwd_dim, act_dim):
    """compulsory DRAM traffic of the fused kernels: state in + out once per launch, action in, obs / reward out"""
    io = 8.0 * (n_obs + rwd_dim + act_dim) + 6
    if wl.startswith("shkadov"):
        return 64.0 * d["nx"] + io
    if wl == "burgers":
        return 48.0 * d["nx"] + io
    if wl == "sloshing":
        return 64.0 * (d["nx"] + 2) + io
    if wl in ("rayleigh", "mixing"):
        return 8 * (d["nx"] + 2) * (d["ny"] + 2) * 8.0 + io
    return 112.0


def load_census():
    p = os.path.join(ROOT, "beacon_b200", "lib", "sass_census.json")
    return json.load(open(p)) if os.path.exists(p) else None


def unit_model(wl, d, sweeps_per_action, census):
    """(fp64 warp-instructions, shared-memory wavefronts) per env-action from the static SASS census x the
    trip counts of this run, and a description of how they were put together."""
    if census is None:
        return None
    if wl.startswith("shkadov"):
        nx = d["nx"]
        for C, T, tag in ((6, 256, "shkadov_6_256_2"), (10, 192, "shkadov_10_192_2"), (6, 512, "shkadov_6_512_1")):
            if C * T >= nx + (C - nx % C) % C:
                break
        c = census[tag]
        off = (C - nx % C) % C
        body = c["substep_unrolled2"]["per_substep"] if (off <= 1 and c["substep_unrolled2"]) else \
            {k: v for k, v in c["substep_bodies"][0].items() if isinstance(v, (int, float))}
        warps = -(-(nx + off) // (32 * C))                     # warps holding lattice points (the others only keep the barrier count)
        n = warps * d["ndt_act"]
        return {"fp64": body["fp64"] * n, "smem": (body.get("smem_wavefronts", 0) + body.get("smem_wavefronts_pred", 0)) * n,
                "how": f"{tag}: {body['fp64']:.0f} fp64 warp-instr per sub-step x {warps} warps x {d['ndt_act']} sub-steps"}
    if wl in ("rayleigh", "mixing"):
        c = census["rayleigh_reg" if wl == "rayleigh" else "mixing_big"]
        warps = 8 if wl == "rayleigh" else 16
        sw, ot, wf = c["per_sweep"], c["substep_other"], c["wavefront_loop"]
        nd = d["ndt_act"]
        trips = (13 if wl == "rayleigh" else 2 * 21) * nd      # wavefront: 6 columns per trip, one warp (mixing: two row passes of 126 steps)
        fp64 = warps * (sweeps_per_action * sw["fp64"] + nd * ot["fp64"]) + trips * wf["fp64"]
        # sweep loop: predicated wavefronts count too (the tile stores of the big kernel are predicated on "thread owns a
        # tile", true for 500 of 512 threads); elsewhere predicated = ghost-cell copies of a few boundary threads, left out
        sw_smem = sw.get("smem_wavefronts", 0) + sw.get("smem_wavefronts_pred", 0)
        smem = warps * (sweeps_per_action * sw_smem + nd * ot.get("smem_wavefronts", 0)) + trips * wf.get("smem_wavefronts", 0)
        return {"fp64": fp64, "smem": smem,
                "how": f"{warps} warps x ({sweeps_per_action:.0f} sweeps x {sw['fp64']:.0f} fp64 / {sw_smem:.0f} smem wavefronts per sweep + "
                       f"{nd} sub-steps x {ot['fp64']} / {ot.get('smem_wavefronts', 0)}) + one-warp transport wavefront; conflict-free wavefronts, counted "
                       f"sweeps only (speculative ones excluded): a lower bound"}
    return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (oracle/ref_bench.py) and the oracle C port (all host threads)
# --------------------------------------------------------------------------------------------
class CpuArm:
    """Steps `B` oracle envs per call with one env per host thread (oracle/beacon_oracle.c)."""

    def __init__(self, env_name, kwargs, B, seed=0):
        import ctypes as C
        from oracle import beacon_oracle as bo
        self.C, self.bo, self.B, self.name = C, bo, B, env_name
        self.lib = bo.lib()
        self.cores = int(self.lib.orc_num_threads())
        self.rng = np.random.default_rng(seed)
        kw = {k: v for k, v in kwargs.items() if k != "per_jet_rwd"}
        self.proto = bo.ENVS[env_name](**kw)
        e = self.proto
        e.reset()
        rep = lambda a: np.ascontiguousarray(np.broadcast_to(a, (B,) + a.shape)).copy()
        if env_name == "shkadov":
            self.st = [rep(e.h), rep(e.q), rep(e.rhsh), rep(e.rhsq), np.zeros((B, e.n_jets)), np.zeros((B, e.n_jets))]
            self.obs, self.rwd, self.blow = np.zeros((B, e.n_jets * e.n_obs)), np.zeros(B), np.zeros(B, dtype=np.uint8)
        elif env_name == "burgers":
            self.st = [rep(e.u), rep(e.up), rep(e.upp)]
            self.obs, self.rwd = np.zeros((B, 5)), np.zeros(B)
        elif env_name == "sloshing":
            self.st = [rep(e.h), rep(e.q), rep(e.rhsh), rep(e.rhsq), np.zeros(B), np.zeros(B)]
            self.obs, self.rwd = np.zeros((B, e.n_obs)), np.zeros(B)
        elif env_name == "lorenz":
            self.st = [rep(e.x), rep(e.fx)]
            self.obs, self.rwd = np.zeros((B, 6)), np.zeros(B)
        else:
            scal = e.T if env_name == "rayleigh" else e.C
            self.st = [rep(e.u), rep(e.v), rep(e.p), rep(scal)]
            self.iters = np.zeros(B, dtype=np.int64)

    def step(self):
        C, e, B, L, rng = self.C, self.proto, self.B, self.lib, self.rng
        P = lambda a: a.ctypes.data_as(C.c_void_p)
        base = self.name
        if base == "shkadov":
            acts, noise = rng.uniform(-1, 1, (B, e.n_jets)), rng.uniform(-e.sigma, e.sigma, (B, e.ndt_act))
            L.orc_shkadov_step_batch(C.byref(e.cfg), B, *[P(a) for a in self.st], P(acts), P(noise), P(self.obs), P(self.rwd), P(self.blow))
        elif base == "burgers":
            acts, noise = rng.uniform(-1, 1, B), rng.uniform(-e.sigma, e.sigma, B)
            L.orc_burgers_step_batch(B, e.nx, C.c_double(e.dx), C.c_double(e.dt), e.ndt_act, e.ctrl_pos, C.c_double(e.amp),
                                     C.c_double(e.u_target), 5, *[P(a) for a in self.st], P(acts), P(noise), P(self.obs), P(self.rwd))
        elif base == "sloshing":
            acts = rng.uniform(-1, 1, B)
            L.orc_sloshing_step_batch(B, e.nx, C.c_double(e.dx), C.c_double(e.dt), e.ndt_act, e.n_interp, C.c_double(e.g),
                                      C.c_double(e.amp), C.c_double(e.alpha), *[P(a) for a in self.st], P(acts), P(self.obs), P(self.rwd))
        elif base == "lorenz":
            acts = rng.integers(0, 3, B).astype(np.int32)
            L.orc_lorenz_step_batch(B, C.c_double(e.sigma), C.c_double(e.rho), C.c_double(e.beta), C.c_double(e.dt), e.ndt_act,
                                    *[P(a) for a in self.st], P(acts), P(self.obs), P(self.rwd))
        elif base == "rayleigh":
            seg = np.stack([e.Th + e.condition(rng.uniform(-1, 1, e.n_sgts)) for _ in range(B)])
            L.orc_mac_solve_batch(C.byref(e.cfg), B, *[P(a) for a in self.st], C.c_double(e.Tc), P(seg), e.n_sgts, e.nx_sgts, None, P(self.iters))
        else:
            wall = np.array([e.get_control(int(a)) for a in rng.integers(0, 4, B)], dtype=np.float64)
            L.orc_mac_solve_batch(C.byref(e.cfg), B, *[P(a) for a in self.st], C.c_double(0.0), None, 0, 0, P(wall), P(self.iters))


def port_sample(wl, seconds):
    """Times the oracle C port on a bounded sample: a few envs per host thread x a few actions."""
    env_name, kwargs = WORKLOADS[wl][0], WORKLOADS[wl][1]
    cores = CpuArm(env_name, kwargs, B=1).cores
    per_env = {"shkadov": 8, "rayleigh": 1, "mixing": 1, "burgers": 64, "sloshing": 64, "lorenz": 65536}[env_name]
    if kwargs.get("n_jets", 0) > 20:
        per_env = 4
    B = 1 if wl == "burgers" else cores * per_env
    arm = CpuArm(env_name, kwargs, B=B)
    arm.step()                                   # warm-up (page faults, thread pool)
    n, t0 = 0, time.perf_counter()
    while True:
        arm.step()
        n += 1
        el = time.perf_counter() - t0
        if el >= seconds or (env_name == "mixing" and n >= 2):
            break
    return {"value": B * n / el, "unit": "env-actions/s", "cores": cores if B > 1 else 1, "kind": "port",
            "sample": f"{B} envs x {n} actions of the same workload, oracle C port (oracle/beacon_oracle.c), {el:.1f} s"}


def cpu_baseline(wl, seconds):
    """The unmodified reference when its modules are reachable (kind "reference", with the C port beside it as
    `port_value`), else the C port (kind "port")."""
    env_name, kwargs = WORKLOADS[wl][0], WORKLOADS[wl][1]
    port = port_sample(wl, min(seconds, 6.0))
    try:
        from oracle import ref_bench
        if ref_bench.available():
            ref = ref_bench.time_reference(env_name, kwargs, seconds, procs=1 if wl == "burgers" else None)
            ref.update(port_value=port["value"], port_cores=port["cores"], port_sample=port["sample"])
            return ref
    except Exception as e:
        port["reference_error"] = repr(e)
    return port


# --------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference arm: the UNMODIFIED reference env classes (numpy + numba) on the host cores, one env per
    process, P = os.cpu_count() processes; a step = every process advances `chunk` actions (a bounded sample of
    the workload: P x chunk env-actions instead of envs_per_gpu).  Rank 0 only."""
    if rank != 0:
        return
    from oracle import ref_bench
    wl = args.env
    env_name, kwargs, defB, defK, desc = WORKLOADS[wl]
    K = args.steps or 10
    budget = 15.0

    def one(wl_):
        en, kw = WORKLOADS[wl_][0], WORKLOADS[wl_][1]
        if ref_bench.available():
            try:
                return ref_bench.time_reference(en, kw, budget, procs=1 if wl_ == "burgers" else None)
            except Exception as e:
                r = port_sample(wl_, budget)
                r["reference_error"] = repr(e)
                return r
        return port_sample(wl_, budget)

    t0 = time.perf_counter()
    main_ = one(wl)
    val = main_["value"]
    P = main_["cores"]
    chunk = max(1, int(round(val * budget / (K * P))))
    line = {"impl": "reference", "metric": "env-actions/sec", "value": val, "unit": "env-actions/s", "n_gpus": args.gpus,
            "steps": K, "warmup": args.warmup, "ms_per_step": 1e3 * P * chunk / val, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[wl][4], "env": wl, "sample_envs_per_step": P, "sample_actions_per_env_per_step": chunk,
                       "note": "reference arm = the unmodified reference env classes (numpy + numba) on the host cores, one env per process; "
                               f"the processes step freely for ~{budget:.0f} s after one untimed (JIT) step; expressed as {K} steps, each a bounded sample of "
                               f"the workload ({P} envs x {chunk} actions)"},
            "cpu_baseline": main_,
            "e2e": {"value": val, "unit": "env-actions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if wl == "shkadov" and args.extras != "none":
        extra = {}
        for w2 in ("rayleigh",):
            r = one(w2)
            extra[w2] = {"value": r["value"], "unit": "env-actions/s", "cpu_baseline": r, "config": {"workload": WORKLOADS[w2][4]}}
        line["workloads"] = extra
    try:
        line["port"] = {wl: port_sample(wl, 6.0)}
    except Exception as e:
        line["port"] = {"error": repr(e)}
    line["wall_seconds"] = time.perf_counter() - t0
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
class Ctx:
    pass


def run_workload(wl, B, K, W, cx, args, headline):
    """Times one workload on this rank's GPU; returns the per-workload dict (rank 0) or None."""
    torch, dist = cx.torch, cx.dist
    from beacon_b200 import BatchedEnv
    env_name, kwargs, _, _, desc = WORKLOADS[wl]
    rank, world, dev = cx.rank, cx.world, cx.dev
    env = BatchedEnv(env_name, batch=B, device=cx.local, seed=1234, env_index_base=rank * B, **kwargs)
    d = env.cfg.d
    g = torch.Generator(device=dev)
    g.manual_seed(1000 + rank)
    n_tot = K + W
    if env.act_is_int:
        hi = 4 if env_name == "mixing" else 3
        actions = torch.randint(0, hi, (n_tot, B), generator=g, device=dev, dtype=torch.int32)
    else:
        actions = torch.rand(n_tot, B, env.act_dim, generator=g, device=dev, dtype=torch.float64) * 2 - 1
    reset = None
    if env_name == "shkadov":
        nw = torch.randint(0, 401, (B,), generator=g, device=dev, dtype=torch.int32)
        env.reset(n_warm=torch.zeros_like(nw), max_warm=0)          # first launch (module load) is not the reset cost
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.reset(n_warm=nw, max_warm=400)
        e1.record()
        torch.cuda.synchronize()
        rs = e0.elapsed_time(e1) * 1e-3
        n_warm_total = int(nw.sum().item())
        reset = {"seconds": rs, "warm_env_actions": n_warm_total, "env_actions_per_s": n_warm_total / rs,
                 "note": "reset with U{0..400} zero-action warm steps per env (shkadov.py:118-123), one launch, longest envs first"}
    else:
        env.reset()
    want_iters = env_name in ("rayleigh", "mixing")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for k in range(W):
        env.step(actions[k], want_iters=want_iters)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    it_sum = torch.zeros((), dtype=torch.int64, device=dev)
    launches0 = env.launches
    with ClockSampler(cx.local) as clk:
        barrier()
        t_wall0 = time.perf_counter()
        for k in range(K):
            cx.flush.zero_()                                 # L2 flush between timed iterations (untimed)
            ev[k][0].record()
            last = env.step(actions[W + k], want_iters=want_iters)
            ev[k][1].record()
            if want_iters:
                it_sum += env.last_iters.sum()
        barrier()
        launches = env.launches - launches0
        # clocks: keep the same kernel running (untimed) until the sampler has seen >= 0.6 s of this load
        k = 0
        while time.perf_counter() - t_wall0 < 0.6:
            env.step(actions[W + (k % K)], want_iters=False)
            k += 1
            if k % 8 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
    if headline and args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = float(sum(ms))
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * B * K / (total_ms_max * 1e-3)
    status_bad = int((env.status != 0).sum().item())
    sweeps = int(it_sum.item()) if want_iters else 0

    # ---- end to end through the public host-buffer API (H2D + step + D2H inside the timed region) ----
    e2e = None
    if not args.no_e2e:
        host_act = actions[:K + W].cpu().pin_memory()
        out = env.alloc_host_outputs()
        for k in range(W):
            env.step_host(host_act[k], out=out)
        barrier()
        t0 = time.perf_counter()
        for k in range(K):
            env.step_host(host_act[W + k], out=out)
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        tt = torch.tensor([el], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        rb = 8
        e2e = {"value": world * B * K / float(tt.item()), "unit": "env-actions/s",
               "h2d_bytes_per_step": int(host_act[0].numel() * host_act[0].element_size()),
               "d2h_bytes_per_step": int(B * env.n_obs * rb + B * env.rwd_dim * rb + 2 * B + 4 * B)}

    # ---- the learner-rank gather inside the timed region (N > 1): NCCL after the step vs the fused peer-memory epilogue ----
    gather = None
    if world > 1 and not args.no_gather:
        from beacon_b200 import dist as bd
        from beacon_b200.peer import LearnerBuffer
        N = world * B

        def timed(fn, n):
            barrier()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for k in range(n):
                fn(k)
            b_.record()
            torch.cuda.synchronize()
            tt = torch.tensor([a.elapsed_time(b_)], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()) * 1e-3

        wait_ev = []

        def nccl_step(k):
            obs, rwd, done, trunc = env.step(actions[W + (k % K)])
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            bd.gather_to_learner(obs, N, dst=0)
            bd.gather_to_learner(rwd, N, dst=0)
            bd.gather_to_learner(done.to(torch.uint8), N, dst=0)
            b_.record()
            wait_ev.append((a, b_))

        nccl_step(0); wait_ev.clear()
        t_nccl = timed(nccl_step, K)
        my_wait = sum(a.elapsed_time(b_) for a, b_ in wait_ev) / K
        waits = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(waits, torch.tensor([my_wait], device=dev, dtype=torch.float64))
        lb = LearnerBuffer(env, N, dst=0)

        def peer_step(k):
            lb.step(actions[W + (k % K)])
            lb.fence()

        peer_step(0)
        t_peer = timed(peer_step, K)
        lb.close()
        gather = {"nccl_gather": {"value": N * K / t_nccl, "unit": "env-actions/s",
                                  "gather_ms_per_step_by_rank": [round(float(w.item()), 4) for w in waits],
                                  "what": "step + dist.gather of obs / rwd / done to rank 0 (NCCL) inside the timed region"},
                  "peer_epilogue": {"value": N * K / t_peer, "unit": "env-actions/s",
                                    "what": "step kernel writes each env's obs / rwd / flag rows into the learner GPU's buffer over NVLink "
                                            "(CUDA IPC mapping), then a 4-byte all-reduce as the completion fence"},
                  "bytes_to_learner_per_step": int((world - 1) * B * (env.n_obs * 8 + env.rwd_dim * 8 + 2)),
                  "note": "back-to-back steps, no L2 flush between them (unlike `value`): compare the two gather variants with each other"}

    if rank != 0:
        return None
    clocks = clk.summary()
    spa = sweeps / (B * K) if want_iters else 0.0
    peak_hbm, peak_src = measured_peak()
    avg_launch_s = (total_ms / K) * 1e-3
    sbytes = s_model_bytes(env_name, d, spa)
    fbytes = f_model_bytes(env_name, d, env.n_obs, env.rwd_dim, env.act_dim)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp)).get("shkadov" if wl == "shkadov_b4096" else wl)
        if tj:
            traffic = float(tj["bytes_per_launch"]) * B / float(tj["grid"])
    n_sm = cx.props.multi_processor_count
    clock_hz = 1e6 * (clocks["sm_mhz"] or clocks["sm_max_mhz"] or 1965.0)
    um = unit_model(env_name, d, spa, cx.census)
    roof = {"bound": "hbm", "achieved": sbytes * B / avg_launch_s / 1e9, "peak": peak_hbm, "unit": "GB/s",
            "frac": sbytes * B / avg_launch_s / 1e9 / peak_hbm, "traffic": traffic}
    if um:
        fp64_rate, smem_rate = um["fp64"] * B / avg_launch_s, um["smem"] * B / avg_launch_s
        fp64_peak, smem_peak = n_sm * 4 * 0.5 * clock_hz, n_sm * 1.0 * clock_hz
        fp64_frac, smem_frac = fp64_rate / fp64_peak, smem_rate / smem_peak
        if smem_frac > fp64_frac:
            roof = {"bound": "smem", "achieved": smem_rate / 1e9, "peak": smem_peak / 1e9, "unit": "Gwavefront/s (128 B shared-memory wavefronts)",
                    "frac": smem_frac, "fp64_frac": fp64_frac}
        else:
            roof = {"bound": "fp64", "achieved": fp64_rate / 1e9, "peak": fp64_peak / 1e9, "unit": "Gwarp-inst/s (fp64 pipe, 2 warp-instr/clk/SM)",
                    "frac": fp64_frac, "smem_frac": smem_frac}
        roof.update({"traffic": traffic, "sm_clock_mhz": clock_hz / 1e6, "sms": n_sm, "model": um["how"],
                     "census": "beacon_b200/lib/sass_census.json (static SASS counts, tools/sass_census.py) x trip counts of this run"})
    roof["hbm"] = {"s_model_effective": {"achieved": sbytes * B / avg_launch_s / 1e9, "peak": peak_hbm, "unit": "GB/s",
                                          "frac": sbytes * B / avg_launch_s / 1e9 / peak_hbm,
                                          "note": "SURVEY.md §8d S-model bytes (%.0f B per env-action): the traffic of an UNFUSED stencil code; sub-steps are fused on chip, "
                                                  "so this may exceed 1 and is not a physical fraction" % sbytes},
                   "f_model_bytes_per_launch": fbytes * B,
                   "traffic_per_launch_ncu": traffic,
                   "traffic_over_f_model": (traffic / (fbytes * B)) if traffic else None,
                   "dram_frac_of_peak": (traffic / avg_launch_s / 1e9 / peak_hbm) if traffic else None,
                   "peak_source": peak_src}
    res = {"value": value, "unit": "env-actions/s", "ms_per_step": total_ms_max / K, "steps": K, "warmup": W,
           "config": {"workload": desc, "envs_per_gpu": B, "global_batch": B * world, "actions_per_launch": 1,
                      "l2": "256 MB flush between timed steps", "noise": "on-device Philox", "status_nonzero_envs": status_bad,
                      **({"jacobi_sweeps_per_action": spa} if want_iters else {})},
           "roofline": roof, "gpu_launches": int(launches), "clocks": clocks}
    if reset:
        res["reset"] = reset
    if e2e:
        res["e2e"] = e2e
    if gather:
        res["e2e_gather"] = gather
    return res


def run_vector_episode(cx, args, B=1024, steps=440):
    """What an agent actually drives: VectorEnv (auto-reset, U{0..400} warm steps per restarted env as in
    shkadov.py:118-123) over more than one 400-action episode, resets included, no host sync in the loop."""
    torch = cx.torch
    from beacon_b200.vector import VectorEnv
    dev = cx.dev
    v = VectorEnv("shkadov", B, n_jets=10, seed=1234, device=cx.local)
    g = torch.Generator(device=dev); g.manual_seed(11)
    acts = torch.rand(8, B, 10, generator=g, device=dev, dtype=torch.float64) * 2 - 1
    v.reset()
    for k in range(3):
        v.step(acts[k])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_done = torch.zeros((), dtype=torch.int64, device=dev)
    a.record()
    for k in range(steps):
        obs, rwd, done, trunc, info = v.step(acts[k % 8])
        n_done += done.sum()
    b.record()
    torch.cuda.synchronize()
    t = a.elapsed_time(b) * 1e-3
    return {"value": B * steps / t, "unit": "env-actions/s (agent-visible steps; the warm steps of the restarts are extra work inside the same time)",
            "steps": steps, "envs_per_gpu": B, "episodes_finished": int(n_done.item()), "seconds": t,
            "config": {"workload": "VectorEnv('shkadov', 1024, n_jets=10): auto-reset with U{0..400} zero-action warm steps, one masked reset launch per step"}}


def run_burgers_single(cx, args, K=200):
    """configs[0]: ONE burgers-v0 env, one 200-action episode: (a) one launch per action, (b) the whole episode as
    one fused launch, (c) a CUDA-graph replay of 200 single-action launches."""
    torch = cx.torch
    from beacon_b200 import BatchedEnv
    dev = cx.dev
    env = BatchedEnv("burgers", batch=1, device=cx.local, seed=1234)
    g = torch.Generator(device=dev); g.manual_seed(7)
    acts = torch.rand(K, 1, 1, generator=g, device=dev, dtype=torch.float64) * 2 - 1
    out = (torch.empty(K, 1, env.n_obs, dtype=torch.float64, device=dev), torch.empty(K, 1, 1, dtype=torch.float64, device=dev),
           torch.empty(K, 1, dtype=torch.uint8, device=dev), torch.empty(K, 1, dtype=torch.uint8, device=dev))
    views = [tuple(o[k:k + 1] for o in out) for k in range(K)]

    def timeit(fn, reps):
        env.reset(); fn(); torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            env.reset()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e-3)
        return statistics.median(ts)

    def per_action():
        for k in range(K):
            env.step_fused(acts[k:k + 1], out=views[k])

    t_single = timeit(per_action, 3)
    t_fused = timeit(lambda: env.step_fused(acts, out=out), 5)
    res = {"config": {"workload": WORKLOADS["burgers"][4], "envs_per_gpu": 1, "episode_actions": K},
           "unit": "env-actions/s", "value": K / t_single,
           "one_launch_per_action": {"value": K / t_single, "us_per_action": 1e6 * t_single / K},
           "fused_episode_one_launch": {"value": K / t_fused, "us_per_action": 1e6 * t_fused / K, "gpu_launches": 1}}
    try:
        env.reset(); torch.cuda.synchronize()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            per_action()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            per_action()
        t_graph = timeit(graph.replay, 5)
        res["cuda_graph_200_launches"] = {"value": K / t_graph, "us_per_action": 1e6 * t_graph / K}
    except Exception as e:
        res["cuda_graph_200_launches"] = {"error": repr(e)[:300]}
    return res


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cx = Ctx()
    cx.torch, cx.dist, cx.rank, cx.world, cx.local, cx.dev = torch, dist, rank, world, local, dev
    cx.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)    # 256 MB > 126 MB L2
    cx.props = torch.cuda.get_device_properties(dev)
    cx.census = load_census()

    wl = args.env
    env_name, kwargs, defB, defK, desc = WORKLOADS[wl]
    B = args.batch or defB
    K = args.steps or defK
    W = max(args.warmup, 3)
    t_start = time.perf_counter()
    main_res = run_workload(wl, B, K, W, cx, args, True)

    extras = args.extras if args.extras is not None else ("all" if (wl == "shkadov" and args.batch is None) else "none")
    names = [] if extras == "none" else (list(DEFAULT_EXTRAS) if extras == "all" else [x for x in extras.split(",") if x])
    workloads = {}
    for w2 in names:
        if w2 == wl:
            continue
        en2, kw2, B2, K2, desc2 = WORKLOADS[w2]
        if w2 == "burgers":
            if rank == 0:
                try:
                    workloads["burgers_single_env"] = run_burgers_single(cx, args)
                except Exception as e:
                    workloads["burgers_single_env"] = {"error": repr(e)[:300]}
                try:
                    workloads["shkadov_vector_env_episode"] = run_vector_episode(cx, args)
                except Exception as e:
                    workloads["shkadov_vector_env_episode"] = {"error": repr(e)[:300]}
            continue
        K2 = min(K2, args.steps) if args.steps else K2
        r = run_workload(w2, B2, K2, W, cx, args, False)
        if rank == 0:
            workloads[w2] = r

    if rank == 0:
        line = {
            "metric": "env-actions/sec", "value": main_res["value"], "unit": "env-actions/s", "n_gpus": world, "steps": main_res["steps"],
            "warmup": W, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {**main_res["config"], "env": wl, "parallelism": f"env-sharded x{world}, no data-path collective in `value`"
                       + ("; `e2e_gather` adds the gather of obs / rewards / flags to the learner rank" if world > 1 else ""),
                       "clock_sampling": "nvidia-smi every 50 ms over the timed region and an untimed continuation of the same steps (>= 0.6 s)"},
            "roofline": main_res["roofline"], "gpu_launches": main_res["gpu_launches"], "clocks": main_res["clocks"],
        }
        for k in ("e2e", "e2e_gather", "reset"):
            if k in main_res:
                line[k] = main_res[k]
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(wl, args.cpu_seconds)
            for w2, r in workloads.items():
                if w2 in ("rayleigh", "mixing", "shkadov_separable") and isinstance(r, dict) and "value" in r:
                    try:
                        r["cpu_baseline"] = cpu_baseline(w2, args.cpu_seconds) if w2 == "rayleigh" else port_sample(w2, min(args.cpu_seconds, 6.0))
                    except Exception as e:
                        r["cpu_baseline"] = {"error": repr(e)[:300]}
        if workloads:
            line["workloads"] = workloads
        line["wall_seconds"] = time.perf_counter() - t_start
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
