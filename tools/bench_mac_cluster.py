"""Throughput of rayleigh / mixing with one environment split over a thread-block cluster (ctas_per_env).

    python tools/bench_mac_cluster.py [--steps 5] [--repeats 3] [--out result.json]

Cases:
  * the grids no single CTA holds (rayleigh 314x50 = L 2 pi, mixing 200x100 and 200x200) at batches with
    B * G a multiple of the B200's 148 SMs, so that the GPU is full;
  * mixing 100x100 at small batches (8, 16, 37 envs) on one CTA per env (mac_big_kernel) against 2 and 4:
    whether spreading an env over idle SMs lowers the latency of a step;
  * rayleigh 100x50 from rest, 16 envs, on the generic mac_kernel at G = 1 (one CTA per env) and on 2, 4, 8
    CTAs: the same grid and the same sweep counts, so the difference of the time per sweep isolates what the
    cluster path adds per sweep (its cluster barrier and DSMEM exchange) net of the work the split saves;
  * the generic mac_kernel at G = 1 on a full GPU (148 envs, one per SM) on rayleigh 100x50, 75x61 (partial
    tiles) and 200x50 (500 tile threads, four transport passes), from rest: the one-CTA throughput of the
    kernel that also runs the clusters, tight enough to show a small change.
Each case: reset, one warm-up action, then `--repeats` windows of `--steps` actions timed with CUDA events
(random actions, one launch each; actions differ between windows).  Per window:
  env_actions_per_s = B * steps / time;
  us_per_sweep      = time of an action / mean sweep count of the batch's envs.  Every phase of the action is
                      in the numerator (predictor, transport, per-sub-step barriers, obs / reward); the Jacobi
                      sweeps are most of it, but this is an upper bound of the cost of one sweep.
Rows give the median and the min / max over the windows.  The GPU name and power limit are read in the same run.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from beacon_b200 import BatchedEnv  # noqa: E402

PAIR = "rayleigh 100x50"
CASES = (
    [("rayleigh 314x50", "rayleigh", dict(init=False, L=2 * math.pi), G, B) for G, B in ((2, 74), (4, 37), (8, 37))]
    + [("mixing 200x100", "mixing", dict(L=2.0), G, B) for G, B in ((2, 74), (4, 37))]
    + [("mixing 200x200", "mixing", dict(L=2.0, H=2.0), 8, 37)]
    + [("mixing 100x100", "mixing", dict(), G, B) for B in (8, 16, 37) for G in (1, 2, 4)]
    + [(PAIR, "rayleigh", dict(init=False, L=2.0, n_sgts=5), G, 16) for G in (1, 2, 4, 8)]
    + [(label, "rayleigh", dict(init=False, L=L, H=H, n_sgts=5), 1, 148)
       for label, L, H in ((PAIR, 2.0, 1.0), ("rayleigh 75x61", 1.5, 1.22), ("rayleigh 200x50", 4.0, 1.0))]
)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr.strip()}


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def run(label, name, kw, G, B, steps, repeats, seed=0):
    env = BatchedEnv(name, batch=B, ctas_per_env=G, **kw)
    rng = np.random.default_rng(seed)

    def act():
        if name == "rayleigh":
            return torch.as_tensor(rng.uniform(-1, 1, (B, env.act_dim)), device=env.device)
        return torch.as_tensor(rng.integers(0, 4, B), dtype=torch.int32, device=env.device)

    env.reset()
    env.step(act())
    rates, per_sweep, ms_act, sweeps = [], [], [], []
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(repeats):
        acts = [act() for _ in range(steps)]
        iters = []
        torch.cuda.synchronize()
        t0.record()
        for a in acts:
            env.step(a, want_iters=True)
            iters.append(env.last_iters[0])
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1)
        sw = float(torch.stack(iters).double().mean())
        rates.append(B * steps / (ms / 1e3)); ms_act.append(ms / steps); sweeps.append(sw)
        per_sweep.append(ms / steps / sw * 1e3)
    ok = int(env.status.max()) == 0
    env.close()
    return {"case": label, "G": G, "B": B, "ctas": B * G, "steps": steps, "repeats": repeats,
            "env_actions_per_s": spread(rates), "ms_per_action": spread(ms_act), "sweeps_per_action": spread(sweeps),
            "us_per_sweep": spread(per_sweep), "status_ok": ok}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    rows = []
    for label, name, kw, G, B in CASES:
        r = run(label, name, kw, G, B, args.steps, args.repeats)
        rows.append(r)
        print(json.dumps(r), flush=True)
    # same grid, same sweep counts: extra time per sweep of the cluster path over the generic one-CTA kernel
    pair = [r for r in rows if r["case"] == PAIR and r["B"] == 16]
    base = next(r for r in pair if r["G"] == 1)["us_per_sweep"]["median"]
    extra = {r["G"]: r["us_per_sweep"]["median"] - base for r in pair if r["G"] > 1}
    print(json.dumps({"case": PAIR, "extra_us_per_sweep_vs_G1": extra}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"gpu": info, "rows": rows, "extra_us_per_sweep_vs_G1": extra}, f, indent=1)


if __name__ == "__main__":
    main()
