"""Per-env physical parameters (rayleigh ra; mixing re, pe): what the per-env kernel instances cost, and what one
launch gains over one handle per value.  Arms are measured in one process, alternating, REPS times each:

  (a) same work: a uniform handle against a per-env handle whose values all equal the default
      (rayleigh B = 4096, mixing B = 1024): the difference is the cost of the per-env instance;
  (b) rayleigh B = 4096 with 16 distinct ra in one per-env handle, against 16 uniform handles of 256 envs
      stepped in turn (one launch each).

Every arm steps its own envs the same number of actions, so the arms' flows (and Jacobi sweep counts) stay
equal across repetitions.  Prints env-actions/s per arm (median, min, max over the repetitions), with the
GPU's name and power limit read in the same run.

    python tools/bench_physics.py [--reps 5] [--steps-ray 4] [--steps-mix 2] [--json OUT]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from beacon_b200 import BatchedEnv  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


class Arm:
    def __init__(self, name, envs, acts):
        self.name, self.envs, self.acts = name, envs, acts
        self.batch = sum(e.batch for e in envs)
        for e in envs:
            e.reset()
        self.rates = []

    def step(self, n):
        for _ in range(n):
            for e, a in zip(self.envs, self.acts):
                e.step(a)

    def time(self, n):
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        self.step(n)
        t1.record()
        t1.synchronize()
        self.rates.append(self.batch * n / (t0.elapsed_time(t1) * 1e-3))


def ray_acts(B, seed):
    return torch.as_tensor(np.random.default_rng(seed).uniform(-1, 1, (B, 10)), device="cuda")


def mix_acts(B, seed):
    return torch.as_tensor(np.random.default_rng(seed).integers(0, 4, B), dtype=torch.int32, device="cuda")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps-ray", type=int, default=4, help="actions per timed window, rayleigh arms")
    ap.add_argument("--steps-mix", type=int, default=2, help="actions per timed window, mixing arms")
    ap.add_argument("--json", default=None, help="also write the results here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_physics needs a CUDA device (B200)")
    info = gpu_info()
    print("gpu:", info)

    BR, BM, NV = 4096, 1024, 16
    ra16 = np.geomspace(1e4, 1e5, NV)
    a_r, a_m = ray_acts(BR, 1), mix_acts(BM, 2)
    groups = {
        "a_rayleigh": ([Arm("uniform", [BatchedEnv("rayleigh", batch=BR)], [a_r]),
                        Arm("per_env_default", [BatchedEnv("rayleigh", batch=BR, ra=np.full(BR, 1e4))], [a_r])], args.steps_ray),
        "a_mixing": ([Arm("uniform", [BatchedEnv("mixing", batch=BM)], [a_m]),
                      Arm("per_env_default", [BatchedEnv("mixing", batch=BM, re=np.full(BM, 100.0), pe=np.full(BM, 1e4))], [a_m])],
                     args.steps_mix),
        "b_rayleigh_16_ra": ([Arm("one_per_env_handle", [BatchedEnv("rayleigh", batch=BR, ra=np.repeat(ra16, BR // NV))], [a_r]),
                              Arm("16_uniform_handles", [BatchedEnv("rayleigh", batch=BR // NV, ra=float(r)) for r in ra16],
                                  [a_r[k * (BR // NV):(k + 1) * (BR // NV)] for k in range(NV)])], args.steps_ray),
    }
    for arms, n in groups.values():      # warm-up: module load, first launches
        for arm in arms:
            arm.step(1)
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for arms, n in groups.values():
            for arm in arms:
                arm.time(n)
    res = {"gpu": info, "reps": args.reps, "groups": {}}
    for g, (arms, n) in groups.items():
        res["groups"][g] = {}
        for arm in arms:
            r = np.array(arm.rates)
            res["groups"][g][arm.name] = {"batch": arm.batch, "actions_per_window": n, "env_actions_per_s_median": float(np.median(r)),
                                          "min": float(r.min()), "max": float(r.max())}
            print(f"{g:18s} {arm.name:20s} B={arm.batch:5d}  env-actions/s median {np.median(r):10.1f}  "
                  f"min {r.min():10.1f}  max {r.max():10.1f}")
        names = [a.name for a in arms]
        m = [res["groups"][g][k]["env_actions_per_s_median"] for k in names]
        print(f"{g:18s} {names[1]} / {names[0]} = {m[1] / m[0]:.4f}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
