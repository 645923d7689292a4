"""The balanced shkadov instance 6/5,256,2 (shkadov_balanced_kernel: threads 0-127 hold 6 points, threads
128-255 hold 5), against the oracle.

The dispatcher puts it first for every lattice whose outlet, aligned to a chunk end, falls in the 5-point
half (768 < nx + off <= 1408, off = (768 - nx) mod 5 <= 4) when the jets are at most one per 6-point chunk
and BEACON_SHKADOV_NOALIGN is unset; both widths then run the unrolled single body, the inlet selects of
thread 0 reaching the points m <= 4.  Each case runs the instance as the dispatcher picks it and forced
with BEACON_SHKADOV_CFG=6/5,256,2, and the launched kernel is read from the profiler.

Mutations these cases are built to catch: the width of warps 4-7 set to 6
(every point beyond 768 moves), the prefix of a0 off by one point, the inlet selects confined to m < 2
(off = 2..4: the phantom points and the inlet keep stale values), the outlet specials compiled into the
6-point body only, the epilogue / store loops writing m >= 5 of a 5-point chunk (the first point of the
next chunk is overwritten), the host offset taken modulo 6.
"""
import numpy as np
import pytest
import torch

from test_gpu_parity import make
from test_gpu_variants import RTOL32, shk_l0, shk_synthetic, shk_vs_oracle

pytestmark = pytest.mark.gpu

BAL = "6/5,256,2"


def bal_off(nx):
    """Phantom shift of the balanced layout, or None if the instance does not take nx."""
    off = (768 - nx) % 5
    return off if 768 < nx + off <= 1408 else None


def kernels_of(fn):
    """Names of the shkadov kernels launched by fn()."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if "shkadov" in e.name and "order_kernel" not in e.name}


def assert_balanced(env, expect=True):
    """env's kernel is (or is not) the balanced one; a plain reset launches it without drawing noise."""
    names = kernels_of(lambda: env.reset())
    assert names and all(("shkadov_balanced_kernel" in n) == expect for n in names), names


def bal_env(nx, n_jets, monkeypatch, forced, B=2, **kw):
    if forced:
        monkeypatch.setenv("BEACON_SHKADOV_CFG", BAL)
    else:
        monkeypatch.delenv("BEACON_SHKADOV_CFG", raising=False)
    env = make("shkadov", B, init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, **kw)
    assert env.cfg.d["nx"] == nx
    return env


# nx, off: the smallest and largest lattice the instance takes, every offset, the reference's 10-jet lattice
CASES = [(769, 4), (1349, 4), (1350, 3), (1351, 2), (1352, 1), (1353, 0), (1408, 0)]


@pytest.mark.parametrize("nx,off", CASES, ids=[f"nx{nx}-off{off}" for nx, off in CASES])
def test_balanced_vs_oracle(nx, off, monkeypatch):
    assert bal_off(nx) == off
    kw = dict(jet_pos=40.0) if nx < 1000 else {}     # 10 jets inside the short lattice
    envs = []
    for forced in (False, True):
        env = bal_env(nx, 10, monkeypatch, forced, **kw)
        assert_balanced(env)
        envs.append(env)
    shk_vs_oracle(envs, nx, 10, 6, seed=nx, **kw)


def test_balanced_20_jets(monkeypatch):
    nx, n_jets, kw = 1400, 20, dict(jet_pos=30.0)
    assert bal_off(nx) == 3
    env = bal_env(nx, n_jets, monkeypatch, False, **kw)
    assert_balanced(env)
    shk_vs_oracle([env], nx, n_jets, 6, seed=11, **kw)


def test_balanced_per_jet_rewards(monkeypatch):
    env = bal_env(1350, 10, monkeypatch, True, per_jet_rwd=True)
    assert_balanced(env)
    shk_vs_oracle([env], 1350, 10, 6, per_jet=True, seed=12)


@pytest.mark.parametrize("nx", [1350, 1352])
def test_balanced_fp32(nx, monkeypatch):
    env = bal_env(nx, 10, monkeypatch, True, dtype=torch.float32)
    assert_balanced(env)
    shk_vs_oracle([env], nx, 10, 6, n_actions=1, rtol=RTOL32, seed=nx + 2)


def test_balanced_fused_equals_single(monkeypatch):
    """K = 3 actions in one launch equal three launches bitwise."""
    nx, n_jets, B, K = 1350, 10, 3, 3
    e1, e2 = (bal_env(nx, n_jets, monkeypatch, True, B=B, seed=5) for _ in range(2))
    assert_balanced(e1)
    hq = [shk_synthetic(nx, b) for b in range(B)]
    for e in (e1, e2):
        e.reset()
        e.set_state("h", np.stack([x[0] for x in hq]))
        e.set_state("q", np.stack([x[1] for x in hq]))
    acts = torch.as_tensor(np.random.default_rng(nx).uniform(-1, 1, (K, B, n_jets)))
    fused = e1.step_fused(acts)
    single = [e2.step(acts[k]) for k in range(K)]
    for i, what in enumerate(("obs", "rwd", "done", "trunc")):
        assert torch.equal(fused[i], torch.stack([s[i] for s in single])), what
    for f in ("h", "q", "rhsh", "rhsq", "u", "up", "stp", "draws"):
        assert torch.equal(e1.get_state(f), e2.get_state(f)), f


def test_balanced_masked_warm_reset_and_batch_of_one(monkeypatch):
    """Masked warm reset with on-device noise: envs outside the mask untouched bitwise, the others equal a
    batch-of-1 env at the same global index bitwise (reset, step and warm reset)."""
    monkeypatch.delenv("BEACON_SHKADOV_CFG", raising=False)
    B, nj, seed = 300, 10, 17
    rng = np.random.default_rng(62)
    nw = rng.integers(0, 41, B)
    mask = rng.random(B) < 0.5
    mask[[0, 150, 299]] = True
    env = make("shkadov", B, n_jets=nj, seed=seed)
    assert env.cfg.d["nx"] == 1350
    assert_balanced(env)
    env.reset()
    acts = torch.as_tensor(rng.uniform(-1, 1, (B, nj)))
    env.step(acts)
    before = {f: env.get_state(f).clone() for f in ("h", "q", "rhsh", "rhsq", "draws", "stp")}
    env.reset(mask=torch.as_tensor(mask), n_warm=torch.as_tensor(nw, dtype=torch.int32))
    after = {f: env.get_state(f) for f in before}
    m = torch.as_tensor(mask, device=after["h"].device)
    for f in before:
        assert torch.equal(after[f][~m], before[f][~m]), f
    for b in (0, 150, 299):
        one = make("shkadov", 1, n_jets=nj, seed=seed, env_index_base=b)
        one.reset()
        one.step(acts[b:b + 1])
        for f in ("h", "q", "rhsh", "rhsq"):
            assert torch.equal(one.get_state(f)[0], before[f][b]), (b, f)
        one.reset(n_warm=torch.tensor([int(nw[b])], dtype=torch.int32))
        for f in before:
            assert torch.equal(one.get_state(f)[0], after[f][b]), (b, f)


def test_balanced_dispatch(monkeypatch):
    """nx = 1350 picks the balanced instance; BEACON_SHKADOV_CFG=6,256,2 still forces the uniform one; lattices
    outside 768 < nx + off <= 1408 keep 6,256,2."""
    monkeypatch.delenv("BEACON_SHKADOV_CFG", raising=False)
    env = make("shkadov", 2, n_jets=10)
    assert env.cfg.d["nx"] == 1350
    assert_balanced(env)
    for nx in (768, 1409):
        assert bal_off(nx) is None
        assert_balanced(bal_env(nx, 10, monkeypatch, False, **(dict(jet_pos=40.0) if nx < 1000 else {})), expect=False)
    monkeypatch.setenv("BEACON_SHKADOV_CFG", "6,256,2")
    env = make("shkadov", 2, n_jets=10)
    names = kernels_of(lambda: env.reset())
    assert names and all("shkadov_kernel<double, 6, 256, 2>" in n for n in names), names


def test_balanced_noalign(monkeypatch):
    """BEACON_SHKADOV_NOALIGN leaves the unaligned general layout, which the balanced instance does not run:
    the dispatcher falls back to 6,256,2 (checked against the oracle), and forcing 6/5,256,2 is refused."""
    from beacon_b200 import BeaconError
    monkeypatch.setenv("BEACON_SHKADOV_NOALIGN", "1")
    env = bal_env(1350, 10, monkeypatch, False)
    assert_balanced(env, expect=False)
    shk_vs_oracle([env], 1350, 10, 6, seed=13)
    with pytest.raises(BeaconError, match="no kernel variant covers"):
        bal_env(1350, 10, monkeypatch, True)
