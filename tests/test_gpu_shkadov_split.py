"""The balanced shkadov instance split at thread 96, 6/5@96,256,2 (shkadov_balanced_kernel<R, 6, 5, 256, 2, 96, 1>:
threads 0-95 hold 6 points, threads 96-255 hold 5), against the oracle.

The split at 96 puts the outlet, aligned to a chunk end, at off = (576 - nx) mod 5; the dispatcher takes this
instance first where that offset is 0 or 1 and the outlet falls in the 5-point part (576 < nx + off <= 1376),
with the jets at most one per 6-point chunk and BEACON_SHKADOV_NOALIGN unset.  The inlet selects of thread 0
then reach m <= 1 only, as in the uniform single body.  Every other lattice of 768 < nx + off <= 1408 keeps the
split at 128 (6/5,256,2).  The reference's 10-jet lattice, nx = 1350, has off = 1 and 1376 slots (26 phantom
points against 58 with the split at 128).  Each case runs the instance as the dispatcher picks it and forced with
BEACON_SHKADOV_CFG=6/5@96,256,2, and the launched kernel is read from the profiler.

Mutations these cases are built to catch: TH left at T/2 in first_point or last_tid (every point beyond 576
moves, or the outlet specials land on the wrong thread), the host offset taken with the split at 128 (off = 3 at
1350: refused by the chunking check or the outlet misaligned), the inlet selects dropped altogether (off = 1:
the phantom point keeps a stale value that feeds the inlet face), the dispatcher taking an off > 1 lattice into
this instance (the inlet reach would miss points 2..4).

The CPU-only test at the end checks the host's dispatch arithmetic (offset, slots, which split) on every lattice
size the balanced layouts can take; it needs no device.
"""
import numpy as np
import pytest
import torch

from test_gpu_parity import make
from test_gpu_variants import RTOL32, shk_l0, shk_synthetic, shk_vs_oracle

T, C, CN = 256, 6, 5
SPLIT96 = "6/5@96,256,2"
SPLIT128 = "6/5,256,2"


def split_dispatch(nx, noalign=False, cfg=None):
    """Mirror of the balanced tries of shkadov.cu (BEACON_SHK_TRY_BAL, in dispatch order): the first split TH whose
    aligned offset off = (TH*C - nx) mod CN is within its inlet reach and puts the outlet in the CN part,
    TH*C < nx + off <= TH*C + (T - TH)*CN.  cfg = None (dispatcher) or the forced split.  Returns (TH, off, slots)
    or None when neither split takes nx (the uniform instances then run).  The jets are assumed to be at most one
    per 6-point chunk (every case here)."""
    if noalign:
        return None
    for th, reach in ((96, 1), (128, CN - 1)):
        if cfg is not None and cfg != th:
            continue
        off = (th * C - nx) % CN
        slots = th * C + (T - th) * CN
        if off <= reach and th * C < nx + off <= slots:
            return th, off, slots
    return None


def last_thread(nx, th, off):
    """The thread whose chunk ends in the outlet point nx - 1 (last_tid of the kernel)."""
    lp = nx - 1 + off
    return th + (lp - th * C) // CN if lp >= th * C else lp // C


# ============================================================================= CPU: host arithmetic
def test_split_dispatch_arithmetic():
    """Offsets, slots and the chosen split for every nx the balanced layouts can take, without a device."""
    assert split_dispatch(1350) == (96, 1, 1376)                 # the 10-jet default: 26 phantom points
    assert split_dispatch(1350, cfg=128) == (128, 3, 1408)       # the split at 128 would hold 58
    assert last_thread(1350, 96, 1) == 250
    taken = {96: [], 128: []}
    for nx in range(500, 1500):
        got = split_dispatch(nx)
        if got is None:
            # neither split: outside 576 < nx + off <= 1408, or the split at 96 with off > 1 and outside the 128 range
            o96, o128 = (576 - nx) % 5, (768 - nx) % 5
            assert not (o96 <= 1 and 576 < nx + o96 <= 1376) and not (768 < nx + o128 <= 1408), nx
            continue
        th, off, slots = got
        taken[th].append(nx)
        assert slots - off >= nx                                  # the host's chunking check
        lt = last_thread(nx, th, off)
        assert th <= lt < T                                       # the outlet chunk is a 5-point one
        assert th * C + (lt - th) * CN - off + CN - 1 == nx - 1   # ... and ends in the outlet point
        assert off <= (1 if th == 96 else CN - 1)                 # within the inlet reach of the instance
        if th == 128:                                             # only lattices the split at 96 cannot take
            assert split_dispatch(nx, cfg=96) is None, nx
    # the split at 96 takes two offsets in five from nx = 580 to 1376, the split at 128 the rest up to 1408
    assert taken[96][0] == 580 and taken[96][-1] == 1376 and len(taken[96]) == 2 * (1376 - 575) // 5
    assert taken[128][0] == 769 and taken[128][-1] == 1408
    assert all((576 - nx) % 5 in (0, 1) for nx in taken[96])
    assert all(nx > 1376 or (576 - nx) % 5 > 1 for nx in taken[128])
    assert split_dispatch(1350, noalign=True) is None


# ============================================================================= GPU: against the oracle
def kernels_of(fn):
    """Names of the shkadov kernels launched by fn()."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if "shkadov" in e.name and "order_kernel" not in e.name}


def assert_split(env, th, dtype="double"):
    """env's kernel is the balanced one split at thread th (None: not a balanced one); a plain reset launches it
    without drawing noise."""
    names = kernels_of(lambda: env.reset())
    if th is None:
        assert names and all("shkadov_balanced_kernel" not in n for n in names), names
    else:
        want = f"shkadov_balanced_kernel<{dtype}, 6, 5, 256, 2, {th}, {1 if th == 96 else 4}>"
        assert names and all(want in n for n in names), names


def split_env(nx, n_jets, monkeypatch, cfg, B=2, **kw):
    if cfg:
        monkeypatch.setenv("BEACON_SHKADOV_CFG", cfg)
    else:
        monkeypatch.delenv("BEACON_SHKADOV_CFG", raising=False)
    env = make("shkadov", B, init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, **kw)
    assert env.cfg.d["nx"] == nx
    return env


# nx, off, jets, kwargs: the smallest and largest lattice the instance takes at both offsets, the 10-jet default
CASES = [(580, 1, 5, dict(jet_pos=40.0)), (581, 0, 5, dict(jet_pos=40.0)), (1350, 1, 10, {}), (1351, 0, 10, {}),
         (1375, 1, 10, {}), (1376, 0, 10, {})]


@pytest.mark.gpu
@pytest.mark.parametrize("nx,off,n_jets,kw", CASES, ids=[f"nx{c[0]}-off{c[1]}" for c in CASES])
def test_split_vs_oracle(nx, off, n_jets, kw, monkeypatch):
    assert split_dispatch(nx) == (96, off, 1376)
    envs = []
    for cfg in (None, SPLIT96):
        env = split_env(nx, n_jets, monkeypatch, cfg, **kw)
        assert_split(env, 96)
        envs.append(env)
    shk_vs_oracle(envs, nx, n_jets, C, seed=nx, **kw)


@pytest.mark.gpu
def test_split_20_jets(monkeypatch):
    nx, n_jets, kw = 1375, 20, dict(jet_pos=30.0)
    assert split_dispatch(nx) == (96, 1, 1376)
    env = split_env(nx, n_jets, monkeypatch, None, **kw)
    assert_split(env, 96)
    shk_vs_oracle([env], nx, n_jets, C, seed=21, **kw)


@pytest.mark.gpu
def test_split_per_jet_rewards(monkeypatch):
    env = split_env(1350, 10, monkeypatch, SPLIT96, per_jet_rwd=True)
    assert_split(env, 96)
    shk_vs_oracle([env], 1350, 10, C, per_jet=True, seed=22)


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [1350, 1351])
def test_split_fp32(nx, monkeypatch):
    env = split_env(nx, 10, monkeypatch, SPLIT96, dtype=torch.float32)
    assert_split(env, 96, "float")
    shk_vs_oracle([env], nx, 10, C, n_actions=1, rtol=RTOL32, seed=nx + 3)


@pytest.mark.gpu
def test_split_fused_equals_single(monkeypatch):
    """K = 3 actions in one launch equal three launches bitwise."""
    nx, n_jets, B, K = 1350, 10, 3, 3
    e1, e2 = (split_env(nx, n_jets, monkeypatch, SPLIT96, B=B, seed=6) for _ in range(2))
    assert_split(e1, 96)
    hq = [shk_synthetic(nx, b) for b in range(B)]
    for e in (e1, e2):
        e.reset()
        e.set_state("h", np.stack([x[0] for x in hq]))
        e.set_state("q", np.stack([x[1] for x in hq]))
    acts = torch.as_tensor(np.random.default_rng(nx + 1).uniform(-1, 1, (K, B, n_jets)))
    fused = e1.step_fused(acts)
    single = [e2.step(acts[k]) for k in range(K)]
    for i, what in enumerate(("obs", "rwd", "done", "trunc")):
        assert torch.equal(fused[i], torch.stack([s[i] for s in single])), what
    for f in ("h", "q", "rhsh", "rhsq", "u", "up", "stp", "draws"):
        assert torch.equal(e1.get_state(f), e2.get_state(f)), f


@pytest.mark.gpu
def test_split_masked_warm_reset_and_batch_of_one(monkeypatch):
    """Masked warm reset with on-device noise: envs outside the mask untouched bitwise, the others equal a
    batch-of-1 env at the same global index bitwise (reset, step and warm reset)."""
    monkeypatch.delenv("BEACON_SHKADOV_CFG", raising=False)
    B, nj, seed = 300, 10, 23
    rng = np.random.default_rng(63)
    nw = rng.integers(0, 41, B)
    mask = rng.random(B) < 0.5
    mask[[0, 151, 299]] = True
    env = make("shkadov", B, n_jets=nj, seed=seed)
    assert env.cfg.d["nx"] == 1350
    assert_split(env, 96)
    env.reset()
    acts = torch.as_tensor(rng.uniform(-1, 1, (B, nj)))
    env.step(acts)
    before = {f: env.get_state(f).clone() for f in ("h", "q", "rhsh", "rhsq", "draws", "stp")}
    env.reset(mask=torch.as_tensor(mask), n_warm=torch.as_tensor(nw, dtype=torch.int32))
    after = {f: env.get_state(f) for f in before}
    m = torch.as_tensor(mask, device=after["h"].device)
    for f in before:
        assert torch.equal(after[f][~m], before[f][~m]), f
    for b in (0, 151, 299):
        one = make("shkadov", 1, n_jets=nj, seed=seed, env_index_base=b)
        assert_split(one, 96)
        one.reset()
        one.step(acts[b:b + 1])
        for f in ("h", "q", "rhsh", "rhsq"):
            assert torch.equal(one.get_state(f)[0], before[f][b]), (b, f)
        one.reset(n_warm=torch.tensor([int(nw[b])], dtype=torch.int32))
        for f in before:
            assert torch.equal(one.get_state(f)[0], after[f][b]), (b, f)


@pytest.mark.gpu
def test_split_dispatch(monkeypatch):
    """The dispatcher picks the split the mirror names: 96 where off <= 1, 128 for the other lattices of
    768 < nx + off <= 1408, neither outside; 6/5,256,2 still forces the split at 128, and 6/5@96,256,2 is refused
    for a lattice with off > 1."""
    from beacon_b200 import BeaconError
    for nx, th in ((700, 96), (1350, 96), (1376, 96), (1352, 128), (1353, 128), (1377, 128), (1408, 128), (768, None)):
        got = split_dispatch(nx)
        assert (got[0] if got else None) == th, nx
        assert_split(split_env(nx, 10, monkeypatch, None, **(dict(jet_pos=40.0) if nx < 1000 else {})), th)
    env = split_env(1350, 10, monkeypatch, SPLIT128)
    assert_split(env, 128)
    shk_vs_oracle([env], 1350, 10, C, n_actions=1, seed=24)
    assert_split(split_env(1351, 10, monkeypatch, SPLIT96), 96)
    with pytest.raises(BeaconError, match="no kernel variant covers"):
        split_env(1352, 10, monkeypatch, SPLIT96)


@pytest.mark.gpu
def test_split_noalign(monkeypatch):
    """BEACON_SHKADOV_NOALIGN leaves the unaligned general layout, which neither split runs: the dispatcher falls
    back to 6,256,2 (checked against the oracle), and forcing 6/5@96,256,2 is refused."""
    from beacon_b200 import BeaconError
    monkeypatch.setenv("BEACON_SHKADOV_NOALIGN", "1")
    env = split_env(1350, 10, monkeypatch, None)
    assert_split(env, None)
    shk_vs_oracle([env], 1350, 10, C, seed=25)
    with pytest.raises(BeaconError, match="no kernel variant covers"):
        split_env(1350, 10, monkeypatch, SPLIT96)
