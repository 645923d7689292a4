"""Parity of the CUDA path (through the C-ABI, libbeacon_b200.so) with the reference.

Two anchors:
  * the committed golden vectors of the UNMODIFIED reference (tests/golden/<env>.npz);
  * the CPU oracle (oracle/, bit-exact restatement of the reference) from identical states on
    fresh seeded inputs, with the state RE-SYNCED from the oracle before every action for the
    chaotic envs (SURVEY.md §4 sensitivity table).
Tolerances (north star): fields <= 1e-10 relative in fp64, <= 1e-5 in fp32; Jacobi sweep counts,
probe indices, flags: exact.
"""
import json

import numpy as np
import pytest
import torch

from oracle import beacon_oracle as bo

pytestmark = pytest.mark.gpu

RTOL64 = 1e-10


def close(a, b, rtol=RTOL64, what="", floor=1e-2):
    """The norm of every field comparison (DESIGN.md §4):
        |a - b| <= rtol * (|b| + floor * scale),     scale = max(1, max|b|)
    floor = 1e-2 (default, solution fields h, q, u, v, p, T, C, observations): every entry agrees to `rtol`
    relative to ITS OWN magnitude, entries below 1 % of the field scale (zeros at walls, u, v << 1) are held to
    an absolute 1e-12 * scale in fp64.
    floor = 1 (right-hand sides rhsh / rhsq, and every fp32 comparison): relative to the field scale.  An rhsq
    entry is a difference of stencil terms of magnitude ~750 (d3o2u divides O(1) differences by 2 dx^3 = 0.016):
    its absolute rounding noise, in the reference as well, is ~1e-12 whatever the size of the result, so a
    per-entry relative bound is not meaningful there; in fp32 one rounding is 6e-8 of the field scale.
    Returns the largest scale-relative error."""
    a = np.asarray(a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if not b.size:
        return 0.0
    scale = max(1.0, float(np.max(np.abs(b))))
    assert np.all(np.isfinite(a)), what
    err = np.abs(a - b)
    lim = rtol * (np.abs(b) + floor * scale)
    worst = int(np.argmax(err - lim))
    assert np.all(err <= lim), (f"{what}: entry {worst}: |a-b| = {err.flat[worst]:.3e} > {rtol:.0e}*(|b| + {floor:g} scale) = {lim.flat[worst]:.3e} "
                               f"(b = {b.flat[worst]:.6e}, scale {scale:.3g})")
    return float(np.max(err)) / scale


def make(name, batch, **kw):
    from beacon_b200 import BatchedEnv
    return BatchedEnv(name, batch=batch, **kw)


def rep(x, B):
    return torch.as_tensor(np.broadcast_to(np.asarray(x), (B,) + np.asarray(x).shape).copy())


# ----------------------------------------------------------------------------- shkadov
@pytest.mark.parametrize("tag,n_jets", [("j10", 10), ("j5", 5), ("j41", 41)])
def test_shkadov_golden(golden, tag, n_jets):
    g = golden("shkadov")
    B = 3
    env = make("shkadov", B, n_jets=n_jets)
    obs0 = env.reset()
    close(obs0, rep(g[f"{tag}_obs0"], B), what="obs0")
    for k in range(g[f"{tag}_actions"].shape[0]):
        obs, rwd, done, trunc = env.step(rep(g[f"{tag}_actions"][k], B), noise=rep(g[f"{tag}_noise"][k], B))
        for f in ("h", "q", "rhsh", "rhsq"):
            close(env.get_state(f), rep(g[f"{tag}_{f}"][k], B), what=f"{f} step {k}", floor=1.0 if f.startswith("rhs") else 1e-2)
        close(obs, rep(g[f"{tag}_obs"][k], B), what="obs")
        close(rwd, rep(g[f"{tag}_rwd"][k], B), rtol=1e-12, what="rwd")
        assert not done.any() and not trunc.any()
    assert int(env.status.max()) == 0


def test_shkadov_integer_tables_bit_exact(golden):
    """probe indices / actuator masks come from host ints: compare with the reference's."""
    from beacon_b200.params import ShkadovCfg
    g = golden("shkadov")
    for row in json.loads(str(g["params_json"])):
        c = ShkadovCfg(init=False, **row["kwargs"])
        for k in ("nx", "ndt_act", "n_act", "n_interp", "jet_pos", "jet_hw", "jet_space", "l_rwd", "n_obs", "l_obs"):
            assert c.d[k] == row[k], (row["kwargs"], k)
        assert c.d["dx"] == row["dx"]
        assert c.jet_mask()[0][1] == row["jet_start"] and c.jet_mask()[0][2] == row["jet_end"]
        assert c.obs_indices()[0, 0] == row["obs_start"]


def test_shkadov_warm_reset_golden(golden):
    g = golden("shkadov")
    B = 2
    env = make("shkadov", B, n_jets=10)
    nw = int(g["warm_n"])
    noise = torch.as_tensor(np.repeat(g["warm_noise"][:, None, :], B, axis=1))
    obs0 = env.reset(n_warm=torch.full((B,), nw), noise=noise)
    close(obs0, rep(g["warm_obs0"], B), what="obs0")
    close(env.get_state("h"), rep(g["warm_h"], B), what="h")
    close(env.get_state("q"), rep(g["warm_q"], B), what="q")
    assert int(env.get_state("stp").max()) == 0


def test_shkadov_vs_oracle_resync():
    """8 envs, different actions and noise, 6 actions, state re-synced from the oracle each action."""
    rng = np.random.default_rng(11)
    B, nj = 8, 10
    env = make("shkadov", B, n_jets=nj)
    orcs = [bo.shkadov(n_jets=nj) for _ in range(B)]
    env.reset()
    for o in orcs:
        o.reset()
        # decorrelate the envs: a few oracle steps with random actions
        for _ in range(2):
            o.step(rng.uniform(-1, 1, nj), noise=rng.uniform(-5e-4, 5e-4, 50))
    for k in range(6):
        for f in ("h", "q", "rhsh", "rhsq", "u", "up"):
            env.set_state(f, np.stack([getattr(o, f) for o in orcs]))
        env.set_state("stp", np.array([o.stp for o in orcs]))
        acts = rng.uniform(-1, 1, (B, nj))
        noise = rng.uniform(-5e-4, 5e-4, (B, 50))
        obs, rwd, done, trunc = env.step(torch.as_tensor(acts), noise=torch.as_tensor(noise))
        ref = [o.step(acts[b], noise=noise[b]) for b, o in enumerate(orcs)]
        for f in ("h", "q", "rhsh", "rhsq"):
            close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), what=f"{f} action {k}", floor=1.0 if f.startswith("rhs") else 1e-2)
        close(obs, np.stack([r[0] for r in ref]), what="obs")
        close(rwd, np.array([r[1] for r in ref]), rtol=1e-12, what="rwd")


@pytest.mark.parametrize("kw,noalign", [
    (dict(n_jets=4, jet_space=5.0), False),      # dense jets (spacing 25 < chunk + jet width): per-point jet table
    (dict(n_jets=4, jet_space=3.0, L0=200.0), False),   # overlapping jets (spacing 15 < 21): generic per-jet loop
    (dict(n_jets=10), True),                     # outlet not aligned to a chunk end: per-point index tests
    (dict(n_jets=20), True),                     # the same on the 10,192,2 instance (nx 1850)
])
def test_shkadov_general_paths_vs_oracle(kw, noalign, monkeypatch):
    """The general (per-point index test) path of the kernel, which the standard configurations no
    longer take: 3 actions from the oracle's state, fields within 1e-10."""
    if noalign:
        monkeypatch.setenv("BEACON_SHKADOV_NOALIGN", "1")
    rng = np.random.default_rng(21)
    B, nj = 2, kw["n_jets"]
    env = make("shkadov", B, **kw)
    orcs = [bo.shkadov(**kw) for _ in range(B)]
    env.reset()
    for o in orcs:
        o.reset()
    for k in range(3):
        for f in ("h", "q", "rhsh", "rhsq", "u", "up"):
            env.set_state(f, np.stack([getattr(o, f) for o in orcs]))
        acts = rng.uniform(-1, 1, (B, nj))
        noise = rng.uniform(-5e-4, 5e-4, (B, 50))
        obs, rwd, done, trunc = env.step(torch.as_tensor(acts), noise=torch.as_tensor(noise))
        ref = [o.step(acts[b], noise=noise[b]) for b, o in enumerate(orcs)]
        for f in ("h", "q", "rhsh", "rhsq"):
            close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), what=f"{f} action {k}", floor=1.0 if f.startswith("rhs") else 1e-2)
        close(obs, np.stack([r[0] for r in ref]), what="obs")
        close(rwd, np.array([r[1] for r in ref]), rtol=1e-12, what="rwd")


def test_shkadov_free_running_return():
    """sigma=0, 10 free-running actions: return within 1e-9 (SURVEY.md §8c)."""
    rng = np.random.default_rng(12)
    env = make("shkadov", 1, n_jets=10, sigma=0.0)
    o = bo.shkadov(n_jets=10)
    env.reset(); o.reset()
    tot_g = tot_o = 0.0
    for k in range(10):
        a = rng.uniform(-1, 1, 10)
        _, r, _, _ = env.step(torch.as_tensor(a[None]), noise=torch.zeros(1, 50, dtype=torch.float64))
        tot_g += float(r[0]); tot_o += o.step(a)[1]
    assert abs(tot_g - tot_o) <= 1e-9 * abs(tot_o)


def test_shkadov_flags_blowup_and_horizon(golden):
    g = golden("shkadov")
    env = make("shkadov", 2, n_jets=2, t_act=0.2, sigma=0.0)
    env.reset()
    flags = []
    for k in range(4):
        _, _, d, t = env.step(torch.zeros(2, 2, dtype=torch.float64))
        flags.append((bool(d[0]), bool(t[0])))
    assert np.array_equal(np.array(flags), g["horizon_flags"])
    env.reset()
    h = env.get_state("h")
    h[1, 300] = 40.0
    env.set_state("h", h)
    _, r, d, t = env.step(torch.zeros(2, 2, dtype=torch.float64))
    assert (bool(d[1]), bool(t[1]), float(r[1])) == (True, False, -1.0)      # shkadov.py:176-180
    assert not bool(d[0]) and int(env.status[1]) & 1 and not int(env.status[0])


def test_shkadov_fused_equals_single_and_host():
    rng = np.random.default_rng(13)
    B, K = 4, 3
    acts = torch.as_tensor(rng.uniform(-1, 1, (K, B, 5)))
    noise = torch.as_tensor(rng.uniform(-5e-4, 5e-4, (K, B, 50)))
    e1, e2, e3, e4 = (make("shkadov", B) for _ in range(4))
    for e in (e1, e2, e3, e4):
        e.reset()
    o1, r1, d1, t1 = e1.step_fused(acts, noise)
    outs = [e2.step(acts[k], noise[k]) for k in range(K)]
    assert torch.equal(o1, torch.stack([o[0] for o in outs])) and torch.equal(r1, torch.stack([o[1] for o in outs]))
    assert torch.equal(e1.get_state("h"), e2.get_state("h")) and torch.equal(e1.get_state("q"), e2.get_state("q"))
    for k in range(K):
        # pageable inputs (staged through device buffers), page-locked outputs (written by the kernel)
        oh, rh, dh, th = e3.step_host(acts[k].numpy(), noise[k].numpy())
        assert np.array_equal(oh.numpy(), outs[k][0].cpu().numpy()) and np.array_equal(rh.numpy(), outs[k][1].cpu().numpy())
        # everything page-locked (the kernel reads and writes the host buffers directly), and everything pageable
        om, rm, dm, tm = e4.step_host(acts[k].pin_memory(), noise[k].pin_memory())
        assert np.array_equal(om.numpy(), oh.numpy()) and np.array_equal(rm.numpy(), rh.numpy())
        assert np.array_equal(dm.numpy(), dh.numpy()) and np.array_equal(tm.numpy(), th.numpy())
    e5 = make("shkadov", B)
    e5.reset()
    op, rp, dp, tp = e5.step_host(acts[0].numpy(), noise[0].numpy(), out=e5.alloc_host_outputs(pinned=False))
    assert np.array_equal(op.numpy(), outs[0][0].cpu().numpy()) and np.array_equal(rp.numpy(), outs[0][1].cpu().numpy())


def test_shkadov_philox_noise_sharding_invariance():
    """On-device noise depends on (seed, global env index, draw) only: a batch of 6 equals two
    shards of 3 with env_index_base 0 and 3; different seeds differ; noise stays inside +-sigma."""
    acts = torch.zeros(2, 6, 5, dtype=torch.float64)
    full = make("shkadov", 6, seed=77)
    a, b = make("shkadov", 3, seed=77, env_index_base=0), make("shkadov", 3, seed=77, env_index_base=3)
    other = make("shkadov", 6, seed=78)
    for e in (full, a, b, other):
        e.reset()
    full.step_fused(acts); a.step_fused(acts[:, :3]); b.step_fused(acts[:, 3:]); other.step_fused(acts)
    hf = full.get_state("h")
    assert torch.equal(hf[:3], a.get_state("h")) and torch.equal(hf[3:], b.get_state("h"))
    assert not torch.equal(hf, other.get_state("h"))
    assert not torch.equal(hf[0], hf[1])
    inlet = hf[:, 0] - 1.0
    assert float(inlet.abs().max()) <= 5.0e-4 and float(inlet.abs().min()) > 0.0


def test_shkadov_per_jet_rewards(golden):
    """separable rewards (shkadov.py:469-481): per-jet vector, same state as the joint env."""
    g = golden("shkadov")
    env = make("shkadov", 1, n_jets=4, per_jet_rwd=True, sigma=0.0)
    obs0 = env.reset()
    close(obs0.reshape(4, 10), g["sep_reset_obs"], what="sep reset obs")
    for k in range(2):
        obs, rwd, d, t = env.step(torch.as_tensor(g["sep_actions"][k][None]), noise=torch.zeros(1, 50, dtype=torch.float64))
        close(obs.reshape(4, 10), g["sep_obs"][4 * k:4 * k + 4], what="sep obs")
        close(rwd.reshape(4), g["sep_rwd"][4 * k:4 * k + 4], rtol=1e-12, what="sep rwd")
    close(env.get_state("h")[0], g["sep_h"], what="h")


# ----------------------------------------------------------------------------- burgers / sloshing / ODEs
def test_burgers_golden(golden):
    g = golden("burgers")
    B = 2
    env = make("burgers", B)
    close(env.reset(), rep(g["obs0"], B), what="obs0")
    for k in range(g["actions"].shape[0]):
        obs, rwd, d, t = env.step(rep(g["actions"][k], B), noise=rep(g["noise"][k:k + 1], B))
        for f in ("u", "up", "upp"):
            close(env.get_state(f), rep(g[f][k], B), what=f"{f} step {k}")
        close(obs, rep(g["obs"][k], B), what="obs")
        close(rwd, rep(g["rwd"][k], B), rtol=1e-12, what="rwd")


def test_burgers_kat_full_episode():
    """configs[0]: one 200-action episode with random actions, single env, against the oracle."""
    rng = np.random.default_rng(14)
    env = make("burgers", 1)
    o = bo.burgers()
    env.reset(); o.reset()
    acts, noise = rng.uniform(-1, 1, (200, 1, 1)), rng.uniform(-0.1, 0.1, (200, 1, 1))
    obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts), torch.as_tensor(noise))
    ref = [o.step(acts[k, 0], noise=float(noise[k, 0, 0])) for k in range(200)]
    close(obs[:, 0], np.stack([r[0] for r in ref]), rtol=1e-9, what="obs trajectory")
    ret_o = sum(r[1] for r in ref)
    assert abs(float(rwd.sum()) - ret_o) <= 1e-9 * abs(ret_o)
    assert [bool(x) for x in done[:, 0]] == [r[2] for r in ref] and bool(done[-1, 0]) and bool(trunc[-1, 0])
    close(env.get_state("u")[0], o.u, rtol=1e-9, what="u")


def test_sloshing_golden(golden):
    g = golden("sloshing")
    B = 2
    env = make("sloshing", B)
    close(env.reset(), rep(g["obs0"], B), what="obs0")
    for k in range(g["actions"].shape[0]):
        obs, rwd, d, t = env.step(rep(g["actions"][k], B))
        for f in ("h", "q", "rhsh", "rhsq"):
            close(env.get_state(f), rep(g[f][k], B), what=f"{f} step {k}", floor=1.0 if f.startswith("rhs") else 1e-2)
        close(obs, rep(g["obs"][k], B), what="obs")
        close(rwd, rep(g["rwd"][k], B), rtol=1e-12, what="rwd")


def test_sloshing_episode_vs_oracle():
    rng = np.random.default_rng(15)
    env = make("sloshing", 3)
    orcs = [bo.sloshing() for _ in range(3)]
    env.reset()
    [o.reset() for o in orcs]
    acts = rng.uniform(-1, 1, (200, 3, 1))
    obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts))
    ref = [[o.step(acts[k, b]) for k in range(200)] for b, o in enumerate(orcs)]
    for b in range(3):
        ret = sum(r[1] for r in ref[b])
        assert abs(float(rwd[:, b].sum()) - ret) <= 1e-9 * abs(ret)
        close(env.get_state("h")[b], orcs[b].h, rtol=1e-9, what="h")
    assert bool(done[-1].all()) and not bool(done[:-1].any())


def test_lorenz_golden_and_resync(golden):
    g = golden("lorenz")
    env = make("lorenz", 2)
    close(env.reset(), rep(g["obs0"], 2), what="obs0")
    o = bo.lorenz()
    o.reset()
    n_exact = 0
    for k, a in enumerate(g["actions"]):
        env.set_state("x", rep(o.x, 2)); env.set_state("fx", rep(o.fx, 2))       # re-sync (chaotic)
        obs, rwd, d, t = env.step(torch.full((2,), int(a)))
        ro = o.step(int(a))
        close(obs, rep(g["obs"][k], 2), what=f"obs step {k}")
        assert float(rwd[0]) == g["rwd"][k] == ro[1]
        n_exact += 1
    # free-running 100 steps: rewards identical (SURVEY.md §8c)
    env.reset(); o.reset()
    acts = np.arange(100) % 3
    _, rwd, done, _ = env.step_fused(torch.as_tensor(acts[:, None].repeat(2, 1)))
    assert [float(x) for x in rwd[:, 0]] == [o.step(int(a))[1] for a in acts]


def test_vortex_golden(golden):
    g = golden("vortex")
    env = make("vortex", 2)
    close(env.reset(), rep(g["obs0"], 2), what="obs0")
    acts = torch.as_tensor(np.repeat(g["actions"][:, None, :], 2, axis=1))
    obs, rwd, d, t = env.step_fused(acts)
    a = obs[:, 0].cpu().numpy()
    assert np.max(np.abs(a - g["obs"]) / (np.abs(g["obs"]) + 1e-12)) < 1e-9
    assert np.max(np.abs(rwd[:, 0].cpu().numpy() - g["rwd"])) <= 1e-9 * np.max(np.abs(g["rwd"]))


# ----------------------------------------------------------------------------- rayleigh / mixing
@pytest.mark.parametrize("name,scal", [("rayleigh", "T"), ("mixing", "C")])
def test_mac2d_golden(golden, name, scal):
    g = golden(name)
    B = 2
    env = make(name, B)
    close(env.reset(), rep(g["obs0"], B), what="obs0")
    for k in range(g["actions"].shape[0]):
        act = rep(g["actions"][k], B)
        obs, rwd, d, t = env.step(act, want_iters=True)
        assert int(env.last_iters[0, 0]) == int(g["itp"][k].sum()), "Jacobi sweep count differs from the reference"
        for f in ("u", "v", "p", scal):
            close(env.get_state(f), rep(g[f][k].reshape(-1), B), what=f"{f} step {k}")
        close(obs, rep(g["obs"][k], B), what="obs")
        close(rwd, rep(g["rwd"][k], B), rtol=1e-12, what="rwd")
    assert int(env.status.max()) == 0


def test_rayleigh_vs_oracle_batch():
    """different actions per env, 3 free-running actions (rayleigh is not chaotic at Ra=1e4)."""
    rng = np.random.default_rng(16)
    B = 4
    env = make("rayleigh", B)
    orcs = [bo.rayleigh() for _ in range(B)]
    env.reset()
    [o.reset() for o in orcs]
    for k in range(3):
        acts = rng.uniform(-1, 1, (B, 10))
        obs, rwd, d, t = env.step(torch.as_tensor(acts), want_iters=True)
        ref = [o.step(acts[b]) for b, o in enumerate(orcs)]
        assert [int(x) for x in env.last_iters[0]] == [int(o.last_iters.sum()) for o in orcs]
        for f in ("u", "v", "p", "T"):
            close(env.get_state(f), np.stack([getattr(o, f).reshape(-1) for o in orcs]), what=f"{f} action {k}")
        close(env.get_state("a"), np.stack([o.a for o in orcs]), rtol=1e-15, what="conditioned action")
        close(obs, np.stack([r[0] for r in ref]), what="obs")
        close(rwd, np.array([r[1] for r in ref]), rtol=1e-12, what="rwd")


def test_probe_indices_bit_exact(golden):
    from beacon_b200.params import MixingCfg, RayleighCfg
    for name, cfg in (("rayleigh", RayleighCfg()), ("mixing", MixingCfg())):
        P = json.loads(str(golden(name)["params_json"]))
        for k, v in P.items():
            assert cfg.d[k] == v, (name, k)
    assert RayleighCfg().probe_indices()[:5] == [(6, 6), (6, 18), (6, 30), (6, 42), (18, 6)]
    assert MixingCfg().d["patch"] == (25, 75, 25, 75)


# ----------------------------------------------------------------------------- fp32 build, C-ABI behaviour
def test_fp32_tolerance(golden):
    g = golden("shkadov")
    env = make("shkadov", 2, n_jets=10, dtype=torch.float32)
    env.reset()
    env.step(rep(g["j10_actions"][0], 2), noise=rep(g["j10_noise"][0], 2))
    close(env.get_state("h"), rep(g["j10_h"][0], 2), rtol=1e-5, what="h fp32", floor=1.0)
    close(env.get_state("q"), rep(g["j10_q"][0], 2), rtol=1e-5, what="q fp32", floor=1.0)
    g = golden("sloshing")
    env = make("sloshing", 2, dtype=torch.float32)
    env.reset()
    env.step(rep(g["actions"][0], 2))
    close(env.get_state("h"), rep(g["h"][0], 2), rtol=1e-5, what="sloshing h fp32", floor=1.0)


def test_capi_errors_are_reported():
    from beacon_b200 import BatchedEnv, BeaconError
    with pytest.raises(BeaconError, match="jets outside"):
        BatchedEnv("shkadov", batch=1, n_jets=3, jet_pos=2.0)
    env = make("lorenz", 2)
    with pytest.raises(ValueError):
        env.step(torch.zeros(3, dtype=torch.int32))
    with pytest.raises(KeyError):
        env.get_state("nope")


# ----------------------------------------------------------------------------- generic 2D kernel (non-default grids)
def test_generic_mac_kernel(monkeypatch, golden):
    """Grids other than the two reference defaults take the generic one-CTA-per-env kernel (phi planes
    in shared memory, fields in global memory): rayleigh from rest on a 100x50 cell against the oracle,
    and — forced with BEACON_MAC_V1 — the reference's mixing golden step; sweep counts exact."""
    env = make("rayleigh", 2, init=False, L=2.0, H=1.0, n_sgts=5)
    o = bo.rayleigh(init=False, L=2.0, H=1.0, n_sgts=5)
    env.reset(); o.reset()
    assert env.cfg.d["nx"] == 100 and env.cfg.d["ny"] == 50
    rng = np.random.default_rng(31)
    for k in range(2):
        a = rng.uniform(-1, 1, 5)
        obs, rwd, d, t = env.step(torch.as_tensor(np.stack([a, a])), want_iters=True)
        ro = o.step(a)
        assert int(env.last_iters[0, 1]) == int(o.last_iters.sum())
        for f in ("u", "v", "p", "T"):
            close(env.get_state(f)[0], getattr(o, f).reshape(-1), what=f"rayleigh 100x50 {f}")
        close(obs[0], ro[0], what="obs")
        close(rwd[1:], np.array([ro[1]]), rtol=1e-12, what="rwd")
    assert int(env.status.max()) == 0
    monkeypatch.setenv("BEACON_MAC_V1", "1")
    g = golden("mixing")
    env = make("mixing", 1)
    env.reset()
    obs, rwd, d, t = env.step(torch.tensor([int(g["actions"][0])], dtype=torch.int32), want_iters=True)
    assert int(env.last_iters[0, 0]) == int(g["itp"][0].sum())
    for f in ("u", "v", "p", "C"):
        close(env.get_state(f)[0], g[f][0].reshape(-1), what=f"mixing generic {f}")
    assert "us" in env.fields          # the generic kernel keeps the starred velocities as state fields


def test_rayleigh_on_the_large_grid_kernel():
    """A 100x100 rayleigh cell takes the large-grid kernel (register-resident Poisson, fields in L2) in its rayleigh
    instantiation — buoyancy term, segment temperatures, Neumann east wall in the residual — which the mixing tests
    do not reach: one action from rest against the oracle, sweep counts exact."""
    env = make("rayleigh", 2, init=False, L=2.0, H=2.0, n_sgts=5)
    o = bo.rayleigh(init=False, L=2.0, H=2.0, n_sgts=5)
    env.reset(); o.reset()
    assert env.cfg.d["nx"] == 100 and env.cfg.d["ny"] == 100
    a = np.random.default_rng(32).uniform(-1, 1, 5)
    obs, rwd, d, t = env.step(torch.as_tensor(np.stack([a, -a])), want_iters=True)
    ro = o.step(a)
    assert int(env.last_iters[0, 0]) == int(o.last_iters.sum())
    for f in ("u", "v", "p", "T"):
        close(env.get_state(f)[0], getattr(o, f).reshape(-1), what=f"rayleigh 100x100 {f}")
    close(obs[0], ro[0], what="obs")
    close(rwd[:1], np.array([ro[1]]), rtol=1e-12, what="rwd")
    assert int(env.status.max()) == 0


def test_mac2d_sweep_counts_soak():
    """More seeds for the data-dependent Jacobi trip counts: the lagged, register-resident solvers must
    stop on exactly the sweep the reference stops on (one sweep more or less changes phi by ~1e-6)."""
    rng = np.random.default_rng(41)
    B, K = 12, 6
    env = make("rayleigh", B)
    orcs = [bo.rayleigh() for _ in range(B)]
    env.reset()
    [o.reset() for o in orcs]
    for k in range(K):
        acts = rng.uniform(-1, 1, (B, 10)) * rng.choice([0.05, 0.5, 1.0, 3.0], size=(B, 1))
        obs, rwd, d, t = env.step(torch.as_tensor(acts), want_iters=True)
        ref = [o.step(acts[b]) for b, o in enumerate(orcs)]
        assert [int(x) for x in env.last_iters[0]] == [int(o.last_iters.sum()) for o in orcs], f"action {k}"
        close(env.get_state("T"), np.stack([o.T.reshape(-1) for o in orcs]), what=f"T action {k}")
        close(env.get_state("p"), np.stack([o.p.reshape(-1) for o in orcs]), what=f"p action {k}")
    env = make("mixing", 4)
    orcs = [bo.mixing() for _ in range(4)]
    env.reset()
    [o.reset() for o in orcs]
    for k in range(3):
        acts = rng.integers(0, 4, 4)
        obs, rwd, d, t = env.step(torch.as_tensor(acts, dtype=torch.int32), want_iters=True)
        ref = [o.step(int(acts[b])) for b, o in enumerate(orcs)]
        assert [int(x) for x in env.last_iters[0]] == [int(o.last_iters.sum()) for o in orcs], f"mixing action {k}"
        close(env.get_state("C"), np.stack([o.C.reshape(-1) for o in orcs]), what=f"C action {k}")
        close(env.get_state("p"), np.stack([o.p.reshape(-1) for o in orcs]), what=f"p action {k}")
        close(rwd, np.array([r[1] for r in ref]), rtol=1e-12, what="rwd")
