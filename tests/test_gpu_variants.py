"""Every kernel instance the host dispatchers can select, against the oracle.

The constructors pick a template instance and a chunk layout from nx, the batch size and the grid
(shkadov.cu BEACON_SHK_TRY, burgers.cu, sloshing.cu, mac2d.cu MacEnv).  The parity tests at the
reference's default sizes reach only the instances those sizes select; here each instance is reached
on purpose.  Each test mirrors the dispatch rule in a small helper and asserts the instance, the
chunk shift `off` and the warp role that its parametrization id names.  Where an environment
variable can force the instance (BEACON_SHKADOV_CFG, BEACON_BURGERS_C4), the forced run is compared
with the oracle too: the constructor throws if the named instance cannot cover the lattice, so a
forced run is guaranteed to execute it.

Norm and tolerances of DESIGN.md §4 (`close` of test_gpu_parity): fp64 fields 1e-10 per action
(floor 1 for rhsh / rhsq), fp32 1e-5 with floor 1, rewards 1e-12; sweep counts, flags and status
bits exact.
"""
import numpy as np
import pytest
import torch

from oracle import beacon_oracle as bo
from test_gpu_parity import close, make, rep

pytestmark = pytest.mark.gpu

RTOL32 = 1e-5


def _ids(cases):
    return [c.id for c in cases]


# ============================================================================= shkadov
SHK_PRODUCTION = ((6, 256, 2), (10, 192, 2), (6, 512, 1), (12, 512, 1))
SHK_TUNING = ((9, 160, 3), (9, 160, 2), (11, 128, 3), (11, 128, 2), (5, 640, 1), (10, 320, 1))


def shk_dispatch(nx, cfg=None):
    """Mirror of BEACON_SHK_TRY in shkadov.cu: the first (C, T, MINB) in this order whose C*T points
    cover nx plus the chunk shift off = (C - nx mod C) mod C; the tuning-only instances take part only
    when BEACON_SHKADOV_CFG = cfg names one.  Warp 0 runs the F_SMALL body when off <= 1 (inlet
    specials confined to m < 3), F_LARGE otherwise (thread 0 holds off phantom points and the inlet).
    Returns ((C, T, MINB), off, role), or (None, None, None) if no instance covers nx."""
    order = SHK_PRODUCTION[:1] + (SHK_TUNING if cfg else ()) + SHK_PRODUCTION[1:]
    for v in order:
        C, T, _ = v
        off = (C - nx % C) % C
        if (cfg is None or v == tuple(cfg)) and C * T >= nx + off:
            return v, off, ("F_SMALL" if off <= 1 else "F_LARGE")
    return None, None, None


def shk_l0(nx, n_jets=10):
    """The L0 whose lattice (shkadov.py:32-33, nx = int(5 (L0 + jet_space (n_jets + 2)))) has nx points."""
    from beacon_b200.params import ShkadovCfg
    base = nx / 5.0 - 10.0 * (n_jets + 2)
    for L0 in (round(base, 1), round(base + 0.1, 1), round(base - 0.1, 1)):
        if ShkadovCfg(init="rest", L0=L0, n_jets=n_jets).d["nx"] == nx:
            return L0
    raise AssertionError(f"no L0 gives nx = {nx} with {n_jets} jets")


def shk_synthetic(nx, row):
    """Multi-scale waves in h and q over the whole lattice (the shipped init field covers nx <= 2900 only,
    and a flat film leaves the limiter and the chunk-edge exchange untested)."""
    i = np.arange(nx, dtype=np.float64)
    p = 0.7 * row
    h = 1.0 + 0.3 * np.sin(2 * np.pi * i / 61 + p) + 0.12 * np.sin(2 * np.pi * i / 17.3 + 2 * p) + 0.04 * np.sin(2 * np.pi * i / 7.9 + 3 * p)
    q = 1.0 + 0.4 * np.sin(2 * np.pi * i / 47 + 1 + p) + 0.15 * np.sin(2 * np.pi * i / 13.1 + 2 + p) + 0.05 * np.sin(2 * np.pi * i / 6.3 + 3 * p)
    return h, q


def assert_minmod_branches(h, q, n):
    """The minmod ratio r = du_k / (du_{k+1} + 1e-8) of the TVD faces takes all three branches (r < 0,
    0 <= r <= 1, r > 1) within the first and within the last n points, for q and for q^2/h."""
    for what, u in (("q", q), ("q2h", q * q / (h + 1.0e-8))):
        d = np.diff(u)
        r = d[:-1] / (d[1:] + 1.0e-8)
        for side, w in (("inlet", r[:n]), ("outlet", r[-n:])):
            assert (w < 0).any() and ((w >= 0) & (w <= 1)).any() and (w > 1).any(), (what, side)


def shk_case(nx, n_jets, variant, off, role):
    return pytest.param(nx, n_jets, variant, off, role, id=f"nx{nx}-j{n_jets}-C{variant[0]}T{variant[1]}MB{variant[2]}-off{off}-{role}")


V6, V10, V6L, V12 = SHK_PRODUCTION
SHK_MATRIX = [
    # 6,256,2: nx + off <= 1536
    shk_case(1350, 10, V6, 0, "F_SMALL"),
    shk_case(1349, 10, V6, 1, "F_SMALL"),
    shk_case(1348, 10, V6, 2, "F_LARGE"),
    shk_case(1351, 10, V6, 5, "F_LARGE"),
    shk_case(1536, 10, V6, 0, "F_SMALL"),       # last nx of 6,256,2
    # 10,192,2: 1537 .. 1920
    shk_case(1537, 10, V10, 3, "F_LARGE"),      # first nx of 10,192,2
    shk_case(1539, 10, V10, 1, "F_SMALL"),
    shk_case(1538, 10, V10, 2, "F_LARGE"),
    shk_case(1541, 10, V10, 9, "F_LARGE"),
    shk_case(1853, 10, V10, 7, "F_LARGE"),
    shk_case(1850, 20, V10, 0, "F_SMALL"),      # 20 jets, default layout
    shk_case(1920, 10, V10, 0, "F_SMALL"),      # last nx of 10,192,2
    # 6,512,1: 1921 .. 3072
    shk_case(1921, 10, V6L, 5, "F_LARGE"),      # first nx of 6,512,1
    shk_case(1925, 10, V6L, 1, "F_SMALL"),
    shk_case(1924, 10, V6L, 2, "F_LARGE"),
    shk_case(3072, 10, V6L, 0, "F_SMALL"),      # last nx of 6,512,1
    # 12,512,1: 3073 .. 6144
    shk_case(3073, 10, V12, 11, "F_LARGE"),     # first nx of 12,512,1: thread 0 holds 11 phantom points and the inlet
    shk_case(3083, 10, V12, 1, "F_SMALL"),
    shk_case(3082, 10, V12, 2, "F_LARGE"),
    shk_case(3850, 60, V12, 2, "F_LARGE"),      # 60 jets, default layout
    shk_case(5550, 94, V12, 6, "F_LARGE"),      # 94 jets: the most the fp64 shared-memory budget takes
    shk_case(6144, 10, V12, 0, "F_SMALL"),      # last nx any instance covers
]
# one lattice per production instance with an F_LARGE warp 0 (off >= 2), for the fp32 and fused-launch cases
SHK_PER_INSTANCE = [shk_case(1351, 10, V6, 5, "F_LARGE"), shk_case(1853, 10, V10, 7, "F_LARGE"),
                    shk_case(1921, 10, V6L, 5, "F_LARGE"), shk_case(3073, 10, V12, 11, "F_LARGE")]


def _check_case(nx, n_jets, variant, off, role, cfg=None):
    assert shk_dispatch(nx, cfg) == (variant, off, role)


def _cfg_env(variant):
    return ",".join(str(x) for x in variant)


def shk_vs_oracle(envs, nx, n_jets, C, n_actions=3, rtol=1e-10, per_jet=False, seed=0, **kw):
    """Synthetic state into every env and the oracle, then n_actions actions with random jet actions and
    explicit inlet noise, each env re-synced from the oracle before each action (the film is chaotic,
    SURVEY.md §4); h, q, rhsh, rhsq, obs, rewards and flags compared after each action.  kw: further
    oracle constructor arguments (delta, jet_pos), the same the envs were made with."""
    B = envs[0].batch
    L0 = shk_l0(nx, n_jets)
    orcs = [bo.shkadov(init=False, L0=L0, n_jets=n_jets, **kw) for _ in range(B)]
    for b, o in enumerate(orcs):
        assert o.nx == nx
        o.h[:], o.q[:] = shk_synthetic(nx, b)
        assert_minmod_branches(o.h, o.q, 3 * C)
    fp32 = envs[0].dtype == torch.float32
    rng = np.random.default_rng(seed)
    for k in range(n_actions):
        acts = rng.uniform(-1, 1, (B, n_jets))
        noise = rng.uniform(-5e-4, 5e-4, (B, 50))
        for env in envs:
            for f in ("h", "q", "rhsh", "rhsq", "u", "up"):
                env.set_state(f, np.stack([getattr(o, f) for o in orcs]))
            env.set_state("stp", np.array([o.stp for o in orcs]))
        outs = [env.step(torch.as_tensor(acts), noise=torch.as_tensor(noise)) for env in envs]
        ref = [o.step(acts[b], noise=noise[b]) for b, o in enumerate(orcs)]
        if per_jet:
            rwd_ref = np.array([[bo.shkadov_separable.get_rwd(o, j) for j in range(n_jets)] for o in orcs])
        else:
            rwd_ref = np.array([r[1] for r in ref])
        for e, (env, (obs, rwd, done, trunc)) in enumerate(zip(envs, outs)):
            tag = f"env {e} action {k}"
            fields = ("h", "q") if fp32 else ("h", "q", "rhsh", "rhsq")
            for f in fields:
                floor = 1.0 if (fp32 or f.startswith("rhs")) else 1e-2
                close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), rtol=rtol, what=f"{f} {tag}", floor=floor)
            close(obs, np.stack([r[0] for r in ref]), rtol=rtol, what=f"obs {tag}", floor=1.0 if fp32 else 1e-2)
            close(rwd, rwd_ref, rtol=RTOL32 if fp32 else 1e-12, what=f"rwd {tag}", floor=1.0 if fp32 else 1e-2)
            assert [bool(x) for x in done] == [r[2] for r in ref] and [bool(x) for x in trunc] == [r[3] for r in ref], tag
            assert int(env.status.max()) == 0, tag
    return orcs


@pytest.mark.parametrize("nx,n_jets,variant,off,role", SHK_MATRIX, ids=_ids(SHK_MATRIX))
def test_shkadov_instance_offset_matrix(nx, n_jets, variant, off, role, monkeypatch):
    """Each production instance at offsets 0, 1, 2 and C-1 and on both sides of each capacity boundary,
    once as the dispatcher picks it and once forced with BEACON_SHKADOV_CFG."""
    _check_case(nx, n_jets, variant, off, role)
    _check_case(nx, n_jets, variant, off, role, cfg=variant)
    kw = dict(init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets)
    natural = make("shkadov", 2, **kw)
    monkeypatch.setenv("BEACON_SHKADOV_CFG", _cfg_env(variant))
    forced = make("shkadov", 2, **kw)
    assert natural.cfg.d["nx"] == nx
    shk_vs_oracle([natural, forced], nx, n_jets, variant[0], seed=nx)


TUNING_CASES = [shk_case(1349, 10, (9, 160, 3), 1, "F_SMALL"), shk_case(1351, 10, (9, 160, 2), 8, "F_LARGE"),
                shk_case(1350, 10, (11, 128, 3), 3, "F_LARGE"), shk_case(1398, 10, (11, 128, 2), 10, "F_LARGE"),
                shk_case(3073, 10, (5, 640, 1), 2, "F_LARGE"), shk_case(3199, 10, (10, 320, 1), 1, "F_SMALL")]


@pytest.mark.parametrize("nx,n_jets,variant,off,role", TUNING_CASES, ids=_ids(TUNING_CASES))
def test_shkadov_tuning_instances(nx, n_jets, variant, off, role, monkeypatch):
    """The instances only BEACON_SHKADOV_CFG selects (tools/sweep_shkadov.py): promoting one to the
    production list must not bring in an unverified kernel."""
    _check_case(nx, n_jets, variant, off, role, cfg=variant)
    monkeypatch.setenv("BEACON_SHKADOV_CFG", _cfg_env(variant))
    env = make("shkadov", 2, init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets)
    shk_vs_oracle([env], nx, n_jets, variant[0], seed=nx)


NOALIGN_CASES = [shk_case(1853, 10, V10, 7, "F_LARGE"), shk_case(3073, 10, V12, 11, "F_LARGE")]


@pytest.mark.parametrize("nx,n_jets,variant,off,role", NOALIGN_CASES, ids=_ids(NOALIGN_CASES))
def test_shkadov_general_path_wide_chunks(nx, n_jets, variant, off, role, monkeypatch):
    """BEACON_SHKADOV_NOALIGN: the general (per-point index test) body at C = 10 and C = 12 — the aligned
    layout of the id is replaced by off = 1 if (nx - 1) mod C == 0 else 0."""
    _check_case(nx, n_jets, variant, off, role, cfg=variant)
    monkeypatch.setenv("BEACON_SHKADOV_NOALIGN", "1")
    kw = dict(init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets)
    natural = make("shkadov", 2, **kw)
    monkeypatch.setenv("BEACON_SHKADOV_CFG", _cfg_env(variant))
    forced = make("shkadov", 2, **kw)
    shk_vs_oracle([natural, forced], nx, n_jets, variant[0], seed=nx + 1)


@pytest.mark.parametrize("nx,n_jets,variant,off,role", SHK_PER_INSTANCE, ids=_ids(SHK_PER_INSTANCE))
def test_shkadov_fp32_per_instance(nx, n_jets, variant, off, role, monkeypatch):
    _check_case(nx, n_jets, variant, off, role, cfg=variant)
    monkeypatch.setenv("BEACON_SHKADOV_CFG", _cfg_env(variant))
    env = make("shkadov", 2, init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, dtype=torch.float32)
    shk_vs_oracle([env], nx, n_jets, variant[0], n_actions=1, rtol=RTOL32, seed=nx + 2)


@pytest.mark.parametrize("nx,n_jets,variant,off,role", SHK_PER_INSTANCE, ids=_ids(SHK_PER_INSTANCE))
def test_shkadov_fused_equals_single_per_instance(nx, n_jets, variant, off, role, monkeypatch):
    """K = 3 actions in one launch equal three launches bitwise (on-device Philox noise: the draw counter
    advances inside the fused launch exactly as across launches)."""
    _check_case(nx, n_jets, variant, off, role, cfg=variant)
    monkeypatch.setenv("BEACON_SHKADOV_CFG", _cfg_env(variant))
    B, K = 3, 3
    kw = dict(init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, seed=5)
    e1, e2 = make("shkadov", B, **kw), make("shkadov", B, **kw)
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
    assert int(e1.get_state("draws")[0, 0]) == K * 50


def test_shkadov_per_jet_rewards_wide_chunks():
    """Separable rewards (shkadov.py:469-481) on the C = 12 instance with thread 0 holding 11 phantom points."""
    nx, n_jets = 3073, 10
    assert shk_dispatch(nx) == (V12, 11, "F_LARGE")
    env = make("shkadov", 2, init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, per_jet_rwd=True)
    assert env.rwd_dim == n_jets
    shk_vs_oracle([env], nx, n_jets, 12, per_jet=True, seed=3)


def test_shkadov_limits():
    """Host-side rejections, never a CUDA error: 95 jets in fp64 exceed the 227 KB shared-memory budget
    (94 fit, test_shkadov_instance_offset_matrix), in fp32 they fit; nx = 6145 has no instance."""
    from beacon_b200 import BeaconError
    with pytest.raises(BeaconError, match="shared-memory budget"):
        make("shkadov", 1, init="rest", n_jets=95)
    env = make("shkadov", 2, init="rest", n_jets=95, dtype=torch.float32)
    nx = env.cfg.d["nx"]
    assert nx == 5600 and shk_dispatch(nx) == (V12, 4, "F_LARGE")
    shk_vs_oracle([env], nx, 95, 12, n_actions=1, rtol=RTOL32, seed=4)
    assert shk_dispatch(6145) == (None, None, None)
    with pytest.raises(BeaconError, match="no kernel variant covers"):
        make("shkadov", 1, init="rest", L0=shk_l0(6145), n_jets=10)
    with pytest.raises(BeaconError, match="no kernel variant covers"):
        make("shkadov", 1, init="rest", L0=shk_l0(6145), n_jets=10, dtype=torch.float32)


def test_shkadov_warm_reset_order_at_scale():
    """3000 envs, masked warm reset with on-device noise: n_warm ~ U{0..400} with ties and a few at 3000
    (the 2048 bins of shkadov_order_kernel then hold ~1.5 warm-up lengths each, and its loops stride
    over the batch).  Every reset env advances its draw counter by exactly n_warm * ndt_act (reset once,
    by its own CTA), the other envs are untouched bitwise, and rows equal a batch-of-1 env at the same
    global index bitwise."""
    B, nj, seed = 3000, 5, 17
    rng = np.random.default_rng(61)
    nw = rng.integers(0, 401, B)
    nw[rng.choice(B, 200, replace=False)] = 137                 # ties
    nw[[7, 1500, 2001, 2999]] = 3000
    nw[0] = 0
    mask = rng.random(B) < 0.5
    mask[[0, 1500, 2999]] = True
    mask[[7, 2001]] = False                                     # a 3000 entry that is not reset
    env = make("shkadov", B, n_jets=nj, seed=seed)
    ndt = env.cfg.d["ndt_act"]
    env.reset()
    acts = torch.as_tensor(rng.uniform(-1, 1, (B, nj)))
    env.step(acts)                                               # every env away from the init state, draws = ndt
    before = {f: env.get_state(f).clone() for f in ("h", "q", "rhsh", "rhsq", "draws", "stp")}
    env.reset(mask=torch.as_tensor(mask), n_warm=torch.as_tensor(nw, dtype=torch.int32))
    after = {f: env.get_state(f) for f in before}

    def draws(t):
        w = t.cpu().numpy().astype(np.int64)
        return (w[:, 0] & 0xFFFFFFFF) | (w[:, 1] << 32)

    d0, d1 = draws(before["draws"]), draws(after["draws"])
    m = torch.as_tensor(mask, device=after["h"].device)
    assert np.array_equal(d1[mask], d0[mask] + nw[mask] * ndt)
    assert np.array_equal(d1[~mask], d0[~mask])
    for f in before:
        assert torch.equal(after[f][~m], before[f][~m]), f
    assert int(after["stp"][m].abs().max()) == 0
    for b in (0, 1500, 2999):
        one = make("shkadov", 1, n_jets=nj, seed=seed, env_index_base=b)
        one.reset()
        one.step(acts[b:b + 1])
        one.reset(n_warm=torch.tensor([int(nw[b])], dtype=torch.int32))
        for f in before:
            assert torch.equal(one.get_state(f)[0], after[f][b]), (b, f)


# ============================================================================= burgers
def burgers_variant(B, forced=False):
    """Mirror of BurgersEnv: (C, T) = (2, 256) for a batch of at most 296 (latency of one env), else
    (4, 128); BEACON_BURGERS_C4 forces (4, 128).  off = 1 if (nx - 1) mod C == 0 else 0 (0 at nx = 500)."""
    return (2, 256) if B <= 296 and not forced else (4, 128)


def burgers_synthetic(B, nx=500):
    """A travelling-wave history u, up, upp (BDF2) over the whole lattice, one phase per row."""
    i = np.arange(nx, dtype=np.float64)
    out = []
    for lag in (0.0, 0.02, 0.04):
        p = 0.7 * np.arange(B, dtype=np.float64)[:, None] - lag
        out.append(0.5 + 0.2 * np.sin(2 * np.pi * i / 53 + p) + 0.06 * np.sin(2 * np.pi * i / 11.7 + 2 * p))
    return out


def burgers_vs_oracle(env, rows, n_actions, rtol=1e-10, seed=0, **kw):
    B = env.batch
    env.reset()
    U = burgers_synthetic(B)
    for f, v in zip(("u", "up", "upp"), U):
        env.set_state(f, v)
    orcs = {b: bo.burgers(**kw) for b in rows}
    for b, o in orcs.items():
        o.reset()
        o.u[:], o.up[:], o.upp[:] = U[0][b], U[1][b], U[2][b]
    fp32 = env.dtype == torch.float32
    floor = 1.0 if fp32 else 1e-2
    rng = np.random.default_rng(seed)
    for k in range(n_actions):
        acts, noise = rng.uniform(-1, 1, (B, 1)), rng.uniform(-0.1, 0.1, (B, 1))
        obs, rwd, done, trunc = env.step(torch.as_tensor(acts), noise=torch.as_tensor(noise))
        ref = {b: o.step(acts[b], noise=float(noise[b, 0])) for b, o in orcs.items()}
        idx = list(rows)
        for f in ("u",) if fp32 else ("u", "up", "upp"):
            close(env.get_state(f)[idx], np.stack([getattr(orcs[b], f) for b in idx]), rtol=rtol, what=f"{f} action {k}", floor=floor)
        close(obs[idx], np.stack([ref[b][0] for b in idx]), rtol=rtol, what=f"obs action {k}", floor=floor)
        close(rwd[idx], np.array([ref[b][1] for b in idx]), rtol=RTOL32 if fp32 else 1e-12, what=f"rwd action {k}", floor=floor)
        assert [bool(done[b]) for b in idx] == [ref[b][2] for b in idx]
        assert [bool(trunc[b]) for b in idx] == [ref[b][3] for b in idx]
    assert int(env.status.max()) == 0


def test_burgers_throughput_instance_batch_300():
    """B = 300 > 296 selects (4, 128) without any switch: per-row actions and noise, three rows against the oracle."""
    assert burgers_variant(300) == (4, 128)
    env = make("burgers", 300)
    burgers_vs_oracle(env, (0, 149, 299), 3, seed=71)


def test_burgers_throughput_instance_full_episode(monkeypatch):
    """The 200-action episode of test_burgers_kat_full_episode on the forced (4, 128) instance, two rows
    with their own actions and noise: return within 1e-9, flags exact, final u within 1e-9."""
    monkeypatch.setenv("BEACON_BURGERS_C4", "1")
    assert burgers_variant(2, forced=True) == (4, 128)
    rng = np.random.default_rng(14)
    B = 2
    env = make("burgers", B)
    orcs = [bo.burgers() for _ in range(B)]
    env.reset()
    [o.reset() for o in orcs]
    acts, noise = rng.uniform(-1, 1, (200, B, 1)), rng.uniform(-0.1, 0.1, (200, B, 1))
    obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts), torch.as_tensor(noise))
    for b, o in enumerate(orcs):
        ref = [o.step(acts[k, b], noise=float(noise[k, b, 0])) for k in range(200)]
        close(obs[:, b], np.stack([r[0] for r in ref]), rtol=1e-9, what=f"obs trajectory row {b}")
        ret_o = sum(r[1] for r in ref)
        assert abs(float(rwd[:, b].sum()) - ret_o) <= 1e-9 * abs(ret_o)
        assert [bool(x) for x in done[:, b]] == [r[2] for r in ref] and [bool(x) for x in trunc[:, b]] == [r[3] for r in ref]
        close(env.get_state("u")[b], o.u, rtol=1e-9, what=f"u row {b}")


def test_burgers_throughput_instance_fp32(monkeypatch):
    """Eight rows: in one action the face right of the inlet meets two same-sign differences (the van Leer
    branch that face must not take, burgers.py:231-243) in only some of the rows' states."""
    monkeypatch.setenv("BEACON_BURGERS_C4", "1")
    env = make("burgers", 8, dtype=torch.float32)
    burgers_vs_oracle(env, range(8), 1, rtol=RTOL32, seed=72)


BURGERS_CTRL = [pytest.param(x, lat, forced, id=f"ctrl{lat}-C{burgers_variant(2, forced)[0]}T{burgers_variant(2, forced)[1]}")
                for x, lat in ((0.02, 5), (1.99, 497)) for forced in (False, True)]


@pytest.mark.parametrize("ctrl_pos,lattice,forced", BURGERS_CTRL, ids=_ids(BURGERS_CTRL))
def test_burgers_control_point_at_the_edges(ctrl_pos, lattice, forced, monkeypatch):
    """ctrl_pos 0.02 (lattice 5: the first legal probe window) and 1.99 (lattice 497: beside the last updated
    point 498 and the outlet copy 499, inside the last chunk) in both instances."""
    if forced:
        monkeypatch.setenv("BEACON_BURGERS_C4", "1")
    env = make("burgers", 2, ctrl_pos=ctrl_pos)
    assert env.cfg.d["ctrl_pos"] == lattice
    burgers_vs_oracle(env, (0, 1), 3, seed=lattice, ctrl_pos=ctrl_pos)


# ============================================================================= sloshing
def sloshing_layout(nx):
    """Mirror of SloshingEnv: nx + 2 cells (ghosts included) in 64 threads x 4; off = 1 when (nx + 1) mod 4 == 0
    so that ghost nx+1 shares a chunk with cell nx.  Returns off, or None above the 255-slot capacity."""
    if nx + 2 > 4 * 64 - 1:
        return None
    return 1 if (nx + 1) % 4 == 0 else 0


def sloshing_L(nx):
    from beacon_b200.params import SloshingCfg
    for L in (round(nx / 80, 4), round((nx + 0.5) / 80, 4)):
        if SloshingCfg(init="rest", L=L).d["nx"] == nx:
            return L
    raise AssertionError(nx)


SLOSH_CASES = [pytest.param(nx, off, id=f"nx{nx}-off{off}") for nx, off in ((80, 0), (203, 1), (251, 1), (253, 0))]


def sloshing_vs_oracle(env, nx, n_actions, rtol, seed):
    B = env.batch
    L = sloshing_L(nx)
    orcs = [bo.sloshing(init=False, L=L) for _ in range(B)]
    for o in orcs:
        o.reset()
        o.h[:] = 1.0                                            # rest, like init="rest"
    obs0 = env.reset()
    close(obs0, np.stack([o.get_obs() for o in orcs]), what="obs0")
    fp32 = env.dtype == torch.float32
    floor = 1.0 if fp32 else 1e-2
    rng = np.random.default_rng(seed)
    for k in range(n_actions):
        acts = rng.choice([-1.0, 1.0], (B, 1)) * rng.uniform(0.5, 1.0, (B, 1))
        obs, rwd, done, trunc = env.step(torch.as_tensor(acts))
        ref = [o.step(acts[b]) for b, o in enumerate(orcs)]
        for f in ("h", "q") if fp32 else ("h", "q", "rhsh", "rhsq"):
            close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), rtol=rtol, what=f"{f} action {k}",
                  floor=1.0 if (fp32 or f.startswith("rhs")) else 1e-2)
        close(obs, np.stack([r[0] for r in ref]), rtol=rtol, what=f"obs action {k}", floor=floor)
        close(rwd, np.array([r[1] for r in ref]), rtol=RTOL32 if fp32 else 1e-12, what=f"rwd action {k}", floor=floor)
        assert [bool(x) for x in done] == [r[2] for r in ref] and [bool(x) for x in trunc] == [r[3] for r in ref]
    assert int(env.status.max()) == 0


@pytest.mark.parametrize("nx,off", SLOSH_CASES, ids=_ids(SLOSH_CASES))
def test_sloshing_chunk_layouts(nx, off):
    """off = 1 (nx = 3 mod 4), the capacity edge (nx 253: 255 of 256 slots, odd n_obs) and a short tank,
    from rest with three exciting actions."""
    assert sloshing_layout(nx) == off
    env = make("sloshing", 2, init="rest", L=sloshing_L(nx))
    assert env.cfg.d["nx"] == nx and env.n_obs == (nx + 1) // 2
    sloshing_vs_oracle(env, nx, 3, 1e-10, seed=nx)


def test_sloshing_off1_fp32():
    assert sloshing_layout(251) == 1
    env = make("sloshing", 2, init="rest", L=sloshing_L(251), dtype=torch.float32)
    sloshing_vs_oracle(env, 251, 1, RTOL32, seed=252)


def test_sloshing_capacity_rejected():
    from beacon_b200 import BeaconError
    for L in (sloshing_L(254), 3.2):
        assert sloshing_layout(int(80 * L)) is None
        with pytest.raises(BeaconError, match="not supported"):
            make("sloshing", 1, init="rest", L=L)


# ============================================================================= mac2d
def mac_dispatch(kind, nx, ny, n_sgts=0, real_bytes=8):
    """Mirror of MacEnv: (kernel, tiles of 4x5 cells, transport passes).  rayleigh 50x50 with n_sgts <= 32:
    mac_reg_kernel; any 100x100 grid: mac_big_kernel; else the generic mac_kernel on one CTA per env (G = 1)
    when two planes fit in shared memory and the 4x5 tiles in 512 threads; else None (rejected)."""
    ld, n = ny + 2, (nx + 2) * (ny + 2)
    tiles = ((nx + 3) // 4) * ((ny + 4) // 5)
    if kind == "rayleigh" and nx == ny == 50 and n_sgts <= 32:
        kernel = "mac_reg_kernel"
    elif nx == ny == 100:
        kernel = "mac_big_kernel"
    elif 2 * n * real_bytes + 1024 <= 220 * 1024 and tiles <= 512:
        kernel = "mac_kernel"
    else:
        return None, tiles, None
    p = 1
    while 3 * ((nx + p - 1) // p) * ld > 2 * n or (nx + p - 1) // p > 32 * 2:
        p += 1
    return kernel, tiles, p


GENERIC_GRIDS = [pytest.param(L, H, nx, ny, tiles, tr_pass, id=f"{nx}x{ny}-tiles{tiles}-pass{tr_pass}")
                 for L, H, nx, ny, tiles, tr_pass in (
                     (1.5, 1.22, 75, 61, 247, 2),       # partial tiles in both directions
                     (4.0, 1.0, 200, 50, 500, 4),       # 500 of the 512 tile threads, four transport passes
                     (1.0, 2.0, 50, 100, 260, 2))]      # tall cell


@pytest.mark.parametrize("L,H,nx,ny,tiles,tr_pass", GENERIC_GRIDS, ids=_ids(GENERIC_GRIDS))
def test_generic_mac_kernel_grids(L, H, nx, ny, tiles, tr_pass):
    """The generic one-CTA-per-env kernel beyond the full-tile 100x50 cell of test_generic_mac_kernel:
    rayleigh from rest, two actions against the oracle, sweep counts exact."""
    assert mac_dispatch("rayleigh", nx, ny, 5) == ("mac_kernel", tiles, tr_pass)
    env = make("rayleigh", 2, init=False, L=L, H=H, n_sgts=5)
    o = bo.rayleigh(init=False, L=L, H=H, n_sgts=5)
    env.reset(); o.reset()
    assert env.cfg.d["nx"] == nx and env.cfg.d["ny"] == ny
    rng = np.random.default_rng(31)
    for k in range(2):
        a = rng.uniform(-1, 1, 5)
        obs, rwd, d, t = env.step(torch.as_tensor(np.stack([a, a])), want_iters=True)
        ro = o.step(a)
        assert [int(x) for x in env.last_iters[0]] == [int(o.last_iters.sum())] * 2, f"action {k}"
        for f in ("u", "v", "p", "T"):
            g = env.get_state(f)
            close(g[0], getattr(o, f).reshape(-1), what=f"rayleigh {nx}x{ny} {f} action {k}")
            assert torch.equal(g[0], g[1]), f"{f}: equal inputs, different rows"
        close(obs[0], ro[0], what="obs")
        close(rwd, np.array([ro[1]] * 2), rtol=1e-12, what="rwd")
    assert int(env.status.max()) == 0


def test_rayleigh_generic_kernel_200x50_fp32():
    """fp32 on the generic kernel's widest grid (500 tile threads, 4 transport passes), from rest: the
    Jacobi iteration meets the reference's tolerance within 5 % of the fp64 sweep count, fields within 1e-5."""
    assert mac_dispatch("rayleigh", 200, 50, 5, real_bytes=4) == ("mac_kernel", 500, 4)
    env = make("rayleigh", 2, init=False, L=4.0, H=1.0, n_sgts=5, dtype=torch.float32)
    o = bo.rayleigh(init=False, L=4.0, H=1.0, n_sgts=5)
    env.reset(); o.reset()
    a = np.random.default_rng(33).uniform(-1, 1, 5)
    obs, rwd, d, t = env.step(torch.as_tensor(np.stack([a, a])).float(), want_iters=True)
    ro = o.step(a)
    assert int(env.status.max()) == 0, "fp32 Poisson iteration hit itmax"
    it, it_ref = int(env.last_iters[0, 0]), int(o.last_iters.sum())
    assert abs(it - it_ref) <= 0.05 * it_ref, (it, it_ref)
    for f in ("u", "v", "T"):
        close(env.get_state(f)[0], getattr(o, f).reshape(-1), rtol=RTOL32, what=f"rayleigh 200x50 {f} fp32", floor=1.0)
    close(obs[0], ro[0], rtol=RTOL32, what="obs fp32", floor=1.0)


REG_CASES = [pytest.param(n, k, acts, id=f"n_sgts{n}-{k}") for n, k, acts in
             ((3, "mac_reg_kernel", 2), (7, "mac_reg_kernel", 2), (32, "mac_reg_kernel", 2), (33, "mac_kernel", 1))]


@pytest.mark.parametrize("n_sgts,kernel,n_actions", REG_CASES, ids=_ids(REG_CASES))
def test_rayleigh_segment_layouts(n_sgts, kernel, n_actions):
    """Heater segments that do not tile the bottom wall (50 // n_sgts columns each, the rest unheated),
    up to the 32 the register kernel takes; 33 falls to the generic kernel.  From the shipped state,
    different actions per env, sweep counts exact."""
    assert mac_dispatch("rayleigh", 50, 50, n_sgts)[0] == kernel
    B = 2
    env = make("rayleigh", B, n_sgts=n_sgts)
    orcs = [bo.rayleigh(n_sgts=n_sgts) for _ in range(B)]
    assert env.cfg.d["nx_sgts"] == 50 // n_sgts
    env.reset()
    [o.reset() for o in orcs]
    rng = np.random.default_rng(n_sgts)
    for k in range(n_actions):
        acts = rng.uniform(-1, 1, (B, n_sgts))
        obs, rwd, d, t = env.step(torch.as_tensor(acts), want_iters=True)
        ref = [o.step(acts[b]) for b, o in enumerate(orcs)]
        assert [int(x) for x in env.last_iters[0]] == [int(o.last_iters.sum()) for o in orcs], f"action {k}"
        for f in ("u", "v", "p", "T"):
            close(env.get_state(f), np.stack([getattr(o, f).reshape(-1) for o in orcs]), what=f"{f} action {k}")
        close(env.get_state("a"), np.stack([o.a for o in orcs]), rtol=1e-15, what="conditioned action")
        close(obs, np.stack([r[0] for r in ref]), what="obs")
        close(rwd, np.array([r[1] for r in ref]), rtol=1e-12, what="rwd")
    assert int(env.status.max()) == 0


def test_smaller_env_keeps_the_shared_memory_limit():
    """The dynamic shared-memory limit is an attribute of the kernel function, shared by every env on that
    instance: creating a smaller env after a larger one must not lower it below what the larger env launches
    with.  mac_kernel: rayleigh 200x50 (168,064 B), then 75x61 (77,616 B); shkadov 6,256,2: nx 1536, then 1350.
    Both envs of each pair are reset and stepped after both were created."""
    assert mac_dispatch("rayleigh", 200, 50, 5)[0] == mac_dispatch("rayleigh", 75, 61, 5)[0] == "mac_kernel"
    kws = [dict(init=False, L=4.0, H=1.0, n_sgts=5), dict(init=False, L=1.5, H=1.22, n_sgts=5)]
    envs = [make("rayleigh", 2, **kw) for kw in kws]
    for env in envs:
        env.reset()
        env.step(torch.zeros(2, 5, dtype=torch.float64))
        assert int(env.status.max()) == 0
    assert shk_dispatch(1536)[0] == shk_dispatch(1350)[0] == V6
    envs = [make("shkadov", 2, init="rest", L0=shk_l0(nx), n_jets=10) for nx in (1536, 1350)]
    for env in envs:
        obs0 = env.reset()
        obs, rwd, d, t = env.step(torch.zeros(2, 10, dtype=torch.float64))
        assert obs.shape == obs0.shape and bool(torch.isfinite(obs).all())


def test_mac2d_grids_rejected():
    """50x200 rayleigh needs 520 tiles of 4x5 cells (512 threads); a 200x100 mixing grid needs more than
    two planes of shared memory: both are host-side rejections."""
    from beacon_b200 import BeaconError
    assert mac_dispatch("rayleigh", 50, 200, 5) == (None, 520, None)
    assert mac_dispatch("mixing", 200, 100)[0] is None
    with pytest.raises(BeaconError, match="grid too large"):
        make("rayleigh", 1, init=False, L=1.0, H=4.0, n_sgts=5)
    with pytest.raises(BeaconError, match="grid too large"):
        make("mixing", 1, L=2.0)
