"""The kernels away from the reference's default run-time values, against the oracle.

The parity and variant suites run every environment at the reference's default physical constants, compare
on-device inlet noise only with other on-device runs and never reach the Poisson iteration cap.  A kernel that
ignored one of these values would pass them.  Here:

  A. physical parameters off their defaults, per kernel instance (the instance each id names is asserted with
     the dispatch mirrors of test_gpu_variants / test_gpu_mac_cluster).  Every case carries a separation
     guard: the oracle run with one parameter back at its default (once per parameter) moves at least one
     compared output by >= 1e3 x its tolerance, so the case fails if the kernel ignores that parameter;
  B. on-device Philox noise against a Python model of the draw, fed to the oracle (fields compared, not the
     noise bits: nvcc may contract -s + 2 s u into an FMA);
  C. the Poisson iteration cap (status bit BEACON_STATUS_POISSON_OVERFLOW) on all five MAC paths, at
     itmax = M (no overflow) and M - 1 (overflow), M being the largest per-sub-step sweep count of the action.

Norm and tolerances of DESIGN.md §4 (`close` of test_gpu_parity): fp64 1e-10 per action, 1e-9 after
free-running episodes, rewards 1e-12; fp32 1e-5 with floor 1; sweep counts, flags and status bits exact.
"""
import functools

import numpy as np
import pytest
import torch

from oracle import beacon_oracle as bo
from test_gpu_mac_cluster import cluster_fit
from test_gpu_parity import close, make
from test_gpu_variants import (RTOL32, SHK_PER_INSTANCE, V6, V12, _cfg_env, _ids, burgers_synthetic, burgers_variant,
                               burgers_vs_oracle, mac_dispatch, shk_dispatch, shk_l0, shk_synthetic,
                               shk_vs_oracle)

pytestmark = pytest.mark.gpu

OVERFLOW = 2            # BEACON_STATUS_POISSON_OVERFLOW
GUARD = 1e3


# ============================================================================= separation guard
def moved(a, b, rtol, floor=1e-2):
    """max |a - b| in units of the `close` bound of b: how far an output moved, in tolerances."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = max(1.0, float(np.max(np.abs(b))))
    return float(np.max(np.abs(a - b) / (rtol * (np.abs(b) + floor * scale))))


def assert_separated(run, params, defaults, rtols):
    """run(**params) -> tuple of outputs compared by the case; rtols: (rtol, floor) per output.  With each
    parameter back at its default, some output must move by >= GUARD tolerances."""
    ref = run(**params)
    for k in params:
        if k not in defaults:
            continue
        alt = run(**{**params, k: defaults[k]})
        m = max(moved(x, y, r, f) for x, y, (r, f) in zip(alt, ref, rtols))
        assert m >= GUARD, f"{k} = {params[k]} vs default {defaults[k]}: outputs move by only {m:.3g} tolerances"


# ============================================================================= A. shkadov
def shk_oracle_once(nx, n_jets, **kw):
    """One action of the oracle from the synthetic state, fixed actions and noise: (h, q, obs, rwd)."""
    o = bo.shkadov(init=False, L0=shk_l0(nx, n_jets), n_jets=n_jets, **kw)
    o.h[:], o.q[:] = shk_synthetic(nx, 0)
    rng = np.random.default_rng(1)
    obs, rwd = o.step(rng.uniform(-1, 1, n_jets), noise=rng.uniform(-5e-4, 5e-4, o.ndt_act))[:2]
    return o.h.copy(), o.q.copy(), obs, np.array([rwd])


SHK_FIELDS = ((1e-10, 1e-2), (1e-10, 1e-2), (1e-10, 1e-2), (1e-12, 1e-2))


def _shk_env(nx, n_jets, variant, monkeypatch, dtype=torch.float64, **kw):
    assert shk_dispatch(nx, variant)[0] == variant
    monkeypatch.setenv("BEACON_SHKADOV_CFG", _cfg_env(variant))
    return make("shkadov", 2, init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, dtype=dtype, **kw)


@pytest.mark.parametrize("nx,n_jets,variant,off,role", SHK_PER_INSTANCE, ids=_ids(SHK_PER_INSTANCE))
def test_shkadov_delta_per_instance(nx, n_jets, variant, off, role, monkeypatch):
    """delta = 0.25 (p5d = 1 / (5 delta) = 0.8 instead of 2) on each production instance."""
    assert shk_dispatch(nx, variant) == (variant, off, role)
    assert_separated(lambda **kw: shk_oracle_once(nx, n_jets, **kw), dict(delta=0.25), dict(delta=0.1), SHK_FIELDS)
    env = _shk_env(nx, n_jets, variant, monkeypatch, delta=0.25)
    shk_vs_oracle([env], nx, n_jets, variant[0], seed=nx + 5, delta=0.25)


def test_shkadov_delta_general_path_and_fp32(monkeypatch):
    """delta = 0.25 on the general (per-point index test) body, and in fp32 on 6,256,2."""
    nx, n_jets = 3073, 10
    assert shk_dispatch(nx) == (V12, 11, "F_LARGE")
    monkeypatch.setenv("BEACON_SHKADOV_NOALIGN", "1")
    env = make("shkadov", 2, init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, delta=0.25)
    shk_vs_oracle([env], nx, n_jets, 12, seed=6, delta=0.25)
    monkeypatch.delenv("BEACON_SHKADOV_NOALIGN")
    assert shk_dispatch(1351) == (V6, 5, "F_LARGE")
    env = _shk_env(1351, 10, V6, monkeypatch, dtype=torch.float32, delta=0.25)
    shk_vs_oracle([env], 1351, 10, 6, n_actions=1, rtol=RTOL32, seed=7, delta=0.25)


def _jet_phase(nx, n_jets, jet_pos, C):
    """(jz0 + off) mod C: where the first jet zone (jz0 = jet_pos - jet_hw) starts inside its chunk; None when
    jet_pos lands on the default's lattice point (the case would not move the jets)."""
    from beacon_b200.params import ShkadovCfg
    cfg = lambda x: ShkadovCfg(init="rest", L0=shk_l0(nx, n_jets), n_jets=n_jets, jet_pos=x).d
    d = cfg(jet_pos)
    assert d["nx"] == nx
    if d["jet_pos"] == cfg(150.0)["jet_pos"]:
        return None
    return (d["jet_pos"] - d["jet_hw"] + (C - nx % C) % C) % C


def _jet_cases():
    out = []
    for nx, variant, phases in ((1100, V6, range(6)), (3100, V12, (0, 1, 11))):
        C = variant[0]
        for ph in phases:               # the first jet_pos above the default 150 with this phase
            jp = next(x for x in (round(150.1 + 0.1 * k, 1) for k in range(200)) if _jet_phase(nx, 5, x, C) == ph)
            out.append(pytest.param(nx, variant, jp, id=f"nx{nx}-C{C}T{variant[1]}-jet_pos{jp}-phase{ph}"))
    # bounds on nx 1100: the first probe on lattice point 0; the reward zone of the last jet ending at nx
    out += [pytest.param(1100, V6, 10.0, id="nx1100-C6T256-jet_pos10.0-first-probe0"),
            pytest.param(1100, V6, 170.0, id="nx1100-C6T256-jet_pos170.0-reward-zone-to-nx")]
    return out


JET_CASES = _jet_cases()


@pytest.mark.parametrize("nx,variant,jet_pos", JET_CASES, ids=_ids(JET_CASES))
def test_shkadov_jet_pos_chunk_phases(nx, variant, jet_pos, monkeypatch):
    """jet_pos moves the jet zones across the chunk boundaries of the aligned layout (5 jets)."""
    from beacon_b200.params import ShkadovCfg
    d = ShkadovCfg(init="rest", L0=shk_l0(nx, 5), n_jets=5, jet_pos=jet_pos).d
    if jet_pos == 10.0:
        assert d["jet_pos"] - d["l_obs"] == 0
    if jet_pos == 170.0:
        assert d["jet_pos"] + 4 * d["jet_space"] + d["l_rwd"] == nx
    assert_separated(lambda **kw: shk_oracle_once(nx, 5, **kw), dict(jet_pos=jet_pos), dict(jet_pos=150.0), SHK_FIELDS)
    env = _shk_env(nx, 5, variant, monkeypatch, jet_pos=jet_pos)
    shk_vs_oracle([env], nx, 5, variant[0], seed=int(10 * jet_pos), jet_pos=jet_pos)


# ============================================================================= A. burgers
BURGERS_DEFAULTS = dict(u_target=0.5, amp=10.0, L=2.0)
# At u_target 0.2, L 1.2 the oracle itself goes non-finite within a 200-action episode from reset (any amp tried,
# 6 to 15) and at amp 15 already within 3 actions from the synthetic state on some rows: that set runs 3 actions.
BURGERS_PARAMS = [pytest.param(dict(u_target=0.8, amp=4.0, L=3.0), 41, 166, 200, id="ut0.8-amp4-L3-ndt41"),
                  pytest.param(dict(u_target=0.2, amp=12.0, L=1.2), 104, 416, 0, id="ut0.2-amp12-L1.2-ndt104")]
BURGERS_INST = [pytest.param(2, id="B2-C2T256"), pytest.param(300, id="B300-C4T128")]


def burgers_oracle_once(**kw):
    o = bo.burgers(**kw)
    o.reset()
    U = burgers_synthetic(1)
    o.u[:], o.up[:], o.upp[:] = U[0][0], U[1][0], U[2][0]
    obs, rwd = o.step(np.array([0.7]), noise=0.05)[:2]
    return o.u.copy(), obs, np.array([rwd])


@pytest.mark.parametrize("B", BURGERS_INST)
@pytest.mark.parametrize("kw,ndt,ctrl,n_episode", BURGERS_PARAMS)
def test_burgers_params(kw, ndt, ctrl, n_episode, B):
    """Reset observation (u_target), a synthetic state for 3 actions and a free-running episode.
    ndt_act 41 is odd: the tail of the kernel's two-sub-step unroll runs."""
    from beacon_b200.params import BurgersCfg
    d = BurgersCfg(**kw).d
    assert (d["ndt_act"], d["ctrl_pos"]) == (ndt, ctrl)
    assert_separated(lambda **k: burgers_oracle_once(**k), kw, BURGERS_DEFAULTS, ((1e-10, 1e-2), (1e-10, 1e-2), (1e-12, 1e-2)))
    assert burgers_variant(B) == ((2, 256) if B == 2 else (4, 128))
    env = make("burgers", B, **kw)
    rows = (0, 1) if B == 2 else (0, 149, 299)
    close(env.reset(), np.full((B, 5), kw["u_target"]), rtol=1e-15, what="reset obs")
    burgers_vs_oracle(env, rows, 3, seed=103, **kw)      # (some seeds drive the oracle itself to NaN at L = 1.2)
    if not n_episode:
        return
    # free-running episode from the reset state, own actions and noise per row
    env.reset()
    rng = np.random.default_rng(ndt)
    acts, noise = rng.uniform(-1, 1, (n_episode, B, 1)), rng.uniform(-0.1, 0.1, (n_episode, B, 1))
    obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts), torch.as_tensor(noise))
    for b in rows:
        o = bo.burgers(**kw)
        o.reset()
        ref = [o.step(acts[k, b], noise=float(noise[k, b, 0])) for k in range(n_episode)]
        close(obs[:, b], np.stack([r[0] for r in ref]), rtol=1e-9, what=f"obs trajectory row {b}")
        ret = sum(r[1] for r in ref)
        assert abs(float(rwd[:, b].sum()) - ret) <= 1e-9 * abs(ret), (b, float(rwd[:, b].sum()), ret)
        assert [bool(x) for x in done[:, b]] == [r[2] for r in ref] and bool(trunc[-1, b])
        close(env.get_state("u")[b], o.u, rtol=1e-9, what=f"u row {b}")
    assert int(env.status.max()) == 0


def test_burgers_params_fp32():
    kw = dict(u_target=0.8, amp=4.0, L=3.0)
    env = make("burgers", 2, dtype=torch.float32, **kw)
    close(env.reset(), np.full((2, 5), 0.8), rtol=RTOL32, what="reset obs fp32", floor=1.0)
    burgers_vs_oracle(env, (0, 1), 1, rtol=RTOL32, seed=9, **kw)


# ============================================================================= A. sloshing
SLOSH_DEFAULTS = dict(g=9.81, amp=5.0, alpha=0.0005)


def slosh_oracle(L, rest, **kw):
    o = bo.sloshing(init=not rest, L=L, **kw)
    o.reset()
    if rest:
        o.h[:] = 1.0
    return o


def slosh_oracle_once(L, rest, **kw):
    o = slosh_oracle(L, rest, **kw)
    for a in (0.9, -0.8, 0.7):
        obs, rwd = o.step(np.array([a]))[:2]
    return o.h.copy(), obs, np.array([rwd])


def sloshing_L(nx):
    from test_gpu_variants import sloshing_L as f
    return f(nx)


# (L, init="rest"?, params, n_actions, layout off)
SLOSH_CASES = [pytest.param(2.5, False, dict(g=4.0, amp=3.0, alpha=0.05), 200, 0, id="shipped-nx200-off0-g4-amp3-alpha0.05-episode"),
               pytest.param(sloshing_L(203), True, dict(g=4.0, amp=3.0, alpha=0.05), 3, 1, id="rest-nx203-off1-g4-amp3-alpha0.05"),
               pytest.param(2.0, True, dict(g=15.0), 3, 0, id="rest-nx160-off0-g15"),
               pytest.param(sloshing_L(203), True, dict(g=15.0), 3, 1, id="rest-nx203-off1-g15")]


@pytest.mark.parametrize("L,rest,kw,n_actions,off", SLOSH_CASES)
def test_sloshing_params(L, rest, kw, n_actions, off):
    from test_gpu_variants import sloshing_layout
    nx = int(80 * L)
    assert sloshing_layout(nx) == off
    assert_separated(lambda **k: slosh_oracle_once(L, rest, **k), kw, SLOSH_DEFAULTS, ((1e-10, 1e-2), (1e-10, 1e-2), (1e-12, 1e-2)))
    B = 2
    env = make("sloshing", B, init="rest" if rest else True, L=L, **kw)
    assert env.cfg.d["nx"] == nx
    orcs = [slosh_oracle(L, rest, **kw) for _ in range(B)]
    close(env.reset(), np.stack([o.get_obs() for o in orcs]), what="obs0")
    rng = np.random.default_rng(nx + n_actions)
    lo, hi = (0.2, 0.5) if n_actions > 3 else (0.5, 1.0)     # the episode stays below the blow-up bound h = 2
    acts = rng.choice([-1.0, 1.0], (n_actions, B, 1)) * rng.uniform(lo, hi, (n_actions, B, 1))
    if n_actions > 3:          # free-running episode: one launch, return and final state within 1e-9
        obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts))
        for b, o in enumerate(orcs):
            ref = [o.step(acts[k, b]) for k in range(n_actions)]
            close(obs[:, b], np.stack([r[0] for r in ref]), rtol=1e-9, what=f"obs trajectory row {b}")
            ret = sum(r[1] for r in ref)
            assert abs(float(rwd[:, b].sum()) - ret) <= 1e-9 * abs(ret), (b, float(rwd[:, b].sum()), ret)
            assert [bool(x) for x in done[:, b]] == [r[2] for r in ref] and [bool(x) for x in trunc[:, b]] == [r[3] for r in ref]
            close(env.get_state("h")[b], o.h, rtol=1e-9, what=f"h row {b}")
        assert bool(done[-1].all()) and not bool(done[:-1].any())
    else:
        for k in range(n_actions):
            obs, rwd, done, trunc = env.step(torch.as_tensor(acts[k]))
            ref = [o.step(acts[k, b]) for b, o in enumerate(orcs)]
            for f in ("h", "q", "rhsh", "rhsq"):
                close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), what=f"{f} action {k}",
                      floor=1.0 if f.startswith("rhs") else 1e-2)
            close(obs, np.stack([r[0] for r in ref]), what=f"obs action {k}")
            close(rwd, np.array([r[1] for r in ref]), rtol=1e-12, what=f"rwd action {k}")
            assert [bool(x) for x in done] == [r[2] for r in ref]
    assert int(env.status.max()) == 0


def test_sloshing_params_fp32():
    L, kw = sloshing_L(251), dict(g=4.0, amp=3.0, alpha=0.05)
    env = make("sloshing", 2, init="rest", L=L, dtype=torch.float32, **kw)
    orcs = [slosh_oracle(L, True, **kw) for _ in range(2)]
    env.reset()
    acts = np.array([[0.9], [-0.6]])
    obs, rwd, _, _ = env.step(torch.as_tensor(acts))
    ref = [o.step(acts[b]) for b, o in enumerate(orcs)]
    for f in ("h", "q"):
        close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), rtol=RTOL32, what=f"{f} fp32", floor=1.0)
    close(rwd, np.array([r[1] for r in ref]), rtol=RTOL32, what="rwd fp32", floor=1.0)


# ============================================================================= A. lorenz / vortex
ODE_ROWS = (0, 127, 128, 255, 256, 299)        # both sides of each 128-thread block; 300 leaves a partial last block
ODE_B = 300


def lorenz_episode(n, seed=0, **kw):
    o = bo.lorenz(**kw)
    o.reset()
    acts = np.random.default_rng(seed).integers(0, 3, n)
    return o, acts, [o.step(int(a)) for a in acts]


@pytest.mark.parametrize("kw", [pytest.param(dict(sigma=6.0, rho=12.0, beta=2.0), id="sigma6-rho12-beta2"),
                                pytest.param(dict(rho=10.0), id="rho10")])
def test_lorenz_params_batch_300(kw):
    """Both parameter sets have a stable fixed point (|x0| stays well away from 0 on the oracle), so whole
    500-action episodes run free: observations within 1e-9, rewards identical, done exactly at the horizon.
    Every row has its own actions and is compared with its own oracle."""
    def run(**k):
        _, _, ref = lorenz_episode(20, **k)
        return (np.stack([r[0] for r in ref]),)
    assert_separated(run, kw, dict(sigma=10.0, rho=28.0, beta=8.0 / 3.0), ((1e-9, 1e-2),))
    env = make("lorenz", ODE_B, **kw)
    env.reset()
    n = env.n_act
    assert n == 500
    acts = np.random.default_rng(3).integers(0, 3, (n, ODE_B))
    obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts, dtype=torch.int32))
    for b in ODE_ROWS:
        o = bo.lorenz(**kw)
        o.reset()
        ref = [o.step(int(a)) for a in acts[:, b]]
        assert min(abs(float(r[0][0])) for r in ref) > 0.01, "x0 comes near the reward switch at 0"
        close(obs[:, b], np.stack([r[0] for r in ref]), rtol=1e-9, what=f"obs row {b}")
        assert [float(x) for x in rwd[:, b]] == [r[1] for r in ref], f"rewards row {b}"
        assert [bool(x) for x in done[:, b]] == [r[2] for r in ref] and bool(done[-1, b]) and bool(trunc[-1, b])


def test_vortex_params_batch_300():
    """re 80, weight 20: 200 free-running actions, each row its own actions and its own oracle."""
    kw = dict(re=80.0, weight=20.0)

    def run(**k):
        o = bo.vortex(**k)
        o.reset()
        rng = np.random.default_rng(0)
        ref = [o.step(rng.uniform(-1, 1, 2)) for _ in range(20)]
        return np.stack([r[0] for r in ref]), np.array([r[1] for r in ref])
    assert_separated(run, kw, dict(re=50.0, weight=50.0), ((1e-9, 1e-2), (1e-9, 1.0)))
    env = make("vortex", ODE_B, **kw)
    env.reset()
    n = 200
    acts = np.random.default_rng(4).uniform(-1, 1, (n, ODE_B, 2))
    obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts))
    for b in ODE_ROWS:
        o = bo.vortex(**kw)
        o.reset()
        ref = [o.step(acts[k, b]) for k in range(n)]
        close(obs[:, b], np.stack([r[0] for r in ref]), rtol=1e-9, what=f"obs row {b}")
        close(rwd[:, b], np.array([r[1] for r in ref]), rtol=1e-9, what=f"rwd row {b}", floor=1.0)
        assert [bool(x) for x in done[:, b]] == [r[2] for r in ref]


# ============================================================================= A. rayleigh / mixing
def mac_oracle(name, **kw):
    o = bo.rayleigh(**kw) if name == "rayleigh" else bo.mixing(**kw)
    o.reset()
    return o


def _key(kw):
    return tuple(sorted(kw.items()))


@functools.lru_cache(maxsize=None)
def mac_reference(name, kwk, acts):
    """Oracle run of each row's action sequence: per row a list of (step result, iters, u, v, p, scalar)."""
    kw = dict(kwk)
    out = []
    for row in acts:
        o = mac_oracle(name, **kw)
        res = []
        for a in row:
            r = o.step(np.array(a) if name == "rayleigh" else a)
            s = o.T if name == "rayleigh" else o.C
            res.append((r, int(o.last_iters.sum()), o.u.reshape(-1).copy(), o.v.reshape(-1).copy(), o.p.reshape(-1).copy(),
                        s.reshape(-1).copy()))
        out.append(res)
    return out


def mac_vs_oracle(env, name, kw, acts, rtol=1e-10):
    """acts: per row a tuple of actions.  Fields, obs, rewards and (fp64) sweep counts after every action."""
    B = env.batch
    fp32 = env.dtype == torch.float32
    ref = mac_reference(name, _key(kw), acts)
    scal = "T" if name == "rayleigh" else "C"
    for k in range(len(acts[0])):
        a = np.array([acts[b][k] for b in range(B)])
        obs, rwd, _, _ = env.step(torch.as_tensor(a, dtype=env.dtype) if name == "rayleigh" else torch.as_tensor(a, dtype=torch.int32),
                                  want_iters=True)
        it_ref = [ref[b][k][1] for b in range(B)]
        if fp32:
            for it, ir in zip(env.last_iters[0].tolist(), it_ref):
                assert abs(it - ir) <= 0.05 * ir, (it, ir)
        else:
            assert [int(x) for x in env.last_iters[0]] == it_ref, f"sweeps action {k}"
        floor = 1.0 if fp32 else 1e-2
        for i, f in enumerate(("u", "v", "p", scal)):
            if fp32 and f == "p":
                continue
            close(env.get_state(f), np.stack([ref[b][k][2 + i] for b in range(B)]), rtol=rtol, what=f"{f} action {k}", floor=floor)
        close(obs, np.stack([ref[b][k][0][0] for b in range(B)]), rtol=rtol, what=f"obs action {k}", floor=floor)
        close(rwd, np.array([ref[b][k][0][1] for b in range(B)]), rtol=RTOL32 if fp32 else 1e-12, what=f"rwd action {k}", floor=floor)
    assert int(env.status.max()) == 0


def _ray_acts(n_sgts, seed):
    rng = np.random.default_rng(seed)
    return tuple(tuple(tuple(rng.uniform(-1, 1, n_sgts)) for _ in range(2)) for _ in range(2))


def _mac_guard(name, kw, defaults, acts):
    def run(**k):
        r = mac_reference(name, _key({**kw, **k}), (acts[0][:1],))[0][0]
        return r[2], r[5], r[0][0]
    assert_separated(run, {k: v for k, v in kw.items() if k in defaults}, defaults, ((1e-10, 1e-2),) * 3)


# (id, ctor kwargs without ra, ra, env var, ctas_per_env, expected kernel, n_sgts)
RAY_CASES = [pytest.param(dict(), 2e4, None, 1, "mac_reg_kernel", 10, id="mac_reg-50x50-shipped-ra2e4"),
             pytest.param(dict(init=False, L=2.0, H=2.0, n_sgts=5), 2e4, None, 1, "mac_big_kernel", 5, id="mac_big-100x100-rest-ra2e4"),
             # ra >= pr / (0.5 / (dt (1/dx^2 + 1/dy^2)))^2 = 7.1e3 keeps the explicit diffusion stable at 50 cells per unit
             pytest.param(dict(init=False, L=2.0, H=1.0, n_sgts=5), 3e4, None, 1, "mac_kernel", 5, id="mac_kernel-G1-100x50-rest-ra3e4"),
             pytest.param(dict(), 2e4, None, 2, "mac_kernel", 10, id="mac_kernel-G2-50x50-shipped-ra2e4")]


@pytest.mark.parametrize("kw,ra,envvar,G,kernel,n_sgts", RAY_CASES)
def test_rayleigh_ra(kw, ra, envvar, G, kernel, n_sgts):
    """ra reaches the kernel through dcoef = sqrt(pr / ra) and tcoef = 1 / sqrt(pr ra): two actions, each env its own."""
    L, H = kw.get("L", 1.0), kw.get("H", 1.0)
    nx, ny = int(50 * L), int(50 * H)
    if G == 1:
        assert mac_dispatch("rayleigh", nx, ny, n_sgts)[0] == kernel
    else:
        assert cluster_fit(nx, ny, G) is not None
    kw = dict(kw, ra=ra)
    acts = _ray_acts(n_sgts, int(ra) + G)
    _mac_guard("rayleigh", kw, dict(ra=1.0e4), acts)
    env = make("rayleigh", 2, ctas_per_env=G, **kw)
    assert ("us" in env.fields) == (kernel == "mac_kernel")
    env.reset()
    mac_vs_oracle(env, "rayleigh", kw, acts)


def test_rayleigh_ra_fp32_mac_reg():
    kw = dict(ra=2e4)
    assert mac_dispatch("rayleigh", 50, 50, 10, real_bytes=4)[0] == "mac_reg_kernel"
    env = make("rayleigh", 2, dtype=torch.float32, **kw)
    env.reset()
    mac_vs_oracle(env, "rayleigh", kw, _ray_acts(10, 20001), rtol=RTOL32)


MIX_KW = dict(re=150.0, pe=5e3, side=0.3, C0=2.5)
MIX_DEFAULTS = dict(re=100.0, pe=10000.0, side=0.5, C0=1.0)
MIX_ACTS = ((2,), (0,))        # action 2 drives the side walls with u_max = re nu / L = 1.5
MIX_CASES = [pytest.param(None, 1, "mac_big_kernel", id="mac_big"),
             pytest.param("BEACON_MAC_V1", 1, "mac_kernel", id="mac_kernel-G1"),
             pytest.param(None, 2, "mac_kernel", id="mac_kernel-G2")]


@pytest.mark.parametrize("envvar,G,kernel", MIX_CASES)
def test_mixing_params(envvar, G, kernel, monkeypatch):
    """re (lid speed u_max = re nu / L and diffusion 1 / re), pe, side and C0 (patch and reward reference) in
    one case: reset observation and C, then one action per env (actions 2 and 0)."""
    if envvar:
        monkeypatch.setenv(envvar, "1")
    if G == 1:
        assert mac_dispatch("mixing", 100, 100)[0] == "mac_big_kernel"     # BEACON_MAC_V1 replaces it with mac_kernel
    else:
        assert cluster_fit(100, 100, G) is not None
    _mac_guard("mixing", MIX_KW, MIX_DEFAULTS, MIX_ACTS)
    env = make("mixing", 2, ctas_per_env=G, **MIX_KW)
    assert ("us" in env.fields) == (kernel == "mac_kernel")
    orc = bo.mixing(**MIX_KW)
    close(env.reset(), np.stack([orc.reset()[0]] * 2), what="reset obs")
    close(env.get_state("C"), np.stack([orc.C.reshape(-1)] * 2), rtol=1e-15, what="reset C")
    mac_vs_oracle(env, "mixing", MIX_KW, MIX_ACTS)


def test_mixing_params_fp32_mac_big():
    env = make("mixing", 2, dtype=torch.float32, **MIX_KW)
    env.reset()
    mac_vs_oracle(env, "mixing", MIX_KW, MIX_ACTS, rtol=RTOL32)


# ============================================================================= B. on-device noise
M32 = 0xFFFFFFFF


def philox(c, k):
    """Philox4x32-10, the test_abi restatement."""
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    c, k = list(c), list(k)
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k[0], p1 & M32, (p0 >> 32) ^ c[3] ^ k[1], p0 & M32]
        k = [(k[0] + W0) & M32, (k[1] + W1) & M32]
    return c


def noise(seed, env, draw, sigma):
    """philox_uniform_pm of common.cuh: key (seed lo, hi), counter (draw lo, hi, env lo, hi), 53 bits."""
    c = philox([draw & M32, (draw >> 32) & M32, env & M32, (env >> 32) & M32], [seed & M32, (seed >> 32) & M32])
    bits = ((c[0] << 32) | c[1]) >> 11
    return -sigma + 2.0 * sigma * (bits * 2.0 ** -53)


def draws_words(d):
    d = np.asarray(d, dtype=np.uint64)
    return np.stack([(d & M32).astype(np.uint32), (d >> np.uint64(32)).astype(np.uint32)], 1).view(np.int32)


def draws_of(t):
    w = t.cpu().numpy().astype(np.int64)
    return [int(x) for x in (w[:, 0] & M32) | (w[:, 1] << 32)]


SEED, BASE = 2 ** 40 + 12345, 2 ** 32 + 7


def test_noise_model_range():
    """The model covers [-sigma, sigma) on both sides and moves with every counter word and both key words."""
    v = [noise(SEED, BASE, d, 1.0) for d in range(2000)]
    assert min(v) < -0.9 and max(v) > 0.9 and all(-1.0 <= x < 1.0 for x in v)
    x = noise(SEED, BASE, 5, 1.0)
    assert len({x, noise(SEED, BASE, 5 + 2 ** 32, 1.0), noise(SEED, BASE + 2 ** 32, 5, 1.0), noise(SEED, BASE + 1, 5, 1.0),
                noise(SEED + 2 ** 32, BASE, 5, 1.0), noise(SEED + 1, BASE, 5, 1.0)}) == 6


def _shk_sync(env, orcs):
    for f in ("h", "q", "rhsh", "rhsq", "u", "up"):
        env.set_state(f, np.stack([getattr(o, f) for o in orcs]))
    env.set_state("stp", np.array([o.stp for o in orcs]))


@pytest.mark.parametrize("dtype", [pytest.param(torch.float64, id="fp64"), pytest.param(torch.float32, id="fp32")])
def test_shkadov_noise_model(dtype):
    """seed and global env index above 32 bits; counters that carry into the high word inside an action
    (2^32 - 20 and 2^33 - 1); K = 3 fused actions per launch, the state re-synced from the oracle before each
    launch; then a warm reset n_warm = [0, 3, 7].  The oracle draws each sub-step's inlet noise from the model
    at draws0 + act ndt_act + i; every counter advances by exactly the draws taken."""
    fp32 = dtype == torch.float32
    B, K, sigma, nj = 3, 1 if fp32 else 3, 2e-3, 5
    env = make("shkadov", B, n_jets=nj, sigma=sigma, seed=SEED, env_index_base=BASE, dtype=dtype)
    ndt = env.cfg.d["ndt_act"]
    assert shk_dispatch(env.cfg.d["nx"])[0] == V6
    env.reset()
    orcs = [bo.shkadov(n_jets=nj) for _ in range(B)]
    for o in orcs:
        o.reset()
    rtol, floor = (RTOL32, 1.0) if fp32 else (1e-9, 1e-2)
    rng = np.random.default_rng(8)
    for launch, start in enumerate(([2 ** 32 - 20, 2 ** 33 - 1, 12345], [2 ** 32 - 20 + 7, 2 ** 40 + 3, 2 ** 32 - 1])):
        _shk_sync(env, orcs)
        env.set_state("draws", draws_words(start))
        acts = rng.uniform(-1, 1, (K, B, nj))
        obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts))
        for b, o in enumerate(orcs):
            ref = []
            for k in range(K):
                nz = [noise(SEED, BASE + b, start[b] + k * ndt + i, sigma) for i in range(ndt)]
                ref.append(o.step(acts[k, b], noise=np.array(nz)))
            tag = f"launch {launch} row {b}"
            close(obs[:, b], np.stack([r[0] for r in ref]), rtol=rtol, what=f"obs {tag}", floor=floor)
            close(rwd[:, b], np.array([r[1] for r in ref]), rtol=rtol, what=f"rwd {tag}", floor=floor)
        for f in ("h", "q"):
            close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), rtol=rtol, what=f"{f} launch {launch}", floor=floor)
        assert draws_of(env.get_state("draws")) == [s + K * ndt for s in start]
    # warm reset: n_warm zero-action steps from the shipped state, noise continuing each env's stream
    nw = [0, 3, 7]
    start = [2 ** 32 - 60, 2 ** 33 - 1, 99]
    env.set_state("draws", draws_words(start))
    env.reset(n_warm=torch.tensor(nw, dtype=torch.int32))
    for b, o in enumerate(orcs):
        cnt = [start[b]]

        def fn(n, b=b, cnt=cnt):
            v = np.array([noise(SEED, BASE + b, cnt[0] + i, sigma) for i in range(n)])
            cnt[0] += n
            return v
        o.noise_fn = fn
        o.reset(n_warm=nw[b])
        assert cnt[0] == start[b] + nw[b] * ndt
    if not fp32:            # seven free-running fp32 actions drift past 1e-5 of the fp64 oracle
        for f in ("h", "q"):
            close(env.get_state(f), np.stack([getattr(o, f) for o in orcs]), rtol=rtol, what=f"{f} after warm reset", floor=floor)
    assert draws_of(env.get_state("draws")) == [s + w * ndt for s, w in zip(start, nw)]


@pytest.mark.parametrize("B,dtype", [pytest.param(2, torch.float64, id="B2-C2T256"), pytest.param(300, torch.float64, id="B300-C4T128"),
                                     pytest.param(2, torch.float32, id="B2-fp32")])
def test_burgers_noise_model(B, dtype):
    """One draw per action at the env's counter: seed and global env index above 32 bits, one counter at
    2^32 - 1 (it carries between two actions), a 20-action fused free run (1 action in fp32)."""
    fp32 = dtype == torch.float32
    sigma, K = 0.03, 1 if fp32 else 20
    env = make("burgers", B, sigma=sigma, seed=SEED, env_index_base=BASE, dtype=dtype)
    env.reset()
    rows = (0, B - 1) if B == 2 else (0, 127, 128, 299)
    start = np.arange(B, dtype=np.uint64) * np.uint64(1000) + np.uint64(2 ** 40)
    start[rows[0]] = 2 ** 32 - 1
    start[rows[-1]] = 2 ** 33 - 3
    env.set_state("draws", draws_words(start))
    acts = np.random.default_rng(B).uniform(-1, 1, (K, B, 1))
    obs, rwd, done, trunc = env.step_fused(torch.as_tensor(acts))
    rtol, floor = (RTOL32, 1.0) if fp32 else (1e-9, 1e-2)
    for b in rows:
        o = bo.burgers(sigma=sigma)
        o.reset()
        ref = [o.step(acts[k, b], noise=noise(SEED, BASE + b, int(start[b]) + k, sigma)) for k in range(K)]
        close(obs[:, b], np.stack([r[0] for r in ref]), rtol=rtol, what=f"obs row {b}", floor=floor)
        close(rwd[:, b], np.array([r[1] for r in ref]), rtol=rtol, what=f"rwd row {b}", floor=floor)
        close(env.get_state("u")[b], o.u, rtol=rtol, what=f"u row {b}", floor=floor)
    assert draws_of(env.get_state("draws")) == [int(s) + K for s in start]


def test_single_env_noise_streams():
    """envs.shkadov: `sigma` reassigned between steps rebuilds the native env (_sync_sigma); the stream goes on
    at the same counter with the new amplitude.  envs.burgers(sigma=, seed=)."""
    from beacon_b200 import envs
    seed = 2 ** 33 + 5
    e = envs.shkadov(seed=seed)
    o = bo.shkadov()
    e.reset(n_warm=0)
    o.reset()
    ndt, draw = o.ndt_act, 0
    rng = np.random.default_rng(10)
    for k, sigma in enumerate((5.0e-4, 5.0e-4, 1.0e-3, 1.0e-3)):
        e.sigma = sigma
        a = rng.uniform(-1, 1, 5)
        obs, rwd = e.step(a)[:2]
        ro = o.step(a, noise=np.array([noise(seed, 0, draw + i, sigma) for i in range(ndt)]))
        draw += ndt
        close(e.h, o.h, rtol=1e-9, what=f"shkadov h action {k} sigma {sigma}")
        close(obs, ro[0], rtol=1e-9, what=f"shkadov obs action {k}")
    e.close()
    sigma = 0.05
    e = envs.burgers(sigma=sigma, seed=seed)
    o = bo.burgers(sigma=sigma)
    e.reset()
    o.reset()
    for k in range(3):
        a = np.array([rng.uniform(-1, 1)])
        obs, rwd = e.step(a)[:2]
        ro = o.step(a, noise=noise(seed, 0, k, sigma))
        close(e.u, o.u, rtol=1e-10, what=f"burgers u action {k}")
        close(np.array([rwd]), np.array([ro[1]]), rtol=1e-12, what=f"burgers rwd action {k}")
    e.close()


# ============================================================================= C. Poisson iteration cap
def capped(name, itmax):
    """The env's parameter class with the Poisson iteration cap set to itmax."""
    from beacon_b200.params import MixingCfg, RayleighCfg

    class Capped(RayleighCfg if name == "rayleigh" else MixingCfg):
        def __post_init__(self):
            super().__post_init__()
            self.d["itmax"] = itmax
    return Capped


def _act(name, a):
    return np.array(a) if name == "rayleigh" else int(a)


def _gpu_act(name, acts):
    if name == "rayleigh":
        return torch.as_tensor(np.array(acts, dtype=np.float64))
    return torch.as_tensor(np.array(acts), dtype=torch.int32)


_RA = tuple(np.random.default_rng(5).uniform(-1, 1, 10))
_RB = tuple(np.random.default_rng(6).uniform(-1, 1, 5))
# id, env, ctor kwargs, env var, G, kernel, A's actions (a1, a2), B's previous action (None: B starts at reset too), B's actions (b1, b2)
CAP_CASES = [pytest.param("rayleigh", dict(), None, 1, "mac_reg_kernel", (_RA, _RA), None, ((0.0,) * 10, (0.0,) * 10), id="mac_reg-rayleigh"),
             pytest.param("rayleigh", dict(init=False, L=2.0, H=2.0, n_sgts=5), None, 1, "mac_big_kernel", (_RB, _RB), _RB,
                          ((0.0,) * 5, (0.0,) * 5), id="mac_big-rayleigh"),
             pytest.param("mixing", dict(), None, 1, "mac_big_kernel", (2, 2), 2, (2, 2), id="mac_big-mixing"),
             pytest.param("rayleigh", dict(), "BEACON_MAC_V1", 1, "mac_kernel", (_RA, _RA), None, ((0.0,) * 10, (0.0,) * 10), id="mac_kernel-G1"),
             pytest.param("rayleigh", dict(), None, 2, "mac_kernel", (_RA, _RA), None, ((0.0,) * 10, (0.0,) * 10), id="mac_kernel-G2")]


@pytest.mark.parametrize("name,kw,envvar,G,kernel,a_acts,b_prev,b_acts", CAP_CASES)
def test_poisson_iteration_cap(name, kw, envvar, G, kernel, a_acts, b_prev, b_acts, monkeypatch):
    """M = env A's largest per-sub-step sweep count in its action (oracle, default cap).  At itmax = M: no
    status bit, sweeps and fields exactly the oracle's.  At itmax = M - 1: bit 2 on env A only (the oracle
    raises there: the reference tests itp > itmax before err > tol), env B (whose largest count is below
    M - 1) still equals the oracle.  A K = 2 launch whose first action overflows keeps the bit, though the same
    second action in a launch of its own clears it.  Fields after
    an overflow are not compared: the kernels carry on with the unconverged iterate, the reference exits."""
    from beacon_b200 import params
    if envvar:
        monkeypatch.setenv(envvar, "1")
    if G == 1:
        nx, ny = int((50 if name == "rayleigh" else 100) * kw.get("L", 1.0)), int((50 if name == "rayleigh" else 100) * kw.get("H", 1.0))
        assert mac_dispatch(name, nx, ny, kw.get("n_sgts", 10))[0] == ("mac_reg_kernel" if envvar else kernel)
    else:
        assert cluster_fit(50, 50, G) is not None
    scal = "T" if name == "rayleigh" else "C"
    # oracle, default cap
    oA = mac_oracle(name, **kw)
    oA.step(_act(name, a_acts[0]))
    M = int(oA.last_iters.max())
    oB = mac_oracle(name, **kw)
    if b_prev is not None:
        oB.step(_act(name, b_prev))
    oB.step(_act(name, b_acts[0]))
    iB = oB.last_iters.copy()
    assert iB.max() < M - 1, (int(iB.max()), M)
    o = mac_oracle(name, **kw)
    o.cfg.itmax = M - 1
    with pytest.raises(RuntimeError, match="max number of iterations"):
        o.step(_act(name, a_acts[0]))
    # B's starting state: one action ahead, taken from an uncapped env
    prev = None
    if b_prev is not None:
        e0 = make(name, 2, ctas_per_env=G, **kw)
        e0.reset()
        e0.step(_gpu_act(name, [b_prev, b_prev]))
        prev = e0.state_dict()

    def env_at(itmax):
        monkeypatch.setitem(params.CFG, name, capped(name, itmax))
        env = make(name, 2, ctas_per_env=G, **kw)
        assert env.cfg.d["itmax"] == itmax
        assert ("us" in env.fields) == (kernel == "mac_kernel")
        env.reset()
        if prev is not None:
            env.load_state_dict(prev)
            env.reset(mask=torch.tensor([1, 0], dtype=torch.uint8))
        return env

    for itmax in (M, M - 1):
        env = env_at(itmax)
        env.step(_gpu_act(name, [a_acts[0], b_acts[0]]), want_iters=True)
        st = [int(x) for x in env.status]
        if itmax == M:
            assert st == [0, 0], (itmax, st)
            assert [int(x) for x in env.last_iters[0]] == [int(oA.last_iters.sum()), int(iB.sum())]
            rows = (0, 1)
        else:
            assert st == [OVERFLOW, 0], (itmax, st)
            assert int(env.last_iters[0, 1]) == int(iB.sum())
            rows = (1,)
        for f in ("u", "v", "p", scal):
            g = env.get_state(f)
            for r in rows:
                close(g[r], getattr(oA if r == 0 else oB, f).reshape(-1), what=f"{f} row {r} itmax {itmax}")
    # K = 2: overflow in the first action only
    e1, e2 = env_at(M - 1), env_at(M - 1)
    acts = [[a_acts[0], b_acts[0]], [a_acts[1], b_acts[1]]]
    e2.step(_gpu_act(name, acts[0]))
    assert [int(x) for x in e2.status] == [OVERFLOW, 0]
    e2.step(_gpu_act(name, acts[1]))
    assert [int(x) for x in e2.status] == [0, 0], "precondition: the second action converges within the cap"
    e1.step_fused(torch.stack([_gpu_act(name, acts[0]), _gpu_act(name, acts[1])]))
    assert [int(x) for x in e1.status] == [OVERFLOW, 0]
