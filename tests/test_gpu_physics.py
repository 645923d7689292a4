"""Per-env physical parameters of rayleigh (ra) and mixing (re, pe): one handle, one launch, each env at its own value.

  * every row of a per-env handle equals a uniform handle created with that row's value, on every MAC kernel path:
    bitwise in fp64 on mac_kernel at G = 1 and over clusters of G = 2 and 4; on mac_reg_kernel and mac_big_kernel
    to 1e-12 with sweep counts, flags and integer fields exact (their per-env instances contract one multiply-add
    differently from the uniform ones, DESIGN.md 3.7);
  * rows away from the default against the oracle (sweep counts exact);
  * the Poisson iteration cap trips on the one env whose value needs more sweeps;
  * set_physics + reset(mask) between launches, checkpoints, sharding and the rejected inputs.
"""
import numpy as np
import pytest
import torch

from test_gpu_mac_cluster import cluster_fit
from test_gpu_params import MIX_KW, OVERFLOW, _key, capped, mac_oracle, mac_reference
from test_gpu_parity import close, make
from test_gpu_variants import mac_dispatch

pytestmark = pytest.mark.gpu

RAS = (1.2e4, 8e3, 3e4, 1e4, 2e4, 1.5e4)                               # shuffled, the default 1e4 among them
MIX = ((150.0, 5e3), (100.0, 1e4), (200.0, 2e4), (120.0, 8e3), (250.0, 1.2e4), (100.0, 6e3))
K = 3


def _acts(name, n_sgts, B, seed):
    rng = np.random.default_rng(seed)
    if name == "rayleigh":
        return torch.as_tensor(rng.uniform(-1, 1, (K, B, n_sgts)))
    return torch.as_tensor(rng.integers(0, 4, (K, B)), dtype=torch.int32)


def run(env, acts):
    """reset, then K fused actions: every output of the launch and every state field."""
    env.reset()
    obs, rwd, done, trunc = env.step_fused(acts.to(env.dtype) if acts.is_floating_point() else acts, want_iters=True)
    out = dict(obs=obs, rwd=rwd, done=done, trunc=trunc, iters=env.last_iters, status=env.status.clone().unsqueeze(0))
    out.update({"state." + f: env.get_state(f).unsqueeze(0) for f in env.fields})
    return {k: v.cpu() for k, v in out.items()}


def row(out, b):
    return {k: v[:, b] for k, v in out.items()}


def assert_rows_equal(got, want, what):
    assert got.keys() == want.keys()
    for k in got:
        assert torch.equal(got[k], want[k]), f"{what}: {k} differs (max {float((got[k].double() - want[k].double()).abs().max()):.3g})"


def assert_rows_close(got, want, what, exact):
    """bitwise when `exact`, else real outputs to 1e-12 (the `close` norm) and integer ones exact"""
    if exact:
        return assert_rows_equal(got, want, what)
    assert got.keys() == want.keys()
    for k in got:
        if got[k].is_floating_point():
            close(got[k], want[k].numpy(), rtol=1e-12, what=f"{what}: {k}")
        else:
            assert torch.equal(got[k], want[k]), f"{what}: {k} differs"


def per_env(name):
    """ctor kwargs of a per-env handle of six envs, and per row the kwargs of the equivalent uniform handle"""
    if name == "rayleigh":
        return dict(ra=list(RAS)), [dict(ra=r) for r in RAS]
    return dict(re=[m[0] for m in MIX], pe=[m[1] for m in MIX]), [dict(re=m[0], pe=m[1]) for m in MIX]


# (name, ctor kwargs, env var, ctas_per_env, expected kernel, n_sgts)
PATHS = [pytest.param("rayleigh", dict(), None, 1, "mac_reg_kernel", 10, id="mac_reg-rayleigh-50x50"),
         pytest.param("rayleigh", dict(init=False, L=2.0, H=2.0, n_sgts=5), None, 1, "mac_big_kernel", 5, id="mac_big-rayleigh-100x100"),
         pytest.param("mixing", dict(), None, 1, "mac_big_kernel", 0, id="mac_big-mixing-100x100"),
         pytest.param("rayleigh", dict(init=False, L=1.5, H=1.22, n_sgts=5), None, 1, "mac_kernel", 5, id="mac_kernel-G1-rayleigh-75x61"),
         pytest.param("mixing", dict(), "BEACON_MAC_V1", 1, "mac_kernel", 0, id="mac_kernel-G1-mixing-100x100"),
         pytest.param("rayleigh", dict(), None, 2, "mac_kernel", 10, id="mac_kernel-G2-rayleigh-50x50"),
         pytest.param("mixing", dict(), None, 2, "mac_kernel", 0, id="mac_kernel-G2-mixing-100x100"),
         pytest.param("mixing", dict(L=2.0), None, 4, "mac_kernel", 0, id="mac_kernel-G4-mixing-200x100")]


def _check_path(name, kw, G, kernel, n_sgts):
    nx, ny = (int((50 if name == "rayleigh" else 100) * kw.get(k, 1.0)) for k in ("L", "H"))
    if G == 1:
        assert mac_dispatch(name, nx, ny, n_sgts)[0] in (kernel, "mac_reg_kernel" if name == "rayleigh" else "mac_big_kernel")
    else:
        assert cluster_fit(nx, ny, G) is not None


@pytest.mark.parametrize("name,kw,envvar,G,kernel,n_sgts", PATHS)
def test_rows_equal_uniform_handles(name, kw, envvar, G, kernel, n_sgts, monkeypatch):
    """Six envs at distinct values in one handle: after reset and K = 3 fused actions, each row's obs, rewards,
    flags, sweep counts, status and state fields equal those of a uniform handle at that row's value (bitwise on
    mac_kernel, see the module docstring)."""
    if envvar:
        monkeypatch.setenv(envvar, "1")
    _check_path(name, kw, G, kernel, n_sgts)
    pk, rows = per_env(name)
    B = len(rows)
    env = make(name, B, ctas_per_env=G, **kw, **pk)
    assert ("us" in env.fields) == (kernel == "mac_kernel")
    acts = _acts(name, n_sgts, B, seed=G + B)
    got = run(env, acts)
    for k in pk:
        assert torch.equal(env.get_physics(k), torch.tensor(pk[k], dtype=torch.float64))
    for b, rk in enumerate(rows):
        ref = run(make(name, 1, ctas_per_env=G, **kw, **rk), acts[:, b:b + 1])
        assert_rows_close(row(got, b), row(ref, 0), f"row {b} {rk}", exact=kernel == "mac_kernel")
    assert int(got["status"].max()) == 0


def test_rows_equal_uniform_handles_fp32():
    """fp32 mac_reg_kernel: each row within 1e-6 (field scale) of a uniform fp32 handle at that row's ra."""
    pk, rows = per_env("rayleigh")
    B = len(rows)
    env = make("rayleigh", B, dtype=torch.float32, **pk)
    acts = _acts("rayleigh", 10, B, seed=32)
    got = run(env, acts)
    for b, rk in enumerate(rows):
        ref = run(make("rayleigh", 1, dtype=torch.float32, **rk), acts[:, b:b + 1])
        for k, v in row(got, b).items():
            if v.is_floating_point():
                close(v, row(ref, 0)[k].numpy(), rtol=1e-6, floor=1.0, what=f"row {b} {k}")
            else:
                assert torch.equal(v, row(ref, 0)[k]), (b, k)


RAY_ORACLE = [pytest.param(dict(), 10, id="mac_reg-50x50"),
              pytest.param(dict(init=False, L=2.0, H=1.0, n_sgts=5), 5, id="mac_kernel-G1-100x50")]


@pytest.mark.parametrize("kw,n_sgts", RAY_ORACLE)
def test_rayleigh_rows_vs_oracle(kw, n_sgts):
    """Two rows at ra 2e4 and 3e4 (test_gpu_params' values) against the oracle run at each row's ra: fields,
    observations, rewards, and the Jacobi sweep counts exact."""
    ras = (2e4, 3e4) if n_sgts == 10 else (3e4, 2.5e4)
    env = make("rayleigh", 2, ra=list(ras), **kw)
    env.reset()
    acts = np.random.default_rng(7).uniform(-1, 1, (2, 2, n_sgts))
    refs = [mac_reference("rayleigh", _key(dict(kw, ra=ra)), (tuple(map(tuple, acts[:, b])),))[0] for b, ra in enumerate(ras)]
    _vs_oracle(env, "rayleigh", torch.as_tensor(acts), refs)


def test_mixing_rows_vs_oracle():
    """mac_big_kernel, rows at (re, pe) = MIX_KW's (150, 5e3) and (120, 8e3), side and C0 of MIX_KW for both."""
    rows = ((MIX_KW["re"], MIX_KW["pe"]), (120.0, 8e3))
    common = {k: v for k, v in MIX_KW.items() if k not in ("re", "pe")}
    env = make("mixing", 2, re=[r[0] for r in rows], pe=[r[1] for r in rows], **common)
    env.reset()
    acts = np.array([[2, 0], [1, 3]])
    refs = [mac_reference("mixing", _key(dict(common, re=re, pe=pe)), (tuple(int(x) for x in acts[:, b]),))[0]
            for b, (re, pe) in enumerate(rows)]
    _vs_oracle(env, "mixing", torch.as_tensor(acts, dtype=torch.int32), refs)


def _vs_oracle(env, name, acts, refs):
    scal = "T" if name == "rayleigh" else "C"
    for k in range(acts.shape[0]):
        obs, rwd, _, _ = env.step(acts[k], want_iters=True)
        assert [int(x) for x in env.last_iters[0]] == [r[k][1] for r in refs], f"sweeps action {k}"
        for i, f in enumerate(("u", "v", "p", scal)):
            close(env.get_state(f), np.stack([r[k][2 + i] for r in refs]), what=f"{f} action {k}")
        close(obs, np.stack([r[k][0][0] for r in refs]), what=f"obs action {k}")
        close(rwd, np.array([r[k][0][1] for r in refs]), rtol=1e-12, what=f"rwd action {k}")
    assert int(env.status.max()) == 0


def test_iteration_cap_trips_on_one_env(monkeypatch):
    """mac_reg_kernel, both envs on the same action: with itmax between the two envs' largest per-sub-step sweep
    counts, only the env whose ra needs more sweeps gets BEACON_STATUS_POISSON_OVERFLOW."""
    from beacon_b200 import params
    a = np.random.default_rng(5).uniform(-1, 1, 10)
    M = {}
    for ra in (1e4, 2e4, 3e4, 5e4):
        o = mac_oracle("rayleigh", ra=ra)
        o.step(a)
        M[ra] = int(o.last_iters.max())
    lo, hi = min(M, key=M.get), max(M, key=M.get)
    assert M[lo] < M[hi] - 1, M
    monkeypatch.setitem(params.CFG, "rayleigh", capped("rayleigh", M[hi] - 1))
    env = make("rayleigh", 2, ra=[hi, lo])
    assert env.cfg.d["itmax"] == M[hi] - 1
    env.reset()
    env.step(torch.as_tensor(np.stack([a, a])))
    assert [int(x) for x in env.status] == [OVERFLOW, 0]
    env = make("rayleigh", 2, ra=[lo, hi])
    env.reset()
    env.step(torch.as_tensor(np.stack([a, a])))
    assert [int(x) for x in env.status] == [0, OVERFLOW]


@pytest.mark.parametrize("name", ["rayleigh", "mixing"])
def test_set_physics_then_masked_reset(name):
    """Rows 1 and 4 get new values and a masked reset between launches: they equal a fresh uniform handle at the
    new value (to 1e-12, integers exact: mac_reg / mac_big); the other rows continue bitwise as in a per-env handle
    that was never touched."""
    pk, rows = per_env(name)
    B = len(rows)
    n_sgts = 10 if name == "rayleigh" else 0
    acts = _acts(name, n_sgts, B, seed=11)
    env, ctl = make(name, B, **pk), make(name, B, **pk)
    for e in (env, ctl):
        e.reset()
        e.step_fused(acts[:1])
    new = {k: np.array(v, dtype=np.float64) for k, v in pk.items()}
    changed = (1, 4)
    for k in new:
        new[k][list(changed)] = {"ra": 2.5e4, "re": 180.0, "pe": 3e4}[k]
    env.set_physics(**new)
    mask = torch.zeros(B, dtype=torch.uint8)
    mask[list(changed)] = 1
    env.reset(mask=mask)
    got = {}
    for e, tag in ((env, "env"), (ctl, "ctl")):
        o, r, d, t = e.step_fused(acts[1:], want_iters=True)
        got[tag] = dict(obs=o.cpu(), rwd=r.cpu(), done=d.cpu(), iters=e.last_iters.cpu(),
                        **{"state." + f: e.get_state(f).unsqueeze(0).cpu() for f in e.fields})
    for b in range(B):
        if b in changed:
            fresh = make(name, 1, **{k: float(v[b]) for k, v in new.items()})
            fresh.reset()
            o, r, d, t = fresh.step_fused(acts[1:, b:b + 1], want_iters=True)
            want = dict(obs=o.cpu(), rwd=r.cpu(), done=d.cpu(), iters=fresh.last_iters.cpu(),
                        **{"state." + f: fresh.get_state(f).unsqueeze(0).cpu() for f in fresh.fields})
            assert_rows_close(row(got["env"], b), row(want, 0), f"changed row {b}", exact=False)   # mac_reg / mac_big
        else:
            assert_rows_equal(row(got["env"], b), row(got["ctl"], b), f"untouched row {b}")
    for k, v in new.items():
        assert torch.equal(env.get_physics(k), torch.as_tensor(v))


@pytest.mark.parametrize("name", ["rayleigh", "mixing"])
def test_checkpoint_round_trip(name):
    """state_dict of a per-env handle -> a new handle created at the default -> load_state_dict: the values come
    along and the next launch is bitwise the original's.  A uniform handle's state dict has only its fields."""
    pk, rows = per_env(name)
    B = len(rows)
    acts = _acts(name, 10 if name == "rayleigh" else 0, B, seed=3)
    env = make(name, B, **pk)
    env.reset()
    env.step_fused(acts[:1])
    sd = env.state_dict()
    assert set(sd) == set(env.fields) | set(pk)
    back = make(name, B)
    assert set(back.state_dict()) == set(back.fields)
    back.load_state_dict(sd)
    for k in pk:
        assert torch.equal(back.get_physics(k), torch.tensor(pk[k], dtype=torch.float64))
    outs = []
    for e in (env, back):
        o, r, d, t = e.step_fused(acts[1:], want_iters=True)
        outs.append([o.cpu(), r.cpu(), e.last_iters.cpu()] + [e.get_state(f).cpu() for f in e.fields])
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def test_make_sharded_slices_per_env_values():
    """Two ranks' handles on one GPU: each holds its shard_range slice of the per-env ra, and its rows equal the
    matching rows of the whole batch in one handle."""
    from beacon_b200.dist import make_sharded, shard_range
    ras = np.array(RAS + (2.2e4,))
    N = len(ras)
    acts = _acts("rayleigh", 10, N, seed=21)
    whole = run(make("rayleigh", N, ra=ras), acts)
    for rank in range(2):
        lo, hi = shard_range(N, rank, 2)
        env = make_sharded("rayleigh", N, rank=rank, world=2, ra=torch.as_tensor(ras))
        assert env.batch == hi - lo
        assert torch.equal(env.get_physics("ra"), torch.as_tensor(ras[lo:hi]))
        part = run(env, acts[:, lo:hi])
        for b in range(hi - lo):
            assert_rows_equal(row(part, b), row(whole, lo + b), f"rank {rank} row {b}")
    with pytest.raises(ValueError, match="per-env values"):
        make_sharded("rayleigh", N + 1, rank=0, world=2, ra=ras)


def test_rejected_inputs_change_nothing():
    """A wrong length, NaN, a value <= 0, an unknown name, ra on mixing and re on shkadov raise, through Python and
    through the C-ABI (BEACON_ERR_INVALID), and leave the values and the launch count as they were."""
    from beacon_b200 import _capi as capi
    ras = np.array(RAS)
    env = make("rayleigh", 6, ra=ras)
    mix = make("mixing", 6)
    launches = env.launches
    for bad in (ras[:5], np.append(ras, 1e4), np.where(np.arange(6) == 2, np.nan, ras), np.where(np.arange(6) == 3, 0.0, ras),
                np.where(np.arange(6) == 0, -1e4, ras), np.where(np.arange(6) == 5, np.inf, ras)):
        with pytest.raises(ValueError):
            env.set_physics(ra=bad)
    with pytest.raises(ValueError):
        env.set_physics(rb=ras)
    with pytest.raises(ValueError):
        env.set_physics(re=ras)
    with pytest.raises(ValueError):
        mix.set_physics(ra=ras)
    with pytest.raises(ValueError):
        mix.set_physics(re=ras, pe=np.where(np.arange(6) == 1, np.nan, ras))   # nothing applied, re included
    with pytest.raises(ValueError):
        make("rayleigh", 6, ra=ras[:4])
    shk = make("shkadov", 2)
    with pytest.raises(ValueError):
        shk.set_physics(re=np.ones(2))
    # the C-ABI checks the same things itself
    L = env._lib
    dp = lambda a: np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(capi.C.POINTER(capi.C.c_double))
    s = env._stream()
    for h, nm, vals in ((env._h, b"ra", np.where(np.arange(6) == 2, np.nan, ras)), (env._h, b"ra", -ras), (env._h, b"re", ras),
                        (env._h, b"xx", ras), (mix._h, b"ra", ras), (shk._h, b"re", np.ones(6))):
        assert L.beacon_env_set_physics(h, nm, dp(vals), s) == -1, nm
    out = np.zeros(6)
    assert L.beacon_env_get_physics(shk._h, b"re", dp(out), s) == -1
    assert env.launches == launches
    assert torch.equal(env.get_physics("ra"), torch.as_tensor(ras))
    assert torch.equal(mix.get_physics("re"), torch.full((6,), 100.0, dtype=torch.float64))
    assert torch.equal(mix.get_physics("pe"), torch.full((6,), 1e4, dtype=torch.float64))
    assert set(mix.state_dict()) == set(mix.fields)            # still uniform: nothing was set
