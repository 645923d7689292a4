"""rayleigh / mixing with one environment split over a thread-block cluster (ctas_per_env = G > 1: the generic
mac_kernel over G CTAs, DESIGN.md §3.6): grids no single CTA holds against the oracle, the cluster path against
the single-CTA kernels on the same grid (for 100x50 that is the same mac_kernel at G = 1), determinism, plumbing,
fp32 and the host-side capacity rule."""
import math

import numpy as np
import pytest
import torch

from oracle import beacon_oracle as bo
from test_gpu_parity import close, make

pytestmark = pytest.mark.gpu

RTOL32 = 1e-5
SMEM = 200 * 1024


def cluster_fit(nx, ny, G, real_bytes=8):
    """Mirror of cluster_misfit / cluster_passes in mac2d.cu: (thickest slab, thinnest slab, transport passes),
    or None when G CTAs cannot hold the grid."""
    ld, smax, smin = ny + 2, -(-nx // G), nx // G
    if G > 8 or smin < 4 or ld > 512 or (-(-smax // 4)) * (-(-ny // 5)) > 512:
        return None
    if 2 * (smax + 2) * ld * real_bytes > SMEM:
        return None
    p = 1
    while -(-smax // p) > 64 or 3 * (-(-smax // p)) * ld * real_bytes > SMEM:
        p += 1
    return smax, smin, p


def oracle(name, **kw):
    return bo.rayleigh(**kw) if name == "rayleigh" else bo.mixing(**kw)


def actions(name, rng, B, n_sgts=None):
    if name == "rayleigh":
        return rng.uniform(-1, 1, (B, n_sgts))
    return rng.integers(0, 4, B)


def as_act(name, a, dtype=torch.float64):
    return torch.as_tensor(a, dtype=dtype) if name == "rayleigh" else torch.as_tensor(a, dtype=torch.int32)


# name, ctor kwargs, (nx, ny), G, (thickest slab, thinnest slab, passes)
LARGE = [pytest.param(*c, id=c[0] + f"-{c[2][0]}x{c[2][1]}-G{c[3]}") for c in (
    ("rayleigh", dict(init=False, H=4.0, n_sgts=5), (50, 200), 2, (25, 25, 1)),
    ("rayleigh", dict(init=False, L=2 * math.pi), (314, 50), 8, (40, 39, 1)),      # 314 = 2 * 40 + 6 * 39
    ("rayleigh", dict(init=False, L=2 * math.pi), (314, 50), 3, (105, 104, 2)),    # two transport passes per slab
    ("mixing", dict(L=2.0), (200, 100), 4, (50, 50, 1)),
    ("mixing", dict(L=2.0, H=2.0), (200, 200), 8, (25, 25, 1)))]


@pytest.mark.parametrize("name,kw,grid,G,slabs", LARGE)
def test_cluster_grids_vs_oracle(name, kw, grid, G, slabs):
    """Grids the one-CTA-per-env kernels reject, two envs with their own actions against the oracle: sweep
    counts exact, fields within 1e-10, reward within 1e-12, status 0."""
    assert cluster_fit(*grid, G) == slabs
    B = 2
    env = make(name, B, ctas_per_env=G, **kw)
    assert (env.cfg.d["nx"], env.cfg.d["ny"]) == grid
    orcs = [oracle(name, **kw) for _ in range(B)]
    obs0 = env.reset()
    close(obs0, np.stack([o.reset()[0] for o in orcs]), what="reset obs")
    rng = np.random.default_rng(G)
    scal = "T" if name == "rayleigh" else "C"
    ns = kw.get("n_sgts", 10)
    for k in range(2):
        a = actions(name, rng, B, ns)
        obs, rwd, d, t = env.step(as_act(name, a), want_iters=True)
        ref = [o.step(a[b] if name == "rayleigh" else int(a[b])) for b, o in enumerate(orcs)]
        assert [int(x) for x in env.last_iters[0]] == [int(o.last_iters.sum()) for o in orcs], f"action {k}"
        for f in ("u", "v", "p", scal):
            close(env.get_state(f), np.stack([getattr(o, f).reshape(-1) for o in orcs]), what=f"{f} action {k}")
        close(obs, np.stack([r[0] for r in ref]), what=f"obs action {k}")
        close(rwd, np.array([r[1] for r in ref]), rtol=1e-12, what=f"rwd action {k}")
    assert int(env.status.max()) == 0


SAME = [pytest.param(*c, G, id=f"{c[0]}-{c[2]}-G{G}") for c in (
    ("rayleigh", dict(), "50x50-reg"),
    ("rayleigh", dict(init=False, L=2.0, n_sgts=5), "100x50-generic"),
    ("mixing", dict(), "100x100-big")) for G in (2, 4)]


@pytest.mark.parametrize("name,kw,tag,G", SAME)
def test_cluster_equals_single_cta(name, kw, tag, G):
    """The same grid on a single-CTA kernel and on G CTAs, three envs with different actions: equal sweep
    counts, fields within 1e-12."""
    nx, ny = (int(x) for x in tag.split("-")[0].split("x"))
    assert cluster_fit(nx, ny, G) is not None
    B = 3
    e1, eg = make(name, B, **kw), make(name, B, ctas_per_env=G, **kw)
    close(eg.reset(), e1.reset().cpu().numpy(), rtol=1e-12, what="reset obs")
    rng = np.random.default_rng(7 + G)
    scal = "T" if name == "rayleigh" else "C"
    for k in range(2):
        a = actions(name, rng, B, kw.get("n_sgts", 10))
        o1, r1, _, _ = e1.step(as_act(name, a), want_iters=True)
        og, rg, _, _ = eg.step(as_act(name, a), want_iters=True)
        assert torch.equal(e1.last_iters, eg.last_iters), (e1.last_iters, eg.last_iters)
        for f in ("u", "v", "p", scal):
            close(eg.get_state(f), e1.get_state(f).cpu().numpy(), rtol=1e-12, what=f"{f} action {k}")
        close(og, o1.cpu().numpy(), rtol=1e-12, what="obs")
        close(rg, r1.cpu().numpy(), rtol=1e-12, what="rwd")
    assert int(eg.status.max()) == 0


def test_cluster_determinism():
    """Equal inputs give bitwise-equal rows; a restored state reproduces the next step bitwise; K = 3 fused
    actions equal three steps bitwise."""
    kw, G = dict(L=2.0), 4
    env = make("mixing", 2, ctas_per_env=G, **kw)
    env.reset()
    a = torch.tensor([2, 2], dtype=torch.int32)
    env.step(a)
    for f in ("u", "v", "p", "C", "obs"):
        g = env.get_state(f)
        assert torch.equal(g[0], g[1]), f
    sd = env.state_dict()
    o1, r1, _, _ = env.step(torch.tensor([0, 3], dtype=torch.int32))
    after = env.state_dict()
    env.load_state_dict(sd)
    o2, r2, _, _ = env.step(torch.tensor([0, 3], dtype=torch.int32))
    assert torch.equal(o1, o2) and torch.equal(r1, r2)
    for k, v in env.state_dict().items():
        assert torch.equal(v, after[k]), k

    acts = torch.tensor([[1, 3], [0, 2], [3, 1]], dtype=torch.int32)
    e1, e2 = make("mixing", 2, ctas_per_env=G, **kw), make("mixing", 2, ctas_per_env=G, **kw)
    e1.reset(); e2.reset()
    of, rf, _, _ = e1.step_fused(acts, want_iters=True)
    for k in range(3):
        o, r, _, _ = e2.step(acts[k], want_iters=True)
        assert torch.equal(o, of[k]) and torch.equal(r, rf[k]), k
        assert torch.equal(e2.last_iters[0], e1.last_iters[k]), k
    for k, v in e1.state_dict().items():
        assert torch.equal(v, e2.state_dict()[k]), k


def test_cluster_plumbing():
    """Masked reset, VectorEnv auto-reset, step_host and a G = 2 checkpoint continued at G = 1."""
    from beacon_b200.vector import VectorEnv
    kw, G = dict(init=False, L=2 * math.pi, n_sgts=10), 4
    env = make("rayleigh", 3, ctas_per_env=G, **kw)
    obs0 = env.reset()
    before_step = env.state_dict()
    a = torch.as_tensor(np.random.default_rng(3).uniform(-1, 1, (3, 10)))
    obs, _, _, _ = env.step(a)
    before = env.state_dict()
    out = obs.clone()
    env.reset(mask=torch.tensor([0, 1, 0], dtype=torch.uint8), out=out)
    after = env.state_dict()
    for k, v in after.items():
        assert torch.equal(v[[0, 2]], before[k][[0, 2]]), k
    assert torch.equal(out[[0, 2]], obs[[0, 2]]) and torch.equal(out[1], obs0[1])
    for f in ("u", "v", "p", "T", "obs", "stp"):
        assert torch.equal(after[f][1], before_step[f][1]), f

    # step_host with pinned buffers equals step
    e1, e2 = make("rayleigh", 3, ctas_per_env=G, **kw), make("rayleigh", 3, ctas_per_env=G, **kw)
    e1.reset(); e2.reset()
    o1, r1, d1, t1 = e1.step(a)
    o2, r2, d2, t2 = e2.step_host(a.clone())
    assert torch.equal(o1.cpu(), o2) and torch.equal(r1.cpu(), r2) and torch.equal(d1.cpu(), d2) and torch.equal(t1.cpu(), t2)

    # VectorEnv: the env at its horizon restarts
    ve = VectorEnv("rayleigh", 2, ctas_per_env=G, **kw)
    r0 = ve.reset()
    n_act = ve.env.n_act
    ve.env.set_state("stp", torch.tensor([[n_act - 1], [0]], dtype=torch.int32))
    o, r, d, t, info = ve.step(a[:2])
    assert d.tolist() == [True, False]
    assert torch.equal(o[0], r0[0]) and not torch.equal(o[1], r0[1])
    assert int(ve.env.get_state("stp")[0, 0]) == 0 and int(ve.env.get_state("stp")[1, 0]) == 1
    ve.close()

    # a G = 2 checkpoint continues on the single-CTA generic kernel (100x50)
    kw2 = dict(init=False, L=2.0, n_sgts=5)
    eg, e1 = make("rayleigh", 2, ctas_per_env=2, **kw2), make("rayleigh", 2, **kw2)
    eg.reset(); e1.reset()
    a2 = torch.as_tensor(np.random.default_rng(5).uniform(-1, 1, (2, 5)))
    eg.step(a2)
    assert set(eg.fields) == set(e1.fields)
    e1.load_state_dict(eg.state_dict())
    a3 = torch.as_tensor(np.random.default_rng(6).uniform(-1, 1, (2, 5)))
    og, rg, _, _ = eg.step(a3)
    o1, r1, _, _ = e1.step(a3)
    for f in ("u", "v", "p", "T"):
        close(eg.get_state(f), e1.get_state(f).cpu().numpy(), rtol=1e-12, what=f"{f} after restore")
    close(og, o1.cpu().numpy(), rtol=1e-12, what="obs after restore")
    close(rg, r1.cpu().numpy(), rtol=1e-12, what="rwd after restore")


def test_cluster_fp32():
    """fp32 on rayleigh 314x50 from rest over 4 CTAs: the sweep count within 5 % of the oracle's, fields
    within 1e-5 of the field scale."""
    kw, G = dict(init=False, L=2 * math.pi, n_sgts=10), 4
    assert cluster_fit(314, 50, G, real_bytes=4) == (79, 78, 2)
    env = make("rayleigh", 2, ctas_per_env=G, dtype=torch.float32, **kw)
    o = bo.rayleigh(**kw)
    env.reset(); o.reset()
    a = np.random.default_rng(33).uniform(-1, 1, 10)
    obs, rwd, d, t = env.step(torch.as_tensor(np.stack([a, a])).float(), want_iters=True)
    ro = o.step(a)
    assert int(env.status.max()) == 0, "fp32 Poisson iteration hit itmax"
    it, it_ref = int(env.last_iters[0, 0]), int(o.last_iters.sum())
    assert abs(it - it_ref) <= 0.05 * it_ref, (it, it_ref)
    for f in ("u", "v", "T"):
        close(env.get_state(f)[0], getattr(o, f).reshape(-1), rtol=RTOL32, what=f"{f} fp32", floor=1.0)
    close(obs[0], ro[0], rtol=RTOL32, what="obs fp32", floor=1.0)


def test_cluster_single_env_and_warmup():
    """The reference-named class and the rayleigh warm-up generator reach the cluster path."""
    from beacon_b200 import envs, fieldio
    e = envs.rayleigh(init=False, L=2 * math.pi, ctas_per_env=8)
    obs, _ = e.reset()
    obs2, rwd, done, trunc, _ = e.step(np.zeros(10))
    assert obs2.shape == obs.shape and np.isfinite(rwd) and not done
    assert e.last_iters > 0 and e.status == 0 and e.T.shape == (316, 52)
    e.close()
    m = envs.mixing(L=2.0, ctas_per_env=4)
    m.reset()
    m.step(2)
    assert m.last_iters > 0 and m.C.shape == (202, 102)
    m.close()
    f = fieldio.generate_init_state("rayleigh", L=2 * math.pi, ctas_per_env=8, n_warmup=2)
    assert set(f) == {"u", "v", "p", "T"} and all(x.shape == (316, 52) for x in f.values())
    assert all(np.isfinite(x).all() for x in f.values()) and np.abs(f["u"]).max() > 0


def test_cluster_rejections():
    """Host-side errors, never a CUDA error: a non-MAC env, more than 8 CTAs, slabs thinner than 4 rows,
    a grid beyond 8 CTAs; the single-CTA message names a cluster size that fits."""
    import ctypes as C

    from beacon_b200 import BeaconError, _capi as capi
    from beacon_b200.params import MixingCfg
    with pytest.raises(ValueError, match="ctas_per_env"):
        make("lorenz", 1, ctas_per_env=2)
    with pytest.raises(BeaconError, match="at most 8"):
        make("mixing", 1, L=2.0, ctas_per_env=9)
    # every constructor grid has nx >= 50, so a thin slab is reached through the C-ABI: 24 rows over 8 CTAs
    assert cluster_fit(24, 24, 8) is None
    L = capi.lib()
    com = capi.Common(1, 0, capi.F64, 0, 0, 0)
    d = MixingCfg().d
    p = capi.MacParams(24, 24, d["ndt_act"], d["n_act"], 0, 0, 1, 1, 1, 4, 4, d["itmax"], 1 / 24, 1 / 24, d["dt"],
                       0.0, 0.0, 0.0, 0.0, 0.0, d["re"], d["pe"], d["u_max"], d["ref_c"], d["tol"], 8)
    h = C.c_void_p()
    C0 = np.zeros(26 * 26)
    rc = L.beacon_mixing_create(C.byref(com), C.byref(p), C0.ctypes.data_as(C.POINTER(C.c_double)), C.byref(h))
    with pytest.raises(BeaconError, match="fewer than 4"):
        capi.check(rc)
    assert all(cluster_fit(400, 400, g) is None for g in range(2, 9))
    with pytest.raises(BeaconError, match="more than 512 tiles"):
        make("mixing", 1, L=4.0, H=4.0, ctas_per_env=8)
    with pytest.raises(BeaconError, match="grid too large"):
        make("mixing", 1, L=4.0, H=4.0)
    assert cluster_fit(200, 100, 2) is not None
    with pytest.raises(BeaconError, match=r"grid too large.*ctas_per_env=2 would fit"):
        make("mixing", 1, L=2.0)
    # the env still works after the failed creations
    env = make("mixing", 1, L=2.0, ctas_per_env=2)
    env.reset()
    env.step(torch.tensor([1], dtype=torch.int32))
    assert int(env.status[0]) == 0
