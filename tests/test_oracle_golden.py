"""The C/numpy oracle replayed on the committed golden vectors of the reference
(tests/golden/<env>.npz, produced by oracle/gen_golden.py from the unmodified
jviquerat/beacon).  Fields must be BIT-EXACT: the oracle follows the reference's
arithmetic operation for operation."""
import json

import numpy as np
import pytest

from oracle import beacon_oracle as bo


def eq(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape
    assert np.array_equal(a, b), f"max abs diff {np.max(np.abs(a - b)):.3e}"


SHK_INTS = ("nx", "ndt_act", "n_act", "n_interp", "jet_pos", "jet_hw", "jet_space", "l_rwd", "n_obs", "l_obs")


def test_shkadov_params_bit_exact(golden):
    g = golden("shkadov")
    for row in json.loads(str(g["params_json"])):
        env = bo.shkadov(init=False, **row["kwargs"])
        for k in SHK_INTS:
            assert getattr(env, k) == row[k], (row["kwargs"], k)
        assert env.dx == row["dx"]
        assert env.jet_pos - env.jet_hw == row["jet_start"] and env.jet_pos + env.l_rwd == row["rwd_end"]
        assert env.jet_pos - env.l_obs == row["obs_start"]


@pytest.mark.parametrize("tag,n_jets", [("j10", 10), ("j5", 5), ("j41", 41)])
def test_shkadov_steps(golden, tag, n_jets):
    g = golden("shkadov")
    env = bo.shkadov(n_jets=n_jets)
    obs0, _ = env.reset()
    eq(obs0, g[f"{tag}_obs0"])
    for k in range(g[f"{tag}_actions"].shape[0]):
        obs, rwd, done, trunc, _ = env.step(g[f"{tag}_actions"][k], noise=g[f"{tag}_noise"][k])
        for f in ("h", "q", "rhsh", "rhsq"):
            eq(getattr(env, f), g[f"{tag}_{f}"][k])
        eq(obs, g[f"{tag}_obs"][k])
        assert rwd == g[f"{tag}_rwd"][k]
        assert not done and not trunc


def test_shkadov_warm_reset(golden):
    g = golden("shkadov")
    env = bo.shkadov(n_jets=10)
    it = iter(g["warm_noise"])
    env.noise_fn = lambda n: next(it)
    obs0, _ = env.reset(n_warm=int(g["warm_n"]))
    eq(obs0, g["warm_obs0"])
    eq(env.h, g["warm_h"])
    eq(env.q, g["warm_q"])
    assert env.stp == int(g["warm_stp"]) == 0


def test_shkadov_kat_and_horizon(golden):
    g = golden("shkadov")
    env = bo.shkadov(n_jets=10)
    env.reset()
    sr = 0.0
    for f in (1.0, -0.5, 1.0):
        sr += env.step(np.linspace(-1, 1, 10) * f)[1]
    assert sr == float(g["kat_sum_rwd"]) and env.h.sum() == float(g["kat_sum_h"]) and env.q.sum() == float(g["kat_sum_q"])
    # SURVEY.md §4 KAT table (values recorded at survey time from the unmodified reference)
    assert sr == -0.016856704466031224
    assert env.h.sum() == 1332.7062381888381 and env.q.sum() == 1346.4015915144832
    env = bo.shkadov(n_jets=2, t_act=0.2)
    env.reset()
    flags = [env.step(np.zeros(2))[2:4] for _ in range(4)]
    assert np.array_equal(np.array(flags), g["horizon_flags"])


def test_shkadov_separable_protocol(golden):
    g = golden("shkadov")
    env = bo.shkadov_separable(n_jets=4)
    eq(np.array([env.reset()[0] for _ in range(4)]), g["sep_reset_obs"])
    obs, rwd, flags = [], [], []
    for k in range(2):
        for j in range(4):
            o, r, d, t, _ = env.step(g["sep_actions"][k])
            obs.append(o); rwd.append(r); flags.append((d, t))
    eq(np.array(obs), g["sep_obs"])
    eq(np.array(rwd), g["sep_rwd"])
    assert np.array_equal(np.array(flags), g["sep_flags"])
    eq(env.h, g["sep_h"])
    eq(env.q, g["sep_q"])


def test_burgers(golden):
    g = golden("burgers")
    P = json.loads(str(g["params_json"]))
    env = bo.burgers()
    for k in ("nx", "ctrl_pos", "ndt_act", "n_act", "n_obs_pts"):
        assert getattr(env, k) == P[k]
    assert env.dx == P["dx"] and env.dt == P["dt"]
    eq(env.reset()[0], g["obs0"])
    for k in range(g["actions"].shape[0]):
        obs, rwd, *_ = env.step(g["actions"][k], noise=float(g["noise"][k]))
        eq(env.u, g["u"][k]); eq(env.up, g["up"][k]); eq(env.upp, g["upp"][k]); eq(obs, g["obs"][k])
        assert rwd == g["rwd"][k]
    env = bo.burgers(sigma=0.0)
    env.reset()
    sr = sum(env.step(np.array([0.3 if k % 2 == 0 else -0.6]))[1] for k in range(20))
    assert sr == float(g["kat_sum_rwd"]) == -0.11846877024941604
    assert env.u.sum() == float(g["kat_sum_u"]) == 251.0452280307368
    eq(env.u[250:255], g["kat_u"])


def test_sloshing(golden):
    g = golden("sloshing")
    P = json.loads(str(g["params_json"]))
    env = bo.sloshing()
    for k in ("nx", "ndt_act", "n_act", "n_interp", "n_obs"):
        assert getattr(env, k) == P[k]
    eq(env.reset()[0], g["obs0"])
    for k in range(g["actions"].shape[0]):
        obs, rwd, *_ = env.step(g["actions"][k])
        for f in ("h", "q", "rhsh", "rhsq"):
            eq(getattr(env, f), g[f][k])
        eq(obs, g["obs"][k])
        assert rwd == pytest.approx(g["rwd"][k], rel=1e-14)   # np.linalg.norm -> BLAS order
    env = bo.sloshing()
    env.reset()
    sr = sum(env.step(np.array([0.5 if k % 2 == 0 else -0.25]))[1] for k in range(5))
    assert sr == pytest.approx(-0.19876715841903386, rel=1e-13)
    assert env.h.sum() == float(g["kat_sum_h"]) == 201.91804846504377
    assert env.q.sum() == float(g["kat_sum_q"]) == -10.390332178211654


def test_lorenz(golden):
    g = golden("lorenz")
    env = bo.lorenz()
    assert env.n_act == int(g["n_act"])
    eq(env.reset()[0], g["obs0"])
    for k, a in enumerate(g["actions"]):
        obs, rwd, *_ = env.step(int(a))
        eq(env.x, g["x"][k]); eq(env.fx, g["fx"][k]); eq(obs, g["obs"][k])
        assert rwd == g["rwd"][k]
    env.reset()
    sr, fl = 0.0, None
    for k in range(500):
        _, r, d, t, _ = env.step(k % 3)
        sr += r
        if k == 9:   # SURVEY.md §4 KAT
            eq(env.x, [-2.659737444682521, -4.401963669325503, 19.073321554161467])
            eq(env.fx, [-17.120198167294266, -19.94139701037164, -39.63498134253869])
    assert sr == float(g["kat500_sum_rwd"]) == 186.0
    assert (d, t) == tuple(g["kat500_last_flags"]) == (True, True)


def test_vortex(golden):
    g = golden("vortex")
    env = bo.vortex()
    assert env.n_act == int(g["n_act"]) and env.ndt_act == int(g["ndt_act"])
    eq(env.reset()[0], g["obs0"])
    for k in range(g["actions"].shape[0]):
        obs, rwd, *_ = env.step(g["actions"][k])
        np.testing.assert_allclose(env.x, g["x"][k], rtol=1e-13, atol=0)
        np.testing.assert_allclose(obs, g["obs"][k], rtol=1e-12, atol=1e-18)
        assert rwd == pytest.approx(g["rwd"][k], rel=1e-9, abs=1e-18)
    env.reset()
    sr = sum(env.step(np.array([0.5, -0.25]))[1] for _ in range(10))
    # SURVEY.md §4 KAT
    np.testing.assert_allclose(env.x, [-0.010474204824095492, -0.0044519423003400675, -0.0003076860892504164,
                                       -0.0028289435961359756], rtol=1e-13, atol=0)
    assert sr == pytest.approx(-0.0021355829919963414, rel=1e-9, abs=1e-18)


@pytest.mark.parametrize("name,scal", [("rayleigh", "T"), ("mixing", "C")])
def test_mac2d(golden, name, scal):
    g = golden(name)
    P = json.loads(str(g["params_json"]))
    env = bo.ENVS[name]()
    for k, v in P.items():
        assert getattr(env, k) == v, k
    eq(env.reset()[0], g["obs0"])
    for k in range(g["actions"].shape[0]):
        obs, rwd, *_ = env.step(g["actions"][k])
        assert np.array_equal(env.last_iters, g["itp"][k]), "Jacobi sweep counts differ"
        for f in ("u", "v", "p", scal):
            eq(getattr(env, f), g[f][k])
        eq(obs, g["obs"][k])
        assert rwd == g["rwd"][k]
    if name == "rayleigh":   # SURVEY.md §4 KAT: r0, r1 of the first two golden actions
        assert g["rwd"][0] == -2.162578835240081 and g["rwd"][1] == -3.1042715751735157
    else:
        assert g["rwd"][0] == -0.3581561537496566 and g["rwd"][1] == -0.35316451436195834
