"""Live A/B of the oracle against the unmodified reference, wherever oracle/refload.py finds a
jviquerat/beacon checkout (REF_ROOT: BEACON_REFERENCE, else its default checkout location, else
the copy oracle/make_ref.py stages under oracle/_ref/); skipped without one.  Longer random
sequences than the golden files; fields bit-exact."""
import warnings

import numpy as np
import pytest

from oracle import beacon_oracle as bo
from oracle import refload

pytestmark = pytest.mark.skipif(not refload.available(), reason=f"no reference checkout at {refload.REF_ROOT} (set BEACON_REFERENCE to a jviquerat/beacon checkout)")
warnings.simplefilter("ignore")


def eq(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert np.array_equal(a, b), f"max abs diff {np.max(np.abs(a - b)):.3e}"


def test_shkadov_random_with_noise():
    rng = np.random.default_rng(7)
    ref, mod = refload.make("shkadov", n_jets=10)
    ref.rand_init = False
    orc = bo.shkadov(n_jets=10)
    eq(ref.reset()[0], orc.reset()[0])
    for k in range(6):
        a = rng.uniform(-1, 1, 10)
        noise = rng.uniform(-5e-4, 5e-4, 50)
        with refload.patched_noise(mod, noise):
            o1, r1, d1, t1, _ = ref.step(a.copy())
        o2, r2, d2, t2, _ = orc.step(a, noise=noise)
        for f in ("h", "q", "rhsh", "rhsq", "rhshp", "rhsqp"):
            eq(getattr(ref, f), getattr(orc, f))
        eq(o1, o2)
        assert r1 == r2 and (d1, t1) == (d2, t2)


def test_shkadov_blowup_flag():
    ref, mod = refload.make("shkadov", n_jets=2)
    ref.rand_init = False
    ref.sigma = 0.0
    orc = bo.shkadov(n_jets=2)
    ref.reset(); orc.reset()
    ref.h[300] = 40.0
    orc.h[300] = 40.0
    o1 = ref.step(np.zeros(2))
    o2 = orc.step(np.zeros(2))
    assert (o1[1], o1[2], o1[3]) == (o2[1], o2[2], o2[3])


def test_rayleigh_random():
    rng = np.random.default_rng(8)
    ref, mod = refload.make("rayleigh")
    orc = bo.rayleigh()
    eq(ref.reset()[0], orc.reset()[0])
    for k in range(3):
        a = rng.uniform(-1, 1, 10)
        o1, r1, *_ = ref.step(a.copy())
        o2, r2, *_ = orc.step(a)
        for f in ("u", "v", "p", "T", "us", "vs", "phi"):
            eq(getattr(ref, f), getattr(orc, f))
        eq(ref.a, orc.a)
        eq(o1, o2)
        assert r1 == r2


def test_mixing_one_action():
    ref, mod = refload.make("mixing")
    orc = bo.mixing()
    eq(ref.reset()[0], orc.reset()[0])
    for a in (3,):
        o1, r1, *_ = ref.step(a)
        o2, r2, *_ = orc.step(a)
        for f in ("u", "v", "p", "C"):
            eq(getattr(ref, f), getattr(orc, f))
        eq(o1, o2)
        assert r1 == r2


def test_burgers_sloshing_lorenz_vortex():
    rng = np.random.default_rng(9)
    ref, mod = refload.make("burgers")
    orc = bo.burgers()
    ref.reset(); orc.reset()
    for k in range(30):
        a, nz = rng.uniform(-1, 1, 1), rng.uniform(-0.1, 0.1, 1)
        with refload.patched_noise(mod, nz):
            o1, r1, *_ = ref.step(a.copy())
        o2, r2, *_ = orc.step(a, noise=float(nz[0]))
        eq(ref.u, orc.u); eq(ref.up, orc.up); eq(ref.upp, orc.upp); eq(o1, o2)
        assert r1 == r2
    ref, mod = refload.make("sloshing")
    orc = bo.sloshing()
    ref.reset(); orc.reset()
    for k in range(30):
        a = rng.uniform(-1, 1, 1)
        o1, r1, *_ = ref.step(a.copy())
        o2, r2, *_ = orc.step(a)
        eq(ref.h, orc.h); eq(ref.q, orc.q); eq(o1, o2)
        assert r1 == pytest.approx(r2, rel=1e-13)
    ref, mod = refload.make("lorenz")
    orc = bo.lorenz()
    ref.reset(); orc.reset()
    for k in range(200):
        a = int(rng.integers(0, 3))
        o1, r1, *_ = ref.step(np.int64(a))
        o2, r2, *_ = orc.step(a)
        eq(o1, o2)
        assert r1 == r2
    ref, mod = refload.make("vortex")
    orc = bo.vortex()
    ref.reset(); orc.reset()
    for k in range(50):
        a = rng.uniform(-1, 1, 2)
        o1, r1, *_ = ref.step(a.copy())
        o2, r2, *_ = orc.step(a)
        np.testing.assert_allclose(o1, o2, rtol=1e-12, atol=1e-18)
        assert r1 == pytest.approx(r2, rel=1e-9, abs=1e-18)
