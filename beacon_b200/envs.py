"""Single-environment classes with the reference's names, constructor signatures and return
tuples (SURVEY.md §8b): `reset() -> (obs, None)`, `step(a) -> (obs, rwd, done, trunc, None)`.

Each one is a batch-of-1 view of `BatchedEnv`; all arithmetic runs in the CUDA library.
Deliberate differences from the reference (documented in DESIGN.md):
  * the caller's action array is never mutated and returned observations are fresh numpy arrays
    (the reference mutates in place, rayleigh.py:165 / shkadov.py:226, and returns views of its
    history buffer, rayleigh.py:260);
  * inlet noise comes from an on-device Philox stream (seedable) instead of numpy's global RNG
    (shkadov.py:204, burgers.py:127); `step(a, noise=...)` injects explicit numbers;
  * shkadov's random warm start draws U{0..rand_steps} from a per-env numpy Generator
    (reference: Python `random.randint`, shkadov.py:120);
  * blow-up / Poisson overflow do not print or exit: see `.status` (bitmask).
Public numpy attributes of the reference (`env.h`, `env.q`, `env.u`, `env.T`, ...) are exposed as
properties that copy the device state to the host.
"""
import numpy as np
import torch

from .batched import BatchedEnv


class _Box:
    def __init__(self, low, high, shape, dtype=np.float32):
        self.low, self.high, self.shape, self.dtype = low, high, shape, dtype


class _Discrete:
    def __init__(self, n):
        self.n = n


class _Single:
    metadata = {"render.modes": ["human"]}
    _name = None
    _fields = ()

    def _make(self, seed=0, device=0, dtype=torch.float64, **kw):
        self._made = dict(seed=seed, device=device, dtype=dtype, **kw)
        self._env = BatchedEnv(self._name, batch=1, device=device, dtype=dtype, seed=seed,
                               init_state=getattr(self, "_init_state", None), **kw)
        self.n_act = self._env.n_act
        self.stp = 0
        d = self._env.cfg.d
        for k in ("nx", "ny", "dx", "dy", "dt", "ndt_act", "n_obs", "n_jets"):
            if k in d and not hasattr(self, k):
                setattr(self, k, d[k])

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        if name in self._fields and name in self._env.fields:
            v = self._env.get_state(name)[0].cpu().numpy()
            shape = self._shape(name)
            return v.reshape(shape) if shape else v
        raise AttributeError(name)

    def _shape(self, name):
        return None

    def set_state(self, **fields):
        for k, v in fields.items():
            self._env.set_state(k, np.asarray(v).reshape(1, -1))

    @property
    def status(self):
        return int(self._env.status[0])

    def _finish(self, obs, rwd, done, trunc):
        self.stp += 1
        r = rwd[0].cpu().numpy()
        return obs[0].cpu().numpy(), (float(r) if r.ndim == 0 else r), bool(done[0]), bool(trunc[0]), None

    def render(self, mode="human", show=False, dump=True):
        raise NotImplementedError("rendering is host-side visualisation, out of scope of the CUDA path (SURVEY.md §2)")

    # ---- on-disk field files in the reference's text format (fieldio.py) -------------------------
    def _dump_arrays(self):
        d = self._env.cfg.d
        if self._name in ("shkadov", "sloshing"):
            return dict(x=d["x"], h=self.h, q=self.q)
        return {k: getattr(self, k) for k in self._fields[:4]}

    def _dump(self, field_name):
        from . import fieldio
        fieldio.dump_fields(self._name, field_name, **self._dump_arrays())

    def load(self, filename):
        """The reference's load(): the file's fields become the INITIAL state used by reset()
        (shkadov.py:364-368, sloshing.py:310-314, rayleigh.py:356-362).  The native env is rebuilt."""
        from . import fieldio
        d = self._env.cfg.d
        f = fieldio.load_fields(self._name, filename, nx=d["nx"] if self._name == "shkadov" else None)
        f.pop("x", None)
        self._init_state = f
        self._rebuild()

    def _rebuild(self):
        self._env.close()
        self._make(**self._made)

    def warmup(self, n=None):
        """Run `n` (default n_warmup) uncontrolled actions on the device, like the reference's
        warmup() (shkadov.py:154-158, rayleigh.py:131-135, sloshing.py:125-129): the previous action is
        repeated, observations and rewards are discarded."""
        d = self._env.cfg.d
        n = d["n_warmup"] if n is None else int(n)
        e = self._env
        a = e.get_state("u" if self._name in ("shkadov", "sloshing") else "a")
        stp = e.get_state("stp")          # the reference's warmup() calls solve() only: the step counter does not move
        left = n
        while left > 0:
            k = min(50, left)
            e.step_fused(a.reshape(1, 1, -1).expand(k, 1, -1).contiguous())
            left -= k
        e.set_state("stp", stp)

    def close(self):
        self._env.close()


class shkadov(_Single):
    """shkadov.py:16-368."""
    _name = "shkadov"
    _fields = ("h", "q", "rhsh", "rhsq", "u", "up")

    def __init__(self, cpu=0, init=True, L0=150.0, n_jets=5, jet_pos=150.0, jet_space=10.0, delta=0.1, t_act=20.0,
                 render_style="dynamic", seed=0, device=0, dtype=torch.float64, _per_jet=False):
        self.n_jets, self.rand_init, self.rand_steps, self.sigma = n_jets, True, 400, 5.0e-4
        self._kw = dict(init=init, L0=L0, n_jets=n_jets, jet_pos=jet_pos, jet_space=jet_space, delta=delta, t_act=t_act,
                        per_jet_rwd=_per_jet)
        self._seed, self._device, self._dtype = seed, device, dtype
        self._make(seed=seed, device=device, dtype=dtype, sigma=self.sigma, **self._kw)
        self._built_sigma = self.sigma
        self._rng = np.random.default_rng(seed)
        n_obs = self._env.cfg.d["n_obs"]
        self.action_space = _Box(-1.0, 1.0, (n_jets,))
        high = np.ones(n_obs * n_jets)
        self.observation_space = _Box(-high, high, (n_obs * n_jets,))

    def _sync_sigma(self):
        # `sigma` is a plain attribute callers overwrite after construction (SURVEY.md §5)
        if self.sigma != self._built_sigma:
            state = self._env.state_dict()
            self._env.close()
            self._make(seed=self._seed, device=self._device, dtype=self._dtype, sigma=self.sigma, **self._kw)
            self._env.load_state_dict(state)
            self._built_sigma = self.sigma

    def reset(self, n_warm=None):
        self._sync_sigma()
        if n_warm is None:
            n_warm = int(self._rng.integers(0, self.rand_steps + 1)) if self.rand_init else 0
        obs = self._env.reset(n_warm=torch.tensor([n_warm], dtype=torch.int32))
        self.stp = 0
        return obs[0].cpu().numpy(), None

    def step(self, u=None, noise=None):
        self._sync_sigma()
        a = self._env.get_state("u") if u is None else torch.as_tensor(np.array(u, dtype=np.float64).reshape(1, -1))
        nz = None if noise is None else torch.as_tensor(np.array(noise, dtype=np.float64).reshape(1, -1))
        return self._finish(*self._env.step(a, noise=nz))


    def dump(self, field_name, jet_name=None):
        """shkadov.py:353-361: columns x, h, q; the current jet actions go to `jet_name`."""
        self._dump(field_name)
        if jet_name is not None:
            np.savetxt(jet_name, self.u, fmt="%.5e")


class shkadov_separable(shkadov):
    """shkadov.py:376-481: one call per jet, the solver advances when count == 0."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, _per_jet=True, **kwargs)
        self.count = 0
        n_obs = self._env.cfg.d["n_obs"]
        self.observation_space = _Box(-np.ones(n_obs), np.ones(n_obs), (n_obs,))
        self._last = None

    def reset(self, n_warm=None):
        if self.count == 0:
            obs, _ = super().reset(n_warm)
            self._obs = obs.reshape(self.n_jets, -1)
        obs = self._obs[self.count].copy()
        self.count = 0 if self.count == self.n_jets - 1 else self.count + 1
        return obs, None

    def step(self, u=None, noise=None):
        if self.count == 0:
            stp = self.stp
            obs, rwd, done, trunc, _ = super().step(u, noise)
            self.stp = stp                                   # advanced after the last jet (:447-449)
            self._last = (obs.reshape(self.n_jets, -1), np.atleast_1d(rwd), done, trunc)
        obs, rwd, done, trunc = self._last
        out = (obs[self.count].copy(), float(rwd[self.count]), done, trunc, None)
        if self.count == self.n_jets - 1:
            self.count = 0
            self.stp += 1
        else:
            self.count += 1
        return out


class burgers(_Single):
    """burgers.py:17-166."""
    _name = "burgers"
    _fields = ("u", "up", "upp")

    def __init__(self, cpu=0, u_target=0.5, amp=10.0, sigma=0.1, ctrl_pos=1.0, L=2.0, seed=0, device=0, dtype=torch.float64):
        self._make(seed=seed, device=device, dtype=dtype, u_target=u_target, amp=amp, sigma=sigma, ctrl_pos=ctrl_pos, L=L)
        self.action_space = _Box(-1.0, 1.0, (1,))
        self.observation_space = _Box(np.zeros(5), np.ones(5), (5,))

    def reset(self):
        self.stp = 0
        return self._env.reset()[0].cpu().numpy(), None

    def step(self, a=None, noise=None):
        act = self._env.get_state("a") if a is None else torch.as_tensor(np.array(a, dtype=np.float64).reshape(1, 1))
        nz = None if noise is None else torch.as_tensor(np.array(noise, dtype=np.float64).reshape(1, 1))
        return self._finish(*self._env.step(act, noise=nz))


class sloshing(_Single):
    """sloshing.py:15-244."""
    _name = "sloshing"
    _fields = ("h", "q", "rhsh", "rhsq", "u", "up")

    def __init__(self, cpu=0, init=True, L=2.5, amp=5.0, alpha=0.0005, g=9.81, device=0, dtype=torch.float64):
        self._make(device=device, dtype=dtype, init=init, L=L, amp=amp, alpha=alpha, g=g)
        n = self._env.n_obs
        self.action_space = _Box(-1.0, 1.0, (1,))
        self.observation_space = _Box(-np.ones(n), np.ones(n), (n,))

    def reset(self):
        self.stp = 0
        return self._env.reset()[0].cpu().numpy(), None

    def step(self, u=None):
        act = self._env.get_state("u") if u is None else torch.as_tensor(np.array(u, dtype=np.float64).reshape(1, 1))
        return self._finish(*self._env.step(act))


    def dump(self, field_name, control_name=None):
        """sloshing.py:298-307: columns x, h, q (interior cells)."""
        self._dump(field_name)
        if control_name is not None:
            np.savetxt(control_name, self.u, fmt="%.5e")


class lorenz(_Single):
    """lorenz.py:18-172."""
    _name = "lorenz"
    _fields = ("x", "fx")

    def __init__(self, cpu=0, sigma=10.0, rho=28.0, beta=8.0 / 3.0, device=0, dtype=torch.float64):
        self._make(device=device, dtype=dtype, sigma=sigma, rho=rho, beta=beta)
        self.action_space = _Discrete(3)
        self.observation_space = _Box(-np.ones(6), np.ones(6), (6,))
        self.u = 1

    def reset(self):
        self.stp, self.u = 0, 1
        return self._env.reset()[0].cpu().numpy(), None

    def step(self, u=None):
        self.u = self.u if u is None else int(u)
        return self._finish(*self._env.step(torch.tensor([self.u], dtype=torch.int32)))


class vortex(_Single):
    """vortex.py:17-208."""
    _name = "vortex"
    _fields = ("x", "fx", "t", "y")

    def __init__(self, cpu=0, re=50.0, weight=50.0, device=0, dtype=torch.float64):
        self._make(device=device, dtype=dtype, re=re, weight=weight)
        self.action_space = _Box(-1.0, 1.0, (2,))
        self.observation_space = _Box(-np.ones(8) * 1.0e-4, np.ones(8) * 1.0e-4, (8,))
        self.u = np.zeros(2)

    def reset(self):
        self.stp, self.u = 0, np.zeros(2)
        return self._env.reset()[0].cpu().numpy(), None

    def step(self, u=None):
        self.u = self.u if u is None else np.array(u, dtype=np.float64)
        return self._finish(*self._env.step(torch.as_tensor(self.u.reshape(1, 2))))


class _Mac(_Single):
    def _shape(self, name):
        d = self._env.cfg.d
        return (d["nx"] + 2, d["ny"] + 2) if name in ("u", "v", "p", "T", "C", "us", "vs") else None

    def reset(self):
        self.stp = 0
        return self._env.reset()[0].cpu().numpy(), None

    @property
    def last_iters(self):
        """sum of Jacobi sweeps of the last action (the reference's `itp`, summed over sub-steps)."""
        return int(self._env.last_iters[0, 0]) if self._env.last_iters is not None else None


class rayleigh(_Mac):
    """rayleigh.py:16-275."""
    _name = "rayleigh"
    _fields = ("u", "v", "p", "T", "a")

    def __init__(self, cpu=0, init=True, L=1.0, H=1.0, n_sgts=10, ra=1.0e4, device=0, dtype=torch.float64, ctas_per_env=1):
        self.n_sgts = n_sgts
        self._make(device=device, dtype=dtype, init=init, L=L, H=H, n_sgts=n_sgts, ra=ra, ctas_per_env=ctas_per_env)
        n = self._env.n_obs
        self.action_space = _Box(-0.75, 0.75, (n_sgts,))
        self.observation_space = _Box(-np.ones(n), np.ones(n), (n,))

    def step(self, a=None):
        act = self._env.get_state("a") if a is None else torch.as_tensor(np.array(a, dtype=np.float64).reshape(1, -1))
        return self._finish(*self._env.step(act, want_iters=True))


    def dump(self, field_name, act_name=None, nusselt_name=None):
        """rayleigh.py:344-353: u, v, p, T stacked; the conditioned action goes to `act_name`.  The Nusselt
        history the reference appends on the host every step (rayleigh.py:273) is not kept here."""
        self._dump(field_name)
        if act_name is not None:
            np.savetxt(act_name, self.a, fmt="%.5e")


class mixing(_Mac):
    """mixing.py:17-264."""
    _name = "mixing"
    _fields = ("u", "v", "p", "C", "us", "vs")

    def __init__(self, cpu=0, L=1.0, H=1.0, re=100.0, pe=10000.0, side=0.5, C0=1.0, device=0, dtype=torch.float64,
                 ctas_per_env=1):
        self._make(device=device, dtype=dtype, L=L, H=H, re=re, pe=pe, side=side, C0=C0, ctas_per_env=ctas_per_env)
        n = self._env.n_obs
        self.action_space = _Discrete(4)
        self.observation_space = _Box(-np.ones(n), np.ones(n), (n,))
        self.a = 1

    def step(self, a=None):
        self.a = self.a if a is None else int(a)
        return self._finish(*self._env.step(torch.tensor([self.a], dtype=torch.int32), want_iters=True))


    def dump(self, field_name, action_name=None):
        """mixing.py:362-373: u, v, p, C stacked; the action is appended to `action_name`."""
        self._dump(field_name)
        if action_name is not None:
            with open(action_name, "a") as f:
                f.write(str(self.a) + "\n")


ENVS = {c.__name__: c for c in (shkadov, shkadov_separable, burgers, sloshing, lorenz, vortex, rayleigh, mixing)}
