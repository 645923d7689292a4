"""BatchedEnv — B independent environments stepped on one B200 through the C-ABI.

Observations, rewards, flags and actions are torch CUDA tensors; the solver state lives inside
the native handle (register/shared-memory resident during a launch, HBM between launches).
PyTorch is only the plumbing here (device memory, streams); all arithmetic is in
libbeacon_b200.so.  There is no CPU path.
"""
import ctypes as C

import numpy as np
import torch

from . import _capi as capi
from .params import CFG


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _host(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x


class BatchedEnv:
    """`BatchedEnv("shkadov", batch=1024, n_jets=10)`; kwargs are the reference ctor's.

    reset(mask=None, n_warm=None) -> obs [B, n_obs]
    step(actions, noise=None)     -> obs [B, n_obs], rwd [B] (or [B, n_jets]), done [B], trunc [B]
    step_fused(actions[K,B,...])  -> same with a leading K axis: K consecutive actions, one launch
    get_state(name) / set_state(name, tensor)

    Per-env physical parameters (rayleigh `ra`; mixing `re`, `pe`): each may be a scalar, as in the
    reference, or a 1-D array / list / tensor of length `batch`, one value per env; set_physics(**values)
    changes them between launches (domain randomisation: draw values for the finished envs, set_physics,
    reset(mask=done)), get_physics(name) reads them back.  All envs of a batch still share one launch.

    ctas_per_env (rayleigh / mixing): how many SMs one environment may occupy.  1 runs each env on one
    CTA (grids up to ~100x100 cells); 2..8 split each env over a thread-block cluster of that many CTAs,
    which reaches larger grids (DESIGN.md §3.6).  The state layout is the same for every value.
    """

    def __init__(self, name, batch, device=0, dtype=torch.float64, seed=0, env_index_base=0, init_state=None,
                 ctas_per_env=1, **kwargs):
        if name not in CFG:
            raise ValueError(f"unknown env '{name}' (have {sorted(CFG)})")
        if dtype not in (torch.float64, torch.float32):
            raise ValueError(f"dtype must be torch.float64 or torch.float32 (the arithmetic types of the kernels), got {dtype}")
        if ctas_per_env != 1 and name not in ("rayleigh", "mixing"):
            raise ValueError(f"ctas_per_env applies to the MAC-grid envs (rayleigh, mixing), not to {name}")
        if not torch.cuda.is_available():
            raise capi.BeaconError("beacon_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.name, self.batch, self.dtype, self.ctas_per_env = name, int(batch), dtype, int(ctas_per_env)
        self.device = torch.device("cuda", device)
        per_env = {}
        for k in capi.PHYSICS.get(name, ()):
            if k in kwargs and np.ndim(_host(kwargs[k])) != 0:
                per_env[k] = self._physics_values(k, kwargs.pop(k))   # the handle is created at the default
        self._per_env_physics = False
        self.cfg = CFG[name](**kwargs)
        d = self.cfg.d
        if init_state:                       # the reference's load(): fields that replace the shipped initial state
            for k, v in init_state.items():
                key = k + "_init"
                if key not in d:
                    raise ValueError(f"{name} has no initial field '{k}'")
                v = np.ascontiguousarray(v, dtype=np.float64)
                if v.shape != np.shape(d[key]):
                    raise ValueError(f"init_state['{k}'] has shape {v.shape}, expected {np.shape(d[key])}")
                d[key] = v
        self._lib = capi.lib()
        com = capi.Common(self.batch, device, capi.F64 if dtype == torch.float64 else capi.F32, 0, seed, env_index_base)
        h = C.c_void_p()
        L = self._lib
        with torch.cuda.device(self.device):
            if name == "shkadov":
                c = self.cfg
                p = capi.ShkadovParams(d["nx"], d["ndt_act"], d["n_act"], d["n_interp"], c.n_jets, d["jet_pos"],
                                       d["jet_hw"], d["jet_space"], d["l_obs"], d["n_obs"], d["obs_stride"],
                                       d["l_rwd"], int(c.per_jet_rwd), 0, d["dx"], d["dt"], c.delta, d["eps"],
                                       d["jet_amp"], c.sigma, -5.0 * d["h_max"], 5.0 * d["h_max"], d["blowup_rwd"])
                capi.check(L.beacon_shkadov_create(C.byref(com), C.byref(p), _dp(d["h_init"]), _dp(d["q_init"]), C.byref(h)))
            elif name == "burgers":
                c = self.cfg
                p = capi.BurgersParams(d["nx"], d["ndt_act"], d["n_act"], d["ctrl_pos"], d["n_obs_pts"], 0, d["dx"],
                                       d["dt"], c.amp, c.sigma, c.u_target)
                capi.check(L.beacon_burgers_create(C.byref(com), C.byref(p), C.byref(h)))
            elif name == "sloshing":
                c = self.cfg
                p = capi.SloshingParams(d["nx"], d["ndt_act"], d["n_act"], d["n_interp"], d["obs_smpl"], d["n_obs"],
                                        d["dx"], d["dt"], c.g, c.amp, c.alpha, -5.0 * d["h_max"], 2.0 * d["h_max"])
                capi.check(L.beacon_sloshing_create(C.byref(com), C.byref(p), _dp(d["h_init"]), _dp(d["q_init"]), C.byref(h)))
            elif name == "lorenz":
                c = self.cfg
                p = capi.LorenzParams(d["ndt_act"], d["n_act"], d["dt"], c.sigma, c.rho, c.beta,
                                      (C.c_double * 3)(*d["x0"]), (C.c_double * 3)(*d["forcing"]))
                capi.check(L.beacon_lorenz_create(C.byref(com), C.byref(p), C.byref(h)))
            elif name == "vortex":
                p = capi.VortexParams(d["ndt_act"], d["n_act"], d["dt"], d["lmbda_re"], d["lmbda_cx"], d["mu_re"],
                                      d["mu_cx"], d["alpha_re"], d["alpha_cx"], d["ire"], d["omega_s"], d["omega_f"],
                                      d["domega"], d["gamma"], d["beta_m"], d["weight"], d["mod_min"], d["mod_max"],
                                      d["phase_min"], d["phase_max"], (C.c_double * 4)(*d["x0"]))
                capi.check(L.beacon_vortex_create(C.byref(com), C.byref(p), C.byref(h)))
            elif name == "rayleigh":
                c = self.cfg
                p = capi.MacParams(d["nx"], d["ny"], d["ndt_act"], d["n_act"], c.n_sgts, d["nx_sgts"], d["nx_obs_pts"],
                                   d["ny_obs_pts"], d["n_obs_steps"], d["nx_obs"], d["ny_obs"], d["itmax"], d["dx"],
                                   d["dy"], d["dt"], d["pr"], d["ra"], d["Tc"], d["Th"], d["C"], 0.0, 0.0, 0.0, 0.0, d["tol"],
                                   self.ctas_per_env)
                arrs = [np.ascontiguousarray(d[k + "_init"], dtype=np.float64) for k in "uvpT"]
                capi.check(L.beacon_rayleigh_create(C.byref(com), C.byref(p), *[_dp(a) for a in arrs], C.byref(h)))
            elif name == "mixing":
                p = capi.MacParams(d["nx"], d["ny"], d["ndt_act"], d["n_act"], 0, 0, d["nx_obs_pts"], d["ny_obs_pts"],
                                   d["n_obs_steps"], d["nx_obs"], d["ny_obs"], d["itmax"], d["dx"], d["dy"], d["dt"],
                                   0.0, 0.0, 0.0, 0.0, 0.0, d["re"], d["pe"], d["u_max"], d["ref_c"], d["tol"], self.ctas_per_env)
                Ci = np.ascontiguousarray(d["C_init"], dtype=np.float64)
                capi.check(L.beacon_mixing_create(C.byref(com), C.byref(p), _dp(Ci), C.byref(h)))
        self._h = h
        info = capi.EnvInfo()
        capi.check(L.beacon_env_info(self._h, C.byref(info)))
        self.info = info
        self.n_obs, self.act_dim, self.rwd_dim, self.n_act = info.n_obs, info.act_dim, info.rwd_dim, info.n_act
        self.act_is_int, self.noise_dim = bool(info.act_is_int), info.noise_dim
        self.fields = {}
        for i in range(info.n_fields):
            nm, cnt, isint = C.c_char_p(), C.c_int64(), C.c_int32()
            capi.check(L.beacon_env_field(self._h, i, C.byref(nm), C.byref(cnt), C.byref(isint)))
            self.fields[nm.value.decode()] = (cnt.value, bool(isint.value))
        self.status = torch.zeros(self.batch, dtype=torch.int32, device=self.device)
        self.last_iters = None
        if per_env:
            self.set_physics(**per_env)

    # ------------------------------------------------------------------------------------
    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.beacon_env_destroy(h)
            self._h = None

    close = __del__

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _real(self, t, shape, what):
        t = torch.as_tensor(t, device=self.device)
        if t.dtype != self.dtype:
            t = t.to(self.dtype)
        t = t.contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"{what}: expected shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    def reset(self, mask=None, n_warm=None, noise=None, max_warm=None, out=None):
        """Envs with mask[b] (all when None) go back to the reset state; shkadov runs n_warm[b]
        zero-action warm steps first (the reference draws random.randint(0,400), shkadov.py:120).

        Returns obs [B, n_obs].  With a mask only the rows of the masked envs are written: pass the
        current observations as `out` to get them merged in place (VectorEnv does); without `out`
        the rows of unmasked envs are NaN — they are NOT observations.
        `max_warm` is an upper bound of n_warm (entries above it are clipped); giving it avoids the
        device->host read of n_warm.max() (no host sync in the call)."""
        B = self.batch
        if out is not None:
            obs = out
            if obs.dtype != self.dtype or tuple(obs.shape) != (B, self.n_obs) or not obs.is_contiguous() or obs.device != self.device:
                raise ValueError(f"reset: out must be a contiguous {self.dtype} tensor of shape {(B, self.n_obs)} on {self.device}")
        elif mask is None:
            obs = torch.empty(B, self.n_obs, dtype=self.dtype, device=self.device)
        else:
            obs = torch.full((B, self.n_obs), float("nan"), dtype=self.dtype, device=self.device)
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            if tuple(m.shape) != (B,):
                raise ValueError("mask must have shape [batch]")
        w, nz = None, None
        if n_warm is not None:
            if self.name != "shkadov":
                raise ValueError("n_warm only applies to shkadov")
            w = torch.as_tensor(n_warm).to(torch.int32)
            if tuple(w.shape) != (B,):
                raise ValueError("n_warm must have shape [batch]")
            if max_warm is None:
                max_warm = int(w.max().item())
            w = w.to(self.device).contiguous()
            max_warm = int(max_warm)
            if noise is not None:
                nz = self._real(noise, (max_warm, B, self.noise_dim), "noise")
        else:
            max_warm = 0
        with torch.cuda.device(self.device):
            capi.check(self._lib.beacon_env_reset(self._h, _ptr(m), _ptr(w), _ptr(nz), max_warm, _ptr(obs), self._stream()))
        return obs

    def step_fused(self, actions, noise=None, want_iters=False, out=None):
        """K consecutive actions in one launch.  actions [K,B,act_dim] real, or [K,B] int.
        `out` = (obs [K,B,n_obs], rwd [K,B,rwd_dim], done uint8 [K,B], trunc uint8 [K,B]) preallocated
        device tensors (no allocation in the call; the flags come back as views of them)."""
        B = self.batch
        actions = torch.as_tensor(actions)
        K = int(actions.shape[0])
        if self.act_is_int:
            a = torch.as_tensor(actions, device=self.device).to(torch.int32).contiguous()
            if tuple(a.shape) != (K, B):
                raise ValueError(f"actions: expected shape {(K, B)}, got {tuple(a.shape)}")
        else:
            a = self._real(actions, (K, B, self.act_dim), "actions")
        nz = None
        if noise is not None:
            if self.noise_dim == 0:
                raise ValueError(f"{self.name} takes no noise")
            nz = self._real(noise, (K, B, self.noise_dim), "noise")
        if out is None:
            obs = torch.empty(K, B, self.n_obs, dtype=self.dtype, device=self.device)
            rwd = torch.empty(K, B, self.rwd_dim, dtype=self.dtype, device=self.device)
            done = torch.empty(K, B, dtype=torch.uint8, device=self.device)
            trunc = torch.empty(K, B, dtype=torch.uint8, device=self.device)
        else:
            obs, rwd, done, trunc = out
            for t, shp, dt, what in ((obs, (K, B, self.n_obs), self.dtype, "obs"), (rwd, (K, B, self.rwd_dim), self.dtype, "rwd"),
                                     (done, (K, B), torch.uint8, "done"), (trunc, (K, B), torch.uint8, "trunc")):
                if t.dtype != dt or tuple(t.shape) != shp or not t.is_contiguous() or t.device != self.device:
                    raise ValueError(f"out.{what}: expected a contiguous {dt} tensor of shape {shp} on {self.device}")
        iters = torch.zeros(K, B, dtype=torch.int64, device=self.device) if want_iters else None
        with torch.cuda.device(self.device):
            capi.check(self._lib.beacon_env_step(self._h, _ptr(a), _ptr(nz), _ptr(obs), _ptr(rwd), _ptr(done), _ptr(trunc),
                                                 _ptr(self.status), _ptr(iters), K, self._stream()))
        self.last_iters = iters
        if self.rwd_dim == 1:
            rwd = rwd[..., 0]
        # the kernels write 0 / 1 flags: a bool view costs no conversion kernels on the stream
        return obs, rwd, done.view(torch.bool), trunc.view(torch.bool)

    def step_into(self, actions, obs_ptr, rwd_ptr, done_ptr, trunc_ptr, noise=None):
        """One gym step whose observation / reward / flag rows are written to RAW device addresses
        (ints): memory this process does not own as torch tensors, e.g. this rank's slice of a
        learner buffer mapped from another GPU (beacon_b200.peer.LearnerBuffer).  Layout as in
        step(): obs [B,n_obs], rwd [B,rwd_dim], done / trunc uint8 [B]."""
        B = self.batch
        if self.act_is_int:
            a = torch.as_tensor(actions, device=self.device).to(torch.int32).contiguous()
            if tuple(a.shape) != (B,):
                raise ValueError(f"actions: expected shape {(B,)}, got {tuple(a.shape)}")
        else:
            a = self._real(actions, (B, self.act_dim), "actions")
        nz = None
        if noise is not None:
            if self.noise_dim == 0:
                raise ValueError(f"{self.name} takes no noise")
            nz = self._real(noise, (B, self.noise_dim), "noise")
        with torch.cuda.device(self.device):
            capi.check(self._lib.beacon_env_step(self._h, _ptr(a), _ptr(nz), C.c_void_p(int(obs_ptr)), C.c_void_p(int(rwd_ptr)),
                                                 C.c_void_p(int(done_ptr)), C.c_void_p(int(trunc_ptr)), _ptr(self.status), None, 1,
                                                 self._stream()))

    def step(self, actions, noise=None, want_iters=False):
        """One gym step for the whole batch. actions [B,act_dim] real or [B] int."""
        a = torch.as_tensor(actions, device=self.device)
        nz = None if noise is None else torch.as_tensor(noise, device=self.device).reshape(1, self.batch, -1)
        o, r, d, t = self.step_fused(a.unsqueeze(0), nz, want_iters)
        return o[0], r[0], d[0], t[0]

    def step_host(self, actions, noise=None, out=None):
        """End-to-end gym step with HOST buffers (numpy / pinned torch CPU tensors): H2D copy of the
        actions, the step kernel, D2H copy of obs/rewards/flags, stream sync — all inside the call
        (beacon_env_step_host).  `out` may hold preallocated pinned tensors (obs, rwd, done, trunc)."""
        B = self.batch

        def host(t, dt, shape, what):
            t = torch.as_tensor(t)
            if t.is_cuda:
                raise ValueError(f"step_host: {what} must be a host buffer")
            if t.dtype != dt:
                t = t.to(dt)
            t = t.contiguous()
            if tuple(t.shape) != tuple(shape):
                raise ValueError(f"step_host: {what}: expected shape {tuple(shape)}, got {tuple(t.shape)}")
            return t

        a = host(actions, torch.int32, (B,), "actions") if self.act_is_int else host(actions, self.dtype, (B, self.act_dim), "actions")
        nz = None
        if noise is not None:
            if self.noise_dim == 0:
                raise ValueError(f"{self.name} takes no noise")
            nz = host(noise, self.dtype, (B, self.noise_dim), "noise")
        if out is None:
            out = self.alloc_host_outputs()
        if len(out) != 5:
            raise ValueError("step_host: out must be (obs, rwd, done, trunc, status) as returned by alloc_host_outputs()")
        obs, rwd, done, trunc, status = out
        # the native side writes B*n_obs*sizeof(real) ... bytes into these buffers: refuse anything else
        for t, dt, shp, what in ((obs, self.dtype, (B, self.n_obs), "obs"), (rwd, self.dtype, (B, self.rwd_dim), "rwd"),
                                 (done, torch.uint8, (B,), "done"), (trunc, torch.uint8, (B,), "trunc"),
                                 (status, torch.int32, (B,), "status")):
            if not isinstance(t, torch.Tensor) or t.is_cuda or t.dtype != dt or tuple(t.shape) != shp or not t.is_contiguous():
                raise ValueError(f"step_host: out.{what} must be a contiguous host {dt} tensor of shape {shp}")
        with torch.cuda.device(self.device):
            capi.check(self._lib.beacon_env_step_host(self._h, _ptr(a), _ptr(nz), _ptr(obs), _ptr(rwd), _ptr(done),
                                                      _ptr(trunc), _ptr(status), self._stream()))
        return obs, (rwd[:, 0] if self.rwd_dim == 1 else rwd), done.bool(), trunc.bool()

    def alloc_host_outputs(self, pinned=True):
        B = self.batch
        mk = lambda *s, dt: torch.empty(*s, dtype=dt, pin_memory=pinned)
        return (mk(B, self.n_obs, dt=self.dtype), mk(B, self.rwd_dim, dt=self.dtype), mk(B, dt=torch.uint8),
                mk(B, dt=torch.uint8), mk(B, dt=torch.int32))

    # ------------------------------------------------------------------------------------
    def get_state(self, name):
        cnt, isint = self.fields[name]
        t = torch.empty(self.batch, cnt, dtype=torch.int32 if isint else self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            capi.check(self._lib.beacon_env_get_state(self._h, name.encode(), _ptr(t), self._stream()))
        return t

    def set_state(self, name, value):
        cnt, isint = self.fields[name]
        t = torch.as_tensor(value, device=self.device).to(torch.int32 if isint else self.dtype).reshape(self.batch, cnt).contiguous()
        with torch.cuda.device(self.device):
            capi.check(self._lib.beacon_env_set_state(self._h, name.encode(), _ptr(t), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()   # `t` may be a temporary

    def state_dict(self):
        """Full device state (binary checkpoint; SURVEY.md §5 'Checkpoint / resume'), including the
        per-env Philox draw counter of the inlet noise ("draws", shkadov / burgers): a restored env
        continues the same noise stream as an uninterrupted one.  A handle with per-env physical
        parameters also carries them ("ra", or "re" and "pe", float64 [B])."""
        sd = {k: self.get_state(k).cpu() for k in self.fields}
        if self._per_env_physics:
            sd.update({k: self.get_physics(k) for k in capi.PHYSICS[self.name]})
        return sd

    def load_state_dict(self, sd):
        phys = {k: v for k, v in sd.items() if k in capi.PHYSICS.get(self.name, ())}
        if phys:
            self.set_physics(**phys)
        for k, v in sd.items():
            if k not in phys:
                self.set_state(k, v)

    # ------------------------------------------------------------------------------------
    def _physics_values(self, name, values):
        if name not in capi.PHYSICS.get(self.name, ()):
            have = capi.PHYSICS.get(self.name)
            raise ValueError(f"{self.name} has no per-env physical parameter '{name}'" +
                             (f" (it has {', '.join(have)})" if have else " (only rayleigh and mixing have them)"))
        v = np.ascontiguousarray(_host(values), dtype=np.float64)
        if v.shape != (self.batch,):
            raise ValueError(f"{name}: expected a scalar or {self.batch} per-env values, got shape {v.shape}")
        if not (np.all(np.isfinite(v)) and np.all(v > 0)):
            raise ValueError(f"{name}: per-env values must be finite and > 0")
        return v

    def set_physics(self, **values):
        """Per-env physical parameters, one array of length `batch` each: rayleigh `ra`; mixing `re`
        (which also sets the wall speed u_max = re nu / L) and `pe`.  Stream-ordered: the values apply from
        the next reset or step.  Every value is checked before any is applied."""
        vals = {k: self._physics_values(k, v) for k, v in values.items()}
        with torch.cuda.device(self.device):
            for k, v in vals.items():
                capi.check(self._lib.beacon_env_set_physics(self._h, k.encode(), _dp(v), self._stream()))
                self._per_env_physics = True

    def get_physics(self, name):
        """float64 [B] CPU tensor of the per-env values of `name` (the handle's scalar for every env
        while none has been set)."""
        self._physics_values(name, np.ones(self.batch))
        out = np.empty(self.batch, dtype=np.float64)
        with torch.cuda.device(self.device):
            capi.check(self._lib.beacon_env_get_physics(self._h, name.encode(), _dp(out), self._stream()))
        return torch.from_numpy(out)

    @property
    def launches(self):
        return int(self._lib.beacon_env_launch_count(self._h))
