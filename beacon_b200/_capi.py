"""ctypes binding of include/beacon_b200.h (libbeacon_b200.so).

There is NO fallback: if the CUDA library is missing or fails to load, importing a symbol from
it raises, and every compute call needs a B200 (sm_100a) device.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libbeacon_b200.so")

F64, F32 = 0, 1
STATUS_BLOWUP, STATUS_POISSON_OVERFLOW, STATUS_NONFINITE = 1, 2, 4
KINDS = {"shkadov": 0, "burgers": 1, "sloshing": 2, "lorenz": 3, "vortex": 4, "rayleigh": 5, "mixing": 6}

_i32, _f64 = C.c_int32, C.c_double


class Common(C.Structure):
    _fields_ = [("batch", _i32), ("device", _i32), ("dtype", _i32), ("reserved", _i32),
                ("seed", C.c_uint64), ("env_index_base", C.c_int64)]


def _struct(name, ints, doubles, extra=()):
    fields = [(n, _i32) for n in ints] + [(n, _f64) for n in doubles] + list(extra)
    return type(name, (C.Structure,), {"_fields_": fields})


ShkadovParams = _struct(
    "ShkadovParams",
    ("nx", "ndt_act", "n_act", "n_interp", "n_jets", "jet_pos", "jet_hw", "jet_space", "l_obs", "n_obs",
     "obs_stride", "l_rwd", "per_jet_rwd", "reserved"),
    ("dx", "dt", "delta", "eps", "jet_amp", "sigma", "blow_lo", "blow_hi", "blowup_rwd"))
BurgersParams = _struct("BurgersParams", ("nx", "ndt_act", "n_act", "ctrl_pos", "n_obs_pts", "reserved"),
                        ("dx", "dt", "amp", "sigma", "u_target"))
SloshingParams = _struct("SloshingParams", ("nx", "ndt_act", "n_act", "n_interp", "obs_smpl", "n_obs"),
                         ("dx", "dt", "g", "amp", "alpha", "blow_lo", "blow_hi"))
LorenzParams = _struct("LorenzParams", ("ndt_act", "n_act"), ("dt", "sigma", "rho", "beta"),
                       (("x0", _f64 * 3), ("forcing", _f64 * 3)))
VortexParams = _struct("VortexParams", ("ndt_act", "n_act"),
                       ("dt", "lmbda_re", "lmbda_cx", "mu_re", "mu_cx", "alpha_re", "alpha_cx", "ire", "omega_s",
                        "omega_f", "domega", "gamma", "beta_m", "weight", "mod_min", "mod_max", "phase_min",
                        "phase_max"), (("x0", _f64 * 4),))
MacParams = _struct("MacParams",
                    ("nx", "ny", "ndt_act", "n_act", "n_sgts", "nx_sgts", "nx_obs_pts", "ny_obs_pts", "n_obs_steps",
                     "nx_obs", "ny_obs", "itmax"),
                    ("dx", "dy", "dt", "pr", "ra", "Tc", "Th", "C", "re", "pe", "u_max", "ref_c", "tol"),
                    (("ctas_per_env", _i32),))


class EnvInfo(C.Structure):
    _fields_ = [(n, _i32) for n in ("kind", "batch", "dtype", "device", "n_obs", "act_dim", "act_is_int", "rwd_dim",
                                    "n_act", "noise_dim", "n_fields", "reserved")]


EXPORTS = (
    "beacon_shkadov_create", "beacon_burgers_create", "beacon_sloshing_create", "beacon_lorenz_create",
    "beacon_vortex_create", "beacon_rayleigh_create", "beacon_mixing_create", "beacon_env_destroy", "beacon_env_info",
    "beacon_env_reset", "beacon_env_step", "beacon_env_step_host", "beacon_env_field", "beacon_env_get_state",
    "beacon_env_set_state", "beacon_env_launch_count", "beacon_last_error", "beacon_version",
    "beacon_peer_alloc", "beacon_peer_export", "beacon_peer_open", "beacon_peer_close", "beacon_peer_free",
    "beacon_env_set_physics", "beacon_env_get_physics",
)
# per-env physical parameters of beacon_env_set_physics, by env
PHYSICS = {"rayleigh": ("ra",), "mixing": ("re", "pe")}
PEER_HANDLE_BYTES = 64

_lib = None


class BeaconError(RuntimeError):
    pass


def lib():
    """Load libbeacon_b200.so; raises if it has not been built (python -m beacon_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BeaconError(f"{LIB_PATH} not found: build the CUDA extension first (python -m beacon_b200.build); "
                          "beacon_b200 has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, dp = C.c_void_p, C.POINTER(_f64)
    L.beacon_shkadov_create.argtypes = [C.POINTER(Common), C.POINTER(ShkadovParams), dp, dp, C.POINTER(vp)]
    L.beacon_burgers_create.argtypes = [C.POINTER(Common), C.POINTER(BurgersParams), C.POINTER(vp)]
    L.beacon_sloshing_create.argtypes = [C.POINTER(Common), C.POINTER(SloshingParams), dp, dp, C.POINTER(vp)]
    L.beacon_lorenz_create.argtypes = [C.POINTER(Common), C.POINTER(LorenzParams), C.POINTER(vp)]
    L.beacon_vortex_create.argtypes = [C.POINTER(Common), C.POINTER(VortexParams), C.POINTER(vp)]
    L.beacon_rayleigh_create.argtypes = [C.POINTER(Common), C.POINTER(MacParams), dp, dp, dp, dp, C.POINTER(vp)]
    L.beacon_mixing_create.argtypes = [C.POINTER(Common), C.POINTER(MacParams), dp, C.POINTER(vp)]
    L.beacon_env_destroy.argtypes = [vp]
    L.beacon_env_destroy.restype = None
    L.beacon_env_info.argtypes = [vp, C.POINTER(EnvInfo)]
    L.beacon_env_reset.argtypes = [vp, vp, vp, vp, _i32, vp, vp]
    L.beacon_env_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, _i32, vp]
    L.beacon_env_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.beacon_env_field.argtypes = [vp, _i32, C.POINTER(C.c_char_p), C.POINTER(C.c_int64), C.POINTER(_i32)]
    L.beacon_env_get_state.argtypes = [vp, C.c_char_p, vp, vp]
    L.beacon_env_set_state.argtypes = [vp, C.c_char_p, vp, vp]
    L.beacon_env_set_physics.argtypes = [vp, C.c_char_p, dp, vp]
    L.beacon_env_get_physics.argtypes = [vp, C.c_char_p, dp, vp]
    L.beacon_env_launch_count.argtypes = [vp]
    L.beacon_env_launch_count.restype = C.c_int64
    L.beacon_peer_alloc.argtypes = [_i32, C.c_uint64, C.POINTER(vp)]
    L.beacon_peer_export.argtypes = [vp, C.c_char_p]
    L.beacon_peer_open.argtypes = [C.c_char_p, _i32, C.POINTER(vp)]
    L.beacon_peer_close.argtypes = [vp]
    L.beacon_peer_free.argtypes = [_i32, vp]
    L.beacon_last_error.restype = C.c_char_p
    L.beacon_version.restype = C.c_char_p
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise BeaconError(f"libbeacon_b200 error {rc}: {lib().beacon_last_error().decode()}")
