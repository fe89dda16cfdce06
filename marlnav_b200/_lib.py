"""ctypes binding of libmarlnav_b200.so (C ABI: include/marlnav_b200.h).

There is no CPU fallback and no JIT: the shared library must have been built
in-tree (``python -m marlnav_b200.build``); loading fails loudly otherwise.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MARLNAV_B200_LIB may point at another build of the same ABI (A/B measurements only)
LIB_PATH = os.environ.get("MARLNAV_B200_LIB") or os.path.join(_HERE, "libmarlnav_b200.so")

ABI_VERSION = 4

# every symbol include/marlnav_b200.h declares
EXPORTS = ("marlnav_abi_version", "marlnav_last_error", "marlnav_obs_size", "marlnav_device_count",
           "marlnav_sizeof_env_params", "marlnav_sizeof_reset_spec", "marlnav_sizeof_io_transform",
           "marlnav_sizeof_actor_spec", "marlnav_sizeof_step_call", "marlnav_step_call_f32",
           "marlnav_host_pipe_create", "marlnav_host_pipe_destroy",
           "marlnav_counter_add", "marlnav_init_f32", "marlnav_observe_f32", "marlnav_step_f32", "marlnav_step_host_f32",
           "marlnav_step_launch_info", "marlnav_actor_sample_f32", "marlnav_act_step_f32", "marlnav_critic_value_f32",
           "marlnav_discounted_returns_f64",
           "marlnav_rollout_last_error")
# every symbol include/marlnav_b200_typed.h declares (16-bit observations; included by marlnav_b200.h)
TYPED_EXPORTS = ("marlnav_observe_typed", "marlnav_step_typed", "marlnav_step_call_typed", "marlnav_step_host_typed")
# every symbol include/marlnav_b200_rollout_typed.h declares (16-bit observations into the actor, the
# critic and the fused actor+step; included by marlnav_b200.h)
ROLLOUT_TYPED_EXPORTS = ("marlnav_actor_sample_typed", "marlnav_critic_value_typed", "marlnav_act_step_typed")
# every symbol include/marlnav_b200_final.h declares (final observations of auto-reset envs and the
# truncation-aware GAE scan; included by marlnav_b200.h)
FINAL_EXPORTS = ("marlnav_step_final_typed", "marlnav_step_call_final_typed", "marlnav_gae_f64")


class _Sized(ctypes.Structure):
    """Every ABI struct starts with ``struct_size`` = its sizeof (checked by the library)."""

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.struct_size = ctypes.sizeof(self)


class EnvParams(_Sized):
    """struct marlnav_env_params"""
    _fields_ = [("struct_size", ctypes.c_uint32)] + [(n, ctypes.c_int32) for n in
                ("num_envs", "num_agents", "num_obstacles", "episode_len")] + \
               [(n, ctypes.c_float) for n in (
                   "min_speed", "max_speed", "min_accel", "max_accel",
                   "risk_factor", "distance_factor", "heading_factor", "target_factor",
                   "soft_factor", "bond_factor",
                   "ob_risk_dist", "ag_risk_dist", "ob_coll_dist", "ag_coll_dist",
                   "agents_min_d", "agents_max_d", "max_at_prop_d", "max_angle_diff",
                   "target_radius", "cap_distance", "bond_sharpness", "ideal_dist", "init_dist",
                   "obst_x_range", "obst_x_mean", "obst_y_range", "obst_y_mean")]


RESET_TMPL_NONNEG, RESET_NOISY_AGENTS = 1, 2


class ResetSpec(_Sized):
    """struct marlnav_reset_spec"""
    _fields_ = [("struct_size", ctypes.c_uint32), ("flags", ctypes.c_int32),
                ("tmpl_states", ctypes.c_void_p), ("tmpl_obstacles", ctypes.c_void_p),
                ("tmpl_target", ctypes.c_void_p),
                ("states_env_stride", ctypes.c_int64), ("obstacles_env_stride", ctypes.c_int64),
                ("target_env_stride", ctypes.c_int64),
                ("alias_first_step", ctypes.c_int32), ("noise_chol", ctypes.c_float),
                ("noise_mult", ctypes.c_float), ("angle_range", ctypes.c_float),
                ("seed", ctypes.c_uint64), ("step_counter", ctypes.c_uint64),
                ("env_id_offset", ctypes.c_uint64), ("step_counter_dev", ctypes.c_void_p)]


class IoTransform(_Sized):
    """struct marlnav_io_transform"""
    _fields_ = [("struct_size", ctypes.c_uint64),
                ("obs_mean", ctypes.c_void_p), ("obs_scale", ctypes.c_void_p),
                ("act_mean", ctypes.c_void_p), ("act_scale", ctypes.c_void_p)]


class ActorSpec(_Sized):
    """struct marlnav_actor_spec"""
    _fields_ = [("struct_size", ctypes.c_uint64)] + \
               [(n, ctypes.c_void_p) for n in ("w1", "b1", "w_mu", "b_mu", "w_std", "b_std")] + \
               [("S", ctypes.c_int32), ("H", ctypes.c_int32), ("seed", ctypes.c_uint64),
                ("counter", ctypes.c_uint64), ("counter_dev", ctypes.c_void_p), ("row_offset", ctypes.c_uint64)]


class StepCall(_Sized):
    """struct marlnav_step_call"""
    _fields_ = [("struct_size", ctypes.c_uint64)] + \
               [(n, ctypes.c_void_p) for n in ("params", "reset", "states", "obstacles", "target", "step_num",
                                               "terminates", "actions", "obs", "rewards", "terminated", "truncated",
                                               "stats", "io", "stream")]


class MarlnavError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library once; raise if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MarlnavError(
            f"{LIB_PATH} is missing. Build it with `python -m marlnav_b200.build` "
            "(nvcc, sm_100a). marlnav_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.marlnav_last_error.restype = ctypes.c_char_p
    lib.marlnav_rollout_last_error.restype = ctypes.c_char_p
    sizeofs = ("marlnav_sizeof_env_params", "marlnav_sizeof_reset_spec", "marlnav_sizeof_io_transform",
               "marlnav_sizeof_actor_spec", "marlnav_sizeof_step_call")
    for name in EXPORTS + TYPED_EXPORTS + ROLLOUT_TYPED_EXPORTS + FINAL_EXPORTS:
        if name in sizeofs:
            getattr(lib, name).restype = ctypes.c_size_t
        elif name == "marlnav_host_pipe_destroy":
            lib.marlnav_host_pipe_destroy.restype = None
        elif name not in ("marlnav_last_error", "marlnav_rollout_last_error"):
            getattr(lib, name).restype = ctypes.c_int
    vp, i32 = ctypes.c_void_p, ctypes.c_int
    lib.marlnav_step_f32.argtypes = [vp] * 15
    lib.marlnav_step_call_f32.argtypes = [vp]
    lib.marlnav_observe_f32.argtypes = [vp] * 6
    lib.marlnav_init_f32.argtypes = [vp] * 8
    lib.marlnav_step_host_f32.argtypes = [vp] * 21
    lib.marlnav_observe_typed.argtypes = [vp] * 5 + [i32, vp]
    lib.marlnav_step_typed.argtypes = [vp] * 9 + [i32] + [vp] * 6
    lib.marlnav_step_call_typed.argtypes = [vp, i32]
    lib.marlnav_step_host_typed.argtypes = [vp] * 21 + [i32]
    lib.marlnav_host_pipe_create.argtypes = [ctypes.POINTER(vp)]
    lib.marlnav_host_pipe_destroy.argtypes = [vp]
    lib.marlnav_act_step_f32.argtypes = [vp] * 18
    lib.marlnav_obs_size.argtypes = [i32, i32]
    i64, u64, f64 = ctypes.c_longlong, ctypes.c_uint64, ctypes.c_double
    lib.marlnav_actor_sample_f32.argtypes = [vp, i64, i32, i32] + [vp] * 7 + [u64, u64, vp, u64] + [vp] * 5
    lib.marlnav_counter_add.argtypes = [vp, u64, vp]
    lib.marlnav_discounted_returns_f64.argtypes = [vp, vp, f64, i32, i64, vp, vp]
    lib.marlnav_critic_value_f32.argtypes = [vp, i64, i32, i32] + [vp] * 6
    lib.marlnav_actor_sample_typed.argtypes = [vp, i32, i64, i32, i32] + [vp] * 7 + [u64, u64, vp, u64] + [vp] * 5
    lib.marlnav_critic_value_typed.argtypes = [vp, i32, i64, i32, i32] + [vp] * 6
    lib.marlnav_act_step_typed.argtypes = [vp] * 12 + [i32] + [vp] * 6
    lib.marlnav_step_final_typed.argtypes = [vp] * 9 + [i32] + [vp] * 7
    lib.marlnav_step_call_final_typed.argtypes = [vp, i32, vp]
    lib.marlnav_gae_f64.argtypes = [vp] * 6 + [f64, f64, i32, i64, vp, vp, vp]
    got = lib.marlnav_abi_version()
    if got != ABI_VERSION:
        raise MarlnavError(f"libmarlnav_b200.so ABI {got} != binding ABI {ABI_VERSION}; rebuild")
    for cls, fn in ((EnvParams, lib.marlnav_sizeof_env_params), (ResetSpec, lib.marlnav_sizeof_reset_spec),
                    (IoTransform, lib.marlnav_sizeof_io_transform), (ActorSpec, lib.marlnav_sizeof_actor_spec),
                    (StepCall, lib.marlnav_sizeof_step_call)):
        if ctypes.sizeof(cls) != fn():
            raise MarlnavError(f"{cls.__name__}: binding layout is {ctypes.sizeof(cls)} bytes, the library's {fn()}")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().marlnav_last_error().decode(errors="replace")
        raise MarlnavError(f"{what} failed (code {rc}): {msg}")
