"""ctypes binding of libmacm.so (include/macm.h) -- the only door from the Python host to the
CUDA kernels.  There is no CPU fallback: if the shared library is missing, or no CUDA device is
present, the host classes raise instead of computing anything themselves."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MACM_LIB") or os.path.join(_HERE, "libmacm.so")   # MACM_LIB: instrumented builds (profiles/)

FLOCK, TDM = 0, 1
REWARD = {"binary": 0, "linear": 1}
ACTION = {"discrete": 0, "continuous": 1}
COORD = {"polar": 0, "cartesian": 1}
DAMPING = {"taylor": 0, "pade": 1, "2.3.0": 0, "2.3.1": 1}
OBS_F32, OBS_F16, OBS_BF16 = 0, 1, 2
OBS_DTYPE = {"float32": OBS_F32, "float16": OBS_F16, "bfloat16": OBS_BF16}   # macm_params.obs_dtype; the torch dtype names
ENV_FRESH, ENV_CONTACT_OVERFLOW, ENV_TOUCH_OVERFLOW = 1, 2, 4
BOTS = {"idle": 0, "forward": 1, "rotate": 2, "diag": 3, "flock": 4, "random": 5, "combat": 6, "circle": 7}
FLAG_REPAIR_MOV_COOLDOWN, FLAG_AUTO_RESET = 1, 2
ENV_EPISODE_SHIFT = 8
ABI_VERSION = 8
MAX_RAYS = 1024   # MACM_MAX_RAYS

i32, f64, u64 = C.c_int32, C.c_double, C.c_uint64


class MacmParams(C.Structure):
    _fields_ = [
        ("env_kind", i32), ("n_envs", i32), ("n_agents", i32), ("n_targets", i32),
        ("max_contacts", i32), ("max_touching", i32),
        ("hz", f64),
        ("velocity_iterations", i32), ("position_iterations", i32), ("warm_starting", i32), ("damping_model", i32),
        ("radius", f64), ("density", f64), ("friction", f64), ("linear_damping", f64),
        ("agent_force", f64), ("agent_rotation_speed", f64), ("time_limit", f64),
        ("reward_mode", i32), ("action_mode", i32), ("coord", i32), ("flags", i32),
        ("reward_radius", f64),
        ("cooldown_atk", f64), ("cooldown_mov_penalty", f64), ("melee_range", f64), ("melee_dmg", f64),
        ("percent_mov_penalty", f64), ("init_health", f64),
        ("start_spread", f64), ("start_x", f64), ("start_y", f64), ("target_mindist", f64), ("target_maxdist", f64),
        ("world_width", f64), ("world_height", f64),
        ("env_index_base", i32), ("obs_dtype", i32),
    ]


BUFFER_NAMES = ("posvel", "angsleep", "fat", "contact_ab", "contact_imp", "contact_count", "env_state", "targets",
                "target_idx", "tdm_state", "team", "obs", "nn_idx", "rewards", "collided", "done", "touch_scratch")


class MacmBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in BUFFER_NAMES]


class MacmBufferSizes(C.Structure):
    _fields_ = [(n, u64) for n in BUFFER_NAMES] + [("obs_dim", i32), ("action_bytes", i32), ("max_contacts", i32),
                                                   ("max_touching", i32)]


class MacmLaunchInfo(C.Structure):
    _fields_ = [(n, i32) for n in ("lanes_per_env", "agents_per_lane", "envs_per_block", "threads_per_block", "blocks",
                                   "smem_bytes_per_block", "blocks_per_sm", "sm_count", "done_step")] + \
               [(n, C.c_float) for n in ("dt", "dt_ratio", "inv_mass", "damping_factor", "binary_d2_threshold")]


# the arrays a reset copies an env's rows to before overwriting them (macm_final_out)
FINAL_NAMES = ("obs", "nn_idx", "tdm_state", "env_state")


class MacmFinalOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in FINAL_NAMES]


class MacmRolloutOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("obs", "nn_idx", "rewards", "collided", "done")] + \
               [("final_" + n, C.c_void_p) for n in FINAL_NAMES]


class MacmRenderArgs(C.Structure):
    _fields_ = [("n_frames", i32), ("height", i32), ("width", i32),
                ("envs", C.c_void_p), ("views", C.c_void_p), ("palette", C.c_void_p), ("out", C.c_void_p)]


class MacmAgentFramesArgs(C.Structure):
    _fields_ = [("n_envs", i32), ("height", i32), ("width", i32), ("half_width", f64),
                ("envs", C.c_void_p), ("palette", C.c_void_p), ("out", C.c_void_p)]


class MacmLidarArgs(C.Structure):
    _fields_ = [("n_envs", i32), ("n_rays", i32), ("max_range", f64), ("fov", f64),
                ("envs", C.c_void_p), ("fraction", C.c_void_p), ("hit", C.c_void_p)]


EXPORTS = ("macm_abi_version", "macm_strerror", "macm_last_cuda_error", "macm_params_default", "macm_create",
           "macm_destroy", "macm_get_buffer_sizes", "macm_get_launch_info", "macm_bind", "macm_reset",
           "macm_sample_reset", "macm_reset_masked", "macm_bind_final", "macm_set_auto_reset_seed", "macm_overflow_count", "macm_pack_actions",
           "macm_step", "macm_rollout", "macm_observe", "macm_bot_actions", "macm_step_host", "macm_step_host_async", "macm_host_sync",
           "macm_host_alloc",
           "macm_host_free", "macm_launch_count", "macm_set_trace", "macm_enable_peer_access", "macm_ipc_open",
           "macm_ipc_close", "macm_device_alloc", "macm_device_free", "macm_render",
           "macm_render_agents", "macm_lidar")


class MacmError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libmacm.so; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MacmError("libmacm.so is missing at %s: build it with `python -c 'import __graft_entry__ as g; "
                            "g.build()'` (nvcc, sm_100a). gym_macm has no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp = C.c_void_p
        L.macm_abi_version.restype = C.c_int
        L.macm_strerror.restype = C.c_char_p
        L.macm_strerror.argtypes = [C.c_int]
        L.macm_last_cuda_error.restype = C.c_char_p
        L.macm_last_cuda_error.argtypes = [vp]
        L.macm_params_default.argtypes = [C.POINTER(MacmParams), C.c_int]
        L.macm_create.argtypes = [C.POINTER(vp), C.POINTER(MacmParams), C.c_int]
        L.macm_destroy.argtypes = [vp]
        L.macm_get_buffer_sizes.argtypes = [vp, C.POINTER(MacmBufferSizes)]
        L.macm_get_launch_info.argtypes = [vp, C.POINTER(MacmLaunchInfo)]
        L.macm_bind.argtypes = [vp, C.POINTER(MacmBuffers)]
        L.macm_reset.argtypes = [vp, vp]
        L.macm_sample_reset.argtypes = [vp, u64, vp]
        L.macm_reset_masked.argtypes = [vp, vp, u64, vp]
        L.macm_bind_final.argtypes = [vp, C.POINTER(MacmFinalOut)]
        L.macm_set_auto_reset_seed.argtypes = [vp, u64]
        L.macm_overflow_count.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), vp]
        L.macm_pack_actions.argtypes = [vp, vp, i32, i32, vp, vp]
        L.macm_step.argtypes = [vp, vp, vp]
        L.macm_rollout.argtypes = [vp, vp, C.c_int32, C.c_int32, u64, C.POINTER(MacmRolloutOut), vp]
        L.macm_observe.argtypes = [vp, vp]
        L.macm_bot_actions.argtypes = [vp, C.c_int, u64, vp, vp]
        L.macm_render.argtypes = [vp, C.POINTER(MacmRenderArgs), vp]
        L.macm_render_agents.argtypes = [vp, C.POINTER(MacmAgentFramesArgs), vp]
        L.macm_lidar.argtypes = [vp, C.POINTER(MacmLidarArgs), vp]
        L.macm_step_host.argtypes = [vp] * 7
        L.macm_step_host_async.argtypes = [vp] * 7
        L.macm_host_sync.argtypes = [vp]
        L.macm_host_alloc.argtypes = [C.POINTER(vp), u64]
        L.macm_host_free.argtypes = [vp]
        L.macm_launch_count.restype = C.c_int64
        L.macm_launch_count.argtypes = [vp]
        L.macm_set_trace.argtypes = [vp, vp]
        L.macm_enable_peer_access.argtypes = [C.c_int, C.c_int]
        L.macm_ipc_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
        L.macm_ipc_close.argtypes = [vp]
        L.macm_device_alloc.argtypes = [C.c_int, u64, C.POINTER(vp), C.c_char_p]
        L.macm_device_free.argtypes = [vp]
        if L.macm_abi_version() != ABI_VERSION:
            raise MacmError("libmacm.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc, handle=None):
    if rc != 0:
        L = lib()
        msg = L.macm_strerror(rc).decode()
        if rc == -2 and handle:
            msg += ": " + L.macm_last_cuda_error(handle).decode()
        raise MacmError("libmacm: %s (status %d)" % (msg, rc))


def default_params(env_kind):
    p = MacmParams()
    check(lib().macm_params_default(C.byref(p), env_kind))
    return p
