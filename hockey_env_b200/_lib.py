"""ctypes binding of include/hockey_b200.h (the C ABI of the CUDA library).

There is no CPU fallback: if the shared library is missing or no CUDA device is present, loading /
creating an env raises -- loudly -- instead of silently running something else.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("HK_LIB_PATH") or os.path.join(_PKG, "libhockey_b200.so")  # override: A/B of builds only

OBS_DIM, ACT_DIM, INFO_DIM, STATS_DIM = 18, 4, 4, 16
N_PAIRS, CONTACT_WORDS = 27, 8
STATE_WORDS = 64 + N_PAIRS * CONTACT_WORDS
HK_OK, HK_E_INVALID, HK_E_CUDA, HK_E_NODEVICE = 0, -1, -2, -3
POLICY_EXTERNAL, POLICY_BASIC_WEAK, POLICY_BASIC_STRONG, POLICY_RANDOM, POLICY_ZERO, POLICY_PER_ENV = 0, 1, 2, 3, 4, 5
STEP_AUTORESET = 1

EXPORTS = [
    "hk_create", "hk_destroy", "hk_num_envs", "hk_reset", "hk_reset_seeded", "hk_step", "hk_step_host", "hk_host_record_bytes", "hk_rollout", "hk_get_obs", "hk_get_info", "hk_get_state",
    "hk_set_state", "hk_set_obs_state", "hk_set_opponent_policies", "hk_set_reset_modes", "hk_get_modes", "hk_get_stats", "hk_clear_stats", "hk_stats_device_ptr", "hk_copy_stats", "hk_debug_phase_cycles", "hk_debug_finish_cycles", "hk_launches_per_step", "hk_debug_lane_trace", "hk_kernel_timing", "hk_kernel_times", "hk_actor_param_bytes", "hk_actor_forward", "hk_actor_pool_scratch_bytes", "hk_actor_forward_pool", "hk_actor_forward_noisy",
    "hk_actor_forward_pool_noisy", "hk_actor_pack", "hk_td3_arena_bytes", "hk_td3_scratch_bytes", "hk_td3_update", "hk_last_error",
    "hk_version",
]


class TD3Batch(C.Structure):
    """hk_td3_batch of include/hockey_b200.h."""
    _fields_ = [("obs", C.c_void_p), ("action", C.c_void_p), ("reward", C.c_void_p), ("next_obs", C.c_void_p),
                ("done", C.c_void_p), ("idx", C.c_void_p), ("prio_weights", C.c_void_p), ("prio_idx", C.c_void_p),
                ("prio_n", C.c_int64)]


class TD3HParams(C.Structure):
    """hk_td3_hparams of include/hockey_b200.h."""
    _fields_ = [(n, C.c_float) for n in ("gamma", "tau_actor", "tau_critic", "lr_actor", "lr_critic", "wd_actor", "wd_critic",
                                         "beta", "target_noise", "target_noise_clip")]


class HockeyLibraryError(RuntimeError):
    pass


_lib = None


def load():
    """Load libhockey_b200.so and declare every export of include/hockey_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise HockeyLibraryError(
            f"{SO_PATH} is missing: build it with `python -m hockey_env_b200.build` "
            "(there is no CPU fallback for the HockeyEnv hot path)")
    L = C.CDLL(SO_PATH)
    vp, i64, u64, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int
    L.hk_create.argtypes = [C.POINTER(vp), i64, i32, i32, i32, u64, i64]
    L.hk_create.restype = i32
    L.hk_destroy.argtypes = [vp]
    L.hk_destroy.restype = i32
    L.hk_num_envs.argtypes = [vp]
    L.hk_num_envs.restype = i64
    L.hk_reset.argtypes = [vp, vp, vp, vp, vp]
    L.hk_reset.restype = i32
    L.hk_reset_seeded.argtypes = [vp, vp, vp, vp, vp, vp]
    L.hk_reset_seeded.restype = i32
    L.hk_step.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.hk_step.restype = i32
    L.hk_step_host.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, i32, vp]
    L.hk_step_host.restype = i32
    L.hk_host_record_bytes.argtypes = [i64, i32, C.POINTER(i64)]
    L.hk_host_record_bytes.restype = i64
    L.hk_set_opponent_policies.argtypes = [vp, vp]
    L.hk_set_opponent_policies.restype = i32
    L.hk_set_reset_modes.argtypes = [vp, vp]
    L.hk_set_reset_modes.restype = i32
    L.hk_get_modes.argtypes = [vp, vp, vp]
    L.hk_get_modes.restype = i32
    L.hk_rollout.argtypes = [vp, i32, i32, i32, vp, vp]
    L.hk_rollout.restype = i32
    L.hk_get_obs.argtypes = [vp, vp, vp, vp]
    L.hk_get_obs.restype = i32
    L.hk_get_info.argtypes = [vp, vp, vp, vp]
    L.hk_get_info.restype = i32
    L.hk_copy_stats.argtypes = [vp, vp, vp]
    L.hk_copy_stats.restype = i32
    L.hk_debug_phase_cycles.argtypes = [vp, vp]
    L.hk_debug_phase_cycles.restype = i32
    L.hk_debug_finish_cycles.argtypes = [vp, vp]
    L.hk_debug_finish_cycles.restype = i32
    L.hk_debug_lane_trace.argtypes = [vp, vp, C.c_int64]
    L.hk_debug_lane_trace.restype = i32
    L.hk_kernel_timing.argtypes = [vp, i32]
    L.hk_kernel_timing.restype = i32
    L.hk_kernel_times.argtypes = [vp, vp, C.POINTER(i64)]
    L.hk_kernel_times.restype = i32
    L.hk_actor_param_bytes.argtypes = []
    L.hk_actor_param_bytes.restype = i32
    L.hk_actor_forward.argtypes = [vp, vp, vp, i32, i64, i32, vp]
    L.hk_actor_forward.restype = i32
    L.hk_actor_pool_scratch_bytes.argtypes = [i64, i32]
    L.hk_actor_pool_scratch_bytes.restype = i64
    L.hk_actor_forward_pool.argtypes = [vp, i32, vp, vp, vp, i32, i64, vp, i32, vp]
    L.hk_actor_forward_pool.restype = i32
    f32 = C.c_float
    L.hk_actor_forward_noisy.argtypes = [vp, vp, vp, i32, i64, u64, vp, f32, f32, i64, i32, vp]
    L.hk_actor_forward_noisy.restype = i32
    L.hk_actor_forward_pool_noisy.argtypes = [vp, i32, vp, vp, vp, i32, i64, vp, u64, vp, f32, f32, i64, i32, vp]
    L.hk_actor_forward_pool_noisy.restype = i32
    L.hk_actor_pack.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp]
    L.hk_actor_pack.restype = i32
    L.hk_td3_arena_bytes.argtypes = []
    L.hk_td3_arena_bytes.restype = i64
    L.hk_td3_scratch_bytes.argtypes = [i32]
    L.hk_td3_scratch_bytes.restype = i64
    L.hk_td3_update.argtypes = [vp, vp, C.POINTER(TD3Batch), i32, C.POINTER(TD3HParams), vp, vp, u64, i32, vp, i32, vp]
    L.hk_td3_update.restype = i32
    L.hk_launches_per_step.argtypes = [vp]
    L.hk_launches_per_step.restype = i32
    L.hk_get_state.argtypes = [vp, vp, vp]
    L.hk_get_state.restype = i32
    L.hk_set_state.argtypes = [vp, vp, vp]
    L.hk_set_state.restype = i32
    L.hk_set_obs_state.argtypes = [vp, vp, vp]
    L.hk_set_obs_state.restype = i32
    L.hk_get_stats.argtypes = [vp, vp, vp]
    L.hk_get_stats.restype = i32
    L.hk_clear_stats.argtypes = [vp, vp]
    L.hk_clear_stats.restype = i32
    L.hk_stats_device_ptr.argtypes = [vp, C.POINTER(vp)]
    L.hk_stats_device_ptr.restype = i32
    L.hk_last_error.restype = C.c_char_p
    L.hk_version.restype = C.c_char_p
    _lib = L
    return L


def check(rc):
    """Map the ABI's error convention onto Python exceptions (ValueError for bad arguments, like the reference's
    mode setter, hockey_env.py:769-779)."""
    if rc == HK_OK:
        return
    msg = load().hk_last_error().decode("utf-8", "replace")
    if rc == HK_E_INVALID:
        raise ValueError(msg)
    raise HockeyLibraryError(f"hockey_b200 error {rc}: {msg}")
