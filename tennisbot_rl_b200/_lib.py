"""ctypes binding of include/tennisbot_b200.h (libtennisbot_b200.so).

The library is the only implementation of the env step in this package: there is no CPU or PyTorch fallback.
Loading fails loudly when the shared object is missing, and tb_create fails when no sm_100 device is usable.
"""
import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("TB_LIB_PATH", PKG / "libtennisbot_b200.so"))  # override: load another build, e.g. to compare two commits

ENV_SWING, ENV_HIT = 0, 1
F32, F64 = 0, 1
STATE_WORDS, INIT_WORDS, NUM_STATS = 32, 8, 10
ACT_RANDOM, ACT_TRACK = 0, 1
POLICY_FLOATS = 9076       # SwingRacket-v0's in-kernel policy (TB_POLICY_FLOATS)
POLICY_FLOATS_HIT = 9324   # Tennisbot-v0's (TB_POLICY_FLOATS_HIT)
ES_FLOATS = 766            # SwingRacket-v0's GatedCNN (TB_ES_FLOATS)
ES_FLOATS_HIT = 858        # Tennisbot-v0's (TB_ES_FLOATS_HIT)
ES_HISTORY = 8             # observations the GatedCNN sees (TB_ES_HISTORY)
CONTROL_FORCE, CONTROL_PID = 0, 1

EV_RACKET_BALL, EV_COURT_BALL, EV_GOAL_BALL, EV_TIMEOUT, EV_BALL_PASSED, EV_NET_BALL, EV_RACKET_LOW = 1, 2, 4, 8, 16, 32, 64
STAT_NAMES = ("episodes", "sum_length", "racket_hits", "goals", "court", "timeouts", "sum_return_q20",
              "sum_return2_q10", "physics_steps", "env_steps")

# every symbol include/tennisbot_b200.h declares (checked by tests/test_abi.py)
EXPORTS = (
    "tb_last_error", "tb_abi_version", "tb_obs_dim", "tb_act_dim", "tb_policy_floats", "tb_num_params", "tb_param_name",
    "tb_scene_constant", "tb_create", "tb_destroy", "tb_set_param", "tb_get_param", "tb_set_control_mode", "tb_reset", "tb_reset_from",
    "tb_step", "tb_rollout", "tb_get_state", "tb_set_state", "tb_stats_device_ptr", "tb_read_stats",
    "tb_reset_host", "tb_step_host", "tb_launch_count", "tb_ff_diagnostics", "tb_set_kernel_timing", "tb_get_kernel_timing",
    "tb_set_policy", "tb_policy_rollout", "tb_es_floats", "tb_es_begin", "tb_es_rollout",
    "tb_es_begin_noise", "tb_es_noise_combine", "tb_es_normalizer_stats",
)


class TbConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("env_kind", C.c_int32), ("precision", C.c_int32), ("device", C.c_int32),
                ("num_envs", C.c_int64), ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
                ("auto_reset", C.c_int32), ("reserved", C.c_int32)]


class TennisbotLibraryError(RuntimeError):
    pass


_lib = None


def load():
    """Load libtennisbot_b200.so (built by `python -m tennisbot_rl_b200.build` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise TennisbotLibraryError(
            f"{LIB_PATH} is missing: build it with `python -m tennisbot_rl_b200.build` "
            "(needs nvcc; there is no CPU fallback for the env step)")
    L = C.CDLL(str(LIB_PATH))
    vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
    L.tb_last_error.restype = C.c_char_p
    L.tb_param_name.restype = C.c_char_p
    L.tb_param_name.argtypes = [i32]
    L.tb_obs_dim.argtypes = [i32]
    L.tb_act_dim.argtypes = [i32]
    if hasattr(L, "tb_policy_floats"):
        L.tb_policy_floats.argtypes = [i32]
    L.tb_scene_constant.argtypes = [C.c_char_p, i32, C.POINTER(dbl)]
    L.tb_create.argtypes = [C.POINTER(TbConfig), C.POINTER(vp)]
    L.tb_destroy.argtypes = [vp]
    L.tb_set_param.argtypes = [vp, C.c_char_p, dbl]
    L.tb_get_param.argtypes = [vp, C.c_char_p, C.POINTER(dbl)]
    L.tb_set_control_mode.argtypes = [vp, i32]
    L.tb_reset.argtypes = [vp, vp, vp, vp]
    L.tb_reset_from.argtypes = [vp, vp, vp, vp, vp]
    L.tb_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.tb_rollout.argtypes = [vp, i32, i32, vp, vp, vp, vp]
    L.tb_get_state.argtypes = [vp, vp, vp]
    L.tb_set_state.argtypes = [vp, vp, vp]
    L.tb_stats_device_ptr.argtypes = [vp, C.POINTER(vp)]
    L.tb_read_stats.argtypes = [vp, vp, i32, vp]
    L.tb_reset_host.argtypes = [vp, vp, vp]
    L.tb_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.tb_launch_count.argtypes = [vp, C.POINTER(i64)]
    if hasattr(L, "tb_ff_diagnostics"):  # absent from older builds loaded through TB_LIB_PATH for comparisons
        L.tb_ff_diagnostics.argtypes = [vp, C.POINTER(i64)]
    if hasattr(L, "tb_set_policy"):
        L.tb_set_policy.argtypes = [vp, vp, i64, vp]
        L.tb_policy_rollout.argtypes = [vp, i32, i32, C.c_uint64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    if hasattr(L, "tb_es_begin"):
        L.tb_es_floats.argtypes = [i32]
        L.tb_es_begin.argtypes = [vp, vp, i64, i64, vp, vp]
        L.tb_es_rollout.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp]
    if hasattr(L, "tb_es_begin_noise"):
        u32, u64 = C.c_uint32, C.c_uint64
        L.tb_es_begin_noise.argtypes = [vp, vp, i64, i64, C.c_float, u64, u32, vp, vp]
        L.tb_es_noise_combine.argtypes = [vp, vp, vp, i64, u64, u32, vp, vp]
        L.tb_es_normalizer_stats.argtypes = [vp, vp, vp]
    L.tb_set_kernel_timing.argtypes = [vp, i32]
    L.tb_get_kernel_timing.argtypes = [vp, C.POINTER(dbl), C.POINTER(dbl), C.POINTER(i64)]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise TennisbotLibraryError(load().tb_last_error().decode())


def scene_constant(name, index=0):
    v = C.c_double()
    check(load().tb_scene_constant(name.encode(), index, C.byref(v)))
    return v.value


def param_names():
    L = load()
    return [L.tb_param_name(i).decode() for i in range(L.tb_num_params())]
