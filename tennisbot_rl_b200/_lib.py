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
SAC_FLOATS = 70672         # SwingRacket-v0's SAC actor (TB_SAC_FLOATS)
SAC_FLOATS_HIT = 70152     # Tennisbot-v0's (TB_SAC_FLOATS_HIT)
SAC_HIDDEN = 256           # TB_SAC_HIDDEN
SAC_SAMPLE, SAC_MEAN, SAC_UNIFORM = 0, 1, 2
SAC_VECNORM = 0x100        # TB_SAC_VECNORM: OR'd into tb_sac_rollout's mode, the normaliser of tb_set_vecnorm applies
VECNORM_OBS, VECNORM_REWARD = 0, 1  # tb_vecnorm_apply's `what`
CONTROL_FORCE, CONTROL_PID = 0, 1
BODY_NONE, BODY_COURT, BODY_NET, BODY_GOAL, BODY_RACKET, BODY_BALL = 0, 1, 2, 3, 4, 5  # TB_BODY_*
RENDER_SKY = (170, 200, 235)                                                           # TB_RENDER_SKY
RENDER_COLORS = ((0, 0, 0), (70, 140, 95), (235, 235, 235), (215, 60, 50), (40, 80, 200), (225, 240, 60))  # by TB_BODY_*
RENDER_LIGHT = (-0.3, 0.4, 1.0)                                                        # TB_RENDER_LIGHT, not normalised
RENDER_MAX_SIZE = 4096
TRACE_MAX_SUBSTEPS = 776   # TB_TRACE_MAX_SUBSTEPS: substeps of SwingRacket-v0's longest env step (Tennisbot-v0's: 1)

EV_RACKET_BALL, EV_COURT_BALL, EV_GOAL_BALL, EV_TIMEOUT, EV_BALL_PASSED, EV_NET_BALL, EV_RACKET_LOW = 1, 2, 4, 8, 16, 32, 64
STAT_NAMES = ("episodes", "sum_length", "racket_hits", "goals", "court", "timeouts", "sum_return_q20",
              "sum_return2_q10", "physics_steps", "env_steps")

class TbSacRing(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("reserved", C.c_int32), ("slots", C.c_int64), ("obs", C.c_void_p),
                ("act", C.c_void_p), ("reward", C.c_void_p), ("next_obs", C.c_void_p), ("done", C.c_void_p)]


class TbCamera(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("width", C.c_int32), ("height", C.c_int32), ("reserved", C.c_int32),
                ("eye", C.c_double * 3), ("target", C.c_double * 3), ("up", C.c_double * 3), ("fov_y_deg", C.c_double)]


class TbVecNorm(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("training", C.c_int32), ("norm_obs", C.c_int32), ("norm_reward", C.c_int32),
                ("clip_obs", C.c_double), ("clip_reward", C.c_double), ("gamma", C.c_double), ("epsilon", C.c_double)]


def vecnorm_words(obs_dim):
    """TB_VECNORM_WORDS: obs mean [obs_dim], obs var [obs_dim], obs count, ret mean, ret var, ret count."""
    return 2 * obs_dim + 4


class TbConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("env_kind", C.c_int32), ("precision", C.c_int32), ("device", C.c_int32),
                ("num_envs", C.c_int64), ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
                ("auto_reset", C.c_int32), ("reserved", C.c_int32)]


_vp, _i32, _u32, _i64, _u64, _dbl = C.c_void_p, C.c_int, C.c_uint32, C.c_int64, C.c_uint64, C.c_double
_str, _dblp, _i64p = C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)
# argument types of every entry point include/tennisbot_b200.h declares (tests/test_abi.py checks the names); all return int
# except those in _STRING_RESULTS
SIGNATURES = {
    "tb_last_error": [], "tb_abi_version": [], "tb_obs_dim": [_i32], "tb_act_dim": [_i32], "tb_policy_floats": [_i32],
    "tb_es_floats": [_i32], "tb_num_params": [], "tb_param_name": [_i32], "tb_scene_constant": [_str, _i32, _dblp],
    "tb_create": [C.POINTER(TbConfig), C.POINTER(_vp)], "tb_destroy": [_vp],
    "tb_set_param": [_vp, _str, _dbl], "tb_get_param": [_vp, _str, _dblp], "tb_set_control_mode": [_vp, _i32],
    "tb_reset": [_vp, _vp, _vp, _vp], "tb_reset_from": [_vp, _vp, _vp, _vp, _vp],
    "tb_step": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp], "tb_rollout": [_vp, _i32, _i32, _vp, _vp, _vp, _vp],
    "tb_set_policy": [_vp, _vp, _i64, _vp], "tb_set_policies": [_vp, _vp, _i64, _i64, _vp],
    "tb_policy_rollout": [_vp, _i32, _i32, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tb_policy_rollout_raw": [_vp, _i32, _i32, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tb_set_vecnorm": [_vp, C.POINTER(TbVecNorm), _vp, _vp], "tb_get_vecnorm": [_vp, _vp, _vp],
    "tb_set_vecnorms": [_vp, C.POINTER(TbVecNorm), _i64, _vp, _vp], "tb_get_vecnorms": [_vp, _vp, _i64, _vp],
    "tb_vecnorm_device_ptr": [_vp, C.POINTER(_vp), _i64p],
    "tb_vecnorm_apply": [_vp, _vp, _i64, _i32, _vp, _vp],
    "tb_es_begin": [_vp, _vp, _i64, _i64, _vp, _vp], "tb_es_rollout": [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tb_es_begin_noise": [_vp, _vp, _i64, _i64, C.c_float, _u64, _u32, _vp, _vp],
    "tb_es_noise_combine": [_vp, _vp, _vp, _i64, _u64, _u32, _vp, _vp], "tb_es_normalizer_stats": [_vp, _vp, _vp],
    "tb_sac_floats": [_i32], "tb_set_sac_actor": [_vp, _vp, _i64, _vp], "tb_set_sac_actors": [_vp, _vp, _i64, _i64, _vp],
    "tb_sac_begin": [_vp, _vp],
    "tb_sac_rollout": [_vp, _i32, _i32, _u64, C.POINTER(TbSacRing), _vp, _vp],
    "tb_render": [_vp, C.POINTER(TbCamera), _vp, _i64, _vp, _vp, _vp, _vp],
    "tb_trace_max_substeps": [_i32], "tb_trace_step": [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tb_get_state": [_vp, _vp, _vp], "tb_set_state": [_vp, _vp, _vp],
    "tb_stats_device_ptr": [_vp, C.POINTER(_vp)], "tb_read_stats": [_vp, _vp, _i32, _vp],
    "tb_reset_host": [_vp, _vp, _vp], "tb_step_host": [_vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tb_launch_count": [_vp, _i64p], "tb_ff_diagnostics": [_vp, _i64p],
    "tb_set_kernel_timing": [_vp, _i32], "tb_get_kernel_timing": [_vp, _dblp, _dblp, _i64p],
}
_STRING_RESULTS = ("tb_last_error", "tb_param_name")
EXPORTS = tuple(SIGNATURES)


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
    for name, argtypes in SIGNATURES.items():
        f = getattr(L, name, None)
        if f is None:  # absent from older builds loaded through TB_LIB_PATH for comparisons
            continue
        f.argtypes = argtypes
        if name in _STRING_RESULTS:
            f.restype = C.c_char_p
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
