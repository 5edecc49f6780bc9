"""ctypes binding of libb747_b200.so (include/b747.h).

The native CUDA library is the product; there is no Python/CPU implementation of the step.
Loading fails loudly if the library has not been built (`python -m b747_rl_ctrl_b200.build`).
"""
import ctypes
import math
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B747_LIB_PATH") or os.path.join(HERE, "lib", "libb747_b200.so")
SCALAR_LIB_PATH = os.path.join(HERE, "lib", "model_simple.so")
LEGACY_LIB_PATH = os.path.join(HERE, "lib", "model.so")   # boundary of the legacy core/model_win64.dll

ABI_VERSION = 2
OK, ERR_ARG, ERR_CUDA, ERR_ALLOC, ERR_STATE = 0, -1, -2, -3, -4
F64, F32 = 0, 1


class B747Error(RuntimeError):
    pass


class Cfg(ctypes.Structure):
    """b747_cfg (include/b747.h)."""
    _fields_ = [
        ("abi_version", ctypes.c_int32), ("device", ctypes.c_int32), ("dtype", ctypes.c_int32),
        ("n_envs", ctypes.c_int32),
        ("obs_type", ctypes.c_int32), ("rew_type", ctypes.c_int32), ("ctrl_type", ctypes.c_int32),
        ("ctrl_mode", ctypes.c_int32), ("reset_ref_mode", ctypes.c_int32), ("disturbance_mode", ctypes.c_int32),
        ("norm_obs", ctypes.c_int32), ("norm_act", ctypes.c_int32), ("use_limiter", ctypes.c_int32),
        ("substeps", ctypes.c_int32), ("auto_reset", ctypes.c_int32), ("env_layer", ctypes.c_int32),
        ("done_tick", ctypes.c_int64), ("env_id_offset", ctypes.c_int64), ("seed", ctypes.c_uint64),
        ("tk", ctypes.c_double), ("action_max", ctypes.c_double), ("vartheta_max", ctypes.c_double),
        ("sample_time", ctypes.c_double), ("rew", ctypes.c_double * 8),
        ("fixed_aero_err", ctypes.c_double * 5), ("has_fixed_aero_err", ctypes.c_int32),
        ("export_signals", ctypes.c_int32), ("track_transfer", ctypes.c_int32), ("record_capacity", ctypes.c_int32),
    ]


class Episode(ctypes.Structure):
    """b747_episode (include/b747.h)."""
    _fields_ = [
        ("state0", ctypes.c_double * 6), ("use_ctrl", ctypes.c_int32), ("oscillating", ctypes.c_int32),
        ("vref_const", ctypes.c_double), ("osc_A", ctypes.c_double * 3), ("osc_f", ctypes.c_double * 3),
        ("h_ref", ctypes.c_double), ("aero_err", ctypes.c_double * 5),
    ]


_lib = None


def load():
    """Load libb747_b200.so and declare prototypes.  Raises B747Error if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B747Error(
            f"{LIB_PATH} is missing: the CUDA extension has not been built "
            "(run `python -m b747_rl_ctrl_b200.build`); there is no CPU fallback")
    L = ctypes.CDLL(LIB_PATH)
    vp, c_int, c_dp = ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_double)
    L.b747_last_error.restype = ctypes.c_char_p
    L.b747_obs_dim.argtypes = [c_int]
    L.b747_done_tick.restype = ctypes.c_int64
    L.b747_done_tick.argtypes = [ctypes.c_double]
    L.b747_create.argtypes = [ctypes.POINTER(Cfg), ctypes.POINTER(vp)]
    L.b747_destroy.argtypes = [vp]
    L.b747_stream.restype = vp
    L.b747_stream.argtypes = [vp]
    L.b747_set_stream.argtypes = [vp, vp]
    L.b747_reset.argtypes = [vp, vp, vp]
    L.b747_reset_to.argtypes = [vp, ctypes.POINTER(Episode), vp]
    L.b747_reset_to_masked.argtypes = [vp, ctypes.POINTER(Episode), vp, vp]
    L.b747_step.argtypes = [vp, vp, vp, vp, vp, vp]
    L.b747_step_host.argtypes = [vp, vp, vp, vp, vp, vp]
    L.b747_set_host_chunks.argtypes = [vp, c_int]
    L.b747_packed_record_floats.argtypes = [c_int]
    L.b747_step_packed.argtypes = [vp, vp, vp, vp]
    L.b747_step_host_packed.argtypes = [vp, vp, vp, vp]
    L.b747_set_host_mode.argtypes = [vp, c_int]
    L.b747_set_seed.argtypes = [vp, ctypes.c_uint64]
    L.b747_model_step.argtypes = [vp, ctypes.c_int32]
    L.b747_model_initialize.argtypes = [vp]
    L.b747_set_param.argtypes = [vp, ctypes.c_char_p, c_dp, c_int]
    L.b747_get_param.argtypes = [vp, ctypes.c_char_p, c_dp, c_int]
    L.b747_n_fields.restype = c_int
    L.b747_field_name.restype = ctypes.c_char_p
    L.b747_field_name.argtypes = [c_int]
    L.b747_field_index.argtypes = [ctypes.c_char_p]
    L.b747_get_field.argtypes = [vp, c_int, vp]
    L.b747_set_field.argtypes = [vp, c_int, vp]
    L.b747_episode_stats.argtypes = [vp, c_dp]
    L.b747_last_episode.argtypes = [vp, vp, vp]
    L.b747_last_episode_of.argtypes = [vp, vp, ctypes.c_int32, vp, vp]
    L.b747_state_bytes.restype = ctypes.c_int64
    L.b747_state_bytes.argtypes = [ctypes.POINTER(Cfg), ctypes.c_int32]
    L.b747_save_state.argtypes = [vp, vp, ctypes.c_int32, vp]
    L.b747_load_state.argtypes = [vp, vp, vp, vp, ctypes.c_int32]
    L.b747_set_env_param.argtypes = [vp, ctypes.c_char_p, vp, vp, ctypes.c_int32]
    L.b747_get_env_param.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_int32, vp]
    L.b747_set_env_param_range.argtypes = [vp, ctypes.c_char_p, c_dp, c_dp, c_int]
    L.b747_launch_count.restype = ctypes.c_int64
    L.b747_launch_count.argtypes = [vp]
    L.b747_synchronize.argtypes = [vp]
    L.b747_transfer_metrics.argtypes = [vp, c_int, c_int, vp]
    L.b747_recorder_n_fields.restype = c_int
    L.b747_recorder_field_name.restype = ctypes.c_char_p
    L.b747_recorder_field_name.argtypes = [c_int]
    L.b747_recorder_read.argtypes = [vp, c_int, vp, ctypes.POINTER(ctypes.c_int32)]
    L.b747_selftest_tables.argtypes = [c_int, c_int, c_dp]
    L.b747_philox4x32.argtypes = [ctypes.POINTER(ctypes.c_uint32)] * 3
    _lib = L
    return L


def check(rc):
    if rc != OK:
        raise B747Error(f"libb747_b200 error {rc}: {load().b747_last_error().decode()}")


def substeps_of(sample_time, dt=0.01):
    """K of Controller.step's loop (core/controller.py:110,261): round(sample_time/dt) with
    Python's round-half-even, sample_time=None meaning dt."""
    st = sample_time if sample_time else dt
    return max(1, round(st / dt))


def done_tick_of(tk):
    """Smallest tick with fl(tick*0.01) >= tk: Controller.is_done (core/controller.py:316-319) with
    model.time == (clockTick0)*stepSize0 (dll@0x172f-0x1747), evaluated on the host in float64 so
    that the kernels compare integers in every arithmetic mode."""
    if tk != tk or math.isinf(tk):
        return 0 if tk < 0 else 2 ** 62
    if tk <= 0:
        return 0
    n = max(0, int(math.floor(tk / 0.01)) - 2)
    while not (n * 0.01 >= tk):
        n += 1
    return n


def reward_constants(rew_type, reward_config=None):
    """The constants ControllerEnv._get_reward_def closes over (env/ctrl_env.py:109-192), as the
    8-slot array b747_cfg.rew carries.  calc_exp_k is tools/general.py:32-33."""
    rc = dict(reward_config or {})
    out = [0.0] * 8
    if rew_type == 0:  # CLASSIC
        k1, k2, k3 = rc.get("k1", 2), rc.get("k2", 2), rc.get("k3", 1)
        kf, kITSE = rc.get("kf", 0.1), rc.get("kITSE", 0.3)
        kt = -math.log(0.8) / 10
        ko = -math.log(0.75) / 0.15
        k0 = rc.get("k0", 2)
        s = k1 + k2 + k3
        out = [k1 / s, k2 / s, k3 / s, k0, kITSE, kf, kt, ko]
    elif rew_type == 1:  # PID_LIKE
        out[0] = rc.get("k", 10)
    elif rew_type == 4:  # TF_REFERENCE
        out[0], out[1], out[2] = rc.get("overshoot_ref", 2), rc.get("tp_ref", 5), rc.get("k", 0.1)
    return [float(x) for x in out]
