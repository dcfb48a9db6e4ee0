"""ctypes binding of libpime_b200.so (the C ABI declared in include/pime_b200.h).

The library is built in-tree by ``build.py`` (nvcc, sm_100a).  Loading fails loudly when it is missing: there is
no Python / CPU fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PIME_B200_LIB") or os.path.join(HERE, "libpime_b200.so")  # override: kernel A/B experiments

OK, EINVAL, ENODEV, ECUDA, ERANGE, ESTATE = 0, -1, -2, -3, -4, -5
REWARD = {"distance": 0, "square_distance": 1, "sparse": 2}
WT_OBS_GOAL, WT_OBS_INTEGRATOR, WT_OBS_STACKING = 0, 1, 2
PH_NO_INTEGRATOR, PH_INTEGRATOR, PH_INTEGRATOR_NOBOUND = 0, 1, 2
ACTOR_PLAIN, ACTOR_MODULAR, CRITIC_ADV = 0, 1, 2
PRECISION_TC, PRECISION_FP32 = 0, 1

vp = C.c_void_p


class WtConfig(C.Structure):
    _fields_ = [("A1", C.c_double), ("A2", C.c_double), ("G", C.c_double), ("sample_t", C.c_double),
                ("n_discrete", C.c_int32), ("max_step", C.c_int32), ("P_max_action", C.c_double),
                ("reward_type", C.c_int32), ("obs_mode", C.c_int32), ("num_stack", C.c_int32), ("reset_from_last_state", C.c_int32),
                ("z1", C.c_double), ("distance_threshold", C.c_double), ("integral_max", C.c_double),
                ("integral_punish", C.c_double), ("noise_scale", C.c_double),
                ("a1_lo", C.c_double), ("a1_hi", C.c_double), ("a2_lo", C.c_double), ("a2_hi", C.c_double),
                ("Kp_lo", C.c_double), ("Kp_hi", C.c_double), ("h_lo", C.c_double), ("h_hi", C.c_double),
                ("r_lo", C.c_double), ("r_hi", C.c_double)]


class WtState(C.Structure):
    _fields_ = [("h1", vp), ("h2", vp), ("r", vp), ("I", vp), ("a1", vp), ("a2", vp), ("Kp", vp), ("t", vp),
                ("episode", vp), ("ep_return", vp), ("frames", vp), ("last_h1", vp), ("last_h2", vp)]


class PhConfig(C.Structure):
    _fields_ = [("reward_type", C.c_int32), ("integrator_mode", C.c_int32), ("max_episode_steps", C.c_int32),
                ("table_len", C.c_int32), ("reset_from_last_state", C.c_int32), ("reserved0", C.c_int32),
                ("act_low", C.c_double), ("act_high", C.c_double), ("sample_t", C.c_double),
                ("mhcl_step", C.c_double), ("distance_threshold", C.c_double), ("integral_max", C.c_double),
                ("integral_punish", C.c_double), ("action_punishment", C.c_double),
                ("kw", C.c_double), ("kchem", C.c_double), ("ka", C.c_double), ("MNaOH", C.c_double), ("MHA", C.c_double),
                ("MNH3", C.c_double), ("qww_lo", C.c_double), ("qww_hi", C.c_double), ("qc_lo", C.c_double),
                ("qc_hi", C.c_double), ("x_lo", C.c_double), ("x_hi", C.c_double), ("r_lo", C.c_double), ("r_hi", C.c_double)]


class PhState(C.Structure):
    _fields_ = [("x", vp), ("y", vp), ("r", vp), ("I", vp), ("A", vp), ("B", vp), ("C", vp), ("qww_V", vp), ("qc_V", vp),
                ("t", vp), ("episode", vp), ("ep_return", vp), ("last_x", vp)]


class ActorConfig(C.Structure):
    _fields_ = [("kind", C.c_int32), ("state_dim", C.c_int32), ("mid_dim", C.c_int32), ("integrator_dim", C.c_int32),
                ("precision", C.c_int32)]


class RolloutArgs(C.Structure):
    _fields_ = [("actor", C.POINTER(ActorConfig)), ("actor_pack", vp), ("a_std_log", C.c_float), ("deterministic", C.c_int32),
                ("priorK_host", C.POINTER(C.c_double)), ("T", C.c_int32), ("auto_reset", C.c_int32),
                ("reward_scale", C.c_double), ("gamma", C.c_double), ("seed", C.c_uint64), ("env_offset", C.c_uint64),
                ("tick0", C.c_uint32), ("keep_params", C.c_uint32), ("eps", vp), ("pnoise1", vp), ("pnoise2", vp),
                ("buf_state", vp), ("buf_other", vp), ("env_action", vp), ("stats", vp), ("status", vp), ("ld", C.c_int64)]


MAX_SEGMENTS = 16


class Schedule(C.Structure):
    _fields_ = [("num_segments", C.c_int32), ("segment_steps", C.c_int32), ("resample_params", C.c_int32),
                ("reserved0", C.c_int32), ("setpoints_host", C.POINTER(C.c_double)), ("metrics", vp)]


POLICY_ACTOR, POLICY_LINEAR = 0, 1


class ScheduleExt(C.Structure):
    _fields_ = [("setpoints_dev", vp), ("policy", C.c_int32), ("reserved0", C.c_int32)]


class StepResponse(C.Structure):
    _fields_ = [("response", vp), ("settle_band", C.c_double)]


class ScheduleGains(C.Structure):
    _fields_ = [("priorK_dev", vp)]


class PpoArgs(C.Structure):
    _fields_ = [("actor", C.POINTER(ActorConfig)), ("theta", vp), ("theta_t", vp), ("adam_m", vp), ("adam_v", vp),
                ("grad_out", vp), ("buf_state", vp), ("buf_action", vp), ("buf_r_sum", vp), ("buf_logprob", vp),
                ("buf_advantage", vp), ("idx", vp), ("batch", C.c_int32), ("ratio_clip", C.c_float),
                ("lambda_entropy", C.c_float), ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("state", vp), ("work", vp), ("loss_ring", vp), ("ring_len", C.c_int32)]


# every symbol include/pime_b200.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = [
    "pime_wt_default_config", "pime_wt_reset_f32", "pime_wt_reset_f64", "pime_wt_step_f32", "pime_wt_step_f64",
    "pime_ph_default_config", "pime_ph_table_build", "pime_ph_update_system_f32", "pime_ph_update_system_f64",
    "pime_ph_reset_f32", "pime_ph_reset_f64", "pime_ph_step_f32", "pime_ph_step_f64",
    "pime_prior_action_f32", "pime_prior_action_f64",
    "pime_actor_param_count", "pime_actor_pack_bytes", "pime_actor_block_list", "pime_actor_pack", "pime_actor_forward",
    "pime_wt_rollout_f32", "pime_wt_rollout_f64", "pime_ph_rollout_f32", "pime_ph_rollout_f64",
    "pime_wt_rollout_schedule_f32", "pime_wt_rollout_schedule_f64", "pime_ph_rollout_schedule_f32", "pime_ph_rollout_schedule_f64",
    "pime_wt_rollout_schedule_ext_f32", "pime_wt_rollout_schedule_ext_f64", "pime_ph_rollout_schedule_ext_f32",
    "pime_ph_rollout_schedule_ext_f64",
    "pime_wt_rollout_schedule_response_f32", "pime_wt_rollout_schedule_response_f64", "pime_ph_rollout_schedule_response_f32",
    "pime_ph_rollout_schedule_response_f64",
    "pime_wt_rollout_schedule_gains_f32", "pime_wt_rollout_schedule_gains_f64", "pime_ph_rollout_schedule_gains_f32",
    "pime_ph_rollout_schedule_gains_f64",
    "pime_gae_scan", "pime_reduce_episode_stats_f32", "pime_reduce_episode_stats_f64",
    "pime_ppo_theta_count", "pime_ppo_theta_layout", "pime_ppo_work_floats", "pime_ppo_transpose", "pime_ppo_step", "pime_ppo_apply_grad",
    "pime_ppo_tc_work_bytes", "pime_ppo_tc_layout", "pime_ppo_grad_tc", "pime_ppo_close_step",
    "pime_wt_rollout_host_f32", "pime_ph_rollout_host_f32", "pime_set_host_slices", "pime_host_slice_plan", "pime_abi_version", "pime_last_error", "pime_device_info", "pime_philox_probe",
]

_lib = None


class PimeError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """The loaded C-ABI library.  Raises if libpime_b200.so has not been built (run build.py / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PimeError(f"{LIB_PATH} is missing: build it with `python {os.path.join(HERE, 'build.py')}` "
                            "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.pime_last_error.restype = C.c_char_p
        L.pime_actor_param_count.restype = C.c_int64
        L.pime_actor_pack_bytes.restype = C.c_int64
        L.pime_ppo_theta_count.restype = C.c_int64
        L.pime_ppo_work_floats.restype = C.c_int64
        L.pime_ppo_tc_work_bytes.restype = C.c_int64
        for name in SYMBOLS:
            getattr(L, name)
        _lib = L
    return _lib


def check(rc: int) -> None:
    """Translate a status code into the exception the reference would raise."""
    if rc == OK:
        return
    msg = lib().pime_last_error().decode("utf-8", "replace")
    if rc == ERANGE:
        raise IndexError(msg or "pH table lookup out of range (reference ph.py:188)")
    if rc == ESTATE:
        raise AssertionError(msg or "Please reset the env first")
    if rc == EINVAL:
        raise ValueError(msg)
    raise PimeError(f"libpime_b200 error {rc}: {msg}")


def ptr(t) -> C.c_void_p:
    """Device (or host) pointer of a torch tensor / None."""
    if t is None:
        return C.c_void_p(None)
    assert t.is_contiguous(), "libpime_b200 needs contiguous tensors"
    return C.c_void_p(t.data_ptr())


def stream_ptr() -> C.c_void_p:
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def wt_config(**kw) -> WtConfig:
    c = WtConfig()
    lib().pime_wt_default_config(C.byref(c))
    for k, v in kw.items():
        if k == "reward_type" and isinstance(v, str):
            v = REWARD[v]
        setattr(c, k, v)
    return c


def ph_config(**kw) -> PhConfig:
    c = PhConfig()
    lib().pime_ph_default_config(C.byref(c))
    for k, v in kw.items():
        if k == "reward_type" and isinstance(v, str):
            v = REWARD[v]
        setattr(c, k, v)
    return c
