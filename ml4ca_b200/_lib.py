"""ctypes binding of libml4ca_b200.so (the C ABI declared in include/ml4ca_b200.h).

There is no CPU fallback: if the shared library is missing this module raises at import of the
first symbol, and every compute entry fails with ML4CA_ERR_NO_DEVICE without a CUDA device.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ML4CA_LIB", os.path.join(_HERE, "libml4ca_b200.so"))   # ML4CA_LIB: tuning variants only

c_f32p = ctypes.c_void_p
c_u8p = ctypes.c_void_p
c_i32p = ctypes.c_void_p
c_stream = ctypes.c_void_p


class EnvCfg(ctypes.Structure):
    """struct ml4ca_env_cfg"""
    _fields_ = [
        ("kind", ctypes.c_int32), ("cont_ang", ctypes.c_int32), ("extended_state", ctypes.c_int32),
        ("n_substeps", ctypes.c_int32), ("max_ep_len", ctypes.c_int32), ("auto_reset", ctypes.c_int32),
        ("reset_acts", ctypes.c_int32), ("hull_model", ctypes.c_int32),
        ("ss_bounds", ctypes.c_float * 6), ("sim_dt", ctypes.c_float), ("step_dt", ctypes.c_float),
        ("reset_fraction", ctypes.c_float), ("actuator_lag_s", ctypes.c_float),
        ("seed", ctypes.c_uint64), ("env_id_offset", ctypes.c_int64),
    ]


class DisturbanceCfg(ctypes.Structure):
    """struct ml4ca_disturbance_cfg"""
    _fields_ = [
        ("current_speed_min", ctypes.c_float), ("current_speed_max", ctypes.c_float),
        ("current_dir_min", ctypes.c_float), ("current_dir_max", ctypes.c_float),
        ("bias_std", ctypes.c_float * 3), ("bias_time_s", ctypes.c_float),
    ]


class WaveCfg(ctypes.Structure):
    """struct ml4ca_wave_cfg"""
    _fields_ = [("sigma", ctypes.c_float * 3), ("omega_min", ctypes.c_float), ("omega_max", ctypes.c_float),
                ("damping", ctypes.c_float)]


class ObserverCfg(ctypes.Structure):
    """struct ml4ca_observer_cfg"""
    _fields_ = [("hull_model", ctypes.c_int32), ("step_dt", ctypes.c_float), ("notch_damping", ctypes.c_float),
                ("wave_damping", ctypes.c_float), ("cutoff_ratio", ctypes.c_float), ("bias_time_s", ctypes.c_float),
                ("k3", ctypes.c_float * 3), ("k4", ctypes.c_float * 3)]


class RefModelCfg(ctypes.Structure):
    """struct ml4ca_refmodel_cfg"""
    _fields_ = [("step_dt", ctypes.c_float), ("zeta", ctypes.c_float * 3), ("omega", ctypes.c_float * 3),
                ("v_max", ctypes.c_float * 3), ("a_max", ctypes.c_float * 3)]


class PolicyCfg(ctypes.Structure):
    """struct ml4ca_policy_cfg"""
    _fields_ = [("obs_dim", ctypes.c_int32), ("act_dim", ctypes.c_int32), ("hidden", ctypes.c_int32),
                ("n_hidden", ctypes.c_int32), ("activation", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class QpOptions(ctypes.Structure):
    """struct ml4ca_qp_options"""
    _fields_ = [("weights", ctypes.c_float * 11), ("reduce_fuel", ctypes.c_int32), ("raw", ctypes.c_int32)]


class Ml4caError(RuntimeError):
    pass


_lib = None

_SIGNATURES = {
    "ml4ca_env_cfg_default": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(EnvCfg)]),
    "ml4ca_env_dims": (ctypes.c_int, [ctypes.POINTER(EnvCfg), ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    "ml4ca_env_create": (ctypes.c_int, [ctypes.POINTER(EnvCfg), ctypes.c_int64, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p)]),
    "ml4ca_env_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ml4ca_env_reset": (ctypes.c_int, [ctypes.c_void_p, c_u8p, ctypes.c_float, c_f32p, c_stream]),
    "ml4ca_env_reset_to": (ctypes.c_int, [ctypes.c_void_p, c_u8p, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_env_set_cut_obs": (ctypes.c_int, [ctypes.c_void_p, c_f32p]),
    "ml4ca_env_set_reset_fraction": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_float]),
    "ml4ca_env_set_ref": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_stream]),
    "ml4ca_env_step": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_u8p, c_stream]),
    "ml4ca_env_observe": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_stream]),
    "ml4ca_env_step_host": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_u8p, c_stream]),
    "ml4ca_env_get_state": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, c_stream]),
    "ml4ca_env_size": (ctypes.c_int64, [ctypes.c_void_p]),
    "ml4ca_env_set_disturbance": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(DisturbanceCfg), c_stream]),
    "ml4ca_env_set_disturbance_state": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_stream]),
    "ml4ca_env_get_disturbance": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_stream]),
    "ml4ca_env_set_waves": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(WaveCfg), c_stream]),
    "ml4ca_env_set_wave_state": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_env_get_waves": (ctypes.c_int, [ctypes.c_void_p, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_env_set_observer": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ObserverCfg), c_f32p, c_f32p, c_stream]),
    "ml4ca_error_frame": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_scale_and_clip": (ctypes.c_int, [ctypes.POINTER(EnvCfg), ctypes.c_int64, c_f32p, c_f32p, ctypes.c_void_p, c_stream]),
    "ml4ca_pinv_pid": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_pinv_allocate": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_observer_cfg_default": (ctypes.c_int, [ctypes.c_int32, ctypes.POINTER(ObserverCfg)]),
    "ml4ca_observer_reset": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_u8p, c_f32p, c_stream]),
    "ml4ca_observer_step": (ctypes.c_int, [ctypes.POINTER(ObserverCfg), ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_u8p,
                                           c_f32p, c_stream]),
    "ml4ca_refmodel_cfg_default": (ctypes.c_int, [ctypes.POINTER(RefModelCfg)]),
    "ml4ca_refmodel_reset": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_stream]),
    "ml4ca_refmodel_step": (ctypes.c_int, [ctypes.POINTER(RefModelCfg), ctypes.c_int64, c_f32p, c_f32p, c_stream]),
    "ml4ca_env_set_refmodel": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(RefModelCfg), c_f32p, c_stream]),
    "ml4ca_pinv_pid_ff": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p,
                                         c_stream]),
    "ml4ca_qp_solve": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, ctypes.c_void_p, c_stream]),
    "ml4ca_qp_options_default": (ctypes.c_int, [ctypes.POINTER(QpOptions)]),
    "ml4ca_qp_solve_ex": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, ctypes.POINTER(QpOptions), c_f32p, ctypes.c_void_p, c_stream]),
    "ml4ca_qp_allocate": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, ctypes.c_void_p, c_stream]),
    "ml4ca_policy_num_params": (ctypes.c_int64, [ctypes.POINTER(PolicyCfg)]),
    "ml4ca_policy_create": (ctypes.c_int, [ctypes.POINTER(PolicyCfg), ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p)]),
    "ml4ca_policy_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ml4ca_policy_params": (ctypes.c_void_p, [ctypes.c_void_p]),
    "ml4ca_policy_refresh": (ctypes.c_int, [ctypes.c_void_p, c_stream]),
    "ml4ca_policy_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, c_f32p, ctypes.c_uint64, ctypes.c_uint32,
                                            ctypes.c_int32, ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_policy_set_step_counter": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "ml4ca_gae": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, c_f32p, c_f32p, c_u8p, c_f32p, ctypes.c_int32, ctypes.c_float, ctypes.c_float,
                                 c_f32p, c_f32p, c_stream]),
    "ml4ca_stats": (ctypes.c_int, [ctypes.c_int64, c_f32p, ctypes.c_void_p, c_stream]),
    "ml4ca_stats5": (ctypes.c_int, [ctypes.c_int64, c_f32p, ctypes.c_void_p, c_stream]),
    "ml4ca_episode_stats": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, c_f32p, c_u8p, c_f32p, c_i32p, ctypes.c_void_p,
                                           ctypes.c_void_p, c_stream]),
    "ml4ca_normalize": (ctypes.c_int, [ctypes.c_int64, c_f32p, ctypes.c_float, ctypes.c_float, c_stream]),
    "ml4ca_ros_state": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_float, c_f32p, c_stream]),
    "ml4ca_ros_action": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_eval_metrics": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.c_float, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_alloc_to_action": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.c_float, c_f32p, c_f32p, c_f32p, c_stream]),
    "ml4ca_policy_describe": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(PolicyCfg), ctypes.POINTER(ctypes.c_int32)]),
    "ml4ca_ppo_grad": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, c_f32p, c_f32p, c_f32p,
                                      c_f32p, c_f32p, ctypes.c_float, c_f32p, ctypes.c_void_p, c_stream]),
    "ml4ca_ppo_grad_ex": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, c_f32p, c_f32p, c_f32p,
                                         c_f32p, c_f32p, ctypes.c_float, c_f32p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                         c_stream]),
    "ml4ca_ppo_ctl_begin": (ctypes.c_int, [ctypes.c_void_p, c_stream]),
    "ml4ca_ppo_ctl_end": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, c_stream]),
    "ml4ca_adam_step_dev": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_float, ctypes.c_float,
                                           ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_int32, ctypes.c_int32,
                                           c_f32p, ctypes.c_float, ctypes.c_float, ctypes.c_void_p, c_stream]),
    "ml4ca_peer_comm_create": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p)]),
    "ml4ca_peer_comm_export": (ctypes.c_int, [ctypes.c_void_p, c_u8p]),
    "ml4ca_peer_comm_connect": (ctypes.c_int, [ctypes.c_void_p, c_u8p]),
    "ml4ca_peer_comm_slab": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]),
    "ml4ca_peer_comm_connect_ptrs": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]),
    "ml4ca_peer_comm_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ml4ca_peer_comm_status": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    "ml4ca_peer_allreduce": (ctypes.c_int, [ctypes.c_void_p, c_f32p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32,
                                            ctypes.c_void_p, ctypes.c_int32, c_stream]),
    "ml4ca_adam_step_peer": (ctypes.c_int, [ctypes.c_void_p, c_f32p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                            ctypes.c_int64, c_f32p, c_f32p, c_f32p, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                            ctypes.c_float, ctypes.c_float, ctypes.c_int32, ctypes.c_int32, ctypes.c_float,
                                            ctypes.c_float, ctypes.c_void_p, c_stream]),
    "ml4ca_ppo_use_fp32": (ctypes.c_int, [ctypes.c_int]),
    "ml4ca_trpo_use_tensor_cores": (ctypes.c_int, [ctypes.c_int]),
    "ml4ca_trpo_policy_mu": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, c_f32p, c_f32p, c_stream]),
    "ml4ca_trpo_kl_grad": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, c_f32p, c_f32p, c_f32p, c_f32p,
                                          ctypes.c_void_p, c_stream]),
    "ml4ca_adam_step": (ctypes.c_int, [ctypes.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, ctypes.c_float, ctypes.c_float,
                                       ctypes.c_float, ctypes.c_float, ctypes.c_int32, ctypes.c_float, c_stream]),
    "ml4ca_last_error": (ctypes.c_char_p, []),
    "ml4ca_version": (ctypes.c_char_p, []),
    "ml4ca_launch_count": (ctypes.c_int64, []),
}


def lib():
    """The loaded library (loads on first use; raises if it has not been built)."""
    global _lib
    if _lib is None:
        if "ML4CA_LIB" not in os.environ:
            # building is not a fallback: the same sm_100a sources, compiled when the library is absent or older than
            # them (nvcc cross-compiles without a GPU; a no-op when the stamp matches)
            from . import build as _build
            try:
                _build.build()
            except FileNotFoundError:   # no nvcc on this box: use the library that travelled with the tree, if any
                pass                    # (compile / link failures propagate: a stale .so must not load silently)
        if not os.path.exists(LIB_PATH):
            raise Ml4caError(
                "libml4ca_b200.so is missing (%s). Build it with `python -m ml4ca_b200.build`; "
                "there is no CPU fallback." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(status, what=""):
    if status != 0:
        msg = lib().ml4ca_last_error().decode("utf-8", "replace")
        raise Ml4caError("%s failed (status %d): %s" % (what or "ml4ca call", status, msg))


def launch_count():
    return int(lib().ml4ca_launch_count())


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
