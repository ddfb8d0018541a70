"""ctypes binding of libouzelum_b200.so (the C ABI declared in include/ouzelum_b200.h).

There is NO fallback: if the shared library is missing or fails to load, importing the package
raises.  Build it with `python __graft_entry__.py` (or `python -m ouzelum_b200.build`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OUZELUM_B200_LIB") or os.path.join(_HERE, "libouzelum_b200.so")   # override: kernel experiments only

OZL_ABI_VERSION = 7


def _header_enum(prefix):
    """`{name: value}` of the enumerators of include/ouzelum_b200.h whose name starts with `prefix` (the header is the one
    statement of such layouts; the library is compiled from the same file)."""
    import re
    with open(os.path.join(_HERE, "..", "include", "ouzelum_b200.h")) as f:
        return {k: int(v) for k, v in re.findall(r"\b(" + prefix + r"\w*)\s*=\s*(\d+)", f.read())}


# privileged critic state written by the step kernels (ozl_set_states_output): slot indices OZL_STATE_* and the row width
STATES_LAYOUT = _header_enum("OZL_STATE")
STATES_WIDTH = STATES_LAYOUT["OZL_STATES_WIDTH"]
# scenario rows applied at every reset (ozl_set_scenarios): slot indices OZL_SCN_* and the row width OZL_SCENARIO_WIDTH
SCENARIO_LAYOUT = _header_enum("OZL_SC")
SCENARIO_WIDTH = SCENARIO_LAYOUT["OZL_SCENARIO_WIDTH"]
# episode records appended by the step kernels (ozl_set_episode_log): slot indices OZL_EPLOG_* and the record width
EPLOG_LAYOUT = _header_enum("OZL_EPLOG")
EPLOG_WIDTH = EPLOG_LAYOUT["OZL_EPLOG_WIDTH"]


DR_NONE, DR_UNIFORM, DR_LOGUNIFORM, DR_GAUSSIAN = 0, 1, 2, 3
DR_SCALING, DR_ADDITIVE = 0, 1
DR_SCHED_NONE, DR_SCHED_LINEAR, DR_SCHED_CONSTANT = 0, 1, 2
DR_PARAMS = ("mass", "ixx", "iyy", "izz", "arm", "thrust_scale", "yaw_km")     # index = OZL_DR_*


class OzlDrParam(C.Structure):
    """Mirror of `struct ozl_dr_param` (include/ouzelum_b200.h)."""
    _fields_ = [("distribution", C.c_int32), ("operation", C.c_int32), ("range", C.c_float * 2),
                ("schedule", C.c_int32), ("schedule_steps", C.c_int32)]

    def to_tuple(self):
        return (self.distribution, self.operation, float(self.range[0]), float(self.range[1]), self.schedule, self.schedule_steps)


class OzlCfg(C.Structure):
    """Mirror of `struct ozl_cfg` (include/ouzelum_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("fault_rotors_lo", C.c_int16), ("fault_rotors_hi", C.c_int16),
        ("num_envs", C.c_int64), ("env_id_base", C.c_int64), ("seed", C.c_uint64),
        ("max_episode_length", C.c_int32), ("target_period", C.c_int32), ("target_fixed", C.c_int32),
        ("substeps", C.c_int32), ("control_freq_inv", C.c_int32),
        ("dt", C.c_float), ("gravity_z", C.c_float), ("clip_actions", C.c_float), ("clip_obs", C.c_float),
        ("thrust_rate", C.c_float), ("thrust_max", C.c_float),
        ("die_dist", C.c_float), ("die_z", C.c_float), ("up_coef", C.c_float),
        ("spawn_base", C.c_float * 3), ("spawn_lo", C.c_float * 3), ("spawn_range", C.c_float * 3),
        ("target_scale", C.c_float * 3), ("target_off", C.c_float * 3),
        ("mass", C.c_float), ("ixx", C.c_float), ("iyy", C.c_float), ("izz", C.c_float),
        ("arm", C.c_float), ("com_z", C.c_float), ("max_angvel", C.c_float),
        ("lin_drag", C.c_float), ("yaw_km", C.c_float),
        ("fault_mode", C.c_int32), ("fault_eff_lo", C.c_float), ("fault_eff_range", C.c_float),
        ("dr_enable", C.c_int32), ("dr", OzlDrParam * 7),
        ("pomdp_mode", C.c_int32), ("pomdp_prob", C.c_float), ("noise_sigma", C.c_float),
        ("collect_metrics", C.c_int32), ("plate_enable", C.c_int32), ("plate_z", C.c_float), ("plate_radius", C.c_float), ("land_cutoff", C.c_float),
        ("wrench_warmup_steps", C.c_int32), ("fault_ramp_steps", C.c_int32),
    ]

    _MULTI_FAULT = ("fault_rotors_lo", "fault_rotors_hi", "fault_ramp_steps")    # meaningful under fault_mode 2 only

    def to_dict(self):
        out = {}
        for name, typ in self._fields_:
            if name.startswith("reserved") or name == "abi_version" or (name in self._MULTI_FAULT and self.fault_mode != 2):
                continue
            v = getattr(self, name)
            if name == "dr":
                out[name] = tuple(d.to_tuple() for d in v)
            else:
                out[name] = tuple(v) if hasattr(v, "__len__") else v
        return out

    def update(self, **kw):
        for k, v in kw.items():
            if k not in dict(self._fields_):
                raise KeyError(f"ozl_cfg has no field {k!r}")
            if k == "dr":                      # {index or name: (distribution, operation, lo, hi[, schedule, schedule_steps])}
                for key, spec in (v.items() if isinstance(v, dict) else enumerate(v)):
                    j = DR_PARAMS.index(key) if isinstance(key, str) else int(key)
                    spec = tuple(spec)
                    spec = spec + (0, 0)[:6 - len(spec)]
                    d = self.dr[j]
                    d.distribution, d.operation, d.schedule, d.schedule_steps = int(spec[0]), int(spec[1]), int(spec[4]), int(spec[5])
                    d.range[0], d.range[1] = float(spec[2]), float(spec[3])
            elif isinstance(v, (tuple, list)):
                getattr(self, k)[:] = [float(x) for x in v]
            else:
                setattr(self, k, v)
        return self


class OzlHostIo(C.Structure):
    """Mirror of `struct ozl_host_io` (include/ouzelum_b200.h)."""
    _fields_ = [("actions_host", C.c_void_p), ("obs_host", C.c_void_p), ("rew_host", C.c_void_p), ("done_host", C.c_void_p),
                ("reset_host", C.c_void_p), ("reset", C.c_void_p), ("progress", C.c_void_p), ("timeout", C.c_void_p), ("ep_ret", C.c_void_p)]


class OzlPvArgs(C.Structure):
    """Mirror of `struct ozl_pv_args` (include/ouzelum_b200.h)."""
    _fields_ = [
        ("n", C.c_int64), ("x9xN", C.c_void_p), ("P81xN", C.c_void_p), ("accel3", C.c_void_p), ("quat4", C.c_void_p),
        ("pos_meas3", C.c_void_p), ("vel_meas3", C.c_void_p), ("pos_mask", C.c_void_p), ("vel_mask", C.c_void_p),
        ("dt", C.c_float), ("acc_var", C.c_float * 3), ("pos_var", C.c_float * 3), ("vel_var", C.c_float * 3),
        ("pos_var_given", C.c_int32), ("vel_var_given", C.c_int32), ("flip_qw", C.c_int32), ("do_predict", C.c_int32),
        ("pos_period", C.c_uint32), ("pos_phase", C.c_uint32), ("vel_period", C.c_uint32), ("vel_phase", C.c_uint32),
        ("iter_base", C.c_uint64),
    ]


class OzlHuskyArgs(C.Structure):
    """Mirror of `struct ozl_husky_args` (include/ouzelum_b200.h)."""
    _fields_ = [
        ("n", C.c_int64), ("pose4", C.c_void_p), ("idx2", C.c_void_p), ("tables204x2", C.c_void_p), ("reset", C.c_void_p),
        ("wheels4", C.c_void_p), ("target3", C.c_void_p), ("seed", C.c_uint64), ("step", C.c_uint64),
        ("step_ptr", C.c_void_p), ("env_id_base", C.c_int64), ("dt", C.c_float), ("dist_thresh", C.c_float), ("kp_lin", C.c_float),
        ("kp_ang", C.c_float), ("ang_thresh", C.c_float), ("x_offset", C.c_float), ("target_z", C.c_float),
        ("respawn_limit", C.c_float),
    ]


class OzlEkfLeeArgs(C.Structure):
    """Mirror of `struct ozl_ekf_lee_args` (include/ouzelum_b200.h)."""
    _fields_ = [
        ("ekf_q4xN", C.c_void_p), ("ekf_P16xN", C.c_void_p), ("pv_x9xN", C.c_void_p), ("pv_P81xN", C.c_void_p),
        ("prev_linvel3", C.c_void_p), ("waypoint3", C.c_void_p), ("target3", C.c_void_p), ("reset", C.c_void_p),
        ("wrench4", C.c_void_p), ("est13", C.c_void_p), ("cmd4", C.c_void_p), ("gains16", C.POINTER(C.c_float)),
        ("dt", C.c_float), ("mg", C.c_float), ("hover_force", C.c_float), ("convergence_steps", C.c_int64),
        ("pomdp_mode", C.c_int32), ("pomdp_prob", C.c_float),
        ("pos_period", C.c_uint32), ("pos_phase", C.c_uint32), ("vel_period", C.c_uint32), ("vel_phase", C.c_uint32),
        ("per_env_triggers", C.c_int32), ("num_envs_total", C.c_int64), ("acc_var", C.c_float * 3), ("pos_var", C.c_float * 3),
        ("ekf_Dt", C.c_double), ("ekf_g_noise", C.c_double),
    ]


class OzlLeeLandedArgs(C.Structure):
    """Mirror of `struct ozl_lee_landed_args` (include/ouzelum_b200.h)."""
    _fields_ = [("gains16", C.POINTER(C.c_float)), ("cmd", C.c_float * 4), ("mg", C.c_float), ("wrench4", C.c_void_p)]


class OzlQuadcopterArgs(C.Structure):
    """Mirror of `struct ozl_quadcopter_args` (include/ouzelum_b200.h)."""
    _fields_ = [
        ("n", C.c_int64), ("actions12", C.c_void_p), ("root13", C.c_void_p), ("dof_pos8", C.c_void_p),
        ("dof_target8", C.c_void_p), ("thrust4", C.c_void_p), ("obs21", C.c_void_p), ("rew", C.c_void_p),
        ("reset", C.c_void_p), ("progress", C.c_void_p), ("timeout", C.c_void_p), ("seed", C.c_uint64), ("step", C.c_uint64),
        ("env_id_base", C.c_int64), ("max_episode_length", C.c_int32), ("substeps", C.c_int32), ("dt", C.c_float),
        ("gravity_z", C.c_float), ("clip_actions", C.c_float), ("clip_obs", C.c_float), ("mass", C.c_float),
        ("ixx", C.c_float), ("iyy", C.c_float), ("izz", C.c_float), ("step_record", C.c_void_p),
    ]


class OzlNoiseLambda(C.Structure):
    """Mirror of `struct ozl_noise_lambda` (include/ouzelum_b200.h)."""
    _fields_ = [("distribution", C.c_int32), ("operation", C.c_int32), ("a", C.c_float), ("b", C.c_float),
                ("a_corr", C.c_float), ("b_corr", C.c_float)]


_P = C.c_void_p
_SIGS = {
    "ozl_abi_version": (C.c_int, []),
    "ozl_cfg_size": (C.c_int, []),
    "ozl_last_error": (C.c_char_p, []),
    "ozl_cfg_default": (C.c_int, [C.POINTER(OzlCfg), C.c_int64]),
    "ozl_create": (C.c_int, [C.POINTER(OzlCfg), C.c_int, C.POINTER(_P)]),
    "ozl_destroy": (C.c_int, [_P]),
    "ozl_reset_all": (C.c_int, [_P, C.c_uint64, _P]),
    "ozl_step": (C.c_int, [_P] * 9),
    "ozl_step_host": (C.c_int, [_P] * 10),
    "ozl_step_host_sync": (C.c_int, [_P, _P, _P]),
    "ozl_step_host_launch": (C.c_int, [_P, _P, _P]),
    "ozl_stream_sync": (C.c_int, [_P]),
    "ozl_step_host_wait": (C.c_int, [_P, _P]),
    "ozl_step_tracking": (C.c_int, [_P] * 10),
    "ozl_step_wrench": (C.c_int, [_P] * 10),
    "ozl_rollout": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P]),
    "ozl_set_states_output": (C.c_int, [_P, _P, C.c_int32]),
    "ozl_set_scenarios": (C.c_int, [_P, _P, C.c_int32, _P]),
    "ozl_set_episode_log": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int32]),
    "ozl_get_state": (C.c_int, [_P] * 6),
    "ozl_set_state": (C.c_int, [_P] * 6),
    "ozl_get_params": (C.c_int, [_P] * 4),
    "ozl_set_params": (C.c_int, [_P] * 4),
    "ozl_get_rotor_eff": (C.c_int, [_P] * 3),
    "ozl_set_rotor_eff": (C.c_int, [_P] * 3),
    "ozl_get_step_count": (C.c_int, [_P, C.POINTER(C.c_uint64), _P]),
    "ozl_set_step_count": (C.c_int, [_P, C.c_uint64, _P]),
    "ozl_metrics_read": (C.c_int, [_P, _P, C.c_int32, _P]),
    "ozl_metrics_xchg_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "ozl_metrics_xchg_destroy": (C.c_int, [_P]),
    "ozl_metrics_xchg_ipc_handle": (C.c_int, [_P, _P]),
    "ozl_metrics_xchg_connect_ipc": (C.c_int, [_P, _P]),
    "ozl_metrics_xchg_box": (C.c_int, [_P, C.POINTER(_P)]),
    "ozl_metrics_xchg_connect_ptrs": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int32)]),
    "ozl_metrics_push": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P]),
    "ozl_metrics_sum": (C.c_int, [_P, _P, _P, _P]),
    "ozl_metrics_xchg_status": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), _P]),
    "ozl_lee_control": (C.c_int, [C.c_int32, C.c_int64, _P, _P, C.POINTER(C.c_float), _P, _P, _P]),
    "ozl_lee_wrench": (C.c_int, [C.c_int32, C.c_int64, _P, _P, C.POINTER(C.c_float), C.c_float, _P, _P]),
    "ozl_pv_init": (C.c_int, [C.c_int64, _P, _P, _P]),
    "ozl_pv_reset": (C.c_int, [C.c_int64, _P, _P, _P, _P]),
    "ozl_pv_step": (C.c_int, [C.POINTER(OzlPvArgs), _P]),
    "ozl_ekf_init": (C.c_int, [C.c_int64, _P, _P, _P]),
    "ozl_ekf_set_q": (C.c_int, [C.c_int64, _P, _P, _P, _P]),
    "ozl_ekf_update": (C.c_int, [C.c_int64, _P, _P, _P, _P, C.c_int32, C.c_double, C.c_double, _P, _P]),
    "ozl_sensor_frontend": (C.c_int, [C.c_int64, _P, _P, _P, C.c_float, C.c_int32, C.c_float, C.c_uint64, C.c_uint64,
                                      C.c_int64, _P]),
    "ozl_waypoint_command": (C.c_int, [C.c_int64, _P, _P, _P, _P, C.c_int32, _P, _P, _P]),
    "ozl_apply_resets": (C.c_int, [_P, _P, _P]),
    "ozl_ekf_lee_step": (C.c_int, [_P, C.POINTER(OzlEkfLeeArgs), _P]),
    "ozl_ekf_lee_landed_step": (C.c_int, [_P] * 10),
    "ozl_step_counter_ptr": (C.c_int, [_P, C.POINTER(C.c_void_p)]),
    "ozl_landing_step": (C.c_int, [_P] * 10),
    "ozl_lee_landed_step": (C.c_int, [_P] * 10),
    "ozl_pomdp_observation": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_uint64, C.c_uint64, C.c_int64,
                                        C.c_int32, _P, _P, _P]),
    "ozl_husky_init": (C.c_int, [C.POINTER(OzlHuskyArgs), _P]),
    "ozl_husky_step": (C.c_int, [C.POINTER(OzlHuskyArgs), _P]),
    "ozl_quadcopter_step": (C.c_int, [C.POINTER(OzlQuadcopterArgs), _P]),
    "ozl_step_record_init": (C.c_int, [_P, C.c_int64, C.c_uint64, _P]),
    "ozl_step_record_read": (C.c_int, [_P, C.POINTER(C.c_uint64), _P]),
    "ozl_pomdp_observation_dev": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_uint64, _P, C.c_int64, C.c_int32,
                                            _P, _P, _P]),
    "ozl_episode_stats": (C.c_int, [C.c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "ozl_noise_lambda_apply": (C.c_int, [C.c_int64, C.c_int32, _P, C.POINTER(OzlNoiseLambda), C.c_float, C.c_uint64, C.c_uint64, _P,
                                         C.c_int64, C.c_uint64, C.c_int64, C.c_int32, _P]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"ouzelum_b200: native library {LIB_PATH} is missing. This framework has no CPU/PyTorch fallback; "
            "build it with `python -c 'import __graft_entry__ as g; g.build()'` from the repo root.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)        # AttributeError if the .so is stale -> loud
        fn.restype = res
        fn.argtypes = args
    v = lib.ozl_abi_version()
    if v != OZL_ABI_VERSION:
        raise RuntimeError(f"ouzelum_b200: library ABI {v} != binding ABI {OZL_ABI_VERSION}; rebuild")
    if lib.ozl_cfg_size() != C.sizeof(OzlCfg):
        raise RuntimeError(f"ouzelum_b200: struct ozl_cfg is {lib.ozl_cfg_size()} bytes in the library but "
                           f"{C.sizeof(OzlCfg)} in the binding; rebuild")
    return lib


lib = _load()


def last_error():
    return (lib.ozl_last_error() or b"").decode()


def check(rc, exc=RuntimeError):
    if rc != 0:
        raise exc(f"ouzelum_b200: {last_error()}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def default_cfg(num_envs, **over):
    cfg = OzlCfg()
    check(lib.ozl_cfg_default(C.byref(cfg), int(num_envs)))
    cfg.update(**over)
    return cfg
