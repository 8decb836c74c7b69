"""ctypes binding of the C ABI in ``include/gpd.h`` (``lib/libgpd_b200.so``).

The product path has no CPU fallback: if the library is missing, :func:`load` raises
``GpdLibraryError`` telling the user to build it; if there is no CUDA device every compute
entry point fails with ``GPD_ERR_NO_DEVICE`` and :func:`check` raises ``GpdError``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .params import DroneParams, PIDParams

_HERE = os.path.dirname(os.path.abspath(__file__))
# GPD_B200_LIB points at another build of the same C ABI (kernel A/B experiments); the default is the in-tree library
LIB_PATH = os.environ.get("GPD_B200_LIB") or os.path.join(_HERE, "lib", "libgpd_b200.so")

GPD_F32, GPD_F64 = 0, 1
ACT_CODES = {"rpm": 0, "pid": 1, "vel": 2, "one_d_rpm": 3, "one_d_pid": 4, "ctrl_rpm": 5, "ctrl_vel": 6}
ENV_CODES = {"ctrl": 0, "hover": 1, "multihover": 2}
MODEL_CODES = {"cf2x": 0, "cf2p": 1, "racer": 2}

#: every symbol include/gpd.h declares (tests check the library exports all of them)
SYMBOLS = [
    "gpd_version", "gpd_last_error", "gpd_device_count", "gpd_create", "gpd_destroy", "gpd_obs_width",
    "gpd_action_width", "gpd_substeps", "gpd_set_init_poses", "gpd_reset", "gpd_step", "gpd_step_host",
    "gpd_reset_host", "gpd_get_state", "gpd_note_latest_obs", "gpd_set_state", "gpd_pid_compute", "gpd_force_ground_effect",
    "gpd_force_drag", "gpd_force_downwash", "gpd_rollout_pid", "gpd_episode_stats", "gpd_grid_size",
    "gpd_set_timeline_buffer", "gpd_count_nonfinite", "gpd_set_targets", "gpd_mirror_alloc", "gpd_mirror_free",
    "gpd_mirror_attach", "gpd_mirror_row", "gpd_step_mirror", "gpd_step_mirror_begin", "gpd_step_mirror_end",
    "gpd_reset_mirror", "gpd_nccl_unique_id", "gpd_nccl_comm_init", "gpd_nccl_comm_destroy", "gpd_adjacency",
    "gpd_set_step_chaining", "gpd_rollout",
]


class GpdLibraryError(RuntimeError):
    pass


class GpdError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgpd_b200 error {code}: {msg}")
        self.code = code


class DroneParamsC(C.Structure):
    _fields_ = [("model", C.c_int32), ("_pad", C.c_int32),
                ("M", C.c_double), ("L", C.c_double), ("THRUST2WEIGHT", C.c_double),
                ("J", C.c_double * 3), ("J_INV", C.c_double * 3),
                ("KF", C.c_double), ("KM", C.c_double),
                ("COLLISION_H", C.c_double), ("COLLISION_R", C.c_double), ("COLLISION_Z_OFFSET", C.c_double),
                ("MAX_SPEED_KMH", C.c_double), ("GND_EFF_COEFF", C.c_double), ("PROP_RADIUS", C.c_double),
                ("DRAG_COEFF", C.c_double * 3),
                ("DW_COEFF_1", C.c_double), ("DW_COEFF_2", C.c_double), ("DW_COEFF_3", C.c_double),
                ("G", C.c_double), ("GRAVITY", C.c_double), ("HOVER_RPM", C.c_double), ("MAX_RPM", C.c_double),
                ("MAX_THRUST", C.c_double), ("MAX_XY_TORQUE", C.c_double), ("MAX_Z_TORQUE", C.c_double),
                ("GND_EFF_H_CLIP", C.c_double),
                ("ROTOR_XYZ", (C.c_double * 3) * 4)]


class PidParamsC(C.Structure):
    _fields_ = [("P_FOR", C.c_double * 3), ("I_FOR", C.c_double * 3), ("D_FOR", C.c_double * 3),
                ("P_TOR", C.c_double * 3), ("I_TOR", C.c_double * 3), ("D_TOR", C.c_double * 3),
                ("PWM2RPM_SCALE", C.c_double), ("PWM2RPM_CONST", C.c_double),
                ("MIN_PWM", C.c_double), ("MAX_PWM", C.c_double),
                ("MIXER", (C.c_double * 3) * 4),
                ("GRAVITY", C.c_double), ("KF", C.c_double)]


class ConfigC(C.Structure):
    _fields_ = [("device", C.c_int32), ("precision", C.c_int32), ("num_envs", C.c_int64),
                ("num_drones", C.c_int32), ("pyb_freq", C.c_int32), ("ctrl_freq", C.c_int32),
                ("env_kind", C.c_int32), ("action_type", C.c_int32), ("physics_flags", C.c_int32),
                ("auto_reset", C.c_int32), ("threads_per_block", C.c_int32),
                ("episode_len_sec", C.c_double), ("speed_limit", C.c_double),
                ("target_pos", C.POINTER(C.c_double)),
                ("drone", DroneParamsC), ("pid", PidParamsC)]


def drone_params_c(p: DroneParams) -> DroneParamsC:
    d = DroneParamsC()
    d.model = MODEL_CODES[p.model.value]
    d.M, d.L, d.THRUST2WEIGHT = p.M, p.L, p.THRUST2WEIGHT_RATIO
    for k in range(3):
        d.J[k] = float(p.J[k, k])
        d.J_INV[k] = float(p.J_INV[k, k])
        d.DRAG_COEFF[k] = float(p.DRAG_COEFF[k])
    d.KF, d.KM = p.KF, p.KM
    d.COLLISION_H, d.COLLISION_R, d.COLLISION_Z_OFFSET = p.COLLISION_H, p.COLLISION_R, p.COLLISION_Z_OFFSET
    d.MAX_SPEED_KMH, d.GND_EFF_COEFF, d.PROP_RADIUS = p.MAX_SPEED_KMH, p.GND_EFF_COEFF, p.PROP_RADIUS
    d.DW_COEFF_1, d.DW_COEFF_2, d.DW_COEFF_3 = p.DW_COEFF_1, p.DW_COEFF_2, p.DW_COEFF_3
    d.G, d.GRAVITY, d.HOVER_RPM, d.MAX_RPM = p.G, p.GRAVITY, p.HOVER_RPM, p.MAX_RPM
    d.MAX_THRUST, d.MAX_XY_TORQUE, d.MAX_Z_TORQUE, d.GND_EFF_H_CLIP = (
        p.MAX_THRUST, p.MAX_XY_TORQUE, p.MAX_Z_TORQUE, p.GND_EFF_H_CLIP)
    for i in range(4):
        for k in range(3):
            d.ROTOR_XYZ[i][k] = float(p.ROTOR_XYZ[i, k])
    return d


def pid_params_c(c: PIDParams) -> PidParamsC:
    o = PidParamsC()
    for k in range(3):
        o.P_FOR[k], o.I_FOR[k], o.D_FOR[k] = float(c.P_COEFF_FOR[k]), float(c.I_COEFF_FOR[k]), float(c.D_COEFF_FOR[k])
        o.P_TOR[k], o.I_TOR[k], o.D_TOR[k] = float(c.P_COEFF_TOR[k]), float(c.I_COEFF_TOR[k]), float(c.D_COEFF_TOR[k])
    o.PWM2RPM_SCALE, o.PWM2RPM_CONST = c.PWM2RPM_SCALE, c.PWM2RPM_CONST
    o.MIN_PWM, o.MAX_PWM = float(c.MIN_PWM), float(c.MAX_PWM)
    mx = np.asarray(c.MIXER_MATRIX, dtype=np.float64)
    for i in range(4):
        for k in range(3):
            o.MIXER[i][k] = float(mx[i, k])
    o.GRAVITY, o.KF = c.GRAVITY, c.KF
    return o


_lib = None


def load(path: str | None = None):
    """Load libgpd_b200.so and declare the prototypes of include/gpd.h.  Raises if it is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise GpdLibraryError(
            f"{p} not found: the CUDA library is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or gym-pybullet-drones-routing_b200/csrc/build.sh (needs nvcc). There is no CPU fallback.")
    L = C.CDLL(p)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    u8p = C.c_void_p
    L.gpd_version.restype = C.c_int
    L.gpd_last_error.restype = C.c_char_p
    L.gpd_device_count.restype = C.c_int
    L.gpd_create.argtypes = [C.POINTER(ConfigC), C.POINTER(vp)]
    L.gpd_destroy.argtypes = [vp]
    L.gpd_destroy.restype = None
    for f in (L.gpd_obs_width, L.gpd_action_width, L.gpd_substeps):
        f.argtypes = [vp]
    L.gpd_set_init_poses.argtypes = [vp, C.POINTER(dbl), C.POINTER(dbl), C.c_int]
    L.gpd_reset.argtypes = [vp, u8p, vp, vp, vp]
    L.gpd_step.argtypes = [vp, vp, vp, vp, vp, u8p, u8p, vp, vp]
    L.gpd_set_step_chaining.argtypes = [vp, C.c_int]
    L.gpd_step_host.argtypes = [vp, vp, vp, vp, u8p, u8p, vp, vp]
    L.gpd_reset_host.argtypes = [vp, u8p, vp, vp]
    L.gpd_get_state.argtypes = [vp, vp, vp, vp, vp, vp]
    L.gpd_note_latest_obs.argtypes = [vp, vp]
    L.gpd_set_state.argtypes = [vp, vp, vp, vp, vp, vp]
    L.gpd_pid_compute.argtypes = [C.c_int, C.c_int, C.POINTER(PidParamsC), i64, dbl,
                                  vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.gpd_force_ground_effect.argtypes = [C.c_int, C.c_int, C.POINTER(DroneParamsC), i64, vp, vp, vp, vp, u8p, vp]
    L.gpd_force_drag.argtypes = [C.c_int, C.c_int, C.POINTER(DroneParamsC), i64, vp, vp, vp, vp, vp]
    L.gpd_force_downwash.argtypes = [C.c_int, C.c_int, C.POINTER(DroneParamsC), i64, i32, vp, vp, vp]
    L.gpd_rollout_pid.argtypes = [vp, i32, vp, i32, vp, vp, vp]
    L.gpd_rollout.argtypes = [vp, i32, vp, vp, vp, vp, u8p, u8p, vp, vp, vp]
    L.gpd_episode_stats.argtypes = [vp, C.POINTER(dbl), C.c_int, vp, vp]
    L.gpd_set_targets.argtypes = [vp, C.POINTER(dbl), C.c_int]
    L.gpd_mirror_alloc.argtypes = [i64, i64, C.POINTER(vp)]
    L.gpd_mirror_free.argtypes = [vp]
    L.gpd_mirror_attach.argtypes = [vp, vp, i64, i64, i64]
    L.gpd_mirror_row.argtypes = [vp]
    L.gpd_mirror_row.restype = i64
    L.gpd_step_mirror.argtypes = [vp, vp, vp, vp, vp, u8p, u8p, vp, C.POINTER(i64), vp]
    L.gpd_step_mirror_begin.argtypes = [vp, vp, vp, vp, vp, u8p, u8p, vp, vp]
    L.gpd_step_mirror_end.argtypes = [vp, C.POINTER(i64), vp]
    L.gpd_reset_mirror.argtypes = [vp, u8p, vp, vp, C.POINTER(i64), vp]
    L.gpd_nccl_unique_id.argtypes = [C.c_char_p]
    L.gpd_nccl_comm_init.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.gpd_nccl_comm_destroy.argtypes = [vp]
    L.gpd_adjacency.argtypes = [vp, dbl, vp, vp]
    L.gpd_grid_size.argtypes = [vp]
    L.gpd_count_nonfinite.argtypes = [vp, C.POINTER(C.c_longlong), vp]
    L.gpd_set_timeline_buffer.argtypes = [vp, vp]
    if path is None:
        _lib = L
    return L


def check(rc: int):
    if rc < 0:
        raise GpdError(rc, load().gpd_last_error().decode("utf-8", "replace"))
    return rc
