"""ctypes binding of libox_b200.so (the C ABI in include/ox_b200.h).

This is the Python stand-in for the `ox_b200-sys` Rust crate (rust/ox_b200-sys/src/lib.rs): one
declaration per exported symbol, nothing else. It fails loudly when the library is missing - there is
no fallback implementation of any kind.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libox_b200.so")

# status codes (ox_status)
OX_OK, OX_ERR_PARSE, OX_ERR_COMPILE, OX_ERR_CUDA, OX_ERR_INVALID, OX_ABSENT, OX_ERR_IO = range(7)

# enums
JNT_FREE, JNT_BALL, JNT_SLIDE, JNT_HINGE = range(4)
OBJ_BODY, OBJ_XBODY, OBJ_JOINT, OBJ_DOF, OBJ_GEOM, OBJ_SITE = 1, 2, 3, 4, 5, 6
OBJ_EQUALITY, OBJ_TENDON, OBJ_ACTUATOR, OBJ_SENSOR, OBJ_PLUGIN = 17, 18, 19, 20, 25
F32, F64 = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
LAYOUT_ENV_MAJOR, LAYOUT_ELEM_MAJOR = 0, 1
MODE_FUSED, MODE_STAGED, MODE_COOP = 0, 1, 2
INT_EULER, INT_RK4, INT_IMPLICIT, INT_IMPLICITFAST = 0, 1, 2, 3

_REAL_FIELDS = [
    "qpos", "qvel", "ctrl", "qfrc_applied", "xfrc_applied", "qacc_warmstart", "time", "act",
    "qacc", "sensordata", "xpos", "xquat", "xmat", "xipos", "ximat", "xanchor", "xaxis", "geom_xpos", "geom_xmat",
    "site_xpos", "site_xmat", "subtree_com", "cinert", "cdof", "qM", "qLD", "qLDiagInv", "cvel", "cdof_dot",
    "qfrc_bias", "qfrc_passive", "actuator_force", "qfrc_actuator", "qfrc_smooth", "qacc_smooth", "qfrc_constraint",
    "con_dist", "con_pos", "con_frame", "efc_J", "efc_pos", "efc_margin", "efc_D", "efc_aref", "efc_force", "act_dot",
    "mocap_pos", "mocap_quat", "eq_active", "ten_length", "ten_J", "qfrc_inverse",
]
FIELD = {name: i for i, name in enumerate(_REAL_FIELDS)}
FIELD.update({"ncon": 100, "nefc": 101, "solver_niter": 102, "diverged": 103, "con_pair": 104})
INT_FIELDS = {"ncon", "nefc", "solver_niter", "diverged", "con_pair"}


class BatchConfig(C.Structure):
    _fields_ = [
        ("nenv", C.c_int32), ("device", C.c_int32), ("precision", C.c_int32), ("mode", C.c_int32),
        ("iterations", C.c_int32), ("ls_iterations", C.c_int32), ("use_graph", C.c_int32), ("block_threads", C.c_int32),
        ("env_id_offset", C.c_int64), ("tolerance", C.c_double), ("specialize", C.c_int32), ("lanes_per_warp", C.c_int32),
        ("coop_solver", C.c_int32), ("reserved_", C.c_int32),
    ]


class ObsSegment(C.Structure):
    _fields_ = [("field", C.c_int32), ("first", C.c_int32), ("count", C.c_int32)]


class RewardTerm(C.Structure):
    _fields_ = [("field", C.c_int32), ("index", C.c_int32), ("kind", C.c_int32), ("reserved_", C.c_int32), ("weight", C.c_double)]


class FinishCond(C.Structure):
    _fields_ = [("field", C.c_int32), ("index", C.c_int32), ("lo", C.c_double), ("hi", C.c_double)]


class TaskSpec(C.Structure):
    _fields_ = [
        ("nobs", C.c_int32), ("obs", C.POINTER(ObsSegment)), ("nreward", C.c_int32), ("reward", C.POINTER(RewardTerm)),
        ("nfinish", C.c_int32), ("finish", C.POINTER(FinishCond)), ("reward_bias", C.c_double), ("time_limit", C.c_double),
        ("discount", C.c_double), ("init_qpos_noise", C.c_double), ("init_qvel_noise", C.c_double), ("seed", C.c_uint64),
        ("frame_skip", C.c_int32), ("auto_reset", C.c_int32),
    ]


REWARD_LINEAR, REWARD_SQUARE, REWARD_ABS = range(3)

# every symbol include/ox_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "ox_last_error_message": (C.c_char_p, []),
    "ox_version": (C.c_char_p, []),
    "ox_model_from_xml_string": (C.c_int32, [C.c_char_p, C.POINTER(_P)]),
    "ox_model_from_xml_path": (C.c_int32, [C.c_char_p, C.POINTER(_P)]),
    "ox_model_free": (None, [_P]),
    "ox_model_serialize": (C.c_int64, [_P, _P, C.c_int64]),
    "ox_model_deserialize": (C.c_int32, [_P, C.c_int64, C.POINTER(_P)]),
    "ox_model_save": (C.c_int32, [_P, C.c_char_p]),
    "ox_model_load": (C.c_int32, [C.c_char_p, C.POINTER(_P)]),
    "ox_model_get_tables": (_P, [_P]),
    "ox_model_int_table": (C.c_int32, [_P, C.c_char_p, C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.c_int32)]),
    "ox_model_real_table": (C.c_int32, [_P, C.c_char_p, C.POINTER(C.POINTER(C.c_double)), C.POINTER(C.c_int32)]),
    "ox_model_size": (C.c_int32, [_P, C.c_char_p]),
    "ox_model_name2id": (C.c_int32, [_P, C.c_int32, C.c_char_p]),
    "ox_model_id2name": (C.c_char_p, [_P, C.c_int32, C.c_int32]),
    "ox_batch_config_default": (None, [C.POINTER(BatchConfig)]),
    "ox_batch_create": (C.c_int32, [_P, C.POINTER(BatchConfig), C.POINTER(_P)]),
    "ox_batch_free": (None, [_P]),
    "ox_batch_nenv": (C.c_int32, [_P]),
    "ox_batch_stream": (_P, [_P]),
    "ox_batch_step": (C.c_int32, [_P, C.c_int32]),
    "ox_batch_forward": (C.c_int32, [_P]),
    "ox_batch_inverse": (C.c_int32, [_P]),
    "ox_batch_step_io": (C.c_int32, [_P, _P, _P, _P, C.c_int32, C.c_int32]),
    "ox_batch_reset": (C.c_int32, [_P, _P]),
    "ox_batch_sync": (C.c_int32, [_P]),
    "ox_batch_ctrl_philox": (C.c_int32, [_P, C.c_int32, C.c_uint64]),
    "ox_batch_set_step_counter": (C.c_int32, [_P, C.c_int64]),
    "ox_batch_ctrl_philox_scale": (C.c_int32, [_P, C.c_double]),
    "ox_group_create": (C.c_int32, [_P, C.POINTER(BatchConfig), C.c_int32, C.POINTER(C.c_int32), C.POINTER(_P)]),
    "ox_group_free": (None, [_P]),
    "ox_group_size": (C.c_int32, [_P]),
    "ox_group_batch": (_P, [_P, C.c_int32]),
    "ox_group_step": (C.c_int32, [_P, C.c_int32]),
    "ox_group_sync": (C.c_int32, [_P]),
    "ox_group_reset": (C.c_int32, [_P]),
    "ox_group_ctrl_philox": (C.c_int32, [_P, C.c_int32, C.c_uint64]),
    "ox_group_stats": (C.c_int32, [_P, C.POINTER(C.c_double)]),
    "ox_group_stats_backend": (C.c_char_p, [_P]),
    "ox_measure_fma_peak": (C.c_int32, [C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "ox_batch_field_size": (C.c_int32, [_P, C.c_int32]),
    "ox_batch_state_size": (C.c_int32, [_P]),
    "ox_batch_get_state": (C.c_int32, [_P, _P, C.c_int32, C.c_int32]),
    "ox_batch_set_state": (C.c_int32, [_P, _P, C.c_int32, C.c_int32]),
    "ox_batch_get_step_counter": (C.c_int64, [_P]),
    "ox_batch_get": (C.c_int32, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32]),
    "ox_batch_set": (C.c_int32, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32]),
    "ox_batch_get_many": (C.c_int32, [_P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(_P), C.c_int32, C.c_int32, C.c_int32]),
    "ox_batch_get1": (C.c_int32, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "ox_batch_set1": (C.c_int32, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "ox_batch_get1_int": (C.c_int32, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "ox_batch_stats": (C.c_int32, [_P, C.POINTER(C.c_double)]),
    "ox_batch_launch_count": (C.c_int64, [_P]),
    "ox_batch_kernel_name": (C.c_char_p, [_P]),
    "ox_batch_jit_note": (C.c_char_p, [_P]),
    "ox_jit_compile": (C.c_int32, [_P, C.c_int32, C.c_char_p, C.c_int32]),
    "ox_spec_count": (C.c_int32, []),
    "ox_spec_name": (C.c_char_p, [C.c_int32]),
    "ox_batch_stage_times": (C.c_int32, [_P, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "ox_stage_name": (C.c_char_p, [C.c_int32]),
    "ox_task_spec_default": (None, [C.POINTER(TaskSpec)]),
    "ox_env_create": (C.c_int32, [_P, C.POINTER(TaskSpec), C.POINTER(_P)]),
    "ox_env_free": (None, [_P]),
    "ox_env_obs_dim": (C.c_int32, [_P]),
    "ox_env_reset": (C.c_int32, [_P, _P, C.c_int32, C.c_int32]),
    "ox_env_step": (C.c_int32, [_P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32]),
    "ox_env_stats": (C.c_int32, [_P, C.POINTER(C.c_double)]),
}

_lib = None


def lib() -> C.CDLL:
    """Load libox_b200.so (built in-tree by __graft_entry__.build()). Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). oxide_control_b200 has no fallback implementation.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the ABI and the header ever disagree
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error() -> str:
    return lib().ox_last_error_message().decode("utf-8", "replace")
