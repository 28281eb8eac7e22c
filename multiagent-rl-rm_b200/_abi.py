"""ctypes mirror of include/rlrm_b200.h (struct layouts and constants). Keep in lock-step with the header;
tests/test_host_logic.py::test_ctypes_structs_match_the_header checks sizes/offsets against a C program compiled from the header."""
from __future__ import annotations

import ctypes as C

ABI_VERSION = 2
MAX_AGENTS = 8
MAX_CELLS = 1024
MAX_RM_STATES = 32
MAX_EVENTS = 63
N_ACTIONS = 4
ACTION_WAIT = 4
EVENT_NONE = 255
NO_TRANSITION = 255

ENV_FROZEN_LAKE, ENV_OFFICE_WORLD = 0, 1
ALGO_QL, ALGO_QRM, ALGO_QLAMBDA = 0, 1, 2
DRIVER_FROZEN_LAKE_MAIN, DRIVER_OFFICE_MAIN = 0, 1
TABLE_F32, TABLE_F64 = 0, 1

SLOT_CELL_SHIFT, SLOT_STEPS_SHIFT, SLOT_TIME_SHIFT, SLOT_RMSTATE_SHIFT, SLOT_FLAGS_SHIFT = 0, 16, 32, 48, 56
FLAG_ACTIVE, FLAG_FAIL, FLAG_DONE, FLAG_TRUNC, FLAG_FIRST = 1, 2, 4, 8, 16

ACTION_NAMES = ("up", "down", "left", "right", "wait")


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("env_kind", C.c_int32),
        ("driver", C.c_int32),
        ("algo", C.c_int32),
        ("width", C.c_int32),
        ("height", C.c_int32),
        ("n_agents", C.c_int32),
        ("n_rm_states", C.c_int32),
        ("n_events", C.c_int32),
        ("rm_final", C.c_int32),
        ("n_qrm_states", C.c_int32),
        ("max_steps", C.c_int32),
        ("stochastic", C.c_int32),
        ("slip_n", C.c_int32),
        ("slip_thr", C.c_uint64 * 3),
        ("slip_outcome", (C.c_uint8 * 4) * 4),
        ("terminate_on_plants", C.c_int32),
        ("terminate_hit_walls", C.c_int32),
        ("hole_penalty", C.c_double),
        ("wall_penalty", C.c_double),
        ("learning_rate", C.c_double),
        ("gamma", C.c_double),
        ("lambd", C.c_double),
        ("epsilon_start", C.c_double),
        ("epsilon_end", C.c_double),
        ("epsilon_decay", C.c_double),
        ("decay_on_reset", C.c_int32),
        ("shared_q", C.c_int32),
        ("seed_lo", C.c_uint32),
        ("seed_hi", C.c_uint32),
        ("instance_offset", C.c_uint32),
        ("per_agent_rm", C.c_int32),
        ("agent_n_rm_states", C.c_int32 * 8),
        ("agent_rm_final", C.c_int32 * 8),
        ("agent_n_qrm", C.c_int32 * 8),
        ("random_starts", C.c_int32),
        ("n_free_cells", C.c_int32),
        ("use_rsh", C.c_int32),
        ("n_actions", C.c_int32),
        ("reserved", C.c_int32),
        ("table_dtype", C.c_int32),
    ]


class Tables(C.Structure):
    _fields_ = [
        ("next_cell", C.c_void_p),
        ("cell_flags", C.c_void_p),
        ("label", C.c_void_p),
        ("delta", C.c_void_p),
        ("rq", C.c_void_p),
        ("rcf", C.c_void_p),
        ("qrm_states", C.c_void_p),
        ("start_cell", C.c_void_p),
        ("free_cells", C.c_void_p),
        ("phi", C.c_void_p),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("active_steps", C.c_uint64),
        ("episodes", C.c_uint32),
        ("successes", C.c_uint32),
        ("return_sum", C.c_double),
        ("last_return", C.c_float),
        ("last_length", C.c_uint32),
    ]


class Eval(C.Structure):
    _fields_ = [
        ("cum_gamma", C.c_double),
        ("disc_return", C.c_double),
        ("return_sum", C.c_double),
        ("return_sqsum", C.c_double),
        ("arps_sum", C.c_double),
        ("len_sum", C.c_uint64),
        ("len_sqsum", C.c_uint64),
        ("episodes", C.c_uint32),
        ("successes", C.c_uint32),
        ("in_success", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class State(C.Structure):
    _fields_ = [
        ("n_instances", C.c_int64),
        ("slot", C.c_void_p),
        ("epsilon", C.c_void_p),
        ("q", C.c_void_p),
        ("e", C.c_void_p),
        ("visits", C.c_void_p),
        ("ep_return", C.c_void_p),
        ("stats", C.c_void_p),
        ("acc_sum", C.c_void_p),
        ("acc_cnt", C.c_void_p),
        ("acc_last", C.c_void_p),
        ("tr_pos", C.c_void_p),
        ("tr_idx", C.c_void_p),
        ("tr_eq", C.c_void_p),
        ("tr_len", C.c_void_p),
        ("tr_work", C.c_void_p),
        ("tr_cap", C.c_int32),
        ("tr_reserved", C.c_int32),
    ]


class StepOut(C.Structure):
    _fields_ = [
        ("prev_cell", C.c_void_p),
        ("cell", C.c_void_p),
        ("prev_q", C.c_void_p),
        ("q", C.c_void_p),
        ("event", C.c_void_p),
        ("executed", C.c_void_p),
        ("renv", C.c_void_p),
        ("rq", C.c_void_p),
        ("reward", C.c_void_p),
        ("env_term", C.c_void_p),
        ("rm_term", C.c_void_p),
        ("term", C.c_void_p),
        ("trunc", C.c_void_p),
        ("cf_q", C.c_void_p),
        ("cf_r", C.c_void_p),
    ]


STEP_OUT_FIELDS = {
    "prev_cell": "uint16",
    "cell": "uint16",
    "prev_q": "uint8",
    "q": "uint8",
    "event": "uint8",
    "executed": "uint8",
    "renv": "float64",
    "rq": "float64",
    "reward": "float64",
    "env_term": "uint8",
    "rm_term": "uint8",
    "term": "uint8",
    "trunc": "uint8",
}

# every symbol include/rlrm_b200.h declares (tests check the built library exports all of them)
EXPORTED_SYMBOLS = (
    "rlrm_abi_version",
    "rlrm_last_error",
    "rlrm_device_count",
    "rlrm_create",
    "rlrm_destroy",
    "rlrm_set_learner",
    "rlrm_set_sweep",
    "rlrm_reset",
    "rlrm_reset_at",
    "rlrm_select_action",
    "rlrm_step",
    "rlrm_rm_step",
    "rlrm_rm_step_agent",
    "rlrm_mdp",
    "rlrm_value_iteration",
    "rlrm_update",
    "rlrm_train",
    "rlrm_train_host",
    "rlrm_evaluate",
    "rlrm_qlambda_materialize",
    "rlrm_launch_count",
    "rlrm_iterate",
    "rlrm_update_list",
    "rlrm_update_list_select",
    "rlrm_merge_replicas",
    "rlrm_stream_sync",
    "rlrm_probe_random_gather",
)


class Hyper(C.Structure):  # rlrm_hyper_t
    _fields_ = [("learning_rate", C.c_double), ("gamma", C.c_double), ("lambd", C.c_double), ("epsilon_end", C.c_double),
                ("epsilon_decay", C.c_double)]


class SelectReq(C.Structure):  # rlrm_select_req_t
    _fields_ = [("state", C.c_uint32), ("best", C.c_uint32), ("epsilon", C.c_double), ("draws", C.c_uint32 * 4), ("seq", C.c_uint32),
                ("action", C.c_uint32), ("done_seq", C.c_uint32), ("pad", C.c_uint32)]


class Experience(C.Structure):
    _fields_ = [("s", C.c_uint32), ("sn", C.c_uint32), ("action", C.c_uint8), ("terminated", C.c_uint8), ("pad", C.c_uint8 * 6),
                ("reward", C.c_double)]
