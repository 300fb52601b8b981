"""ctypes mirror of include/evgsim.h and the loader of libevgsim.so.

The reference has no FFI (pure Python), so this file IS the binding a maintainer would add to
call the CUDA path from ``gym_everglades/envs/everglades_env.py`` (see INTEGRATION.md).
There is no fallback: if the shared library is missing or CUDA is unavailable, loading or
``evg_create`` raises — nothing here computes a game step on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os

MAX_NODES = 32
MAX_UNIT_TYPES = 8
NUM_GROUPS = 12
MAX_GROUP_UNITS = 16
MAX_ACTIONS = 7
NUM_PLAYERS = 2
ABI_VERSION = 1

AUTORESET_OFF, AUTORESET_TERMINAL, AUTORESET_NEXT = 0, 1, 2
STATUS_IN_PROGRESS, STATUS_TIME_EXPIRED, STATUS_BASE_CAPTURE, STATUS_ANNIHILATION = 0, 1, 2, 3
SHAPE_NORMALIZED_SCORE, SHAPE_BASIC, SHAPE_PENALIZE_LONG, SHAPE_SHORT_GAMES = 0, 1, 2, 3
AGENT_EXTERNAL, AGENT_RANDOM, AGENT_BASE_RUSH, AGENT_SWARM = 0, 1, 2, 3
OBS_F32, OBS_I16, OBS_WIRE = 0, 1, 2
WIRE_NODE0 = 4
MLP_IN_PAD, MLP_CHUNK, MLP_OUT_PAD = 128, 192, 144
PPO_IN_PAD, PPO_MAX_LATENT, PPO_OUT_PAD = 128, 256, 144
VALUE_OUT_PAD = 16
BIND_RECORDS, BIND_HEALTH, BIND_STATS, BIND_TABLES, BIND_AGENTS, BIND_COUNT = 0, 1, 2, 3, 4, 5

_N1 = MAX_NODES + 1


class EvgConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("n_nodes", C.c_int32),
        ("n_unit_types", C.c_int32),
        ("turn_limit", C.c_int32),
        ("capture_bonus", C.c_int32),
        ("max_score", C.c_int32),
        ("auto_reset", C.c_int32),
        ("reserved0", C.c_int32),
        ("node_control_points", C.c_int32 * _N1),
        ("node_defense", C.c_double * _N1),
        ("node_team_start", C.c_int8 * _N1),
        ("node_has_defense", C.c_uint8 * _N1),
        ("node_has_observe", C.c_uint8 * _N1),
        ("node_has_defend", C.c_uint8 * _N1),
        ("edge_distance", (C.c_uint8 * _N1) * _N1),
        ("p1_node_map", C.c_uint8 * _N1),
        ("unit_armor", C.c_double * MAX_UNIT_TYPES),
        ("unit_damage", C.c_int32 * MAX_UNIT_TYPES),
        ("unit_speed", C.c_int32 * MAX_UNIT_TYPES),
        ("unit_control", C.c_int32 * MAX_UNIT_TYPES),
        ("unit_cost", C.c_int32 * MAX_UNIT_TYPES),
        ("group_type", (C.c_uint8 * NUM_GROUPS) * NUM_PLAYERS),
        ("group_size", (C.c_uint8 * NUM_GROUPS) * NUM_PLAYERS),
    ]


class EvgGroupState(C.Structure):
    _fields_ = [
        ("location", C.c_int16),
        ("travel_destination", C.c_int16),
        ("distance_remaining", C.c_int16),
        ("ready", C.c_uint8),
        ("moving", C.c_uint8),
        ("destroyed", C.c_uint8),
        ("count", C.c_uint8),
        ("arrival", C.c_int32),
        ("avg_health", C.c_int32),
    ]


class EvgEnvState(C.Structure):
    _fields_ = [
        ("turn", C.c_int32),
        ("episode", C.c_int32),
        ("control_state", C.c_int16 * _N1),
        ("controlled_by", C.c_int8 * _N1),
        ("pad1", C.c_int8 * 5),
        ("groups", (EvgGroupState * NUM_GROUPS) * NUM_PLAYERS),
        ("health", ((C.c_double * MAX_GROUP_UNITS) * NUM_GROUPS) * NUM_PLAYERS),
    ]


class EvgLayout(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int64),
        ("obs_len", C.c_int32),
        ("record_bytes", C.c_int32),
        ("health_slots", C.c_int32),
        ("action_bytes", C.c_int32),
        ("records_bytes", C.c_int64),
        ("health_bytes", C.c_int64),
        ("stats_bytes", C.c_int64),
        ("tables_bytes", C.c_int64),
        ("agents_bytes", C.c_int64),
    ]


class EvgEpisodeStats(C.Structure):
    _fields_ = [
        ("episodes", C.c_int64),
        ("wins", C.c_int64 * 2),
        ("ties", C.c_int64),
        ("total_turns", C.c_int64),
        ("total_score", C.c_int64 * 2),
        ("status_count", C.c_int64 * 4),
        ("env_turns", C.c_int64),
        ("fought_unit_slots", C.c_int64),
    ]


def env_state_dtype():
    """numpy structured dtype with exactly the memory layout of EvgEnvState."""
    import numpy as np

    grp = np.dtype([("location", "<i2"), ("travel_destination", "<i2"), ("distance_remaining", "<i2"),
                    ("ready", "u1"), ("moving", "u1"), ("destroyed", "u1"), ("count", "u1"),
                    ("arrival", "<i4"), ("avg_health", "<i4")], align=True)
    dt = np.dtype([("turn", "<i4"), ("episode", "<i4"), ("control_state", "<i2", (_N1,)),
                   ("controlled_by", "i1", (_N1,)), ("pad1", "i1", (5,)),
                   ("groups", grp, (NUM_PLAYERS, NUM_GROUPS)),
                   ("health", "<f8", (NUM_PLAYERS, NUM_GROUPS, MAX_GROUP_UNITS))], align=True)
    assert dt.itemsize == C.sizeof(EvgEnvState), (dt.itemsize, C.sizeof(EvgEnvState))
    return dt


class EvgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("libevgsim error %d: %s" % (code, msg))
        self.code = code


LIB_NAME = "libevgsim.so"
_lib = None


def lib_path() -> str:
    """The in-tree library; EVGSIM_LIB names another build of the same sources (kernel A/B runs, tools/ab_variants.sh)."""
    return os.environ.get("EVGSIM_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)


# every symbol include/evgsim.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("evg_default_config", C.c_int, [C.POINTER(EvgConfig)]),
    ("evg_create", C.c_int, [C.POINTER(EvgConfig), C.c_int64, C.c_uint64, C.c_int64, C.c_int, C.POINTER(_P)]),
    ("evg_destroy", C.c_int, [_P]),
    ("evg_layout", C.c_int, [_P, C.POINTER(EvgLayout)]),
    ("evg_bind", C.c_int, [_P, C.POINTER(_P), C.c_int32]),
    ("evg_reset", C.c_int, [_P, _P, _P, _P]),
    ("evg_step", C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_step_agents", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_rollout", C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_step_host", C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_obs_row_bytes", C.c_int, [_P, C.c_int32]),
    ("evg_reset_fmt", C.c_int, [_P, C.c_int32, _P, _P, _P, _P]),
    ("evg_step_fmt", C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_step_host_fmt", C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_export_state", C.c_int, [_P, C.c_int64, C.c_int64, _P, _P]),
    ("evg_import_state", C.c_int, [_P, C.c_int64, C.c_int64, _P, _P]),
    ("evg_episode_stats", C.c_int, [_P, C.POINTER(EvgEpisodeStats), _P]),
    ("evg_agent_random", C.c_int, [_P, _P, C.c_int32, _P]),
    ("evg_agents", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P]),
    ("evg_decode_dqn", C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P]),
    ("evg_decode_indices", C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    ("evg_policy_mlp", C.c_int, [_P, _P, C.c_int64, _P, _P, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
    ("evg_policy_ppo", C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    ("evg_policy_rppo", C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    ("evg_policy_mlp_fmt", C.c_int, [_P, C.c_int32, _P, C.c_int64, _P, _P, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
    ("evg_policy_ppo_fmt", C.c_int, [_P, C.c_int32, _P, C.c_int32, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    ("evg_policy_rppo_fmt", C.c_int, [_P, C.c_int32, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      _P, _P, _P, _P, _P]),
    ("evg_policy_ppo_logp", C.c_int, [_P, C.c_int32, _P, C.c_int32, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    ("evg_policy_rppo_logp", C.c_int, [_P, C.c_int32, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                       _P, _P, _P, _P, _P, _P, _P]),
    ("evg_policy_value", C.c_int, [_P, C.c_int32, _P, C.c_int64, C.c_int32, _P, _P, _P, _P, C.c_int32, _P, _P]),
    ("evg_wire_expand", C.c_int, [_P, _P, C.c_int64, _P, C.c_int64, C.c_int32, _P, _P, _P, _P]),
    ("evg_gae", C.c_int, [_P, C.c_int32, C.c_int64, C.c_int32, _P, _P, _P, _P, C.c_float, C.c_float, _P, _P, _P]),
    ("evg_ppo_loss", C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_float, _P, _P, _P, _P, _P]),
    ("evg_ppo_loss_grad", C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_float, _P, _P, _P, _P]),
    ("evg_rppo_train_pack", C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    ("evg_rppo_train_forward", C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_rppo_train_backward", C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_pack_mlp", C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    ("evg_pack_ppo", C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    ("evg_pack_rppo", C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    ("evg_pack_value", C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P]),
    ("evg_decode_dqn_layout",C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    ("evg_shape_reward", C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P]),
    ("evg_step_kernel_kind", C.c_int, [_P]),
    ("evg_launch_count", C.c_int64, [_P]),
    ("evg_last_error", C.c_char_p, []),
    ("evg_abi_version", C.c_int, []),
]


def load():
    """dlopen the in-tree libevgsim.so (built by __graft_entry__.build()); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.isfile(path):
        raise ImportError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback for the game step)" % path)
    lib = C.CDLL(path)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the .so does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    if lib.evg_abi_version() != ABI_VERSION:
        raise ImportError("libevgsim ABI %d != binding ABI %d" % (lib.evg_abi_version(), ABI_VERSION))
    assert C.sizeof(EvgConfig) > 0
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        raise EvgError(code, (load().evg_last_error() or b"").decode("utf-8", "replace"))
