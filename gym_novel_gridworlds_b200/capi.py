"""ctypes binding of the C-ABI in include/ngw.h (libngw_b200.so, built in-tree under csrc/).

No CPU fallback exists: if the CUDA library is missing or cannot be loaded, `load_library()` raises."""
import ctypes as C
import os

from . import opcodes as oc

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libngw_b200.so')
ABI_VERSION = 13
OBS_I32, OBS_U8, OBS_HITS = 0, 1, 2
RNG_PHILOX, RNG_NUMPY = 0, 1


class ActionEntryC(C.Structure):
    _fields_ = [('op', C.c_uint8), ('arg', C.c_uint8), ('variant', C.c_uint8), ('reserved', C.c_uint8),
                ('layers', C.c_uint8 * oc.MAX_LAYERS)]


class RecipeC(C.Structure):
    _fields_ = [('n_inputs', C.c_uint8),
                ('in_item', C.c_uint8 * oc.MAX_RECIPE_INPUTS),
                ('in_qty', C.c_uint8 * oc.MAX_RECIPE_INPUTS),
                ('out_item', C.c_uint8), ('out_qty', C.c_uint8), ('needs_table', C.c_uint8),
                ('reward_ok', C.c_int32),
                ('cost_missing', C.c_float), ('cost_no_table', C.c_float), ('cost_ok', C.c_float)]


class ResetOpC(C.Structure):
    _fields_ = [('kind', C.c_uint8), ('a', C.c_uint8), ('b', C.c_uint8), ('lo', C.c_uint8), ('hi', C.c_uint8),
                ('reserved', C.c_uint8 * 3)]


class ConfigC(C.Structure):
    _fields_ = [
        ('n_items', C.c_int32), ('n_actions', C.c_int32),
        ('actions', ActionEntryC * oc.MAX_ACTIONS),
        ('unbreakable_mask', C.c_uint32), ('entity_mask', C.c_uint32),
        ('break_reward_mask', C.c_uint32), ('reserved_mask', C.c_uint32),
        ('id_wall', C.c_uint8), ('id_crafting_table', C.c_uint8), ('id_tree_log', C.c_uint8),
        ('id_tree_tap', C.c_uint8), ('id_rubber', C.c_uint8), ('id_wool', C.c_uint8), ('id_string', C.c_uint8),
        ('id_goal', C.c_uint8), ('id_wooden_axe', C.c_uint8), ('id_iron_axe', C.c_uint8), ('id_fence', C.c_uint8),
        ('id_fire_wall', C.c_uint8), ('id_crate', C.c_uint8), ('reserved0', C.c_uint8 * 3),
        ('crate_add', C.c_uint8 * oc.MAX_ITEMS),
        ('reward_intermediate', C.c_int32), ('reward_done', C.c_int32), ('reward_firewall', C.c_int32),
        ('n_recipes', C.c_int32),
        ('recipes', RecipeC * oc.MAX_RECIPES),
        ('n_beams', C.c_int32), ('max_range', C.c_int32), ('n_lidar_items', C.c_int32),
        ('lidar_slot', C.c_int8 * oc.MAX_ITEMS),
        ('n_inv_obs', C.c_int32),
        ('inv_obs_item', C.c_uint8 * oc.MAX_ITEMS),
        ('beam_lut', C.c_void_p),
        ('n_place', C.c_int32),
        ('place_item', C.c_uint8 * oc.MAX_PLACE), ('place_qty', C.c_uint8 * oc.MAX_PLACE),
        ('n_reset_ops', C.c_int32),
        ('reset_ops', ResetOpC * oc.MAX_RESET_OPS),
        ('reset_obs_after_ops', C.c_int32),
    ]


class StateViewC(C.Structure):
    _fields_ = [('map', C.c_void_p), ('pose', C.c_void_p), ('inventory', C.c_void_p), ('cfg_id', C.c_void_p),
                ('episode', C.c_void_p), ('ep_len', C.c_void_p), ('error_flags', C.c_void_p),
                ('inv_stride', C.c_int32), ('obs_dim', C.c_int32),
                ('n_envs', C.c_int64), ('n_envs_padded', C.c_int64),
                ('map_size', C.c_int32), ('n_configs', C.c_int32),
                ('obs_format', C.c_int32), ('obs_row_bytes', C.c_int32)]


class RolloutRecordC(C.Structure):
    """struct ngw_rollout_record (include/ngw.h): the per-step buffers a rollout fills, [max_steps][n_envs_padded]."""
    _fields_ = [('max_steps', C.c_int32), ('obs', C.c_void_p), ('reward', C.c_void_p), ('step_cost', C.c_void_p),
                ('done', C.c_void_p), ('result', C.c_void_p), ('truncated', C.c_void_p), ('final_obs', C.c_void_p)]


# name -> (restype, argtypes); the same list is checked against include/ngw.h by the CPU test-suite
EXPORTS = {
    'ngw_create': (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(ConfigC), C.c_int32, C.c_int64, C.c_int32,
                             C.c_int32, C.c_int64, C.c_uint64]),
    'ngw_destroy': (None, [C.c_void_p]),
    'ngw_last_error': (C.c_char_p, []),
    'ngw_abi_version': (C.c_int, []),
    'ngw_state': (C.c_int, [C.c_void_p, C.POINTER(StateViewC)]),
    'ngw_set_obs_format': (C.c_int, [C.c_void_p, C.c_int32]),
    'ngw_lidar_path': (C.c_int, [C.POINTER(ConfigC), C.c_int32]),
    'ngw_set_env_configs': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    'ngw_load_state': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    'ngw_export_state': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    'ngw_reset': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'ngw_set_reset_rng': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    'ngw_load_rng_state': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    'ngw_export_rng_state': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    'ngw_step': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                           C.c_int32, C.c_int32, C.c_void_p]),
    'ngw_step_many': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    'ngw_set_message_buffer': (C.c_int, [C.c_void_p, C.c_void_p]),
    'ngw_set_episode_end_buffers': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    'ngw_set_rollout_record': (C.c_int, [C.c_void_p, C.POINTER(RolloutRecordC)]),
    'ngw_step_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int32, C.c_int32]),
    'ngw_rollout': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    'ngw_rollout_policy': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                     C.c_void_p]),
    'ngw_step_host_begin': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int32, C.c_int32]),
    'ngw_step_host_end': (C.c_int, [C.c_void_p]),
    'ngw_observe': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    'ngw_agent_map': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    'ngw_stats': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    'ngw_launch_count': (C.c_int64, [C.c_void_p]),
    'ngw_concurrent_launch_count': (C.c_int64, [C.c_void_p]),
}

_lib = None


class StepItem(C.Structure):
    """struct ngw_step_item (include/ngw.h): one handle's pointers in an ngw_step_many call."""
    _fields_ = [('h', C.c_void_p), ('actions', C.c_void_p), ('obs', C.c_void_p), ('reward', C.c_void_p),
                ('done', C.c_void_p), ('step_cost', C.c_void_p), ('result', C.c_void_p)]


def load_library(path=None):
    """dlopen libngw_b200.so and declare every export.  Fails loudly — there is no other backend."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(
            "CUDA extension %s is missing. Build it with `python __graft_entry__.py` (or "
            "`make -C gym_novel_gridworlds_b200/csrc`); this package has no CPU or PyTorch fallback." % p)
    lib = C.CDLL(p)
    for name, (restype, argtypes) in EXPORTS.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.ngw_abi_version() != ABI_VERSION:
        raise RuntimeError("libngw_b200.so ABI %d != python binding %d: rebuild" % (lib.ngw_abi_version(), ABI_VERSION))
    if path is None:
        _lib = lib
    return lib


def check(lib, rc):
    if rc != 0:
        msg = lib.ngw_last_error()
        raise RuntimeError("libngw_b200: " + (msg.decode() if msg else "error %d" % rc))
