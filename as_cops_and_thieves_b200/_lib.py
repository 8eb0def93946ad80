"""ctypes binding of ``libcat_b200.so`` (C ABI in ``include/cat_b200.h``).

Fails loudly: if the shared library is missing it is built with nvcc; if that is impossible, or a
compute entry point is called without a CUDA device, an exception is raised.  There is no CPU or
PyTorch fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import build as _build

CAT_ABI_VERSION = 9
CAT_MAX_AGENTS = 8
CAT_MAX_RAYS = 128
CAT_MAX_MAPS = 8
CAT_WALL_SLOTS = 4
CAT_NEAR_SLOTS = 4
CAT_SCRIPT_NONE = 0
CAT_SCRIPT_RANDOM = 1
CAT_SCRIPT_CHASE = 2
CAT_SCRIPT_EVADE = 3


class CatError(RuntimeError):
    pass


class CatMapDesc(C.Structure):
    _fields_ = [
        ("n_hulls", C.c_int32), ("n_edges", C.c_int32),
        ("hull_off", C.c_void_p), ("vert", C.c_void_p), ("normal", C.c_void_p), ("edge_len", C.c_void_p),
        ("hull_bb", C.c_void_p),
        ("n_cops", C.c_int32), ("n_thieves", C.c_int32),
        ("init_pos", C.c_void_p), ("region_off", C.c_void_p), ("regions", C.c_void_p),
        ("grid_x0", C.c_double), ("grid_y0", C.c_double), ("cell", C.c_double),
        ("nx", C.c_int32), ("ny", C.c_int32),
        ("con_cell_off", C.c_void_p), ("con_cell_hulls", C.c_void_p),
        ("view_cell_off", C.c_void_p), ("view_cell_edges", C.c_void_p), ("view_range", C.c_double),
    ]


class CatParams(C.Structure):
    _fields_ = [
        ("dt", C.c_double), ("max_step_count", C.c_int32),
        ("unit_velocity", C.c_double), ("unit_mass", C.c_double), ("unit_size", C.c_double),
        ("max_speed", C.c_double), ("termination_radius", C.c_double),
        ("ray_length", C.c_double), ("ray_radius", C.c_double), ("wall_radius", C.c_double),
        ("n_rays", C.c_int32), ("iterations", C.c_int32),
        ("collision_slop", C.c_double), ("collision_bias", C.c_double),
        ("collision_persistence", C.c_int32), ("stale_shape_cache", C.c_int32),
        ("auto_reset", C.c_int32), ("seed", C.c_uint64), ("ray_list_cell", C.c_double),
    ]


class CatStepIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("actions_kind", C.c_int32), ("reset_mask", C.c_void_p),
        ("shared_dist", C.c_void_p), ("shared_type", C.c_void_p), ("team_pos", C.c_void_p),
        ("obs_f32", C.c_void_p), ("state_f32", C.c_void_p), ("hit_point", C.c_void_p),
        ("record", C.c_void_p), ("record_world_stride", C.c_int32),
        ("critic_f32", C.c_void_p), ("obs_bf16", C.c_void_p), ("critic_bf16", C.c_void_p), ("record_packed_types", C.c_int32),
        ("final_record", C.c_void_p), ("final_record_world_stride", C.c_int32),
        ("final_obs_f32", C.c_void_p), ("final_state_f32", C.c_void_p), ("final_critic_f32", C.c_void_p),
    ]


class CatEpisodeTotals(C.Structure):
    _fields_ = [
        ("episodes", C.c_uint64), ("captures", C.c_uint64), ("timeouts", C.c_uint64), ("length_sum", C.c_uint64),
        ("length_min_key", C.c_uint32), ("length_max_key", C.c_uint32),
        ("return_sum", C.c_double * CAT_MAX_AGENTS), ("return_sq_sum", C.c_double * CAT_MAX_AGENTS),
        ("return_min_key", C.c_uint32 * CAT_MAX_AGENTS), ("return_max_key", C.c_uint32 * CAT_MAX_AGENTS),
    ]


class CatEpisodeStatsIO(C.Structure):
    _fields_ = [("acc", C.c_void_p), ("episode_return", C.c_void_p), ("episode_length", C.c_void_p), ("totals", C.c_void_p)]


class CatWorldParams(C.Structure):
    _fields_ = [("unit_velocity", C.c_float * 2), ("max_speed", C.c_float * 2), ("termination_radius", C.c_float),
                ("max_step_count", C.c_int32)]


class CatWorldParamRanges(C.Structure):
    _fields_ = [("lo", CatWorldParams), ("hi", CatWorldParams), ("draw", C.c_int32)]


class CatWorldParamsIO(C.Structure):
    _fields_ = [("params", C.c_void_p), ("ranges", C.c_void_p)]


class CatScriptIO(C.Structure):
    _fields_ = [("mode", C.c_void_p), ("decisions", C.c_void_p)]


class CatRecordLayout(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("bytes", "off_dist", "off_type", "off_reward", "off_terminated",
                                         "off_truncated", "off_winner", "type_bits")]


class CatEnvInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_worlds", "n_agents", "n_cops", "n_thieves", "n_rays", "n_hulls", "n_edges", "state_dim",
        "record_words", "map_blob_bytes", "smem_bytes_per_cta", "warps_per_cta", "grid", "n_pairs",
        "ray_list_cells", "ray_list_nx", "ray_list_ny")] + [("ray_list_cell", C.c_float), ("ray_list_bytes", C.c_int64)]


class CatStateView(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "pos", "vel", "vbias", "tc", "step_count", "episode", "wall_hull", "wall_age", "wall_jn",
        "pair_age", "pair_jn")]


class CatRenderIO(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32), ("world", C.c_void_p), ("n_elements", C.c_int64), ("map_of", C.c_void_p),
        ("pos", C.c_void_p), ("pos_stride", C.c_int64), ("ray_dist", C.c_void_p), ("ray_dist_stride", C.c_int64),
        ("ray_type", C.c_void_p), ("ray_type_stride", C.c_int64), ("downsample", C.c_int32),
        ("agent_radius", C.c_double), ("frames", C.c_void_p),
    ]


#: every symbol ``include/cat_b200.h`` declares
EXPORTS = (
    "cat_abi_version", "cat_last_error", "cat_env_create", "cat_env_create_multi", "cat_env_destroy", "cat_env_info",
    "cat_env_map_info", "cat_env_create_swappable", "cat_env_set_map", "cat_map_blob_bytes", "cat_ray_lists_device",
    "cat_env_record_layout", "cat_env_packed_record_layout", "cat_env_overflow_counts", "cat_ray_lists_host",
    "cat_env_set_seed", "cat_env_state_bytes", "cat_env_init_state", "cat_env_reset", "cat_env_step", "cat_env_step_host", "cat_env_observe",
    "cat_env_get_state", "cat_env_set_state", "cat_env_attach_episode_stats", "cat_env_attach_world_params",
    "cat_env_attach_scripts", "cat_gae", "cat_adv_normalize",
    "cat_renderer_create", "cat_renderer_destroy", "cat_renderer_frame_size", "cat_render", "cat_ray_directions",
)

_LIB = None


def lib_path() -> Path:
    return _build.LIB


def load():
    """Load (building first if needed) the CUDA extension.  Raises if it cannot be had."""
    global _LIB
    if _LIB is not None:
        return _LIB
    import os
    override = os.environ.get("CAT_B200_LIB")  # developer knob: load a tuning variant of the extension
    path = Path(override) if override else _build.build()
    L = C.CDLL(str(path))
    for name in EXPORTS:
        if not hasattr(L, name):
            raise CatError(f"{path} does not export {name}")
    L.cat_abi_version.restype = C.c_int
    if L.cat_abi_version() != CAT_ABI_VERSION:
        raise CatError(f"ABI mismatch: library {L.cat_abi_version()} != binding {CAT_ABI_VERSION}")
    L.cat_last_error.restype = C.c_char_p
    L.cat_env_create.argtypes = [C.POINTER(CatMapDesc), C.POINTER(CatParams), C.c_int32, C.c_int64, C.c_int32,
                                 C.POINTER(C.c_void_p)]
    L.cat_env_create_multi.argtypes = [C.POINTER(CatMapDesc), C.c_int32, C.POINTER(C.c_int32), C.POINTER(CatParams), C.c_int64,
                                       C.c_int32, C.POINTER(C.c_void_p)]
    L.cat_env_create_swappable.argtypes = [C.POINTER(CatMapDesc), C.c_int32, C.POINTER(C.c_int32), C.POINTER(CatParams), C.c_int32,
                                           C.c_int64, C.c_int32, C.POINTER(C.c_void_p)]
    L.cat_env_set_map.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CatMapDesc), C.c_void_p]
    L.cat_map_blob_bytes.argtypes = [C.POINTER(CatMapDesc), C.POINTER(CatParams), C.POINTER(C.c_int32)]
    L.cat_env_destroy.argtypes = [C.c_void_p]
    L.cat_env_info.argtypes = [C.c_void_p, C.POINTER(CatEnvInfo)]
    L.cat_env_map_info.argtypes = [C.c_void_p, C.c_int32, C.POINTER(CatEnvInfo)]
    L.cat_env_set_seed.argtypes = [C.c_void_p, C.c_uint64]
    L.cat_env_state_bytes.restype = C.c_size_t
    L.cat_env_state_bytes.argtypes = [C.c_void_p]
    L.cat_env_init_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    for fn in (L.cat_env_reset, L.cat_env_step, L.cat_env_observe):
        fn.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(CatStepIO), C.c_void_p]
    L.cat_env_step_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    L.cat_ray_lists_host.argtypes = [C.POINTER(CatMapDesc), C.c_int32, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double * 5),
                                     C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.POINTER(C.c_int64)]
    L.cat_ray_lists_device.argtypes = L.cat_ray_lists_host.argtypes + [C.c_int32]
    L.cat_env_record_layout.argtypes = [C.c_void_p, C.POINTER(CatRecordLayout)]
    L.cat_env_packed_record_layout.argtypes = [C.c_void_p, C.POINTER(CatRecordLayout)]
    L.cat_env_overflow_counts.argtypes = [C.c_void_p, C.POINTER(C.c_uint64 * 2), C.c_int32]
    for fn in (L.cat_env_get_state, L.cat_env_set_state):
        fn.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(CatStateView), C.c_void_p]
    L.cat_env_attach_episode_stats.argtypes = [C.c_void_p, C.POINTER(CatEpisodeStatsIO)]
    L.cat_env_attach_world_params.argtypes = [C.c_void_p, C.POINTER(CatWorldParamsIO)]
    L.cat_env_attach_scripts.argtypes = [C.c_void_p, C.POINTER(CatScriptIO)]
    L.cat_gae.argtypes = [C.c_void_p] * 7 + [C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_void_p]
    L.cat_adv_normalize.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    L.cat_renderer_create.argtypes = [C.POINTER(CatMapDesc), C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int32,
                                      C.POINTER(C.c_void_p)]
    L.cat_renderer_destroy.argtypes = [C.c_void_p]
    L.cat_renderer_frame_size.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.cat_render.argtypes = [C.c_void_p, C.POINTER(CatRenderIO), C.c_void_p]
    L.cat_ray_directions.argtypes = [C.c_int32, C.c_void_p]
    _LIB = L
    return L


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().cat_last_error()
        raise CatError(f"{what} failed ({status}): {msg.decode() if msg else ''}")


def np_ptr(a: np.ndarray) -> C.c_void_p:
    return a.ctypes.data_as(C.c_void_p)
