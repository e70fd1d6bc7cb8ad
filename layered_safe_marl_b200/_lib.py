"""ctypes binding of include/lsm_b200.h. There is NO CPU fallback: if the CUDA library is missing
or no device is present, construction of the environment raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import _build


class LsmConfig(C.Structure):
    _fields_ = [('dynamics', C.c_int32), ('num_agents', C.c_int32), ('num_landmarks', C.c_int32),
                ('episode_length', C.c_int32), ('num_total_episode', C.c_int32),
                ('num_internal_step', C.c_int32), ('flags', C.c_uint32), ('num_obstacles', C.c_int32),
                ('world_size', C.c_double), ('dt', C.c_double), ('coordination_range', C.c_double),
                ('dist_thresh', C.c_double), ('heading_thresh', C.c_double), ('speed_thresh', C.c_double),
                ('goal_speed_min', C.c_double), ('goal_speed_max', C.c_double),
                ('separation_distance_target', C.c_double), ('engagement_distance_ref', C.c_double),
                ('engagement_ref_separation', C.c_double), ('cbf_rate', C.c_double),
                ('agent_max_speed', C.c_double), ('goal_rew', C.c_double),
                ('safety_violation_rew', C.c_double), ('hj_value_rew', C.c_double),
                ('potential_conflict_rew', C.c_double), ('diff_from_filtered_action_rew', C.c_double),
                ('min_reward', C.c_double), ('max_reward', C.c_double),
                ('act_tab0', C.c_double * 5), ('act_tab1', C.c_double * 5)]


class LsmGridDesc(C.Structure):
    _fields_ = [('ndim', C.c_int32), ('shape', C.c_int32 * 5), ('periodic', C.c_int32 * 5),
                ('_pad', C.c_int32), ('lo', C.c_double * 5), ('hi', C.c_double * 5),
                ('separation_distance', C.c_double), ('ttr_max', C.c_double),
                ('values', C.c_void_p), ('grads', C.c_void_p)]


class LsmBuffers(C.Structure):
    _fields_ = [('num_envs', C.c_int64), ('env_id_base', C.c_int64),
                ('agent_f64', C.c_void_p), ('agent_i32', C.c_void_p), ('landmarks', C.c_void_p),
                ('env_f64', C.c_void_p), ('env_i32', C.c_void_p),
                ('obs', C.c_void_p), ('node_obs', C.c_void_p), ('adj', C.c_void_p),
                ('reward', C.c_void_p), ('done', C.c_void_p), ('safe_action', C.c_void_p),
                ('ep_info', C.c_void_p), ('reward_individual', C.c_void_p),
                ('term_f64', C.c_void_p), ('term_i32', C.c_void_p), ('term_env_f64', C.c_void_p),
                ('obstacles', C.c_void_p)]


class LsmTuning(C.Structure):
    _fields_ = [('chunks', C.c_int32), ('pair_placement', C.c_int32), ('packed_grid', C.c_int32), ('use_graph', C.c_int32)]


class LsmLaunchInfo(C.Structure):
    _fields_ = [('grid_blocks', C.c_int32), ('block_threads', C.c_int32), ('warps_per_block', C.c_int32),
                ('envs_per_warp', C.c_int32), ('smem_bytes_per_block', C.c_int32), ('regs_per_thread', C.c_int32),
                ('blocks_per_sm', C.c_int32), ('sm_count', C.c_int32), ('specialised', C.c_int32),
                ('emit_block_threads', C.c_int32), ('emit_smem_bytes_per_block', C.c_int32),
                ('emit_regs_per_thread', C.c_int32), ('emit_blocks_per_sm', C.c_int32),
                ('pair_regs_per_thread', C.c_int32), ('launches_per_step', C.c_int32), ('emit_record_bytes', C.c_int32),
                ('chunks', C.c_int32), ('pair_placement', C.c_int32), ('graph_replays', C.c_int32),
                ('graph_captures', C.c_int32)]


class LsmHostIo(C.Structure):
    _fields_ = [('obs', C.c_void_p), ('node_obs', C.c_void_p), ('adj', C.c_void_p), ('reward', C.c_void_p),
                ('done', C.c_void_p), ('adj_base_staging', C.c_void_p), ('adj_keep_staging', C.c_void_p),
                ('threads', C.c_int32), ('chunks', C.c_int32), ('cached_stores', C.c_int32), ('_reserved', C.c_int32)]


class LsmFilterIo(C.Structure):
    _fields_ = [('num_rows', C.c_int64), ('num_slots', C.c_int32), ('_reserved', C.c_int32),
                ('ego', C.c_void_p), ('others', C.c_void_p), ('ego_action', C.c_void_p), ('other_actions', C.c_void_p),
                ('active', C.c_void_p), ('separation_distance', C.c_void_p), ('safe_action', C.c_void_p),
                ('filtered', C.c_void_p), ('index', C.c_void_p), ('value', C.c_void_p)]


class LsmLookupIo(C.Structure):
    _fields_ = [('num_points', C.c_int64), ('rel', C.c_void_p), ('ego', C.c_void_p), ('other', C.c_void_p),
                ('separation_distance', C.c_void_p), ('value', C.c_void_p), ('grad', C.c_void_p), ('rel_out', C.c_void_p)]


class LsmRecordEmitIo(C.Structure):
    _fields_ = [('num_items', C.c_int64), ('num_records', C.c_int64), ('records', C.c_void_p), ('record', C.c_void_p),
                ('observer', C.c_void_p), ('node_obs', C.c_void_p), ('adj', C.c_void_p)]


class LsmRecordEdgesIo(C.Structure):
    _fields_ = [('num_items', C.c_int64), ('num_records', C.c_int64), ('records', C.c_void_p), ('record', C.c_void_p),
                ('observer', C.c_void_p), ('counts', C.c_void_p), ('offsets', C.c_void_p), ('edge_index', C.c_void_p),
                ('edge_attr', C.c_void_p), ('capacity', C.c_int64)]


class LsmReturnsIo(C.Structure):
    """include/lsm_b200_ppo.h lsm_returns_io."""
    _fields_ = [('T', C.c_int64), ('columns', C.c_int64), ('rewards', C.c_void_p), ('value_preds', C.c_void_p),
                ('next_value', C.c_void_p), ('masks', C.c_void_p), ('bad_masks', C.c_void_p), ('returns', C.c_void_p),
                ('advantages', C.c_void_p), ('active_masks', C.c_void_p), ('value_scale', C.c_void_p),
                ('value_shift', C.c_void_p), ('scratch', C.c_void_p), ('stats64', C.c_void_p), ('stats', C.c_void_p),
                ('gamma', C.c_float), ('gamma_lambda', C.c_float), ('use_gae', C.c_int32),
                ('use_proper_time_limits', C.c_int32)]


class LsmHjProblem(C.Structure):
    """include/lsm_b200_hj.h lsm_hj_problem."""
    _fields_ = [('dynamics', C.c_int32), ('shape', C.c_int32 * 5), ('lo', C.c_double * 5), ('hi', C.c_double * 5),
                ('cfl', C.c_double)]


class LsmHjTtrProblem(C.Structure):
    """include/lsm_b200_hj.h lsm_hj_ttr_problem."""
    _fields_ = [('shape', C.c_int32 * 4), ('lo', C.c_double * 4), ('hi', C.c_double * 4), ('cfl', C.c_double)]


EXPORTED_SYMBOLS = ('lsm_abi_version', 'lsm_last_error', 'lsm_create', 'lsm_destroy', 'lsm_set_value_grid',
                    'lsm_set_ttr_grid', 'lsm_bind_buffers', 'lsm_get_launch_info', 'lsm_step', 'lsm_reset',
                    'lsm_observe', 'lsm_emit_only', 'lsm_invalidate', 'lsm_set_output_buffers', 'lsm_edge_list',
                    'lsm_debug_timeline', 'lsm_rollout_insert', 'lsm_math_eval', 'lsm_math_eval_device', 'lsm_set_tuning',
                    'lsm_set_compact_adjacency', 'lsm_expand_adjacency_host', 'lsm_set_edge_output', 'lsm_world_graph', 'lsm_fetch_host', 'lsm_step_host',
                    'lsm_episode_stats', 'lsm_debug_pair_values', 'lsm_safety_filter', 'lsm_hj_lookup',
                    'lsm_copy_records', 'lsm_emit_from_records', 'lsm_edges_from_records')

PPO_EXPORTED_SYMBOLS = ('lsm_ppo_abi_version', 'lsm_ppo_last_error', 'lsm_compute_returns', 'lsm_returns_scratch_bytes')

HJ_EXPORTED_SYMBOLS = ('lsm_hj_abi_version', 'lsm_hj_last_error', 'lsm_hj_work_bytes', 'lsm_hj_dissipation',
                       'lsm_hj_solve', 'lsm_hj_ttr_work_bytes', 'lsm_hj_ttr_dissipation', 'lsm_hj_ttr_solve')

_libs = {}          # one CDLL per path: the product library and the per-shape libraries (_build.build_shape)


def lib_path() -> str:
    return _build.LIB_PATH


def load(path: Optional[str] = None):
    """Load liblsm_b200.so (building it first if the sources are newer), or with `path` the library at that path (a
    per-shape library of _build.build_shape). One CDLL per path and process. Raises if unavailable."""
    key = path
    if key in _libs:
        return _libs[key]
    if path is None:
        path = _build.LIB_PATH
        alt = os.environ.get('LSM_LIB')     # A/B builds: another build of the sources (see _build.build)
        if alt:
            path = alt
        elif _build.needs_build():
            try:
                _build.build()
            except Exception as exc:  # no nvcc on the box and no prebuilt library: fail loudly
                if not os.path.exists(path):
                    raise RuntimeError(f"liblsm_b200.so is missing and could not be built: {exc}") from exc
    lib = C.CDLL(path)
    lib.lsm_abi_version.restype = C.c_int
    lib.lsm_last_error.restype = C.c_char_p
    lib.lsm_create.argtypes = [C.POINTER(LsmConfig), C.POINTER(C.c_void_p)]
    lib.lsm_destroy.argtypes = [C.c_void_p]
    lib.lsm_set_value_grid.argtypes = [C.c_void_p, C.POINTER(LsmGridDesc)]
    lib.lsm_set_ttr_grid.argtypes = [C.c_void_p, C.POINTER(LsmGridDesc)]
    lib.lsm_bind_buffers.argtypes = [C.c_void_p, C.POINTER(LsmBuffers)]
    lib.lsm_get_launch_info.argtypes = [C.c_void_p, C.POINTER(LsmLaunchInfo)]
    lib.lsm_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.c_void_p]
    lib.lsm_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.c_void_p]
    lib.lsm_observe.argtypes = [C.c_void_p, C.c_void_p]
    lib.lsm_emit_only.argtypes = [C.c_void_p, C.c_void_p]
    lib.lsm_invalidate.argtypes = [C.c_void_p]
    lib.lsm_set_output_buffers.argtypes = [C.c_void_p] + [C.c_void_p] * 5
    lib.lsm_edge_list.argtypes = [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]
    lib.lsm_debug_timeline.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.lsm_debug_pair_values.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lsm_rollout_insert.argtypes = [C.c_void_p] * 7
    lib.lsm_set_tuning.argtypes = [C.c_void_p, C.POINTER(LsmTuning)]
    lib.lsm_set_compact_adjacency.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lsm_expand_adjacency_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    lib.lsm_fetch_host.argtypes = [C.c_void_p, C.POINTER(LsmHostIo), C.c_void_p]
    lib.lsm_step_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.POINTER(LsmHostIo), C.c_void_p]
    lib.lsm_set_edge_output.argtypes = [C.c_void_p] * 5 + [C.c_int64, C.c_int]
    lib.lsm_world_graph.argtypes = [C.c_void_p] * 5 + [C.c_int64, C.c_void_p]
    lib.lsm_episode_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lsm_safety_filter.argtypes = [C.c_void_p, C.POINTER(LsmFilterIo), C.c_void_p]
    lib.lsm_hj_lookup.argtypes = [C.c_void_p, C.POINTER(LsmLookupIo), C.c_void_p]
    lib.lsm_copy_records.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lsm_emit_from_records.argtypes = [C.c_void_p, C.POINTER(LsmRecordEmitIo), C.c_void_p]
    lib.lsm_edges_from_records.argtypes = [C.c_void_p, C.POINTER(LsmRecordEdgesIo), C.c_void_p]
    lib.lsm_math_eval.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    lib.lsm_math_eval_device.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    for name in EXPORTED_SYMBOLS:
        if name not in ('lsm_abi_version', 'lsm_last_error'):
            getattr(lib, name).restype = C.c_int
    _libs[key] = lib
    return lib


def load_ppo():
    """Load liblsm_b200_ppo.so (include/lsm_b200_ppo.h), building it first if the sources are newer. Once per process."""
    key = _build.PPO_LIB_PATH
    if key in _libs:
        return _libs[key]
    if _build.needs_build(key, _build.PPO_DEPS):
        try:
            _build.build_ppo()
        except Exception as exc:
            if not os.path.exists(key):
                raise RuntimeError(f"liblsm_b200_ppo.so is missing and could not be built: {exc}") from exc
    lib = C.CDLL(key)
    lib.lsm_ppo_abi_version.restype = C.c_int
    lib.lsm_ppo_last_error.restype = C.c_char_p
    lib.lsm_compute_returns.argtypes = [C.POINTER(LsmReturnsIo), C.c_void_p]
    lib.lsm_compute_returns.restype = C.c_int
    lib.lsm_returns_scratch_bytes.argtypes = [C.c_int64]
    lib.lsm_returns_scratch_bytes.restype = C.c_int64
    lib.lsm_last_error = lib.lsm_ppo_last_error      # check(rc, what, lib) reads this library's own error string
    _libs[key] = lib
    return lib


def load_hj():
    """Load liblsm_b200_hj.so (include/lsm_b200_hj.h), building it first if the sources are newer. Once per process."""
    key = _build.HJ_LIB_PATH
    if key in _libs:
        return _libs[key]
    if _build.needs_build(key, _build.HJ_DEPS):
        try:
            _build.build_hj()
        except Exception as exc:
            if not os.path.exists(key):
                raise RuntimeError(f"liblsm_b200_hj.so is missing and could not be built: {exc}") from exc
    lib = C.CDLL(key)
    lib.lsm_hj_abi_version.restype = C.c_int
    lib.lsm_hj_last_error.restype = C.c_char_p
    lib.lsm_hj_work_bytes.argtypes = [C.POINTER(LsmHjProblem)]
    lib.lsm_hj_work_bytes.restype = C.c_int64
    lib.lsm_hj_dissipation.argtypes = [C.POINTER(LsmHjProblem), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.lsm_hj_dissipation.restype = C.c_int
    lib.lsm_hj_solve.argtypes = [C.POINTER(LsmHjProblem), C.c_void_p, C.POINTER(C.c_double), C.c_int32, C.c_void_p,
                                 C.c_void_p, C.c_void_p]
    lib.lsm_hj_solve.restype = C.c_int
    lib.lsm_hj_ttr_work_bytes.argtypes = [C.POINTER(LsmHjTtrProblem)]
    lib.lsm_hj_ttr_work_bytes.restype = C.c_int64
    lib.lsm_hj_ttr_dissipation.argtypes = [C.POINTER(LsmHjTtrProblem), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.lsm_hj_ttr_dissipation.restype = C.c_int
    lib.lsm_hj_ttr_solve.argtypes = [C.POINTER(LsmHjTtrProblem), C.c_void_p, C.c_double, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]
    lib.lsm_hj_ttr_solve.restype = C.c_int
    lib.lsm_last_error = lib.lsm_hj_last_error       # check(rc, what, lib) reads this library's own error string
    _libs[key] = lib
    return lib


def check(rc: int, what: str, lib=None):
    """Raise on a non-zero return code; the message is `lsm_last_error` of `lib`, the library that returned `rc` (default:
    the product library)."""
    if rc != 0:
        msg = (lib if lib is not None else load()).lsm_last_error()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
