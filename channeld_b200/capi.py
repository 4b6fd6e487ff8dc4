"""ctypes binding of the C ABI in include/chd_gpu.h (libchd_b200.so).

This is the only way Python reaches the kernels: tests, bench.py and the controller mirror all call through
these entry points — the same ones a cgo shim binds (INTEGRATION.md).  There is no CPU fallback: if the
library is missing it is built; if it cannot be loaded, importing fails loudly.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)
f64p = C.POINTER(C.c_double)

OK, ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_STATE = 0, 1, 2, 3, 4
AOI_SPOTS, AOI_BOX, AOI_SPHERE, AOI_CONE = 1, 2, 4, 8
Q_OK, Q_ERR_OUT_OF_WORLD, Q_ERR_BAD_STEP, Q_ERR_ITER_BOUND, Q_ERR_ANGLE_RANGE, Q_ERR_CAPACITY, Q_ERR_MISSING_ARRAY = 0, 1, 2, 5, 6, 7, 8
DUE_VOID = 0xFFFFFFFF
TICK_BUILD, TICK_EMIT, TICK_FANOUT, TICK_ALL = 1, 2, 4, 7
TICK_EARLY_RESULTS = 8
OVF_PAIRS, OVF_WINDOW, OVF_VISIBLE, OVF_DUE, OVF_BORDER, OVF_RING = 1, 2, 4, 8, 16, 32
PF_HAD_FIRST, PF_NEW, PF_SKIP_SELF = 1, 2, 4


class GridCfg(C.Structure):
    _fields_ = [
        ("world_offset_x", C.c_double), ("world_offset_z", C.c_double),
        ("grid_width", C.c_double), ("grid_height", C.c_double),
        ("grid_cols", C.c_uint32), ("grid_rows", C.c_uint32),
        ("server_cols", C.c_uint32), ("server_rows", C.c_uint32),
        ("server_interest_border_size", C.c_uint32), ("channel_id_start", C.c_uint32),
    ]


class Limits(C.Structure):
    _fields_ = [
        ("max_entities", C.c_uint32), ("max_subscribers", C.c_uint32), ("max_queries", C.c_uint32),
        ("max_spots", C.c_uint32), ("max_pairs", C.c_uint64), ("max_window_cells", C.c_uint64),
        ("max_visible", C.c_uint64), ("max_ring_entries", C.c_uint32), ("max_due", C.c_uint32),
        ("default_fanout_interval_ms", C.c_uint32), ("default_fanout_delay_ms", C.c_int32),
    ]


class QueryBatch(C.Structure):
    _fields_ = [
        ("n", C.c_uint32), ("sub", C.c_void_p), ("kind", C.c_void_p),
        ("sph_cx", C.c_void_p), ("sph_cz", C.c_void_p), ("sph_r", C.c_void_p),
        ("box_cx", C.c_void_p), ("box_cz", C.c_void_p), ("box_ex", C.c_void_p), ("box_ez", C.c_void_p),
        ("cone_cx", C.c_void_p), ("cone_cz", C.c_void_p), ("cone_dx", C.c_void_p), ("cone_dz", C.c_void_p),
        ("cone_angle", C.c_void_p), ("cone_r", C.c_void_p),
        ("spot_off", C.c_void_p), ("spot_ndist", C.c_void_p), ("spot_x", C.c_void_p), ("spot_z", C.c_void_p),
        ("spot_dist", C.c_void_p),
    ]


class BroadcastBatch(C.Structure):
    _fields_ = [("n", C.c_uint32), ("channel_id", C.c_void_p), ("broadcast", C.c_void_p), ("sender_conn_id", C.c_void_p),
                ("client_conn_id", C.c_void_p)]


BC_ALL_BUT_SENDER, BC_ALL_BUT_OWNER, BC_ALL_BUT_CLIENT, BC_ALL_BUT_SERVER, BC_ADJACENT_CHANNELS = 4, 8, 16, 32, 64
CONN_SERVER, CONN_CLIENT = 1, 2


class Due(C.Structure):
    _fields_ = [
        ("sub", C.c_uint32), ("channel_id", C.c_uint32), ("kind", C.c_uint32), ("n_selected", C.c_uint32),
        ("first_sel", C.c_uint32), ("last_sel", C.c_uint32), ("sel_hash", C.c_uint64),
        ("last_message_index", C.c_uint64), ("window_hi", C.c_int64),
    ]


DUE_DTYPE = np.dtype([("sub", "<u4"), ("channel_id", "<u4"), ("kind", "<u4"), ("n_selected", "<u4"),
                      ("first_sel", "<u4"), ("last_sel", "<u4"), ("sel_hash", "<u8"),
                      ("last_message_index", "<u8"), ("window_hi", "<i8")])
assert DUE_DTYPE.itemsize == C.sizeof(Due) == 48


class ResultBuffers(C.Structure):
    _fields_ = [
        ("pair_off", C.c_void_p), ("pair_channel", C.c_void_p), ("pair_dist", C.c_void_p), ("pair_interval_ms", C.c_void_p),
        ("pair_cap", C.c_uint64),
        ("new_sub", C.c_void_p), ("new_channel", C.c_void_p), ("unsub_sub", C.c_void_p), ("unsub_channel", C.c_void_p),
        ("diff_cap", C.c_uint64),
        ("due", C.c_void_p), ("due_cap", C.c_uint32),
        ("handover_entity", C.c_void_p), ("handover_src", C.c_void_p), ("handover_dst", C.c_void_p), ("handover_cap", C.c_uint32),
        ("query_status", C.c_void_p), ("status_cap", C.c_uint32),
        ("vis_off", C.c_void_p), ("vis_entity", C.c_void_p), ("vis_cap", C.c_uint64),
        ("cell_start", C.c_void_p), ("sorted_entity", C.c_void_p), ("entity_cap", C.c_uint32),
    ]


class TickSummary(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_uint64), ("n_visible", C.c_uint64), ("n_entities_in_world", C.c_uint32),
        ("n_query_errors", C.c_uint32), ("n_sub_new", C.c_uint32), ("n_unsub", C.c_uint32), ("n_kept", C.c_uint32),
        ("n_due", C.c_uint32), ("n_handover", C.c_uint32), ("overflow", C.c_uint32),
        ("required_pairs", C.c_uint64), ("required_window_cells", C.c_uint64), ("required_visible", C.c_uint64),
        ("required_due", C.c_uint32), ("reserved", C.c_uint32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


# every symbol include/chd_gpu.h declares (checked by tests/test_abi.py against the header text)
SYMBOLS = [
    "chd_abi_version", "chd_default_limits", "chd_create", "chd_destroy", "chd_last_error", "chd_set_stream", "chd_sync",
    "chd_alloc_pinned", "chd_free_pinned", "chd_device_numa_node", "chd_cell_of", "chd_cell_of_valid", "chd_set_entities", "chd_prefetch_entities", "chd_set_entities_f32", "chd_prefetch_entities_f32", "chd_prefetch_queries", "chd_prefetch_rings", "chd_adopt_prefetched", "chd_entity_buffers", "chd_set_entity_count",
    "chd_assign_cells", "chd_build", "chd_set_subscribers", "chd_query_channel_ids", "chd_update_interest",
    "chd_emit_visible", "chd_set_rings", "chd_fanout_tick", "chd_summary", "chd_tick", "chd_begin_interest", "chd_get_cells", "chd_get_pairs",
    "chd_get_query_status", "chd_get_diff", "chd_get_visible", "chd_get_visible_slot", "chd_get_due", "chd_fetch_results", "chd_get_handover", "chd_device_view",
    "chd_set_slab", "chd_set_entity_ids", "chd_export_border", "chd_import_halo", "chd_due_classes", "chd_set_subscriber_types", "chd_adjacent_broadcast", "chd_get_adjacent_channels",
    "chd_get_regions", "chd_damping_interval_ms", "chd_launch_count", "chd_profile_enable", "chd_profile_get", "chd_profile_timeline", "chd_enable_graphs",
    "chd_graph_launch_count",
    "chd_add_subscribers", "chd_remove_subscribers", "chd_fetch_results_async", "chd_fetch_wait", "chd_rings_init", "chd_rings_append", "chd_get_rings", "chd_set_channel_start_times", "chd_set_payload_bytes", "chd_assemble_payloads", "chd_frame_packets", "chd_comm_unique_id", "chd_comm_init", "chd_comm_info", "chd_comm_destroy", "chd_tick_sharded", "chd_collective_count", "chd_comm_exchange_mode", "chd_comm_use_collective", "chd_migrate_out", "chd_migrate_in", "chd_get_rehome",
    "chd_visible_delta_enable", "chd_visible_delta", "chd_get_visible_delta",
]
STAGE_BUILD, STAGE_INTEREST, STAGE_EMIT, STAGE_EMIT_KERNEL, STAGE_FANOUT, STAGE_TICK, STAGE_EXPORT, STAGE_EXCHANGE, STAGE_IMPORT, STAGE_READBACK = range(10)
(VIEW_CELL_START, VIEW_SORTED_ENTITY, VIEW_ENT_CELL, VIEW_PAIR_OFF, VIEW_PAIR_CHANNEL, VIEW_PAIR_DIST, VIEW_VIS_OFF, VIEW_VIS_ENTITY,
 VIEW_DUE, VIEW_ENTER_OFF, VIEW_ENTER_ENTITY, VIEW_LEAVE_OFF, VIEW_LEAVE_ENTITY) = range(13)  # chd_device_view

_lib = None


def lib():
    """Loads (building first if stale) libchd_b200.so.  Raises if that is impossible: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build()
    if os.environ.get("CHD_EXPERIMENT_LIB"):  # tools/ only: an experiment build of the same sources (different tile constants)
        path = os.environ["CHD_EXPERIMENT_LIB"]
    L = C.CDLL(path)
    vp = C.c_void_p
    L.chd_abi_version.restype = C.c_uint32
    L.chd_default_limits.restype = None
    L.chd_default_limits.argtypes = [C.POINTER(GridCfg), C.c_uint32, C.c_uint32, C.POINTER(Limits)]
    L.chd_create.restype = C.c_int
    L.chd_create.argtypes = [C.POINTER(GridCfg), C.POINTER(Limits), C.c_int, C.POINTER(vp)]
    L.chd_destroy.restype = None
    L.chd_destroy.argtypes = [vp]
    L.chd_last_error.restype = C.c_char_p
    L.chd_last_error.argtypes = [vp]
    L.chd_set_stream.restype = C.c_int
    L.chd_set_stream.argtypes = [vp, vp]
    L.chd_sync.restype = C.c_int
    L.chd_sync.argtypes = [vp]
    L.chd_alloc_pinned.restype = vp
    L.chd_alloc_pinned.argtypes = [C.c_uint64]
    L.chd_device_numa_node.restype = C.c_int
    L.chd_device_numa_node.argtypes = [C.c_int]
    L.chd_free_pinned.restype = None
    L.chd_free_pinned.argtypes = [vp]
    L.chd_cell_of.restype = C.c_int
    L.chd_cell_of.argtypes = [vp, vp, vp, C.c_uint32, vp]
    L.chd_cell_of_valid.restype = C.c_int
    L.chd_cell_of_valid.argtypes = [vp, vp, vp, C.c_uint32, vp, vp]
    L.chd_set_entities.restype = C.c_int
    L.chd_set_entities.argtypes = [vp, vp, vp, C.c_uint32]
    L.chd_prefetch_entities.restype = C.c_int
    L.chd_prefetch_entities.argtypes = [vp, vp, vp, C.c_uint32]
    L.chd_set_entities_f32.restype = C.c_int
    L.chd_set_entities_f32.argtypes = [vp, vp, vp, C.c_uint32]
    L.chd_prefetch_entities_f32.restype = C.c_int
    L.chd_prefetch_entities_f32.argtypes = [vp, vp, vp, C.c_uint32]
    L.chd_prefetch_queries.restype = C.c_int
    L.chd_prefetch_queries.argtypes = [vp, vp]
    L.chd_prefetch_rings.restype = C.c_int
    L.chd_prefetch_rings.argtypes = [vp, vp, C.c_uint32, vp, vp, vp, vp]
    L.chd_adopt_prefetched.restype = C.c_int
    L.chd_adopt_prefetched.argtypes = [vp]
    L.chd_entity_buffers.restype = C.c_int
    L.chd_entity_buffers.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), u32p]
    L.chd_set_entity_count.restype = C.c_int
    L.chd_set_entity_count.argtypes = [vp, C.c_uint32]
    L.chd_assign_cells.restype = C.c_int
    L.chd_assign_cells.argtypes = [vp]
    L.chd_build.restype = C.c_int
    L.chd_build.argtypes = [vp]
    L.chd_set_subscribers.restype = C.c_int
    L.chd_set_subscribers.argtypes = [vp, vp, C.c_uint32]
    L.chd_query_channel_ids.restype = C.c_int
    L.chd_query_channel_ids.argtypes = [vp, C.POINTER(QueryBatch), vp, vp, vp, vp, C.c_uint64]
    L.chd_update_interest.restype = C.c_int
    L.chd_update_interest.argtypes = [vp, C.POINTER(QueryBatch), C.c_int64]
    L.chd_emit_visible.restype = C.c_int
    L.chd_emit_visible.argtypes = [vp]
    L.chd_set_rings.restype = C.c_int
    L.chd_set_rings.argtypes = [vp, vp, C.c_uint32, vp, vp, vp, vp]
    L.chd_fanout_tick.restype = C.c_int
    L.chd_fanout_tick.argtypes = [vp, C.c_int64]
    L.chd_summary.restype = C.c_int
    L.chd_summary.argtypes = [vp, C.POINTER(TickSummary)]
    L.chd_begin_interest.restype = C.c_int
    L.chd_begin_interest.argtypes = [vp, C.POINTER(QueryBatch), C.c_int64, C.c_int]
    L.chd_tick.restype = C.c_int
    L.chd_tick.argtypes = [vp, C.POINTER(QueryBatch), C.c_int64, C.c_uint32, C.POINTER(TickSummary)]
    L.chd_get_cells.restype = C.c_int
    L.chd_get_cells.argtypes = [vp, vp, vp]
    L.chd_get_pairs.restype = C.c_int
    L.chd_get_pairs.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.chd_get_query_status.restype = C.c_int
    L.chd_get_query_status.argtypes = [vp, vp, C.c_uint32]
    L.chd_get_diff.restype = C.c_int
    L.chd_get_diff.argtypes = [vp, vp, vp, vp, vp]
    L.chd_get_visible.restype = C.c_int
    L.chd_get_visible.argtypes = [vp, vp, vp]
    L.chd_fetch_results.restype = C.c_int
    L.chd_fetch_results.argtypes = [vp, C.POINTER(ResultBuffers), C.POINTER(TickSummary)]
    L.chd_get_visible_slot.restype = C.c_int
    L.chd_get_visible_slot.argtypes = [vp, C.c_uint32, vp, C.c_uint64, u64p]
    L.chd_get_due.restype = C.c_int
    L.chd_get_due.argtypes = [vp, vp, C.c_uint32]
    L.chd_get_handover.restype = C.c_int
    L.chd_get_handover.argtypes = [vp, vp, vp, vp, C.c_uint32]
    L.chd_device_view.restype = C.c_int
    L.chd_device_view.argtypes = [vp, C.c_int, C.POINTER(vp), u64p]
    L.chd_set_slab.restype = C.c_int
    L.chd_set_slab.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32]
    L.chd_set_entity_ids.restype = C.c_int
    L.chd_set_entity_ids.argtypes = [vp, vp, C.c_uint32]
    L.chd_export_border.restype = C.c_int
    L.chd_export_border.argtypes = [vp, vp, C.c_uint32, u32p]
    L.chd_import_halo.restype = C.c_int
    L.chd_import_halo.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32]
    L.chd_due_classes.restype = C.c_int
    L.chd_due_classes.argtypes = [vp, vp, vp, vp, C.c_uint32, u32p]
    L.chd_set_subscriber_types.restype = C.c_int
    L.chd_set_subscriber_types.argtypes = [vp, vp, C.c_uint32]
    L.chd_adjacent_broadcast.restype = C.c_int
    L.chd_adjacent_broadcast.argtypes = [vp, C.POINTER(BroadcastBatch), vp, vp, vp, C.c_uint64]
    L.chd_get_adjacent_channels.restype = C.c_uint32
    L.chd_get_adjacent_channels.argtypes = [C.POINTER(GridCfg), C.c_uint32, vp]
    L.chd_get_regions.restype = C.c_int
    L.chd_get_regions.argtypes = [C.POINTER(GridCfg), vp, vp, vp, vp, vp, vp]
    L.chd_damping_interval_ms.restype = C.c_uint32
    L.chd_damping_interval_ms.argtypes = [C.c_uint32, C.c_uint32]
    L.chd_launch_count.restype = C.c_uint64
    L.chd_launch_count.argtypes = [vp]
    L.chd_enable_graphs.restype = C.c_int
    L.chd_enable_graphs.argtypes = [vp, C.c_int]
    L.chd_graph_launch_count.restype = C.c_uint64
    L.chd_graph_launch_count.argtypes = [vp]
    L.chd_profile_enable.restype = C.c_int
    L.chd_profile_enable.argtypes = [vp, C.c_int]
    L.chd_profile_timeline.restype = C.c_int
    L.chd_profile_timeline.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.chd_profile_get.restype = C.c_int
    L.chd_profile_get.argtypes = [vp, C.c_int, C.POINTER(C.c_double), u64p]
    L.chd_fetch_results_async.restype = C.c_int
    L.chd_fetch_results_async.argtypes = [vp, C.POINTER(ResultBuffers), vp]
    L.chd_fetch_wait.restype = C.c_int
    L.chd_fetch_wait.argtypes = [vp, C.POINTER(TickSummary)]
    L.chd_rings_init.restype = C.c_int
    L.chd_rings_init.argtypes = [vp, C.c_uint32]
    L.chd_rings_append.restype = C.c_int
    L.chd_rings_append.argtypes = [vp, vp, C.c_uint32, vp, vp]
    L.chd_get_rings.restype = C.c_int
    L.chd_get_rings.argtypes = [vp, vp, vp, vp, vp, vp, C.c_uint32]
    L.chd_set_channel_start_times.restype = C.c_int
    L.chd_set_channel_start_times.argtypes = [vp, vp]
    L.chd_set_payload_bytes.restype = C.c_int
    L.chd_set_payload_bytes.argtypes = [vp, vp, C.c_uint32, vp, vp, vp, vp, C.c_uint32]
    L.chd_assemble_payloads.restype = C.c_int
    L.chd_assemble_payloads.argtypes = [vp, u32p, vp, C.c_uint32, vp, C.c_uint64, u64p]
    L.chd_frame_packets.restype = C.c_int
    L.chd_frame_packets.argtypes = [vp, vp, vp, vp, vp, vp, C.c_uint64, u64p, u32p]
    L.chd_add_subscribers.restype = C.c_int
    L.chd_add_subscribers.argtypes = [vp, vp, vp, C.c_uint32]
    L.chd_remove_subscribers.restype = C.c_int
    L.chd_remove_subscribers.argtypes = [vp, vp, C.c_uint32]
    L.chd_comm_unique_id.restype = C.c_int
    L.chd_comm_unique_id.argtypes = [vp]
    L.chd_comm_init.restype = C.c_int
    L.chd_comm_init.argtypes = [vp, vp, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
    L.chd_migrate_out.restype = C.c_int
    L.chd_migrate_out.argtypes = [vp, vp, C.c_uint32]
    L.chd_migrate_in.restype = C.c_int
    L.chd_migrate_in.argtypes = [vp, C.c_uint32, C.c_uint32, vp, vp, C.c_uint32]
    L.chd_get_rehome.restype = C.c_int
    L.chd_get_rehome.argtypes = [vp, vp, vp, C.c_uint32, u32p]
    L.chd_comm_info.restype = C.c_int
    L.chd_comm_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), u32p, u32p, u32p, C.POINTER(C.c_int)]
    L.chd_comm_destroy.restype = C.c_int
    L.chd_comm_destroy.argtypes = [vp]
    L.chd_tick_sharded.restype = C.c_int
    L.chd_tick_sharded.argtypes = [vp, C.POINTER(QueryBatch), C.c_int64, C.c_uint32, C.POINTER(TickSummary)]
    L.chd_collective_count.restype = C.c_uint64
    L.chd_collective_count.argtypes = [vp]
    L.chd_comm_exchange_mode.restype = C.c_int
    L.chd_comm_exchange_mode.argtypes = [vp]
    L.chd_comm_use_collective.restype = C.c_int
    L.chd_comm_use_collective.argtypes = [vp, C.c_int]
    L.chd_visible_delta_enable.restype = C.c_int
    L.chd_visible_delta_enable.argtypes = [vp, C.c_uint64]
    L.chd_visible_delta.restype = C.c_int
    L.chd_visible_delta.argtypes = [vp]
    L.chd_get_visible_delta.restype = C.c_int
    L.chd_get_visible_delta.argtypes = [vp, vp, vp, C.c_uint64, vp, vp, C.c_uint64, u64p, u64p]
    _lib = L
    return L


def lib_path():
    return _build.LIB


def ptr(a):
    """numpy array / torch tensor / int / None -> raw address (host or device)."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return a.ctypes.data
    if hasattr(a, "data_ptr"):  # torch tensor (host pinned or cuda)
        assert a.is_contiguous()
        return a.data_ptr()
    raise TypeError(type(a))


class ChdError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("chd status %d: %s" % (status, msg))
        self.status = status
