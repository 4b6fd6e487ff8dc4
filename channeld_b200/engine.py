"""Thin object wrapper over the C ABI (include/chd_gpu.h).  No compute happens in Python: every method is one
C call; results come back as numpy arrays copied by the library.  Inputs may be numpy arrays (host), torch
tensors (pinned host or CUDA) or raw addresses.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import ChdError, GridCfg, Limits, QueryBatch, TickSummary, ptr

SPATIAL_CHANNEL_ID_START = 0x10000  # settings.go:94
ENTITY_CHANNEL_ID_START = 0x80000   # settings.go:95


def grid_cfg(offx, offz, w, h, cols, rows, server_cols=1, server_rows=1, border=0, id_start=SPATIAL_CHANNEL_ID_START):
    return GridCfg(float(offx), float(offz), float(w), float(h), int(cols), int(rows), int(server_cols), int(server_rows),
                   int(border), int(id_start))


def make_batch(n, sub=None, kind=None, sphere=None, box=None, cone=None, spots=None, keep=None):
    """Builds a chd_query_batch.  sphere=(cx,cz,r) box=(cx,cz,ex,ez) cone=(cx,cz,dx,dz,angle,r) are tuples of
    arrays; spots=(spot_off, spot_ndist, x, z, dist).  Arrays are kept alive in `keep` (a list)."""
    keep = keep if keep is not None else []
    b = QueryBatch()
    b.n = int(n)

    def f64(a):
        if a is None:
            return None
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a, np.float64)
        keep.append(a)
        return ptr(a)

    def u32(a):
        if a is None:
            return None
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a, np.uint32)
        keep.append(a)
        return ptr(a)

    b.sub = u32(sub)
    if kind is not None:
        if isinstance(kind, np.ndarray):
            kind = np.ascontiguousarray(kind, np.uint8)
        keep.append(kind)
        b.kind = ptr(kind)
    if sphere is not None:
        b.sph_cx, b.sph_cz, b.sph_r = (f64(a) for a in sphere)
    if box is not None:
        b.box_cx, b.box_cz, b.box_ex, b.box_ez = (f64(a) for a in box)
    if cone is not None:
        b.cone_cx, b.cone_cz, b.cone_dx, b.cone_dz, b.cone_angle, b.cone_r = (f64(a) for a in cone)
    if spots is not None:
        off, ndist, x, z, dist = spots
        b.spot_off, b.spot_ndist, b.spot_x, b.spot_z, b.spot_dist = u32(off), u32(ndist), f64(x), f64(z), u32(dist)
    return b, keep


class Engine:
    def __init__(self, cfg, n_entities, n_subscribers, device=0, **limit_overrides):
        self.L = capi.lib()
        self.cfg = cfg
        lim = Limits()
        self.L.chd_default_limits(C.byref(cfg), int(n_entities), int(n_subscribers), C.byref(lim))
        for k, v in limit_overrides.items():
            if not hasattr(lim, k):
                raise KeyError(k)
            setattr(lim, k, v)
        self.lim = lim
        h = C.c_void_p()
        st = self.L.chd_create(C.byref(cfg), C.byref(lim), int(device), C.byref(h))
        if st != capi.OK:
            raise ChdError(st, self.L.chd_last_error(None).decode())
        self.h = h
        self.n_cells = cfg.grid_cols * cfg.grid_rows
        self.n_slots = 0
        self._keep = []

    def close(self):
        if getattr(self, "h", None):
            self.L.chd_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, st):
        if st != capi.OK:
            raise ChdError(st, self.L.chd_last_error(self.h).decode())

    # ---- plumbing
    def set_stream(self, cuda_stream):
        self._ck(self.L.chd_set_stream(self.h, cuda_stream))

    def sync(self):
        self._ck(self.L.chd_sync(self.h))

    # ---- GetChannelId (batched)
    def cell_of(self, x, z, with_valid=False):
        x = np.ascontiguousarray(x, np.float64)
        z = np.ascontiguousarray(z, np.float64)
        out = np.zeros(len(x), np.uint32)
        if with_valid:
            ok = np.zeros(len(x), np.uint8)
            self._ck(self.L.chd_cell_of_valid(self.h, ptr(x), ptr(z), len(x), ptr(out), ptr(ok)))
            return out, ok.astype(bool)
        self._ck(self.L.chd_cell_of(self.h, ptr(x), ptr(z), len(x), ptr(out)))
        return out

    # ---- entities / build
    def set_entities(self, x, z, n=None):
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, np.float64)
            z = np.ascontiguousarray(z, np.float64)
        n = len(x) if n is None else n
        self._keep = [x, z]  # async H2D: keep alive until the next call
        self._ck(self.L.chd_set_entities(self.h, ptr(x), ptr(z), int(n)))

    def prefetch_entities(self, x, z, n=None):
        """Start the H2D upload of the NEXT tick's positions (overlaps the tick in flight); see chd_prefetch_entities."""
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, np.float64)
            z = np.ascontiguousarray(z, np.float64)
        n = len(x) if n is None else n
        self._keep_prefetch = [x, z]
        self._ck(self.L.chd_prefetch_entities(self.h, ptr(x), ptr(z), int(n)))

    def set_entities_f32(self, x, z, n=None):
        """Positions that are floats at the source (unrealpb.FVector): uploaded as floats, widened exactly on the device."""
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, np.float32)
            z = np.ascontiguousarray(z, np.float32)
        n = len(x) if n is None else n
        self._keep = [x, z]
        self._ck(self.L.chd_set_entities_f32(self.h, ptr(x), ptr(z), int(n)))

    def prefetch_entities_f32(self, x, z, n=None):
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, np.float32)
            z = np.ascontiguousarray(z, np.float32)
        n = len(x) if n is None else n
        self._keep_prefetch = [x, z]
        self._ck(self.L.chd_prefetch_entities_f32(self.h, ptr(x), ptr(z), int(n)))

    def adopt_prefetched(self):
        self._ck(self.L.chd_adopt_prefetched(self.h))
        self._keep = getattr(self, "_keep_prefetch", None)

    def set_entity_ids(self, gid):
        if gid is None:
            self._ck(self.L.chd_set_entity_ids(self.h, None, 0))
            return
        if isinstance(gid, np.ndarray):
            gid = np.ascontiguousarray(gid, np.uint32)
        self._keep_gid = gid
        self._ck(self.L.chd_set_entity_ids(self.h, ptr(gid), len(gid)))

    def entity_buffers(self):
        dx, dz, n = C.c_void_p(), C.c_void_p(), C.c_uint32()
        self._ck(self.L.chd_entity_buffers(self.h, C.byref(dx), C.byref(dz), C.byref(n)))
        return dx.value, dz.value, n.value

    def set_entity_count(self, n):
        self._ck(self.L.chd_set_entity_count(self.h, int(n)))

    def assign_cells(self):
        self._ck(self.L.chd_assign_cells(self.h))

    def build(self):
        self._ck(self.L.chd_build(self.h))

    # ---- subscribers / interest
    def set_subscribers(self, conn_id):
        conn_id = np.ascontiguousarray(conn_id, np.uint32)
        self._keep_conn = conn_id
        self._ck(self.L.chd_set_subscribers(self.h, ptr(conn_id), len(conn_id)))
        self.n_slots = len(conn_id)

    def add_subscribers(self, slots, conn_ids):
        slots = np.ascontiguousarray(slots, np.uint32)
        conn_ids = np.ascontiguousarray(conn_ids, np.uint32)
        self._ck(self.L.chd_add_subscribers(self.h, ptr(slots), ptr(conn_ids), len(slots)))
        if len(slots):
            self.n_slots = max(self.n_slots, int(slots.max()) + 1)

    def remove_subscribers(self, slots):
        slots = np.ascontiguousarray(slots, np.uint32)
        self._ck(self.L.chd_remove_subscribers(self.h, ptr(slots), len(slots)))

    def query_channel_ids(self, batch, cap=None):
        """-> (status[n], off[n+1], channel_id[], dist[])"""
        n = batch.n
        cap = int(cap if cap is not None else self.lim.max_pairs)
        status = np.zeros(n, np.uint32)
        off = np.zeros(n + 1, np.uint32)
        ids = np.zeros(cap, np.uint32)
        dist = np.zeros(cap, np.uint32)
        self._ck(self.L.chd_query_channel_ids(self.h, C.byref(batch), ptr(status), ptr(off), ptr(ids), ptr(dist), cap))
        t = int(off[n]) if n else 0
        return status, off, ids[:t].copy(), dist[:t].copy()

    def update_interest(self, batch, now_ns):
        self._ck(self.L.chd_update_interest(self.h, C.byref(batch) if batch is not None else None, int(now_ns)))

    def emit_visible(self):
        self._ck(self.L.chd_emit_visible(self.h))

    def set_rings(self, ring_off, arrival, sender, index, channel_msg_index=None):
        ring_off = np.ascontiguousarray(ring_off, np.uint32)
        arrival = np.ascontiguousarray(arrival, np.int64)
        sender = np.ascontiguousarray(sender, np.uint32)
        index = np.ascontiguousarray(index, np.uint64)
        cmi = None if channel_msg_index is None else np.ascontiguousarray(channel_msg_index, np.uint64)
        self._keep_ring = [ring_off, arrival, sender, index, cmi]
        self._ck(self.L.chd_set_rings(self.h, ptr(ring_off), int(ring_off[-1]), ptr(arrival), ptr(sender), ptr(index), ptr(cmi)))

    def fanout_tick(self, t_ns):
        self._ck(self.L.chd_fanout_tick(self.h, int(t_ns)))

    def summary(self):
        s = TickSummary()
        self._ck(self.L.chd_summary(self.h, C.byref(s)))
        return s

    def begin_interest(self, batch, t_ns, with_fanout=True):
        """batch None = the batch handed over by prefetch_queries + adopt_prefetched."""
        self._ck(self.L.chd_begin_interest(self.h, C.byref(batch) if batch is not None else None, int(t_ns), int(bool(with_fanout))))

    def prefetch_queries(self, batch, keep=None):
        self._keep_pf_q = (batch, keep)
        self._ck(self.L.chd_prefetch_queries(self.h, C.byref(batch)))

    def prefetch_rings(self, ring_off, arrival, sender, index, channel_msg_index=None):
        ring_off = np.ascontiguousarray(ring_off, np.uint32)
        arrival = np.ascontiguousarray(arrival, np.int64)
        sender = np.ascontiguousarray(sender, np.uint32)
        index = np.ascontiguousarray(index, np.uint64)
        cmi = None if channel_msg_index is None else np.ascontiguousarray(channel_msg_index, np.uint64)
        self._keep_pf_ring = [ring_off, arrival, sender, index, cmi]
        self._ck(self.L.chd_prefetch_rings(self.h, ptr(ring_off), int(ring_off[-1]), ptr(arrival), ptr(sender), ptr(index), ptr(cmi)))

    def tick(self, batch, t_ns, flags=capi.TICK_ALL, want_summary=True):
        s = TickSummary() if want_summary else None
        self._ck(self.L.chd_tick(self.h, C.byref(batch) if batch is not None else None, int(t_ns), int(flags),
                                 C.byref(s) if s is not None else None))
        return s

    # ---- results
    def get_cells(self):
        cs = np.zeros(self.n_cells + 1, np.uint32)
        self._ck(self.L.chd_get_cells(self.h, ptr(cs), None))
        se = np.zeros(int(cs[-1]), np.uint32)
        self._ck(self.L.chd_get_cells(self.h, None, ptr(se)))
        return cs, se

    def get_pairs(self, n_pairs=None):
        if n_pairs is None:
            off = np.zeros(self.n_slots + 1, np.uint32)
            self._ck(self.L.chd_get_pairs(self.h, ptr(off), None, None, None, None, None, None))
            n_pairs = int(off[-1])
        P = int(n_pairs)
        off = np.zeros(self.n_slots + 1, np.uint32)
        ch = np.zeros(P, np.uint32); dist = np.zeros(P, np.uint32); iv = np.zeros(P, np.uint32)
        fl = np.zeros(P, np.uint8); last = np.zeros(P, np.int64); li = np.zeros(P, np.uint64)
        self._ck(self.L.chd_get_pairs(self.h, ptr(off), ptr(ch), ptr(dist), ptr(iv), ptr(fl), ptr(last), ptr(li)))
        return dict(off=off, channel=ch, dist=dist, interval=iv, flags=fl, last=last, last_index=li)

    def get_query_status(self, n):
        st = np.zeros(n, np.uint32)
        self._ck(self.L.chd_get_query_status(self.h, ptr(st), n))
        return st

    def get_diff(self, n_new, n_unsub):
        a = np.zeros(n_new, np.uint32); b = np.zeros(n_new, np.uint32)
        c = np.zeros(n_unsub, np.uint32); d = np.zeros(n_unsub, np.uint32)
        self._ck(self.L.chd_get_diff(self.h, ptr(a), ptr(b), ptr(c), ptr(d)))
        return (a, b), (c, d)

    def get_visible(self, n_visible=None):
        off = np.zeros(self.n_slots + 1, np.uint64)
        self._ck(self.L.chd_get_visible(self.h, ptr(off), None))
        V = int(off[-1]) if n_visible is None else int(n_visible)
        ve = np.zeros(V, np.uint32)
        self._ck(self.L.chd_get_visible(self.h, None, ptr(ve)))
        return off, ve

    def get_visible_slot(self, slot, cap=1 << 20):
        out = np.zeros(cap, np.uint32)
        n = C.c_uint64()
        self._ck(self.L.chd_get_visible_slot(self.h, int(slot), ptr(out), cap, C.byref(n)))
        if n.value > cap:
            return self.get_visible_slot(slot, int(n.value))
        return out[:n.value].copy()

    # ---- per-subscriber visibility deltas (chd_visible_delta)
    def enable_visible_delta(self, cap):
        """Allocates the baseline and cap entries for each of the enter / leave lists (call again to grow; the baseline is kept)."""
        self._ck(self.L.chd_visible_delta_enable(self.h, int(cap)))

    def visible_delta(self):
        """Enqueues the delta since the previous call (stream-ordered, no host synchronisation)."""
        self._ck(self.L.chd_visible_delta(self.h))

    def get_visible_delta(self):
        """-> (enter_off[S+1], enter_entity[], leave_off[S+1], leave_entity[]) of the last visible_delta, as numpy arrays.
        Raises ChdError (ERR_CAPACITY) if that call overflowed its capacity."""
        _, n_off = self.device_view(capi.VIEW_ENTER_OFF)
        eo, lo = np.zeros(n_off, np.uint64), np.zeros(n_off, np.uint64)
        ne, nl = C.c_uint64(), C.c_uint64()
        self._ck(self.L.chd_get_visible_delta(self.h, ptr(eo), None, 0, ptr(lo), None, 0, C.byref(ne), C.byref(nl)))
        ee, le = np.zeros(ne.value, np.uint32), np.zeros(nl.value, np.uint32)
        self._ck(self.L.chd_get_visible_delta(self.h, None, ptr(ee), ne.value, None, ptr(le), nl.value, None, None))
        return eo, ee, lo, le

    def get_due(self, n_due):
        out = np.zeros(int(n_due), capi.DUE_DTYPE)
        if n_due:
            self._ck(self.L.chd_get_due(self.h, ptr(out), int(n_due)))
        return out

    def get_handover(self, n):
        a = np.zeros(n, np.uint32); b = np.zeros(n, np.uint32); c = np.zeros(n, np.uint32)
        self._ck(self.L.chd_get_handover(self.h, ptr(a), ptr(b), ptr(c), n))
        return a, b, c

    def due_classes(self, n_due):
        """Window classes of the last fan-out pass -> (class_of[n_due], class_rep[n_classes], class_count[n_classes])."""
        of = np.zeros(n_due, np.uint32)
        rep = np.zeros(max(n_due, 1), np.uint32)
        cnt = np.zeros(max(n_due, 1), np.uint32)
        n = C.c_uint32(0)
        self._ck(self.L.chd_due_classes(self.h, ptr(of), ptr(rep), ptr(cnt), len(rep), C.byref(n)))
        return of, rep[:n.value], cnt[:n.value]

    def set_subscriber_types(self, conn_type):
        if conn_type is None:
            self._ck(self.L.chd_set_subscriber_types(self.h, None, 0))
            return
        t = np.ascontiguousarray(conn_type, np.uint8)
        self._ck(self.L.chd_set_subscriber_types(self.h, ptr(t), len(t)))

    def adjacent_broadcast(self, channel_id, broadcast, sender_conn_id=None, client_conn_id=None, cap=None):
        """BroadcastType_ADJACENT_CHANNELS recipient sets (message.go:188-239) -> (status[n], off[n+1], slot[])."""
        ch = np.ascontiguousarray(channel_id, np.uint32)
        bc = np.ascontiguousarray(broadcast, np.uint32)
        n = len(ch)
        snd = None if sender_conn_id is None else np.ascontiguousarray(sender_conn_id, np.uint32)
        cli = None if client_conn_id is None else np.ascontiguousarray(client_conn_id, np.uint32)
        b = capi.BroadcastBatch()
        b.n, b.channel_id, b.broadcast, b.sender_conn_id, b.client_conn_id = n, ptr(ch), ptr(bc), ptr(snd), ptr(cli)
        cap = int(cap if cap is not None else max(1, 9 * n * max(self.n_slots, 1)))
        cap = min(cap, 1 << 26)
        status, off, slot = np.zeros(n, np.uint32), np.zeros(n + 1, np.uint32), np.zeros(cap, np.uint32)
        self._ck(self.L.chd_adjacent_broadcast(self.h, C.byref(b), ptr(status), ptr(off), ptr(slot), cap))
        return status, off, slot[:off[-1]]

    def device_view(self, which):
        p, n = C.c_void_p(), C.c_uint64()
        self._ck(self.L.chd_device_view(self.h, which, C.byref(p), C.byref(n)))
        return p.value, n.value

    # ---- instrumentation
    def launch_count(self):
        return int(self.L.chd_launch_count(self.h))

    def enable_graphs(self, on=True):
        self._ck(self.L.chd_enable_graphs(self.h, int(bool(on))))

    def graph_launch_count(self):
        return int(self.L.chd_graph_launch_count(self.h))

    def profile_enable(self, on=True):
        """True / 1: every stage; 2: the emit kernel only; False / 0: off."""
        self._ck(self.L.chd_profile_enable(self.h, 2 if on == 2 else int(bool(on))))

    def profile_get(self, stage):
        ms, n = C.c_double(), C.c_uint64()
        self._ck(self.L.chd_profile_get(self.h, int(stage), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def profile_timeline(self, stage):
        a, b = C.c_double(), C.c_double()
        self._ck(self.L.chd_profile_timeline(self.h, int(stage), C.byref(a), C.byref(b)))
        return a.value, b.value

    # ---- multi-GPU: the NCCL exchange behind the C ABI
    @staticmethod
    def comm_unique_id():
        buf = (C.c_uint8 * 128)()
        st = capi.lib().chd_comm_unique_id(buf)
        if st != capi.OK:
            raise ChdError(st, "chd_comm_unique_id failed (libnccl.so.2 missing?)")
        return bytes(buf)

    def comm_init(self, unique_id, rank, world, halo_cols, border_capacity, migrate_subscribers=0, migrate_pairs=0):
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        self._ck(self.L.chd_comm_init(self.h, buf, int(rank), int(world), int(halo_cols), int(border_capacity), int(migrate_subscribers),
                                      int(migrate_pairs)))

    def migrate_out(self, slots):
        slots = np.ascontiguousarray(slots, np.uint32)
        self._ck(self.L.chd_migrate_out(self.h, ptr(slots), len(slots)))

    def migrate_in(self, src_rank, first_index, slots, conn_ids):
        slots = np.ascontiguousarray(slots, np.uint32)
        conn_ids = np.ascontiguousarray(conn_ids, np.uint32)
        self._ck(self.L.chd_migrate_in(self.h, int(src_rank), int(first_index), ptr(slots), ptr(conn_ids), len(slots)))
        if len(slots):
            self.n_slots = max(self.n_slots, int(slots.max()) + 1)

    def get_rehome(self, cap=1 << 20):
        gid, dst, n = np.zeros(cap, np.uint32), np.zeros(cap, np.uint32), C.c_uint32()
        self._ck(self.L.chd_get_rehome(self.h, ptr(gid), ptr(dst), cap, C.byref(n)))
        k = min(n.value, cap)
        return gid[:k].copy(), dst[:k].copy(), n.value

    def comm_info(self):
        r, w, ver = C.c_int(), C.c_int(), C.c_int()
        lo, hi, halo = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self._ck(self.L.chd_comm_info(self.h, C.byref(r), C.byref(w), C.byref(lo), C.byref(hi), C.byref(halo), C.byref(ver)))
        return dict(rank=r.value, world=w.value, col_lo=lo.value, col_hi=hi.value, halo=halo.value, nccl_version=ver.value)

    def tick_sharded(self, batch, t_ns, flags=capi.TICK_ALL, want_summary=True):
        s = TickSummary() if want_summary else None
        self._ck(self.L.chd_tick_sharded(self.h, C.byref(batch) if batch is not None else None, int(t_ns), int(flags),
                                         C.byref(s) if s is not None else None))
        return s

    def collective_count(self):
        return int(self.L.chd_collective_count(self.h))

    def exchange_mode(self):
        """0 no communicator, 1 ncclAllGather per tick, 2 peer windows (stores over NVLink + flags, no collective on the tick path)."""
        return int(self.L.chd_comm_exchange_mode(self.h))

    def use_collective(self, on=True):
        self._ck(self.L.chd_comm_use_collective(self.h, 1 if on else 0))

    # ---- multi-GPU slab
    def set_slab(self, col_lo, col_hi, halo):
        self._ck(self.L.chd_set_slab(self.h, int(col_lo), int(col_hi), int(halo)))

    def export_border(self, d_records, cap_records, want_count=True):
        """want_count=False keeps the call free of host synchronisation (overflow shows up in the next summary)."""
        if not want_count:
            self._ck(self.L.chd_export_border(self.h, ptr(d_records), int(cap_records), None))
            return None
        n = C.c_uint32()
        self._ck(self.L.chd_export_border(self.h, ptr(d_records), int(cap_records), C.byref(n)))
        return n.value

    def import_halo(self, d_records, n_records, skip_first, skip_count):
        self._ck(self.L.chd_import_halo(self.h, ptr(d_records), int(n_records), int(skip_first), int(skip_count)))
