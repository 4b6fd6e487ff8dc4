"""Per-subscriber visibility deltas (chd_visible_delta) against set differences of ORACLE visible lists at consecutive states.
The expected lists are never taken from the engine's own chd_get_visible: they come from tests/_oracle.py (sphere_tick), put into
the canonical order (enter: current cell asc, entity asc; leave: baseline cell asc, entity asc; per slot).
Run on the B200 box:  python -m pytest tests/test_gpu_visible_delta.py -m gpu
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

S0 = 65536
MS = 1_000_000


@pytest.fixture(scope="module")
def chd():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from channeld_b200 import capi, engine, synth

    capi.lib()

    class NS:
        pass

    ns = NS()
    ns.capi, ns.engine, ns.synth = capi, engine, synth
    return ns


def _og(wc):
    from tests._oracle import make_grid

    return make_grid(wc.offx, wc.offz, wc.w, wc.h, wc.cols, wc.rows, wc.server_cols, wc.server_rows)


def _keys(off, ent):
    """(slot << 32 | entity) per visible entry, slot-major: the oracle's lists are already in (cell asc, entity asc) order."""
    off = np.asarray(off, np.int64)
    slot = np.repeat(np.arange(len(off) - 1, dtype=np.uint64), np.diff(off))
    return (slot << np.uint64(32)) | np.asarray(ent, np.uint64)


def _oracle_keys(oracle, wc, ex, ez, cx, cz, r):
    """Oracle visible lists as keys, and the oracle's whole result."""
    w = oracle.sphere_tick(_og(wc), ex, ez, cx, cz, r)
    return _keys(w["vis_off"], w["vis_entity"]), w


def _expected(now, base, S):
    """enter = now \\ base, leave = base \\ now, each in its own state's order, as CSRs over S slots."""
    def csr(k):
        slot = (k >> np.uint64(32)).astype(np.int64)
        off = np.zeros(S + 1, np.uint64)
        off[1:] = np.cumsum(np.bincount(slot, minlength=S)[:S])
        return off, (k & np.uint64(0xFFFFFFFF)).astype(np.uint32)

    eo, ee = csr(now[~np.isin(now, base)])
    lo, le = csr(base[~np.isin(base, now)])
    return eo, ee, lo, le


def _check(got, want, what=""):
    for g, w, name in zip(got, want, ("enter_off", "enter", "leave_off", "leave")):
        np.testing.assert_array_equal(g, w, err_msg="%s %s" % (what, name))


def _engine(chd, wc, n_max, S, cap, **kw):
    e = chd.engine.Engine(wc.cfg(), n_max, S, **kw)
    e.set_subscribers(np.arange(1, S + 1, dtype=np.uint32))
    e.enable_visible_delta(cap)
    return e


def _tick(chd, e, ex, ez, cx, cz, r, t, emit=False, sub=None):
    e.set_entities(ex, ez)
    S = len(cx)
    batch, keep = chd.engine.make_batch(S, sub=np.arange(S, dtype=np.uint32) if sub is None else sub, sphere=(cx, cz, r))
    flags = chd.capi.TICK_BUILD | chd.capi.TICK_FANOUT | (chd.capi.TICK_EMIT if emit else 0)
    return e.tick(batch, t, flags)


def _follow(wc, ex, ez, S):
    """queries that follow their pawns: subscriber j stands on entity j * (N // S)"""
    N = len(ex)
    idx = (np.arange(S, dtype=np.int64) * max(N // S, 1)) % N
    return ex[idx].copy(), ez[idx].copy(), np.full(S, wc.radius)


def _world(chd, name, n, s):
    wc = chd.synth.scaled(chd.synth.CONFIGS[name], n, s)
    ex, ez = chd.synth.entities(wc)
    return wc, ex, ez


def test_first_call_is_the_whole_view(chd, oracle):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    cx, cz, r = _follow(wc, ex, ez, S)
    now, w = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
    e = _engine(chd, wc, len(ex), S, len(now) + 16)
    _tick(chd, e, ex, ez, cx, cz, r, MS)
    e.visible_delta()
    eo, ee, lo, le = e.get_visible_delta()
    np.testing.assert_array_equal(eo, w["vis_off"])
    np.testing.assert_array_equal(ee, w["vis_entity"])
    assert len(le) == 0 and not lo.any()
    e.close()


def _pair_keys(w):
    """(slot << 32 | channel id) of every oracle subscription"""
    off = w["pair_off"].astype(np.int64)
    slot = np.repeat(np.arange(len(off) - 1, dtype=np.uint64), np.diff(off))
    return (slot << np.uint64(32)) | w["pair_cell"].astype(np.uint64)


def _pair_kinds(prev, cur):
    """(new cells, dropped cells) over all slots between two oracle states"""
    a, b = _pair_keys(prev), _pair_keys(cur)
    return int((~np.isin(b, a)).sum()), int((~np.isin(a, b)).sum())


def test_six_ticks_match_oracle_differences(chd, oracle):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    e = _engine(chd, wc, len(ex), S, 1 << 22)
    base = np.zeros(0, np.uint64)
    prev_w = None
    og = _og(wc)
    new_cells = dropped = kept_movers = 0
    for tick in range(6):
        if tick:
            ex, ez = chd.synth.move_entities(wc, ex, ez, tick, 400.0)
        cx, cz, r = _follow(wc, ex, ez, S)
        now, w = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
        assert (w["status"] == 0).all()
        _tick(chd, e, ex, ez, cx, cz, r, (tick + 1) * 33 * MS)
        e.visible_delta()
        got = e.get_visible_delta()
        _check(got, _expected(now, base, S), "tick %d" % tick)
        if prev_w is not None:
            n, d = _pair_kinds(prev_w, w)
            new_cells += n
            dropped += d
            # enter entries whose current cell the slot was already subscribed to: movers into a kept cell
            slot = np.repeat(np.arange(S, dtype=np.uint64), np.diff(got[0].astype(np.int64)))
            cell = oracle.cell_of(og, ex, ez)[got[1]].astype(np.uint64)
            kept_movers += int(np.isin((slot << np.uint64(32)) | cell, _pair_keys(prev_w)).sum())
        base, prev_w = now, w
    assert new_cells > 0 and dropped > 0 and kept_movers > 0, (new_cells, dropped, kept_movers)
    e.close()


def test_every_other_tick_spans_two_ticks(chd, oracle):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    e = _engine(chd, wc, len(ex), S, 1 << 22)
    base = np.zeros(0, np.uint64)
    keys = []
    back_and_forth = 0
    for tick in range(6):
        if tick:
            ex, ez = chd.synth.move_entities(wc, ex, ez, tick, 400.0)
        cx, cz, r = _follow(wc, ex, ez, S)
        now, _ = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
        keys.append(now)
        _tick(chd, e, ex, ez, cx, cz, r, (tick + 1) * 33 * MS)
        if tick % 2 == 0:
            e.visible_delta()
            _check(e.get_visible_delta(), _expected(now, base, S), "tick %d" % tick)
            if tick:  # entries that left at tick-1 and came back at tick: in neither list
                mid = keys[-2]
                back_and_forth += int(np.isin(base[~np.isin(base, mid)], now).sum())
            base = now
    assert back_and_forth > 0
    e.close()


def test_entities_leave_and_enter_the_world_and_n_changes(chd, oracle):
    wc, ex0, ez0 = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    e = _engine(chd, wc, 40_000, S, 1 << 22)
    base = np.zeros(0, np.uint64)
    x_hi = wc.offx + wc.w * wc.cols
    for step, n in enumerate([30_000, 24_000, 36_000, 36_000, 28_000]):
        wc2 = chd.synth.scaled(wc, n, S)
        ex, ez = chd.synth.entities(wc2)
        ex, ez = chd.synth.move_entities(wc2, ex, ez, step, 300.0)
        out = np.arange(n) % (97 + step) == 0  # a different set leaves the world every step
        ex = np.where(out, x_hi + 5.0, ex)
        cx, cz, r = _follow(wc, ex0, ez0, S)  # fixed queries: the view changes only through the entities
        now, w = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
        _tick(chd, e, ex, ez, cx, cz, r, (step + 1) * 33 * MS)
        e.visible_delta()
        _check(e.get_visible_delta(), _expected(now, base, S), "step %d n=%d" % (step, n))
        base = now
    e.close()


def test_removed_subscribers_and_failing_queries(chd, oracle):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    e = _engine(chd, wc, len(ex), S, 1 << 22)
    cx, cz, r = _follow(wc, ex, ez, S)
    base, w = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
    _tick(chd, e, ex, ez, cx, cz, r, MS)
    e.visible_delta()
    e.get_visible_delta()
    # a failing query (centre out of the world) keeps the slot's subscriptions: no delta for that slot; the others move
    cx2, cz2 = cx + 900.0, cz.copy()
    cx2[::7] = wc.offx - 10.0
    now, w2 = _oracle_keys(oracle, wc, ex, ez, cx2, cz2, r)
    bad = np.nonzero(w2["status"])[0]
    assert set(range(0, S, 7)) <= set(bad.tolist())
    now = now[~np.isin((now >> np.uint64(32)).astype(np.int64), bad)]
    kept = base[np.isin((base >> np.uint64(32)).astype(np.int64), bad)]  # same positions: the kept view is unchanged
    both = np.concatenate([now, kept])
    now = both[np.argsort(both >> np.uint64(32), kind="stable")]  # slot-major again, each slot's own order untouched
    _tick(chd, e, ex, ez, cx2, cz2, r, 2 * MS)
    e.visible_delta()
    got = e.get_visible_delta()
    _check(got, _expected(now, base, S), "failing queries")
    assert all(got[0][s] == got[0][s + 1] and got[2][s] == got[2][s + 1] for s in bad)
    base = now
    # chd_remove_subscribers: the removed slots' whole views leave (applied by the next interest update; an empty batch will do)
    gone = np.array([1, 5, 100, S - 1], np.uint32)
    e.remove_subscribers(gone)
    empty, keep = chd.engine.make_batch(0, sub=np.zeros(0, np.uint32), sphere=(np.zeros(0), np.zeros(0), np.zeros(0)))
    e.tick(empty, 3 * MS, chd.capi.TICK_BUILD | chd.capi.TICK_FANOUT)
    e.visible_delta()
    now = base[~np.isin((base >> np.uint64(32)).astype(np.int64), gone)]
    got = e.get_visible_delta()
    _check(got, _expected(now, base, S), "remove")
    assert len(got[3]) > 0 and len(got[1]) == 0
    base = now
    # chd_set_subscribers resets every slot: everything leaves
    e.set_subscribers(np.arange(1, S + 1, dtype=np.uint32))
    e.visible_delta()
    _check(e.get_visible_delta(), _expected(np.zeros(0, np.uint64), base, S), "set_subscribers")
    e.close()


def test_emit_does_not_change_the_delta(chd):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    out = {}
    for emit in (False, True):
        e = _engine(chd, wc, len(ex), S, 1 << 22, max_visible=1 << 23)
        x, z = ex, ez
        res = []
        for tick in range(3):
            if tick:
                x, z = chd.synth.move_entities(wc, x, z, tick, 400.0)
            cx, cz, r = _follow(wc, x, z, S)
            _tick(chd, e, x, z, cx, cz, r, (tick + 1) * 33 * MS, emit=emit)
            e.visible_delta()
            res.append(e.get_visible_delta())
        out[emit] = res
        e.close()
    for a, b in zip(out[False], out[True]):
        _check(a, b, "emit")


def test_overflow_is_transactional(chd, oracle):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    empty = np.zeros(0, np.uint64)
    cx, cz, r = _follow(wc, ex, ez, S)
    first, _ = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
    e = _engine(chd, wc, len(ex), S, len(first) // 2)
    L, ne, nl = e.L, C.c_uint64(), C.c_uint64()
    _tick(chd, e, ex, ez, cx, cz, r, MS)
    e.visible_delta()
    eo = np.zeros(S + 1, np.uint64)
    assert L.chd_get_visible_delta(e.h, chd.capi.ptr(eo), None, 0, None, None, 0, C.byref(ne), C.byref(nl)) == chd.capi.ERR_CAPACITY
    assert (ne.value, nl.value) == (len(first), 0)
    np.testing.assert_array_equal(eo, _expected(first, empty, S)[0])  # the offsets are valid
    s = e.summary()
    assert s.overflow == 0
    # the baseline did not advance: the next delta is still taken against the empty baseline
    x2, z2 = chd.synth.move_entities(wc, ex, ez, 1, 400.0)
    cx2, cz2, r2 = _follow(wc, x2, z2, S)
    mid, _ = _oracle_keys(oracle, wc, x2, z2, cx2, cz2, r2)
    s2 = _tick(chd, e, x2, z2, cx2, cz2, r2, 2 * MS)
    assert s2.overflow == 0
    e.visible_delta()
    assert L.chd_get_visible_delta(e.h, None, None, 0, None, None, 0, C.byref(ne), C.byref(nl)) == chd.capi.ERR_CAPACITY
    assert (ne.value, nl.value) == (len(mid), 0)
    # grow to the required size and call again: the whole delta since the old baseline
    e.enable_visible_delta(ne.value)
    e.visible_delta()
    _check(e.get_visible_delta(), _expected(mid, empty, S), "after re-enable")
    assert e.summary().as_dict() == s2.as_dict()
    # and from now on the baseline moves again
    x3, z3 = chd.synth.move_entities(wc, x2, z2, 2, 400.0)
    cx3, cz3, r3 = _follow(wc, x3, z3, S)
    now, _ = _oracle_keys(oracle, wc, x3, z3, cx3, cz3, r3)
    _tick(chd, e, x3, z3, cx3, cz3, r3, 3 * MS)
    e.visible_delta()
    _check(e.get_visible_delta(), _expected(now, mid, S), "warm")
    e.close()


def test_handover_shape(chd, oracle):
    """256 x 256 cells of 100 x 100, half of the entities jump one cell (SURVEY §8d #5) at 400 000 / 4 000"""
    wc, ex, ez = _world(chd, "handover", 400_000, 4_000)
    S, N = wc.n_subscribers, len(ex)
    og = _og(wc)
    e = _engine(chd, wc, N, S, 1 << 22)
    base = np.zeros(0, np.uint64)
    for tick in range(3):
        if tick:
            i = np.arange(N, dtype=np.uint64)
            jump = chd.synth.uniform(wc.seed + 50 + tick, i, 0) < 0.5
            axis = chd.synth.uniform(wc.seed + 51 + tick, i, 0) < 0.5
            sign = np.where(chd.synth.uniform(wc.seed + 52 + tick, i, 0) < 0.5, -1.0, 1.0)
            ex = np.where(jump & axis, ex + sign * wc.w, ex)
            ez = np.where(jump & ~axis, ez + sign * wc.h, ez)
        cx, cz, r = _follow(wc, ex, ez, S)
        if tick:  # a pawn that jumped out of the world keeps its query where it was (a failing query keeps its subscriptions)
            out = oracle.cell_of(og, cx, cz) == 0
            cx, cz = np.where(out, px, cx), np.where(out, pz, cz)
        px, pz = cx, cz
        now, w = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
        assert (w["status"] == 0).all()
        _tick(chd, e, ex, ez, cx, cz, r, (tick + 1) * 33 * MS)
        e.visible_delta()
        _check(e.get_visible_delta(), _expected(now, base, S), "tick %d" % tick)
        base = now
    e.close()


@pytest.mark.parametrize("name", ["benchmark", "handover"])  # 225 cells (one radix pass per mover sort) and 65536 (two)
def test_moving_crowd_with_a_large_entity_capacity(chd, oracle, name):
    """A crowd of 80 % of the entities, spread over 2 x 2 cells, moves one cell along x per tick for 4 ticks: most movers share a
    few destination (and source) cells.  max_entities > 2^21, so the mover sorts take the build's shared-memory scatter."""
    N, S = 100_000, 128
    wc, ex, ez = _world(chd, name, N, S)
    rng = np.random.default_rng(3)
    crowd = rng.uniform(size=N) < 0.8
    ex = np.where(crowd, wc.offx + (3.0 + rng.uniform(0.01, 1.99, N)) * wc.w, ex)
    ez = np.where(crowd, wc.offz + (3.0 + rng.uniform(0.01, 1.99, N)) * wc.h, ez)
    e = _engine(chd, wc, (2 << 20) + 4099, S, 1 << 23)
    base = np.zeros(0, np.uint64)
    for tick in range(5):
        if tick:
            ex = np.where(crowd, ex + wc.w, ex)
        cx, cz, r = _follow(wc, ex, ez, S)
        now, w = _oracle_keys(oracle, wc, ex, ez, cx, cz, r)
        assert (w["status"] == 0).all()
        _tick(chd, e, ex, ez, cx, cz, r, (tick + 1) * 33 * MS)
        e.visible_delta()
        got = e.get_visible_delta()
        _check(got, _expected(now, base, S), "tick %d" % tick)
        if tick:
            assert len(got[1]) > 0 and len(got[3]) > 0
        base = now
    e.close()


def test_enabled_delta_changes_no_other_result(chd):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    res = {}
    for on in (False, True):
        e = chd.engine.Engine(wc.cfg(), len(ex), S, max_visible=1 << 23)
        e.set_subscribers(np.arange(1, S + 1, dtype=np.uint32))
        if on:
            e.enable_visible_delta(1 << 22)
        x, z = ex, ez
        out = []
        for tick in range(3):
            if tick:
                x, z = chd.synth.move_entities(wc, x, z, tick, 400.0)
            cx, cz, r = _follow(wc, x, z, S)
            ring = chd.synth.update_rings(wc, tick, (tick + 1) * 33 * MS, 33 * MS, 4, S)
            e.set_rings(*ring[1:])
            e.set_entities(x, z)
            batch, keep = chd.engine.make_batch(S, sub=np.arange(S, dtype=np.uint32), sphere=(cx, cz, r))
            s = e.tick(batch, (tick + 1) * 33 * MS, chd.capi.TICK_ALL)
            if on:
                e.visible_delta()
                e.get_visible_delta()
            p = e.get_pairs(s.n_pairs)
            voff, vis = e.get_visible()
            due = np.sort(e.get_due(s.n_due), order=["sub", "channel_id", "window_hi"])  # SETs: canonical order
            ho = np.stack(e.get_handover(s.n_handover), 1)
            ho = ho[np.argsort(ho[:, 0])]
            out.append((s.as_dict(), p, voff, vis, due, ho))
        res[on] = out
        e.close()
    for a, b in zip(res[False], res[True]):
        assert a[0] == b[0]
        for k in a[1]:
            np.testing.assert_array_equal(a[1][k], b[1][k])
        for x, y in zip(a[2:], b[2:]):
            np.testing.assert_array_equal(x, y)
    assert sum(r[0]["n_due"] for r in res[True]) > 0 and sum(r[0]["n_handover"] for r in res[True]) > 0


def test_slab_engine_is_refused(chd):
    wc, ex, ez = _world(chd, "benchmark", 30_000, 3_000)
    S = wc.n_subscribers
    e = _engine(chd, wc, len(ex), S, 1 << 20)
    cx, cz, r = _follow(wc, ex, ez, S)
    _tick(chd, e, ex, ez, cx, cz, r, MS)
    e.visible_delta()
    e.set_slab(0, wc.cols, 1)
    with pytest.raises(chd.capi.ChdError) as ei:
        e.visible_delta()
    assert ei.value.status == chd.capi.ERR_STATE
    e.close()
