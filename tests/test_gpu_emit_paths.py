"""Every copy path of the expanded visible lists (chd_emit.cuh), and the cell-CSR build, on clustered worlds (tests/_worlds.py).
Everything is compared bit-exact with the CPU oracle: pair offsets, channels and dists, the visible offsets, the WHOLE visible
list and the query statuses.  Each test first asserts with _worlds.emit_plan that its world reaches the branch it targets
(tests/test_worlds.py checks the same on a machine without a GPU).
Run on the B200 box:  python -m pytest tests/test_gpu_emit_paths.py -m gpu
"""
import ctypes as C

import numpy as np
import pytest

from tests import _worlds as W

pytestmark = pytest.mark.gpu

S0 = W.S0
MS = 1_000_000


@pytest.fixture(scope="module")
def chd():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from channeld_b200 import capi, engine

    capi.lib()

    class NS:
        pass

    ns = NS()
    ns.capi, ns.engine = capi, engine
    return ns


def _engine(chd, world, n_max, S, max_visible, max_pairs=1 << 16):
    e = chd.engine.Engine(world.cfg(), n_max, S, max_visible=int(max_visible), max_pairs=int(max_pairs), max_window_cells=1 << 22)
    e.set_subscribers(np.arange(1, S + 1, dtype=np.uint32))
    return e


def _want(oracle, world, q, **kw):
    """(oracle result, emit plan)"""
    w = oracle.sphere_tick(world.og(), world.x, world.z, *q)
    return w, W.emit_plan(world.n, world.cells, w["pair_off"], w["pair_cell"], W.cell_counts(oracle, world), **kw)


def _batch(chd, q):
    S = len(q[0])
    return chd.engine.make_batch(S, sub=np.arange(S, dtype=np.uint32), sphere=q)


def _tick(chd, e, world, q, t, direct=False):
    """direct: chd_tick builds and updates the interest, chd_emit_visible writes the lists; else the overlapped emit of chd_tick"""
    e.set_entities(world.x, world.z)
    batch, keep = _batch(chd, q)
    if direct:
        e.tick(batch, t, chd.capi.TICK_BUILD, want_summary=False)
        e.emit_visible()
        return e.summary()
    return e.tick(batch, t, chd.capi.TICK_BUILD | chd.capi.TICK_EMIT)


def _check(e, s, want, what=""):
    S = len(want["status"])
    assert s.overflow == 0, what
    assert s.n_pairs == len(want["pair_cell"]) and s.n_visible == len(want["vis_entity"]), what
    pairs = e.get_pairs(s.n_pairs)
    np.testing.assert_array_equal(pairs["off"].astype(np.uint64), want["pair_off"], err_msg=what)
    np.testing.assert_array_equal(pairs["channel"], want["pair_cell"], err_msg=what)
    np.testing.assert_array_equal(pairs["dist"], want["pair_dist"], err_msg=what)
    voff, vis = e.get_visible()
    np.testing.assert_array_equal(voff, want["vis_off"], err_msg=what)
    np.testing.assert_array_equal(vis, want["vis_entity"], err_msg=what)
    np.testing.assert_array_equal(e.get_query_status(S), want["status"], err_msg=what)


def _one_tick(chd, oracle, world, q):
    want, plan = _want(oracle, world, q)
    e = _engine(chd, world, world.n, len(q[0]), plan["V"] + 4096, len(want["pair_cell"]) + 1024)
    s = _tick(chd, e, world, q, 33 * MS)
    _check(e, s, want)
    e.close()
    return plan


def test_cta_general_tiles_shared_table(chd, oracle):
    w, (q,) = W.world_general()
    _, plan = _want(oracle, w, q)
    assert plan["kernel"] == "cta" and plan["general_smem"] > 0 and len(plan["phases"]) == 16
    _one_tick(chd, oracle, w, q)


@pytest.mark.parametrize("n", [2_097_152, 2_400_000])  # the build's plain scatter, and its shared-memory scatter (N > 2^21)
def test_cta_general_tiles_per_entry_search(chd, oracle, n):
    w, (q,) = W.world_search(n)
    _, plan = _want(oracle, w, q)
    assert plan["kernel"] == "cta" and plan["general_search"] > 0 and plan["max_general_pairs"] > W.EMIT_SMEM_PAIRS
    _one_tick(chd, oracle, w, q)


def test_warp_path_on_a_clustered_world(chd, oracle):
    w, (q,) = W.world_warp()
    _, plan = _want(oracle, w, q)
    assert plan["kernel"] == "warp" and plan["warp_smem"] > 0 and plan["warp_search"] > 0
    _one_tick(chd, oracle, w, q)


def test_kernel_switch_across_ticks(chd, oracle):
    """warp -> CTA x 3 -> warp -> CTA on one engine.  Ticks 1, 3 and 5 take the overlapped emit on the same pair buffer, so the
    CTA preparation is captured as a graph at tick 3 and replayed at tick 5 while general tiles exist (the general-tile list
    must be emptied by the copy kernel of every tick); ticks 2 and 4 go through chd_emit_visible."""
    worlds, q = W.world_switch()
    wants = [_want(oracle, w, q) for w in worlds]
    assert [p["kernel"] for _, p in wants] == ["warp", "cta", "cta", "cta", "warp", "cta"]
    assert all(p["general_smem"] > 0 for _, p in wants if p["kernel"] == "cta")
    e = _engine(chd, worlds[0], max(w.n for w in worlds), len(q[0]), max(p["V"] for _, p in wants) + 4096)
    for k, (w, (want, plan)) in enumerate(zip(worlds, wants)):
        s = _tick(chd, e, w, q, (k + 1) * 33 * MS, direct=k in (2, 4))
        _check(e, s, want, "tick %d (%s)" % (k, plan["kernel"]))
    e.close()


def test_copy_grid_under_estimate(chd, oracle):
    """The CTA grid is sized from the previous tick's visible count: a tick with eight times that count loops over the tiles the
    grid does not cover, and the next small tick leaves most CTAs without a tile."""
    w, qs = W.world_underestimate()
    wants = [_want(oracle, w, q) for q in qs]
    small, big = wants[0][1], wants[1][1]
    max_visible = big["V"] + 4096
    assert big["V"] >= 8 * small["V"] and big["n_tiles"] > W.cta_grid(small["V"], max_visible)
    assert wants[2][1]["n_tiles"] < W.cta_grid(big["V"], max_visible)
    e = _engine(chd, w, w.n, len(qs[0][0]), max_visible)
    for k, (q, (want, plan)) in enumerate(zip(qs, wants)):
        s = _tick(chd, e, w, q, (k + 1) * 33 * MS)  # (the summary read sets the next grid)
        _check(e, s, want, "tick %d" % k)
    e.close()


def test_visible_overflow_on_the_cta_path(chd, oracle):
    """V >= 2 * max_visible: the tick reports CHD_OVF_VISIBLE with valid offsets and writes no list; the next tick that fits is
    bit-exact on the same engine.  (The partition pass must not describe tiles past the descriptor buffer.)"""
    w, (big, fits) = W.world_overflow()
    mv = W.OVERFLOW_MAX_VISIBLE
    want, plan = _want(oracle, w, big, max_visible=mv)
    assert plan["kernel"] == "cta" and plan["V"] >= 2 * mv and plan["n_tiles"] > plan["desc_capacity"]
    S = len(big[0])
    e = _engine(chd, w, w.n, S, mv)
    e.set_entities(w.x, w.z)
    batch, keep = _batch(chd, big)
    s = chd.capi.TickSummary()
    st = e.L.chd_tick(e.h, C.byref(batch), 33 * MS, chd.capi.TICK_BUILD | chd.capi.TICK_EMIT, C.byref(s))
    assert st == chd.capi.ERR_CAPACITY
    assert s.overflow == chd.capi.OVF_VISIBLE and s.required_visible == s.n_visible == plan["V"]
    voff = np.zeros(S + 1, np.uint64)
    e._ck(e.L.chd_get_visible(e.h, chd.capi.ptr(voff), None))
    np.testing.assert_array_equal(voff, want["vis_off"])
    pairs = e.get_pairs(s.n_pairs)
    np.testing.assert_array_equal(pairs["channel"], want["pair_cell"])
    want2, plan2 = _want(oracle, w, fits, max_visible=mv)
    assert plan2["kernel"] == "cta" and 0 < plan2["V"] <= mv
    s2 = _tick(chd, e, w, fits, 66 * MS)
    _check(e, s2, want2, "the tick after the overflow")
    e.close()


@pytest.mark.parametrize("case", W.EDGE_CASES)
def test_cta_edge_shapes(chd, oracle, case):
    """V = 0; V = 3 * 4096 exactly and + 1, 2, 3 (a last tile of 1-3 entries); a last tile that ends in a run of empty pairs;
    failing queries (no pairs) between working ones."""
    w = W.edge_world()
    q = W.edge_queries(w, case)
    _, plan = _want(oracle, w, q)
    assert plan["kernel"] == "cta"
    if W.edge_expected_v(case) is not None:
        assert plan["V"] == W.edge_expected_v(case)
    if case == "trailing_empty":
        assert plan["trailing_empty"] >= 16
    _one_tick(chd, oracle, w, q)


# ----------------------------------------------------------------- the cell-CSR build under skew

def _skewed(case, cols, rows, n, seed):
    C_ = cols * rows
    counts = np.zeros(C_, np.int64)
    n_out = 0
    if case == "one_cell":
        counts[C_ // 2 + 7] = n
    elif case == "last_cell_and_out":  # out-of-world entities sort after the last cell (key C)
        n_out = n // 10
        counts[C_ - 1] = n - n_out
    elif case == "all_out_but_one":
        n_out = n - 1
        counts[5] = 1
    else:  # lognormal cell sizes, a third of the cells empty
        rng = np.random.default_rng(seed)
        p = np.exp(rng.normal(0.0, 2.0, C_)) * (rng.uniform(size=C_) > 0.33)
        counts = rng.multinomial(n, p / p.sum())
    return W.clustered(cols, rows, counts, seed, n_out=n_out)


def _check_cells(e, s, oracle, world, what):
    ids = oracle.cell_of(world.og(), world.x, world.z)
    valid = np.nonzero(ids)[0]
    order = valid[np.argsort(ids[valid], kind="stable")]
    cs, se = e.get_cells()
    np.testing.assert_array_equal(cs, np.concatenate([[0], np.cumsum(np.bincount(ids[valid] - S0, minlength=world.cells))]), err_msg=what)
    np.testing.assert_array_equal(se, order.astype(np.uint32), err_msg=what)
    assert s.n_entities_in_world == len(valid), what
    return ids


@pytest.mark.parametrize("n", [1_000_003, 2_200_001])  # the build's plain scatter, and its shared-memory scatter (N > 2^21)
@pytest.mark.parametrize("grid", [(32, 31), (256, 256)])  # 992 cells: one radix pass; 65536 cells: two
@pytest.mark.parametrize("case", ["one_cell", "last_cell_and_out", "all_out_but_one", "lognormal"])
def test_build_under_skew(chd, oracle, case, grid, n):
    """The complete cell CSR against a stable sort of the oracle's cell ids; then a seeded 30 % of the entities jumps into cell 0
    and the handover list must be exactly the entities whose cell changed."""
    cols, rows = grid
    w = _skewed(case, cols, rows, n, 60 + cols)
    e = chd.engine.Engine(w.cfg(), n, 1)
    e.set_entities(w.x, w.z)
    s = e.tick(None, MS, chd.capi.TICK_BUILD)
    prev = _check_cells(e, s, oracle, w, "%s first build" % case)
    rng = np.random.default_rng(7)
    crowd = rng.uniform(size=n) < 0.3
    w.x = np.where(crowd, w.offx + rng.uniform(0.1, 0.9, n) * w.w, w.x)
    w.z = np.where(crowd, w.offz + rng.uniform(0.1, 0.9, n) * w.h, w.z)
    e.set_entities(w.x, w.z)
    s = e.tick(None, 2 * MS, chd.capi.TICK_BUILD)
    ids = _check_cells(e, s, oracle, w, "%s after the move" % case)
    moved = np.nonzero(prev != ids)[0]
    assert s.n_handover == len(moved) > 0
    he, hs, hd = e.get_handover(s.n_handover)
    order = np.argsort(he)
    np.testing.assert_array_equal(he[order], moved.astype(np.uint32))
    np.testing.assert_array_equal(hs[order], prev[moved])
    np.testing.assert_array_equal(hd[order], ids[moved])
    e.close()
