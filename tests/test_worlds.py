"""CPU checks of tests/_worlds.py: emit_plan() on hand-built pair lists with known answers, and, for every world of
tests/test_gpu_emit_paths.py, that the oracle's pairs reach the kernel branch the GPU test targets (so that a later change of a
threshold cannot quietly turn one of those tests into a duplicate of another)."""
import numpy as np
import pytest

from tests import _worlds as W

S0 = W.S0
N_CTA = 600_000  # 16 x 16 cells: 2343 per cell, the CTA path


def _plan(counts, pair_cells, n_own=N_CTA, cells=256, **kw):
    """one subscriber whose pairs are cells `pair_cells` (in order)"""
    counts = np.asarray(counts, np.int64)
    pc = np.asarray(pair_cells, np.int64) + S0
    return W.emit_plan(n_own, cells, np.array([0, len(pc)]), pc, counts, **kw)


def test_kernel_choice_follows_the_average_density():
    assert W.emit_uses_cta_tiles(2048 * 256, 256) and not W.emit_uses_cta_tiles(2048 * 256 - 1, 256)
    assert W.emit_uses_cta_tiles(4 << 20, 1024) and not W.emit_uses_cta_tiles((4 << 20) + 1, 1024)


def test_two_segments_make_a_simple_tile():
    counts = np.zeros(256, np.int64)
    counts[:2] = [3000, 1096]  # exactly one tile: the second segment ends it
    p = _plan(counts, [0, 1])
    assert (p["kernel"], p["n_tiles"], p["simple"], p["simple_two"], p["general_smem"], p["general_search"]) == ("cta", 1, 1, 1, 0, 0)
    assert p["phases"] == [(0, 0)]  # end0 = 3000; the second cell starts at 3000 in the CSR: (3000 - 3000) & 3
    counts[0], counts[2] = 3001, 2000
    assert _plan(counts, [0, 1])["phases"] == [(1, 0)]
    p = _plan(counts, [0, 2])  # cell 1 (1096 entities) is skipped: the second segment starts at 4097 in the CSR
    assert p["phases"] == [(1, (3001 - 4097) & 3)]
    counts[1] = 5000  # the second segment runs past the tile: still simple, and the next tile holds one segment
    p = _plan(counts, [0, 1])
    assert (p["n_tiles"], p["simple"], p["simple_two"], p["general_smem"]) == (2, 2, 1, 0)


def test_three_segments_make_a_general_tile():
    counts = np.zeros(256, np.int64)
    counts[:3] = [3000, 500, 4000]
    p = _plan(counts, [0, 1, 2])
    assert (p["n_tiles"], p["simple"], p["general_smem"], p["general_search"], p["max_general_pairs"]) == (2, 1, 1, 0, 3)


def test_257_empty_pairs_make_a_per_entry_tile():
    counts = np.zeros(1024, np.int64)
    counts[0], counts[500], counts[501] = 2000, 1, 4000  # three segments in the first tile, empty cells 1..499 between
    for k, branch in ((254, "general_search"), (253, "general_smem")):  # the tile's pairs: 2000, k empty, 1, 4000 (the next tile's first)
        p = _plan(counts, np.r_[0, 1:k + 1, 500, 501], n_own=1024 * 2048, cells=1024)
        assert p["kernel"] == "cta" and p[branch] == 1 and p["max_general_pairs"] == k + 3
        assert p["general_smem"] + p["general_search"] == 1 and p["simple"] == 1
    # empty pairs alone do not make a tile general: the partition skips them
    p = _plan(counts, np.r_[0, 1:300, 501], n_own=1024 * 2048, cells=1024)
    assert p["general_smem"] + p["general_search"] == 0 and p["simple_two"] == 1


def test_trailing_empty_pairs_count_in_the_last_tile():
    counts = np.zeros(256, np.int64)
    counts[:2] = [4096, 100]
    p = _plan(counts, np.arange(40))  # cells 2..39 are empty
    assert p["trailing_empty"] == 38 and p["n_tiles"] == 2
    # tile 1 holds 100 entries of pair 1 and then the 38 empty pairs: 39 pairs, one segment
    assert p["simple"] == 2 and p["general_smem"] == 0


def test_warp_tiles():
    counts = np.zeros(256, np.int64)
    counts[:70] = 1  # 70 one-entry pairs share one 1024-entry tile
    counts[70] = 5000
    p = _plan(counts, np.arange(71), n_own=1000)
    assert p["kernel"] == "warp" and p["n_tiles"] == 5 and p["warp_search"] == 1 and p["warp_smem"] == 4


def test_grid_from_the_last_visible_count():
    assert W.cta_grid(0, 1 << 20) == 256
    assert W.cta_grid(4096 * 100, 1 << 30) == (4096 * 100 + 4096 * 100 // 32) // 4096 + 64
    assert W.cta_grid(1 << 30, 1 << 20) == 256


# ----------------------------------------------------------------- the GPU tests' worlds reach their branches

def _oracle_plan(oracle, world, q, **kw):
    r = oracle.sphere_tick(world.og(), world.x, world.z, *q)
    return W.emit_plan(world.n, world.cells, r["pair_off"], r["pair_cell"], W.cell_counts(oracle, world), **kw), r


def test_world_general(oracle):
    w, (q,) = W.world_general()
    p, r = _oracle_plan(oracle, w, q)
    assert w.n // w.cells >= 2048 and p["kernel"] == "cta"
    assert p["general_smem"] > 0 and len(p["phases"]) == 16
    assert p["V"] < 30_000_000 and (r["status"] == 0).all()


@pytest.mark.parametrize("n", [2_097_152, 2_400_000])
def test_world_search(oracle, n):
    w, (q,) = W.world_search(n)
    p, _ = _oracle_plan(oracle, w, q)
    assert w.n == n and p["kernel"] == "cta" and p["general_search"] > 0 and p["max_general_pairs"] > 256
    assert p["V"] < 30_000_000


def test_world_warp(oracle):
    w, (q,) = W.world_warp()
    p, _ = _oracle_plan(oracle, w, q)
    assert p["kernel"] == "warp" and p["warp_smem"] > 0 and p["warp_search"] > 0


def test_world_switch(oracle):
    worlds, q = W.world_switch()
    plans = [_oracle_plan(oracle, w, q)[0] for w in worlds]
    assert [p["kernel"] for p in plans] == ["warp", "cta", "cta", "cta", "warp", "cta"]
    assert all(p["general_smem"] > 0 for p in plans if p["kernel"] == "cta")


def test_world_underestimate(oracle):
    w, qs = W.world_underestimate()
    small, big, small2 = (_oracle_plan(oracle, w, q)[0] for q in qs)
    assert small["kernel"] == big["kernel"] == "cta"
    assert big["V"] >= 8 * small["V"] > 0
    max_visible = big["V"] + 4096
    assert big["n_tiles"] > W.cta_grid(small["V"], max_visible)  # the copy kernel loops
    assert small2["n_tiles"] < W.cta_grid(big["V"], max_visible)  # surplus CTAs exit


def test_world_overflow(oracle):
    w, (big, fits) = W.world_overflow()
    mv = W.OVERFLOW_MAX_VISIBLE
    p, _ = _oracle_plan(oracle, w, big, max_visible=mv)
    assert p["kernel"] == "cta" and p["V"] >= 2 * mv
    assert p["n_tiles"] > p["desc_capacity"]  # tiles below V do not fit the descriptor buffer
    f, _ = _oracle_plan(oracle, w, fits, max_visible=mv)
    assert 0 < f["V"] <= mv and f["kernel"] == "cta"


@pytest.mark.parametrize("case", W.EDGE_CASES)
def test_edge_world(oracle, case):
    w = W.edge_world()
    p, r = _oracle_plan(oracle, w, W.edge_queries(w, case))
    assert p["kernel"] == "cta"
    if W.edge_expected_v(case) is not None:
        assert p["V"] == W.edge_expected_v(case)
    if case == "failing":
        assert r["status"][[1, 3, 5]].all() and not r["status"][[0, 2, 4, 6, 7]].any()
        assert p["V"] > 0
    else:
        assert (r["status"] == 0).all()
    if case == "trailing_empty":
        assert p["trailing_empty"] >= 16
