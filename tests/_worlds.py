"""Clustered test worlds, and a numpy mirror of how the emit stage cuts the visible lists into tiles.  Test infrastructure
only: nothing under channeld_b200/ may import this module.

A game world is not uniform: towns, crowds and empty sea.  The emit stage picks its copy kernel from the AVERAGE density
(chd_tick.cu emit_uses_cta_tiles), so a clustered world sends tiny and empty cells through the CTA-tile kernels, which is
what their general branches exist for.  emit_plan() says which kernel and which branch every tile takes, so that each GPU
test can assert that its world reaches the branch it targets.
"""
from dataclasses import dataclass

import numpy as np

from channeld_b200.engine import SPATIAL_CHANNEL_ID_START, grid_cfg
from tests._oracle import make_grid

S0 = SPATIAL_CHANNEL_ID_START

# chd_types.cuh / chd_tick.cu
EMIT_TILE = 4096            # CTA tile (entries)
EMIT_SMEM_PAIRS = 256       # pairs of a general CTA tile held in shared memory
EMIT_WARP_TILE = 1024       # warp tile (entries)
EMIT_WARP_SMEM_PAIRS = 64   # pairs of a warp tile held in shared memory
CTA_MIN_PER_CELL = EMIT_TILE // 2
CTA_MAX_BUILD_BYTES = 64 << 20  # 16 bytes per built entity: the four phase copies of the cell CSR stay L2-resident


@dataclass
class World:
    cols: int
    rows: int
    w: float
    h: float
    offx: float
    offz: float
    x: np.ndarray
    z: np.ndarray

    @property
    def cells(self):
        return self.cols * self.rows

    @property
    def n(self):
        return len(self.x)

    def cfg(self):
        return grid_cfg(self.offx, self.offz, self.w, self.h, self.cols, self.rows)

    def og(self):
        return make_grid(self.offx, self.offz, self.w, self.h, self.cols, self.rows)

    def centre(self, cell):
        """centre of cell index `cell` (index = col + row * cols, the channel order)"""
        cell = np.asarray(cell)
        return self.offx + (cell % self.cols + 0.5) * self.w, self.offz + (cell // self.cols + 0.5) * self.h

    def whole(self):
        """(cx, cz, r) of a sphere that covers every cell"""
        W, H = self.cols * self.w, self.rows * self.h
        return self.offx + W / 2, self.offz + H / 2, 0.55 * float(np.hypot(W, H))


def clustered(cols, rows, counts, seed, w=100.0, h=100.0, n_out=0):
    """Seeded world with counts[c] entities uniform inside cell c (c = col + row * cols), plus n_out entities outside the world.
    Entity ids (array positions) are shuffled, so the build's sort really reorders them."""
    counts = np.asarray(counts, np.int64)
    assert counts.shape == (cols * rows,) and (counts >= 0).all()
    rng = np.random.default_rng(seed)
    offx, offz = -cols * w / 2, -rows * h / 2
    cell = np.repeat(np.arange(cols * rows), counts)
    # (inside the cell with a margin: the cell of a position is exact, no rounding at a border)
    x = offx + (cell % cols + rng.uniform(0.02, 0.98, len(cell))) * w
    z = offz + (cell // cols + rng.uniform(0.02, 0.98, len(cell))) * h
    if n_out:
        x = np.concatenate([x, offx + cols * w + rng.uniform(1.0, 50.0, n_out)])
        z = np.concatenate([z, offz + rng.uniform(0.0, rows * h, n_out)])
    perm = rng.permutation(len(x))
    return World(cols, rows, float(w), float(h), offx, offz, x[perm], z[perm])


def band_counts(cols, rows, bands, seed):
    """Per-cell counts by row band: bands = [(first_row, end_row, lo, hi)], counts uniform in [lo, hi]; rows in no band are empty."""
    rng = np.random.default_rng(seed)
    counts = np.zeros(cols * rows, np.int64)
    for r0, r1, lo, hi in bands:
        counts[r0 * cols:r1 * cols] = rng.integers(lo, hi + 1, (r1 - r0) * cols)
    return counts


def cell_counts(oracle, world):
    """entities per cell, from the oracle's GetChannelId"""
    ids = oracle.cell_of(world.og(), world.x, world.z)
    return np.bincount(ids[ids != 0].astype(np.int64) - S0, minlength=world.cells)


def emit_uses_cta_tiles(n_own, cells):
    return n_own // max(cells, 1) >= CTA_MIN_PER_CELL and n_own * 16 <= CTA_MAX_BUILD_BYTES


def cta_grid(vis_estimate, max_visible):
    """CTAs the copy kernel is launched with (chd_tick.cu emit_kernel_enqueue)"""
    cap_tiles = -(-max_visible // EMIT_TILE)
    tiles = min(cap_tiles, (vis_estimate + vis_estimate // 32) // EMIT_TILE + 64) if vis_estimate else cap_tiles
    return max(tiles, 1)


def emit_plan(n_own, cells, pair_off, pair_cell, cell_counts, vis_estimate=0, max_visible=None, id_start=S0):
    """Which copy kernel a tick runs, and which branch each of its tiles takes (chd_emit.cuh emit_partition_kernel and the copy
    kernels).  pair_off / pair_cell: the oracle's pair CSR (channel ids); cell_counts: entities per cell index."""
    pair_cell = np.asarray(pair_cell, np.int64) - id_start
    n = int(pair_off[-1])
    counts = np.asarray(cell_counts, np.int64)
    cs = np.concatenate([[0], np.cumsum(counts)])
    vcnt = counts[pair_cell[:n]]
    voff = np.concatenate([[0], np.cumsum(vcnt)])
    V = int(voff[-1])
    cta = emit_uses_cta_tiles(n_own, cells)
    nonempty = np.nonzero(vcnt)[0]
    out = dict(kernel="cta" if cta else "warp", V=V, n_pairs=n,
               trailing_empty=int(n - 1 - nonempty[-1]) if len(nonempty) else n)
    tile = EMIT_TILE if cta else EMIT_WARP_TILE
    n_tiles = -(-V // tile)
    out["n_tiles"] = n_tiles
    base = np.arange(n_tiles, dtype=np.int64) * tile
    p0 = np.searchsorted(voff[1:], base, side="right")  # the pair whose list holds the tile's first entry
    p1 = np.append(p0[1:], n - 1)
    cnt = p1 - p0 + 1
    if not cta:
        out.update(warp_smem=int((cnt <= EMIT_WARP_SMEM_PAIRS).sum()), warp_search=int((cnt > EMIT_WARP_SMEM_PAIRS).sum()))
        return out
    tile_len = np.minimum(tile, V - base)
    e0 = voff[p0 + 1]
    end0 = np.minimum(tile, e0 - base)
    two = end0 < tile_len
    q = np.searchsorted(voff[1:], np.where(two, e0, 0), side="right")  # next non-empty pair
    q = np.minimum(q, n - 1)
    end1 = np.where(two, np.minimum(tile, voff[q + 1] - base), end0)
    general = end1 < tile_len
    simple2 = two & ~general
    ph1 = (end0 - cs[pair_cell[q]]) & 3  # phase of the second segment's source: (0 - (cell_start - end0)) & 3
    out.update(simple=int((~general).sum()), simple_two=int(simple2.sum()),
               phases=sorted(set(zip((end0[simple2] & 3).tolist(), ph1[simple2].tolist()))),
               general_smem=int((general & (cnt <= EMIT_SMEM_PAIRS)).sum()),
               general_search=int((general & (cnt > EMIT_SMEM_PAIRS)).sum()),
               max_general_pairs=int(cnt[general].max()) if general.any() else 0)
    if max_visible is not None:
        out["grid"] = cta_grid(vis_estimate, max_visible)
        out["desc_capacity"] = -(-max_visible // EMIT_TILE) + 8
    return out


# ----------------------------------------------------------------- the worlds of tests/test_gpu_emit_paths.py
# Cells are 100 x 100.  Every builder returns (world, [query sets]); a query set is (cx, cz, r), one sphere per subscriber slot.

def _tiny(world, cells):
    """spheres that see exactly cell `cells` each"""
    cx, cz = world.centre(np.asarray(cells))
    return cx, cz, np.full(len(cx), 10.0)


def bands16(seed, dense=(4096, 9000)):
    """16 x 16: rows 0-5 dense, 6-9 medium (10-2000), 10-12 sparse (0-7), 13-15 empty"""
    counts = band_counts(16, 16, [(0, 6, *dense), (6, 10, 10, 2000), (10, 13, 0, 7)], seed)
    return clustered(16, 16, counts, seed)


def mixed_queries(world, seed, n_whole=6, n_local=300):
    """whole-world spheres, local spheres anywhere, and spheres on the band edges (rows 6, 10 and 13)"""
    rng = np.random.default_rng(seed + 100)
    W, H = world.cols * world.w, world.rows * world.h
    wx, wz, wr = world.whole()
    lx = world.offx + rng.uniform(0, W, n_local)
    lz = world.offz + rng.uniform(0, H, n_local)
    lr = rng.uniform(20.0, 120.0, n_local)
    ex = np.tile(world.offx + (np.arange(16) + 0.5) * world.w, 3)
    ez = np.repeat(world.offz + np.array([6.0, 10.0, 13.0]) * world.h, 16)
    er = np.full(len(ex), 80.0)
    cx = np.concatenate([np.full(n_whole, wx), lx, ex])
    cz = np.concatenate([np.full(n_whole, wz), lz, ez])
    r = np.concatenate([np.full(n_whole, wr), lr, er])
    perm = rng.permutation(len(cx))  # whole-world slots between the others
    return cx[perm], cz[perm], r[perm]


def world_general(seed=11):
    """CTA path, general tiles with at most 256 pairs (shared-memory segment table), all 16 simple-tile phase combinations"""
    w = bands16(seed)
    return w, [mixed_queries(w, seed)]


def search_world(n, seed=12):
    """32 x 32 with rows 10-19 near-empty (0-3 entities: 320 consecutive cells in channel order) and the other rows sharing the
    rest of the n entities evenly"""
    counts = band_counts(32, 32, [(10, 20, 0, 3)], seed)
    dense = np.r_[0:320, 640:1024]
    q, m = divmod(n - int(counts.sum()), len(dense))
    counts[dense] = q
    counts[dense[np.random.default_rng(seed).permutation(len(dense))[:m]]] += 1
    return clustered(32, 32, counts, seed)


def world_search(n):
    """CTA path (n / 1024 cells >= 2048), a tile with more than 256 pairs (per-entry binary search)"""
    w = search_world(n)
    wx, wz, wr = w.whole()
    rng = np.random.default_rng(13)
    lx = w.offx + rng.uniform(0, 3200, 64)
    lz = w.offz + rng.uniform(0, 3200, 64)
    # 128 consecutive slots with small spheres inside the near-empty band: hundreds of pairs of a few entries in one tile, whose
    # cells do not follow each other in the CSR (a row jump, a new slot)
    bx = w.offx + rng.uniform(100, 3100, 128)
    bz = w.offz + rng.uniform(1100, 1900, 128)
    cx = np.concatenate([np.full(5, wx), bx, lx])
    cz = np.concatenate([np.full(5, wz), bz, lz])
    r = np.concatenate([np.full(5, wr), np.full(128, 60.0), np.full(64, 60.0)])
    return w, [(cx, cz, r)]


def world_warp():
    """the same shapes below 2048 entities per cell: the warp kernel, tiles with <= 64 and > 64 pairs"""
    return world_search(1_200_000)


def world_switch():
    """one 16 x 16 engine whose entity count crosses the CTA threshold: warp, CTA x 3, warp, CTA"""
    worlds = []
    for k, cta in enumerate([False, True, True, True, False, True]):
        worlds.append(bands16(20 + k, dense=(4096, 9000) if cta else (1500, 3000)))
    return worlds, mixed_queries(worlds[0], 20, n_whole=4, n_local=200)


def world_underestimate():
    """16 x 16 CTA world; slots 0-5 see an empty cell (small V) or the whole world (V at least 8 times larger)"""
    w = bands16(30)
    rng = np.random.default_rng(31)
    local = _tiny(w, rng.integers(0, 96, 58))
    empty = _tiny(w, np.full(6, 15 * 16 + 3))
    wx, wz, wr = w.whole()
    small = tuple(np.concatenate([a, b]) for a, b in zip(empty, local))
    big = tuple(np.concatenate([np.full(6, v), b]) for v, b in zip((wx, wz, wr), local))
    return w, [small, big, small]


OVERFLOW_MAX_VISIBLE = 1 << 20


def world_overflow():
    """16 x 16 CTA world: a tick with V >= 2 * OVERFLOW_MAX_VISIBLE, then one that fits"""
    w, (big,) = world_general(40)
    rng = np.random.default_rng(41)
    fits = _tiny(w, rng.integers(96, 256, len(big[0])))  # one medium, sparse or empty cell each
    return w, [big, fits]


EDGE_X = 17                                      # dense cell of exactly 3 * 4096 entities
EDGE_Y = {1: 10 * 16 + 4, 2: 10 * 16 + 9, 3: 11 * 16 + 2}  # sparse cells of 1, 2, 3 entities
EDGE_CASES = ["failing", "v0", "k4096", "k4096+1", "k4096+2", "k4096+3", "trailing_empty"]


def edge_world():
    counts = band_counts(16, 16, [(0, 10, 3000, 5000), (10, 12, 0, 7)], 50)
    counts[EDGE_X] = 3 * EMIT_TILE
    for k, c in EDGE_Y.items():
        counts[c] = k
    return clustered(16, 16, counts, 50)


def edge_queries(world, case):
    """8 slots; the slots a case does not use see one empty cell"""
    S = 8
    cells = np.full(S, 14 * 16 + 5)
    cx, cz, r = _tiny(world, cells)
    if case == "failing":  # centres outside the world between working slots
        cx, cz, r = _tiny(world, [EDGE_X, 0, 40, 1, 90, 2, 77, 3])
        cx[[1, 3, 5]] = world.offx - 25.0
        r[[0, 2, 4, 6, 7]] = 90.0
    elif case == "v0":
        cx, cz = world.centre(14 * 16 + np.arange(S))  # spheres over rows 13-15 only
        r = np.full(S, 120.0)
    elif case.startswith("k4096"):
        d = int(case[6:]) if "+" in case else 0
        cx[0], cz[0] = world.centre(EDGE_X)
        if d:
            cx[3], cz[3] = world.centre(EDGE_Y[d])
    elif case == "trailing_empty":  # the last slot: one dense row, the sparse rows, then empty rows to the end
        cx[7], cz[7] = world.offx + 8 * world.w, world.offz + 12.5 * world.h
        r[7] = 350.0
    return cx, cz, r


def edge_expected_v(case):
    return {"v0": 0, "k4096": 3 * EMIT_TILE, "k4096+1": 3 * EMIT_TILE + 1, "k4096+2": 3 * EMIT_TILE + 2,
            "k4096+3": 3 * EMIT_TILE + 3}.get(case)
