// chd_emit.cuh — expanded per-subscriber visible-entity lists (SURVEY.md §8 a14): for every subscription pair
// (subscriber, cell), in pair order, copy the cell's entity list out of the cell CSR.  This is the dominant
// HBM term of a tick (8V bytes algorithmic: read 4V + write 4V; V ~ 4.9e8 on the benchmark config).
//
// Decomposition: the OUTPUT array is cut into fixed tiles of EMIT_TILE entries (load-balanced regardless of
// how entities are distributed over cells).  A partition pass records the first pair of each tile; one CTA copies one
// tile.  Every thread moves 16-byte chunks: stores are fully coalesced; loads are co-aligned 16-byte reads out of the
// L2-resident phase copies of the cell CSR (4 x 4 B x N: 16 MB at 1 M entities, far below the 126 MB L2).
// History (profiles/README.md): v1 4-byte moves, issue-bound, 0.75 ms -> v2/v3 phase-matched 16-byte moves on a persistent
// grid of warp tiles, 0.355 ms -> this shape (round 2).
#pragma once
#include "chd_types.cuh"

namespace chd {


// scan input functor: visible entries of pair p = size of its cell's list (computed on the fly by the offset scan)
struct PairVcountIn {
    const uint32_t* pair_cell;
    const uint32_t* cell_start;
    __device__ __forceinline__ uint64_t operator()(uint64_t p) const {
        const uint32_t c = pair_cell[p];
        return (uint64_t)(cell_start[c + 1] - cell_start[c]);
    }
};

// tile descriptors + first_pair[t] (the pair whose output interval [voff[p], voff[p+1]) contains entry t*EMIT_TILE);
// also vis_off[s] = voff[pair_off[s]] and the V / overflow bookkeeping (one launch)
__global__ void __launch_bounds__(256)
    emit_partition_kernel(const uint32_t* __restrict__ n_pairs_ptr, uint64_t pair_cap, const uint64_t* __restrict__ voff,
                          const uint32_t* __restrict__ pair_cell, const uint32_t* __restrict__ cell_start, uint32_t* __restrict__ first_pair,
                          TileDesc* __restrict__ desc, uint32_t stride, uint64_t max_tiles, uint32_t n_slots, const uint32_t* __restrict__ pair_off,
                          uint64_t* __restrict__ vis_off, uint64_t vis_cap, Counters* __restrict__ ctr, unsigned long long* bump_epoch,
                          uint32_t tile, uint32_t* __restrict__ general_tiles, uint32_t* __restrict__ n_general) {
    const uint64_t n = min((uint64_t)*n_pairs_ptr, pair_cap);
    // last kernel of the emit preparation: open the NEXT execution's scan epoch (the scan of this one has completed)
    if (bump_epoch && blockIdx.x == 0 && threadIdx.x == 0) *bump_epoch = chd_next_epoch(*bump_epoch);
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s <= n_slots; s += (uint64_t)gridDim.x * blockDim.x) {
        vis_off[s] = voff[min((uint64_t)pair_off[s], n)];
        if (s == n_slots) {
            const uint64_t V = voff[n];
            ctr->n_visible = V;
            ctr->required_visible = V;
            if (V > vis_cap) atomicOr(&ctr->overflow, (uint32_t)CHD_OVF_VISIBLE);
        }
    }
    const uint64_t V = voff[n];
    // A visible overflow writes no list, so no tile is described.  This is also what keeps the loop below in bounds: max_tiles
    // counts the smaller 1024-entry warp tiles of vis_cap, while desc and general_tiles hold the 4096-entry CTA tiles of vis_cap
    // (+8); with V > vis_cap the CTA tiles below V would write up to three times those buffers' size past their end.
    if (V > vis_cap) return;
    for (uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; p < n; p += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t b = voff[p], e = voff[p + 1];
        if (e == b) continue;
        if (!desc) {  // warp-tile kernel: only the first pair of every tile
            for (uint64_t t = (b + tile - 1) / tile; t * tile < e && t < max_tiles; t++) first_pair[t] = (uint32_t)p;
            continue;
        }
        const uint32_t cs = cell_start[pair_cell[p]];
        for (uint64_t t = (b + tile - 1) / tile; t * tile < e && t < max_tiles; t++) {
            const uint64_t base = t * tile;
            const uint32_t tile_len = (uint32_t)min((uint64_t)tile, V - base);
            TileDesc d;
            d.p0 = (uint32_t)p;
            // bases are phase-adjusted: the entry that lands on tile slot o is sorted4[base + o] and base + o is a multiple of 4
            // whenever o is (copy k of the CSR payload holds element i at k * stride + k + i, stride % 4 == 0)
            const uint32_t s0 = cs + (uint32_t)(base - b), ph0 = (0u - s0) & 3u;
            d.src0 = ph0 * stride + ph0 + s0;
            const uint32_t end0 = (uint32_t)min((uint64_t)tile, e - base);
            uint32_t end1 = end0;
            d.src1 = 0;
            if (end0 < tile_len) {  // the pair ends inside this tile: the second segment is the next non-empty pair
                uint64_t q = p + 1;
                while (q < n && voff[q + 1] == e) q++;
                if (q < n) {
                    const uint32_t s1 = cell_start[pair_cell[q]] - end0, ph1 = (0u - s1) & 3u;  // (wraps: only base + o, o >= end0, is used)
                    d.src1 = ph1 * stride + ph1 + s1;
                    end1 = (uint32_t)min((uint64_t)tile, voff[q + 1] - base);
                }
            }
            d.ends = end0 | (end1 << 16) | (end1 < tile_len ? 0x80000000u : 0u);
            desc[t] = d;
            first_pair[t] = (uint32_t)p;
            if (end1 < tile_len) general_tiles[atomicAdd(n_general, 1u)] = (uint32_t)t;  // more than two segments: the general pass
        }
    }
}

// General path of one tile: more than two pairs' lists intersect it (cells smaller than a tile).
__device__ __forceinline__ void emit_tile_general(uint64_t t, uint64_t n_tiles, uint64_t V, uint32_t p0, const uint32_t* __restrict__ n_pairs_ptr,
                                               uint64_t pair_cap, const uint64_t* __restrict__ voff, const uint32_t* __restrict__ pair_cell,
                                               const uint32_t* __restrict__ cell_start, const uint32_t* __restrict__ sorted4, uint32_t stride,
                                               const uint32_t* __restrict__ first_pair, uint32_t* __restrict__ vis_entity, uint32_t* s_end,
                                               uint32_t* s_src) {
    const uint32_t tid = threadIdx.x;
    const uint64_t base = t * EMIT_TILE;
    const uint32_t tile_len = (uint32_t)min((uint64_t)EMIT_TILE, V - base);
    uint32_t* __restrict__ out = vis_entity + base;
    const uint64_t np = min((uint64_t)*n_pairs_ptr, pair_cap);
    const uint32_t p1 = (t + 1 < n_tiles) ? first_pair[t + 1] : (uint32_t)(np - 1);
    const uint32_t cnt = p1 - p0 + 1;
    if (cnt <= EMIT_SMEM_PAIRS) {
        __syncthreads();  // the previous tile's readers are done (only when the loop runs more than once)
        if (tid < cnt) {
            const uint64_t b = voff[p0 + tid], e = voff[p0 + tid + 1];
            const uint32_t c = pair_cell[p0 + tid];
            s_end[tid] = (uint32_t)min((uint64_t)EMIT_TILE, e > base ? e - base : 0);
            s_src[tid] = cell_start[c] + (uint32_t)(b < base ? base - b : 0);
        }
        __syncthreads();
        for (int r = 0; r < EMIT_ROWS; r++) {
            const uint32_t o = (r * EMIT_THREADS + tid) * 4;  // first entry of this 16-byte chunk
            if (o >= tile_len) continue;
            uint32_t lo = 0, hi = cnt - 1;  // first k with s_end[k] > o (exists: s_end[cnt-1] >= tile_len > o)
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (s_end[mid] > o) hi = mid; else lo = mid + 1;
            }
            const uint32_t k = lo;
            const uint32_t beg = k == 0 ? 0u : s_end[k - 1];
            const uint32_t sidx = s_src[k] + (o - beg);
            if (o + 4 <= s_end[k]) {
                const uint32_t ph = (0u - sidx) & 3u;  // whole chunk inside one segment: phase copy (-sidx) & 3
                __stcs(reinterpret_cast<uint4*>(out + o), __ldg(reinterpret_cast<const uint4*>(sorted4 + ph * stride + ph + sidx)));
            } else {
                uint32_t kk = k;  // the chunk straddles a segment boundary (or the end of the list): entry by entry
                for (uint32_t j = 0; j < 4 && o + j < tile_len; j++) {
                    while (s_end[kk] <= o + j) kk++;
                    const uint32_t bb = kk == 0 ? 0u : s_end[kk - 1];
                    out[o + j] = __ldg(sorted4 + s_src[kk] + (o + j - bb));
                }
            }
        }
    } else {
        // more than EMIT_SMEM_PAIRS pairs inside one tile (tiny / empty cells): per-entry binary search
        for (uint32_t o = tid; o < tile_len; o += EMIT_THREADS) {
            const uint64_t go = base + o;
            uint64_t lo = p0, hi = p1;  // last p in [p0,p1] with voff[p] <= go
            while (lo < hi) {
                const uint64_t mid = (lo + hi + 1) >> 1;
                if (voff[mid] <= go) lo = mid; else hi = mid - 1;
            }
            const uint32_t c = pair_cell[lo];
            vis_entity[go] = sorted4[cell_start[c] + (uint32_t)(go - voff[lo])];
        }
    }
}

// One CTA per 16 KB tile of the output (EMIT_TILE = 4096 entries: EMIT_ROWS rows of 256 x 16 bytes), dispatched by the
// hardware block scheduler.  Measured on B200 (tools/write_probe.cu, profiles/r2_write_probe.json): the same streaming copy
// out of an L2-resident pool runs at 6.96 TB/s of writes with one CTA per 16 KB chunk, against 6.2 TB/s with a persistent
// grid that walks the chunks round-robin (the round-1 shape) and 7.48 TB/s for a pure fill; 4 rows per thread beat 1 (more
// loads in flight), streaming stores (st.global.cs) beat write-back ones by 15 % (the write stream does not evict the
// L2-resident sources).
// This kernel copies the SIMPLE tiles only (at most two segments: everything a thread needs is the 16-byte descriptor
// {base0, base1, ends, p0}; the bases are phase-adjusted so every move is a co-aligned LDG.128 -> STG.128) and nothing else
// lives in it, so that it fits 32 registers = 8 CTAs (all 64 warps) per SM; tiles with more segments are listed by the
// partition pass and copied by emit_visible_general_kernel.  The loop only runs more than once if the host under-estimated
// the tile count when it sized the grid.
__global__ void __launch_bounds__(EMIT_THREADS, CHD_EMIT_MIN_BLOCKS)
    emit_visible_kernel(const unsigned long long* __restrict__ n_visible_ptr, const uint32_t* __restrict__ sorted4, const TileDesc* __restrict__ desc,
                        uint32_t* __restrict__ vis_entity, uint64_t vis_cap) {
    // V (published by the partition pass) and the CTA's descriptor are loaded back to back: two independent round trips to L2 in
    // flight at once (volatile asm: the compiler would otherwise sink the descriptor load below the early exits)
    const uint64_t V = *n_visible_ptr;
    uint4 dw;
    {
        const TileDesc* dp = desc + blockIdx.x;
        asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(dw.x), "=r"(dw.y), "=r"(dw.z), "=r"(dw.w) : "l"(dp));
    }
    if (V == 0 || V > vis_cap) return;
    const uint32_t n_tiles = (uint32_t)((V + EMIT_TILE - 1) / EMIT_TILE);
    const uint32_t tid4 = threadIdx.x * 4;
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        if (t != blockIdx.x) dw = __ldg(reinterpret_cast<const uint4*>(desc + t));
        if (dw.z & 0x80000000u) continue;  // CTA-uniform: a general tile
        const uint32_t end0 = dw.z & 0x7FFFu, end1 = (dw.z >> 16) & 0x7FFFu;  // a simple tile's second segment reaches the end of the tile / list
        uint32_t* __restrict__ out = vis_entity + (uint64_t)t * EMIT_TILE;
        uint4 v[EMIT_ROWS];
        uint32_t whole = 0;
#pragma unroll
        for (int r = 0; r < EMIT_ROWS; r++) {
            const uint32_t o = r * (EMIT_THREADS * 4) + tid4;
            const bool in0 = o + 4 <= end0, in1 = o >= end0 && o + 4 <= end1;
            if (in0 || in1) {
                // 32-bit index arithmetic ON PURPOSE: base1 is stored minus end0 and may have wrapped below zero; base1 + o wraps back
                const uint32_t si = (in0 ? dw.x : dw.y) + o;
                v[r] = __ldg(reinterpret_cast<const uint4*>(sorted4 + si));
                whole |= 1u << r;
            }
        }
#pragma unroll
        for (int r = 0; r < EMIT_ROWS; r++)
            if (whole & (1u << r)) __stcs(reinterpret_cast<uint4*>(out + r * (EMIT_THREADS * 4) + tid4), v[r]);
#pragma unroll
        for (int r = 0; r < EMIT_ROWS; r++) {
            const uint32_t o = r * (EMIT_THREADS * 4) + tid4;
            if (!(whole & (1u << r)) && o < end1)  // the chunk straddles the segment boundary / the end of the list: entry by entry
                for (uint32_t j = 0; j < 4 && o + j < end1; j++) {
                    const uint32_t si = (o + j < end0 ? dw.x : dw.y) + o + j;  // (32-bit wrap, as above)
                    out[o + j] = __ldg(sorted4 + si);
                }
        }
    }
}

// The tiles the partition pass listed as general (more than two segments): segment table in shared memory, binary search per row.
__global__ void __launch_bounds__(EMIT_THREADS)
    emit_visible_general_kernel(const uint32_t* __restrict__ general_tiles, uint32_t* __restrict__ n_general_ptr,
                                const uint32_t* __restrict__ n_pairs_ptr, uint64_t pair_cap, const unsigned long long* __restrict__ n_visible_ptr,
                                const uint64_t* __restrict__ voff, const uint32_t* __restrict__ pair_cell, const uint32_t* __restrict__ cell_start,
                                const uint32_t* __restrict__ sorted4, uint32_t stride, const uint32_t* __restrict__ first_pair,
                                uint32_t* __restrict__ vis_entity, uint64_t vis_cap) {
    __shared__ uint32_t s_end[EMIT_SMEM_PAIRS];  // end of pair (p0+k) relative to the tile base, clamped to EMIT_TILE
    __shared__ uint32_t s_src[EMIT_SMEM_PAIRS];  // source index of the pair's entry that lands on max(voff[p], tile base)
    // n_general_ptr[0] = list length (appended by the partition pass), [1] = blocks that have read it: the last one to arrive
    // empties the list for the next partition pass (which is ordered after this kernel)
    __shared__ uint32_t s_n;
    if (threadIdx.x == 0) {
        s_n = n_general_ptr[0];
        __threadfence();
        if (atomicAdd(n_general_ptr + 1, 1u) == gridDim.x - 1) {
            n_general_ptr[0] = 0;
            n_general_ptr[1] = 0;
        }
    }
    __syncthreads();
    const uint32_t n_general = s_n;
    const uint64_t V = *n_visible_ptr;
    if (n_general == 0 || V == 0 || V > vis_cap) return;
    const uint64_t n_tiles = (V + EMIT_TILE - 1) / EMIT_TILE;
    for (uint32_t i = blockIdx.x; i < n_general; i += gridDim.x) {
        const uint32_t t = general_tiles[i];
        emit_tile_general(t, n_tiles, V, first_pair[t], n_pairs_ptr, pair_cap, voff, pair_cell, cell_start, sorted4, stride, first_pair, vis_entity, s_end, s_src);
    }
}


// General kernel (round 1's shape): a persistent grid, every WARP owns whole 4 KB tiles (no block barrier anywhere), the segment
// table of a tile lives in a warp-private slice of shared memory.  Used when cells are small against a 16 KB tile (many segments
// per tile: config #5's 152 entities per cell) or when the CSR payload does not fit the L2 (config #3: the copy is then DRAM-bound
// on both sides and this shape reaches 0.95 of the copy peak, where the CTA-tile kernel above reaches 0.80).
__global__ void __launch_bounds__(EMIT_THREADS, 4)
    emit_visible_warp_kernel(const uint32_t* __restrict__ n_pairs_ptr, uint64_t pair_cap, const uint64_t* __restrict__ voff,
                        const uint32_t* __restrict__ pair_cell, const uint32_t* __restrict__ cell_start,
                        const uint32_t* __restrict__ sorted4, uint32_t stride, const uint32_t* __restrict__ first_pair,
                        uint32_t* __restrict__ vis_entity, uint64_t vis_cap) {
    __shared__ uint32_t s_end_all[EMIT_WARP_WARPS][EMIT_WARP_SMEM_PAIRS];  // end of pair (p0+k) relative to the tile base, clamped to EMIT_WARP_TILE
    __shared__ uint32_t s_src_all[EMIT_WARP_WARPS][EMIT_WARP_SMEM_PAIRS];  // source index of the pair's entry that lands on max(voff[p], tile base)
    const uint64_t np = min((uint64_t)*n_pairs_ptr, pair_cap);
    if (np == 0) return;
    const uint64_t V = voff[np];
    if (V > vis_cap) return;
    const uint64_t n_tiles = (V + EMIT_WARP_TILE - 1) / EMIT_WARP_TILE;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t* s_end = s_end_all[w];
    uint32_t* s_src = s_src_all[w];
    const uint64_t warp_id = (uint64_t)blockIdx.x * EMIT_WARP_WARPS + w, n_warps = (uint64_t)gridDim.x * EMIT_WARP_WARPS;
    for (uint64_t t = warp_id; t < n_tiles; t += n_warps) {
        const uint64_t base = t * EMIT_WARP_TILE;
        const uint32_t p0 = first_pair[t];
        const uint32_t p1 = (t + 1 < n_tiles) ? first_pair[t + 1] : (uint32_t)(np - 1);
        const uint32_t cnt = p1 - p0 + 1;
        const uint32_t tile_len = (uint32_t)min((uint64_t)EMIT_WARP_TILE, V - base);
        uint32_t* __restrict__ out = vis_entity + base;
        if (cnt <= EMIT_WARP_SMEM_PAIRS) {
            __syncwarp();  // the previous tile's readers are done
            for (uint32_t k = lane; k < cnt; k += 32) {
                const uint64_t b = voff[p0 + k], e = voff[p0 + k + 1];
                const uint32_t c = pair_cell[p0 + k];
                s_end[k] = (uint32_t)min((uint64_t)EMIT_WARP_TILE, e > base ? e - base : 0);
                s_src[k] = cell_start[c] + (uint32_t)(b < base ? base - b : 0);
            }
            __syncwarp();
            uint32_t k = 0;  // segment cursor of this lane (its chunks ascend)
            uint32_t src[EMIT_WARP_CHUNKS];  // element index into sorted4 (multiple of 4), or 0xFFFFFFFF
            // phase 1: resolve every chunk's source (nullptr = handled element-wise / out of range)
#pragma unroll
            for (int it = 0; it < EMIT_WARP_CHUNKS; it++) {
                const uint32_t o = (it * 32 + lane) * 4;  // first entry of this 16-byte chunk
                src[it] = 0xFFFFFFFFu;
                if (o < tile_len) {
                    while (s_end[k] <= o) k++;  // terminates: s_end[cnt-1] >= tile_len > o
                    const uint32_t beg = k == 0 ? 0u : s_end[k - 1];
                    const uint32_t sidx = s_src[k] + (o - beg);
                    if (o + 4 <= s_end[k]) {
                        // whole chunk inside one segment: co-aligned 16-byte move out of phase copy (-sidx)&3
                        const uint32_t ph = (0u - sidx) & 3u;
                        src[it] = ph * stride + ph + sidx;
                    } else {
                        // the chunk straddles a segment boundary (or the end of the list): entry by entry
                        uint32_t kk = k;
                        for (uint32_t j = 0; j < 4 && o + j < tile_len; j++) {
                            while (s_end[kk] <= o + j) kk++;
                            const uint32_t bb = kk == 0 ? 0u : s_end[kk - 1];
                            out[o + j] = __ldg(sorted4 + s_src[kk] + (o + j - bb));
                        }
                    }
                }
            }
            // phase 2: all loads in flight, phase 3: streaming stores
            uint4 v[EMIT_WARP_CHUNKS];
#pragma unroll
            for (int it = 0; it < EMIT_WARP_CHUNKS; it++)
                if (src[it] != 0xFFFFFFFFu) v[it] = __ldg(reinterpret_cast<const uint4*>(sorted4 + src[it]));
#pragma unroll
            for (int it = 0; it < EMIT_WARP_CHUNKS; it++)
                if (src[it] != 0xFFFFFFFFu) __stcs(reinterpret_cast<uint4*>(out + (it * 32 + lane) * 4), v[it]);
        } else {
            // more than EMIT_WARP_SMEM_PAIRS pairs inside one tile (tiny / empty cells): per-entry binary search
            for (uint32_t o = lane; o < tile_len; o += 32) {
                const uint64_t go = base + o;
                uint64_t lo = p0, hi = p1;  // last p in [p0,p1] with voff[p] <= go
                while (lo < hi) {
                    const uint64_t mid = (lo + hi + 1) >> 1;
                    if (voff[mid] <= go) lo = mid; else hi = mid - 1;
                }
                const uint32_t c = pair_cell[lo];
                vis_entity[go] = sorted4[cell_start[c] + (uint32_t)(go - voff[lo])];
            }
        }
    }
}


}  // namespace chd
