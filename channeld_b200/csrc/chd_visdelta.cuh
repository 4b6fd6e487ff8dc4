// chd_visdelta.cuh — kernels of the per-subscriber visibility deltas (chd_visible_delta, include/chd_gpu.h).
//
// V(s) = { e : cell(e) in C(s) } is never materialised.  Two states are compared: NOW (the cell keys / cell CSR of the last
// chd_build, the current pair CSR) and the BASELINE (copies of the same arrays taken at the end of the last successful call).
//   enter(s) = V_now(s) \ V_base(s): for every current pair (s, c): if c was not in C_base(s), the whole cell c of the current
//              CSR is a candidate, otherwise only the entities that moved INTO c since the baseline; a candidate e is kept
//              if cell_base(e) is not in C_base(s).
//   leave(s) = V_base(s) \ V_now(s): the mirror image over the baseline pairs, the baseline cell CSR and the movers OUT of
//              each cell, tested against C_now(s).
// A work item is one pair (one warp); counts -> look-back scan -> the same sweep writes with a warp ballot, so the output is in
// (cell asc, entity asc) order per slot and byte-for-byte deterministic.
#pragma once
#include "chd_types.cuh"

namespace chd {

// One side of the delta.  ENTER: the current pairs against the baseline; LEAVE: the baseline pairs against the current state.
struct VdSide {
    const uint32_t *sub, *cell, *n_pairs;  // the pairs swept: owning slot, cell index, live count (device)
    const uint32_t *o_off, *o_cell, *o_S;  // the other state's pair CSR by slot (channel-sorted), its slot count (device)
    const uint32_t *cs, *ents;             // this state's cell CSR: whole-cell segments
    const uint32_t *mv_start, *mv_ent;     // movers into (ENTER) / out of (LEAVE) each cell, entity id ascending
    const uint32_t *o_key, *o_n;           // the other state's cell key per entity and its entity count (device)
    uint32_t cells;
};

__device__ __forceinline__ bool vd_contains(const uint32_t* __restrict__ a, uint32_t lo, uint32_t hi, uint32_t x) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1, v = a[mid];
        if (v == x) return true;
        if (v < x) lo = mid + 1;
        else hi = mid;
    }
    return false;
}

static __global__ void vd_begin_kernel(VdState* st, unsigned long long* epoch, uint32_t n_now, uint32_t S_now, const uint32_t* __restrict__ cur_off) {
    *epoch = chd_next_epoch(*epoch);
    st->n_now = n_now;
    st->S_now = S_now;
    st->P_now = cur_off[S_now];
    st->ovf = 0;
}

// an entity is a mover when its cell key differs between the two states (entities beyond a state's count are in no cell)
struct VdMoverFlag {
    const uint32_t *key_now, *key_base;
    const VdState* st;
    uint32_t cells;
    __device__ __forceinline__ uint32_t now(uint64_t i) const { return i < st->n_now ? key_now[i] : cells; }
    __device__ __forceinline__ uint32_t base(uint64_t i) const { return i < st->n_base ? key_base[i] : cells; }
    __device__ __forceinline__ bool operator()(uint64_t i) const { return now(i) != base(i); }
};
struct VdMoverSink {
    VdMoverFlag f;
    uint32_t *ent, *dst_key, *src_key, *count;
    __device__ __forceinline__ void operator()(uint64_t i, uint32_t k) const {
        ent[k] = (uint32_t)i;
        dst_key[k] = f.now(i);
        src_key[k] = f.base(i);
    }
    __device__ __forceinline__ void total(uint32_t n) const { *count = n; }
};

// CSR offsets of the movers sorted by cell: start[c] = #keys < c for c in [0, cells + 1] (lower bound: one thread per cell, so a
// sparse key set costs no serial gap filling)
static __global__ void __launch_bounds__(256) vd_bounds_kernel(const uint32_t* __restrict__ sorted_key, const uint32_t* __restrict__ n_ptr, uint32_t cells,
                                                               uint32_t* __restrict__ start) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > cells + 1) return;
    uint32_t lo = 0, hi = *n_ptr;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (sorted_key[mid] < c) lo = mid + 1;
        else hi = mid;
    }
    start[c] = lo;
}

// WRITE = false: cnt[p] = entries pair p contributes.  WRITE = true: writes them at off[p] (skipped when the delta overflowed).
template <bool WRITE>
__global__ void __launch_bounds__(256) vd_pairs_kernel(VdSide a, const VdState* __restrict__ st, uint32_t* __restrict__ cnt,
                                                       const unsigned long long* __restrict__ off, uint32_t* __restrict__ out) {
    if (WRITE && st->ovf) return;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t n_pairs = *a.n_pairs, o_S = *a.o_S, o_n = *a.o_n;
    const uint32_t nw = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < n_pairs; p += nw) {
        const uint32_t s = a.sub[p], c = a.cell[p];
        const uint32_t ob = a.o_off[min(s, o_S)], oe = s < o_S ? a.o_off[s + 1] : ob;
        const bool kept = vd_contains(a.o_cell, ob, oe, c);
        const uint32_t b = kept ? a.mv_start[c] : a.cs[c];
        const uint32_t len = (kept ? a.mv_start[c + 1] : a.cs[c + 1]) - b;
        const uint32_t* __restrict__ list = (kept ? a.mv_ent : a.ents) + b;
        const uint64_t o = WRITE ? off[p] : 0;
        uint32_t k = 0;
        for (uint32_t i0 = 0; i0 < len; i0 += 32) {
            const uint32_t i = i0 + lane;
            bool keep = false;
            uint32_t ent = 0;
            if (i < len) {
                ent = list[i];
                const uint32_t x = ent < o_n ? a.o_key[ent] : a.cells;
                keep = x >= a.cells || !vd_contains(a.o_cell, ob, oe, x);
            }
            const uint32_t m = __ballot_sync(0xffffffffu, keep);
            if (WRITE && keep) out[o + k + __popc(m & lt)] = ent;
            k += __popc(m);
        }
        if (!WRITE && lane == 0) cnt[p] = k;
    }
}

// per-slot CSR offsets from the per-pair ones, totals and the overflow decision (thread 0)
static __global__ void __launch_bounds__(256) vd_offsets_kernel(VdState* st, uint32_t S_out, const uint32_t* __restrict__ cur_off,
                                                                const uint32_t* __restrict__ base_off, const unsigned long long* __restrict__ epoff,
                                                                const unsigned long long* __restrict__ lpoff, uint64_t cap, unsigned long long* __restrict__ enter_off,
                                                                unsigned long long* __restrict__ leave_off) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > S_out) return;
    const uint32_t Sn = st->S_now, Sb = st->S_base;
    enter_off[s] = epoff[cur_off[min(s, Sn)]];
    leave_off[s] = lpoff[base_off[min(s, Sb)]];
    if (s == 0) {
        const unsigned long long ne = epoff[st->P_now], nl = lpoff[st->P_base];
        st->n_enter = ne;
        st->n_leave = nl;
        st->ovf = (ne > cap || nl > cap) ? 1u : 0u;
    }
}

// The current state becomes the baseline (skipped on the device when the delta overflowed).  blockIdx.y selects the array.
struct VdSnap {
    const uint32_t *key, *cs, *sorted, *off, *cell, *sub;
    uint32_t *b_key, *b_cs, *b_sorted, *b_off, *b_cell, *b_sub;
    uint32_t cells;
};
static __global__ void __launch_bounds__(256) vd_snapshot_kernel(VdState* st, VdSnap a) {
    if (st->ovf) return;
    const uint32_t* src;
    uint32_t* dst;
    uint64_t n;
    switch (blockIdx.y) {
        case 0: src = a.key; dst = a.b_key; n = st->n_now; break;
        case 1: src = a.cs; dst = a.b_cs; n = (uint64_t)a.cells + 2; break;
        case 2: src = a.sorted; dst = a.b_sorted; n = a.cs[a.cells]; break;
        case 3: src = a.off; dst = a.b_off; n = (uint64_t)st->S_now + 1; break;
        case 4: src = a.cell; dst = a.b_cell; n = st->P_now; break;
        default: src = a.sub; dst = a.b_sub; n = st->P_now; break;
    }
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[i];
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {  // nothing in this kernel reads the baseline counts
        st->n_base = st->n_now;
        st->S_base = st->S_now;
        st->P_base = st->P_now;
    }
}

}  // namespace chd
