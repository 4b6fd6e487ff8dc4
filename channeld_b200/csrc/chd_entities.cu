// chd_entities.cu — entity positions, GetChannelId per entity, spatial-hash build (cell CSR + phase copies).
#include "chd_engine.h"

#include "chd_build.cuh"
#include "chd_misc.cuh"

// assign: when set, the pass's histogram kernel also computes the keys from the positions (first pass of a single-GPU build)
struct FusedAssign {
    const double *x, *z;
    uint32_t* key;
    const uint32_t* prev;
    HandoverOut ho;
};
template <int BINS>
static chd_status sort_pass(chd_engine* e, uint32_t* hist, const ScanSite& site, const uint32_t* key_in, const uint32_t* val_in, uint32_t n,
                            const uint32_t* n_ptr, uint32_t per_block, uint32_t nblocks, uint32_t shift, uint32_t bits, uint32_t* key_out,
                            uint32_t* val_out, ScatterExtras ex, unsigned long long* bump, const FusedAssign* assign = nullptr, int half = 0) {
    // half: 0 = the whole pass, 1 = histogram + scan only, 2 = scatter only (single-pass builds are split so that the emit
    // preparation, which needs only the cell counts, overlaps the scatter)
    const uint32_t mask = (1u << bits) - 1u;
    if (half == 2) goto scatter;
    if (assign)
        assign_hist_kernel<BINS><<<nblocks, BUILD_THREADS, 0, e->stream>>>(e->g, assign->x, assign->z, n, assign->key, assign->prev, assign->ho, per_block, mask,
                                                                           hist, nblocks, bump);
    else
        radix_hist_kernel<BINS><<<nblocks, BUILD_THREADS, 0, e->stream>>>(key_in, n, n_ptr, per_block, shift, mask, hist, nblocks, bump);
    KCHECK(e);
    SCAN(e, exclusive_scan_1p<uint32_t, uint32_t>(hist, hist, (uint64_t)BINS * nblocks, site, e->stream));
    if (half == 1) return CHD_OK;
scatter:
    // bandwidth-bound regime: reorder each tile by digit in shared memory first (coalesced runs); small inputs are latency-bound
    // and take the plain scatter (fewer barriers per tile)
    if (n > (2u << 20))
        radix_scatter_sorted_kernel<BINS><<<nblocks, BUILD_THREADS, 0, e->stream>>>(key_in, val_in, n, n_ptr, per_block, shift, mask, hist, nblocks,
                                                                                   key_out, val_out, ex);
    else
        radix_scatter_kernel<BINS><<<nblocks, BUILD_THREADS, 0, e->stream>>>(key_in, val_in, n, n_ptr, per_block, shift, mask, hist, nblocks,
                                                                            key_out, val_out, ex);
    KCHECK(e);
    return CHD_OK;
}

static chd_status sort_pass_fused(chd_engine* e, uint32_t* hist, const ScanSite& site, const uint32_t* key_in, const uint32_t* val_in, uint32_t n,
                                  const uint32_t* n_ptr, uint32_t per_block, uint32_t nblocks, uint32_t shift, uint32_t bits, uint32_t* key_out,
                                  uint32_t* val_out, ScatterExtras ex, unsigned long long* bump, const FusedAssign* assign, int half = 0) {
    if (bits <= 8) return sort_pass<256>(e, hist, site, key_in, val_in, n, n_ptr, per_block, nblocks, shift, bits, key_out, val_out, ex, bump, assign, half);
    return sort_pass<1024>(e, hist, site, key_in, val_in, n, n_ptr, per_block, nblocks, shift, bits, key_out, val_out, ex, bump, assign, half);
}

chd_status chd_sort_pass_any(chd_engine* e, uint32_t* hist, const ScanSite& site, const uint32_t* key_in, const uint32_t* val_in,
                                uint32_t n, const uint32_t* n_ptr, uint32_t per_block, uint32_t nblocks, uint32_t shift, uint32_t bits,
                                uint32_t* key_out, uint32_t* val_out, ScatterExtras ex,
                                unsigned long long* bump) {
    return sort_pass_fused(e, hist, site, key_in, val_in, n, n_ptr, per_block, nblocks, shift, bits, key_out, val_out, ex, bump, nullptr);
}

extern "C" {

/* ------------------------------------------------------------------ entities / build ---- */

chd_status chd_cell_of(chd_engine* e, const double* x, const double* z, uint32_t n, uint32_t* out) {
    return chd_cell_of_valid(e, x, z, n, out, nullptr);
}

chd_status chd_cell_of_valid(chd_engine* e, const double* x, const double* z, uint32_t n, uint32_t* out, uint8_t* out_valid) {
    if (!e || (n && (!x || !z || !out))) return CHD_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lk(e->mu);
    CU(e, cudaSetDevice(e->device));
    // chunked through the tmp buffers (they are free outside chd_build)
    double *dx = nullptr, *dz = nullptr;
    uint32_t* dk = nullptr;
    uint8_t* dv = nullptr;
    const uint32_t chunk = 1u << 20;
    CU(e, cudaMallocAsync((void**)&dx, sizeof(double) * chunk, e->stream));
    CU(e, cudaMallocAsync((void**)&dz, sizeof(double) * chunk, e->stream));
    CU(e, cudaMallocAsync((void**)&dk, sizeof(uint32_t) * chunk, e->stream));
    if (out_valid) CU(e, cudaMallocAsync((void**)&dv, chunk, e->stream));
    HandoverOut ho{};
    for (uint32_t b = 0; b < n; b += chunk) {
        const uint32_t m = n - b < chunk ? n - b : chunk;
        CU(e, cudaMemcpyAsync(dx, x + b, sizeof(double) * m, cudaMemcpyDefault, e->stream));
        CU(e, cudaMemcpyAsync(dz, z + b, sizeof(double) * m, cudaMemcpyDefault, e->stream));
        assign_cells_kernel<<<blocks_for(m, 256), 256, 0, e->stream>>>(e->g, dx, dz, m, dk, nullptr, ho, nullptr);
        KCHECK(e);
        cell_key_to_id_kernel<<<blocks_for(m, 256), 256, 0, e->stream>>>(dk, m, e->g.cells, e->g.id_start, dv);
        KCHECK(e);
        CU(e, cudaMemcpyAsync(out + b, dk, sizeof(uint32_t) * m, cudaMemcpyDefault, e->stream));
        if (out_valid) CU(e, cudaMemcpyAsync(out_valid + b, dv, m, cudaMemcpyDefault, e->stream));
    }
    CU(e, cudaFreeAsync(dx, e->stream));
    CU(e, cudaFreeAsync(dz, e->stream));
    CU(e, cudaFreeAsync(dk, e->stream));
    if (dv) CU(e, cudaFreeAsync(dv, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    return CHD_OK;
}

chd_status chd_set_entities(chd_engine* e, const double* x, const double* z, uint32_t n) {
    if (!e || (n && (!x || !z))) return CHD_ERR_INVALID;
    if (n > e->lim.max_entities) {
        e->fail("chd_set_entities: %u > max_entities %u", n, e->lim.max_entities);
        return CHD_ERR_CAPACITY;
    }
    CU(e, cudaSetDevice(e->device));
    if (n != e->n_own) e->have_prev_key = false;
    if (n && chd_is_device_ptr(e, x) && chd_is_device_ptr(e, z)) {
        e->pos_x = x;  // device-resident producer: read in place
        e->pos_z = z;
    } else {
        CU(e, cudaMemcpyAsync(e->d_x, x, sizeof(double) * n, cudaMemcpyDefault, e->stream));
        CU(e, cudaMemcpyAsync(e->d_z, z, sizeof(double) * n, cudaMemcpyDefault, e->stream));
        e->pos_x = e->d_x;
        e->pos_z = e->d_z;
    }
    e->n_own = n;
    e->n_halo = 0;
    e->halo_on_device = false;
    e->assigned = false;
    e->entities_dirty = true;
    return CHD_OK;
}

chd_status chd_prefetch_entities(chd_engine* e, const double* x, const double* z, uint32_t n) {
    if (!e || (n && (!x || !z))) return CHD_ERR_INVALID;
    if (n > e->lim.max_entities) {
        e->fail("chd_prefetch_entities: %u > max_entities %u", n, e->lim.max_entities);
        return CHD_ERR_CAPACITY;
    }
    CU(e, cudaSetDevice(e->device));
    const int back = e->pos_buf ^ 1;
    {
        chd_status st = chd_ensure_upload_stream(e);
        if (st != CHD_OK) return st;
    }
    if (!e->d_xb[back]) {  // the second pair of position buffers exists only for hosts that prefetch
        if (!dalloc(e, &e->d_xb[back], e->lim.max_entities) || !dalloc(e, &e->d_zb[back], e->lim.max_entities)) return CHD_ERR_CUDA;
    }
    // the back pair was last read by the cell assignment of an earlier tick
    if (e->pos_read_recorded[back]) CU(e, cudaStreamWaitEvent(e->up_stream, e->ev_pos_read[back], 0));
    CU(e, cudaMemcpyAsync(e->d_xb[back], x, sizeof(double) * n, cudaMemcpyDefault, e->up_stream));
    CU(e, cudaMemcpyAsync(e->d_zb[back], z, sizeof(double) * n, cudaMemcpyDefault, e->up_stream));
    CU(e, cudaEventRecord(e->ev_upload, e->up_stream));
    e->staged = true;
    e->staged_n = n;
    return CHD_OK;
}

// float uploads (see widen_positions_kernel): the floats land in a staging buffer (or are read in place when they already live on
// the device) and are widened into the double buffers on the same stream, so everything downstream is unchanged.
static chd_status widen_upload(chd_engine* e, int which, const float* x, const float* z, uint32_t n, double* dx, double* dz, cudaStream_t s) {
    if (!n) return CHD_OK;
    const float *sx = x, *sz = z;
    if (!(chd_is_device_ptr(e, x) && chd_is_device_ptr(e, z))) {
        if (!e->d_pos_f32[which] && !dalloc(e, &e->d_pos_f32[which], 2ull * e->lim.max_entities + 8)) return CHD_ERR_CUDA;
        float* stage_x = e->d_pos_f32[which];
        float* stage_z = stage_x + (((size_t)e->lim.max_entities + 3) & ~(size_t)3);
        CU(e, cudaMemcpyAsync(stage_x, x, sizeof(float) * n, cudaMemcpyDefault, s));
        CU(e, cudaMemcpyAsync(stage_z, z, sizeof(float) * n, cudaMemcpyDefault, s));
        sx = stage_x;
        sz = stage_z;
    } else if ((((uintptr_t)x) | ((uintptr_t)z)) & 15) {
        e->fail("float positions on the device must be 16-byte aligned");
        return CHD_ERR_INVALID;
    }
    widen_positions_kernel<<<blocks_for((n + 3) / 4, 256), 256, 0, s>>>(sx, sz, dx, dz, n);
    KCHECK(e);
    return CHD_OK;
}

chd_status chd_set_entities_f32(chd_engine* e, const float* x, const float* z, uint32_t n) {
    if (!e || (n && (!x || !z))) return CHD_ERR_INVALID;
    if (n > e->lim.max_entities) {
        e->fail("chd_set_entities_f32: %u > max_entities %u", n, e->lim.max_entities);
        return CHD_ERR_CAPACITY;
    }
    CU(e, cudaSetDevice(e->device));
    if (n != e->n_own) e->have_prev_key = false;
    chd_status st = widen_upload(e, 0, x, z, n, e->d_x, e->d_z, e->stream);
    if (st != CHD_OK) return st;
    e->pos_x = e->d_x;
    e->pos_z = e->d_z;
    e->n_own = n;
    e->n_halo = 0;
    e->halo_on_device = false;
    e->assigned = false;
    e->entities_dirty = true;
    return CHD_OK;
}

chd_status chd_prefetch_entities_f32(chd_engine* e, const float* x, const float* z, uint32_t n) {
    if (!e || (n && (!x || !z))) return CHD_ERR_INVALID;
    if (n > e->lim.max_entities) {
        e->fail("chd_prefetch_entities_f32: %u > max_entities %u", n, e->lim.max_entities);
        return CHD_ERR_CAPACITY;
    }
    CU(e, cudaSetDevice(e->device));
    const int back = e->pos_buf ^ 1;
    {
        chd_status st = chd_ensure_upload_stream(e);
        if (st != CHD_OK) return st;
    }
    if (!e->d_xb[back]) {
        if (!dalloc(e, &e->d_xb[back], e->lim.max_entities) || !dalloc(e, &e->d_zb[back], e->lim.max_entities)) return CHD_ERR_CUDA;
    }
    if (e->pos_read_recorded[back]) CU(e, cudaStreamWaitEvent(e->up_stream, e->ev_pos_read[back], 0));
    chd_status st = widen_upload(e, 1, x, z, n, e->d_xb[back], e->d_zb[back], e->up_stream);
    if (st != CHD_OK) return st;
    CU(e, cudaEventRecord(e->ev_upload, e->up_stream));
    e->staged = true;
    e->staged_n = n;
    return CHD_OK;
}

chd_status chd_entity_buffers(chd_engine* e, double** d_x, double** d_z, uint32_t* n) {
    if (!e) return CHD_ERR_INVALID;
    if (d_x) *d_x = e->d_x;
    if (d_z) *d_z = e->d_z;
    if (n) *n = e->n_own;
    e->pos_x = e->d_x;
    e->pos_z = e->d_z;
    e->assigned = false;  // the caller may write positions
    e->entities_dirty = true;
    return CHD_OK;
}

chd_status chd_set_entity_count(chd_engine* e, uint32_t n) {
    if (!e || n > e->lim.max_entities) return CHD_ERR_INVALID;
    if (n != e->n_own) e->have_prev_key = false;
    e->n_own = n;
    e->n_halo = 0;
    e->halo_on_device = false;
    e->assigned = false;
    e->entities_dirty = true;
    return CHD_OK;
}

chd_status chd_set_entity_ids(chd_engine* e, const uint32_t* gid, uint32_t n) {
    if (!e || n > e->lim.max_entities) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    if (!gid) {
        e->have_gid = false;
        return CHD_OK;
    }
    CU(e, cudaMemcpyAsync(e->d_gid, gid, sizeof(uint32_t) * n, cudaMemcpyDefault, e->stream));
    e->have_gid = true;
    e->entities_dirty = true;
    return CHD_OK;
}

// The engine's position buffers are double-buffered for chd_prefetch_entities: remember (outside any graph capture)
// the last kernel that read the front pair, so an upload into it can be ordered after that read.
chd_status chd_note_pos_read(chd_engine* e) {
    if (e->pos_x != e->d_x || !e->ev_pos_read[e->pos_buf]) return CHD_OK;
    CU(e, cudaEventRecord(e->ev_pos_read[e->pos_buf], e->stream));
    e->pos_read_recorded[e->pos_buf] = true;
    return CHD_OK;
}

chd_status chd_assign_cells_impl(chd_engine* e);

chd_status chd_assign_cells(chd_engine* e) {
    if (!e) return CHD_ERR_INVALID;
    {
        chd_status gs_ = chd_fetch_guard(e);
        if (gs_ != CHD_OK) return gs_;
    }
    const bool was_assigned = e->assigned;
    chd_status st = chd_assign_cells_impl(e);
    if (st == CHD_OK && !was_assigned) st = chd_note_pos_read(e);
    return st;
}

// host-side half of a cell assignment: the key buffers swap (handover detection compares against the keys of the previous
// assignment, same entity count; swapped, never copied), the handover counter is zeroed.  Returns the previous keys or nullptr.
static chd_status assign_prepare(chd_engine* e, uint32_t** prev_out, HandoverOut* ho) {
    uint32_t* prev = nullptr;
    if (e->have_prev_key) {
        uint32_t* t = e->d_key;
        e->d_key = e->d_prev_key;
        e->d_prev_key = t;
        prev = e->d_prev_key;
    }
    *ho = HandoverOut{e->d_ho_entity, e->d_ho_src, e->d_ho_dst, &e->d_ctr->n_handover, e->ho_cap};
    CU(e, cudaMemsetAsync(&e->d_ctr->n_handover, 0, 4, e->stream));
    *prev_out = prev;
    return CHD_OK;
}

chd_status chd_assign_cells_impl(chd_engine* e) {
    CU(e, cudaSetDevice(e->device));
    if (e->assigned) return CHD_OK;
    uint32_t* prev = nullptr;
    HandoverOut ho{};
    chd_status st = assign_prepare(e, &prev, &ho);
    if (st != CHD_OK) return st;
    if (e->n_own) {
        assign_cells_kernel<<<blocks_for(e->n_own, 256), 256, 0, e->stream>>>(e->g, e->pos_x ? e->pos_x : e->d_x, e->pos_z ? e->pos_z : e->d_z,
                                                                              e->n_own, e->d_key, prev, ho, e->assign_bump);
        KCHECK(e);
        e->have_prev_key = true;
        e->assign_bump = nullptr;  // consumed
    }
    e->assigned_since_build = true;  // (cleared by chd_build once the cell CSR matches the keys again)
    e->n_halo = 0;
    e->assigned = true;
    return CHD_OK;
}

// part: 0 = the whole build; single-pass builds only: 1 = cell assignment + histogram + scan + CSR offsets, 2 = scatter (+ phase
// copies).  The cell CSR offsets are final after part 1.
static chd_status build_enqueue(chd_engine* e, bool with_assign, int part = 0) {
    chd_status st;
    FusedAssign fa{};
    const FusedAssign* fap = nullptr;
    if (with_assign) {
        if (!e->assigned && e->n_own && !e->halo_on_device) {
            // single-GPU build: GetChannelId per entity is fused into the first pass's histogram kernel
            uint32_t* prev = nullptr;
            HandoverOut ho{};
            st = assign_prepare(e, &prev, &ho);
            if (st != CHD_OK) return st;
            fa = FusedAssign{e->pos_x ? e->pos_x : e->d_x, e->pos_z ? e->pos_z : e->d_z, e->d_key, prev, ho};
            fap = &fa;
            e->have_prev_key = true;
            e->n_halo = 0;
            e->assigned = true;
        } else {
            st = chd_assign_cells_impl(e);
            if (st != CHD_OK) return st;
        }
    }
    // multi-GPU: the halo count stays on the device (d_n_build = own + kept halo records); launches are sized for
    // the entity capacity and blocks beyond the live length idle.
    const uint32_t* n_ptr = e->halo_on_device ? e->d_n_build : nullptr;
    const uint32_t n = e->halo_on_device ? e->lim.max_entities : e->n_own + e->n_halo;
    const uint32_t C = e->g.cells;
    uint32_t bits = 1;
    while ((1u << bits) < C + 1) bits++;  // keys are in [0, C]
    const uint32_t passes = bits <= 10 ? 1 : 2;
    const uint32_t bits0 = passes == 1 ? bits : (bits + 1) / 2, bits1 = bits - bits0;
    // contiguous slice per block, multiple of the tile
    uint32_t per_block = (n + e->build_blocks - 1) / e->build_blocks;
    per_block = ((per_block + BUILD_TILE - 1) / BUILD_TILE) * BUILD_TILE;
    if (per_block == 0) per_block = BUILD_TILE;
    uint32_t nblocks = (n + per_block - 1) / per_block;
    if (nblocks == 0) nblocks = 1;
    const uint32_t* vals = e->have_gid ? e->d_gid : nullptr;
    // Phase copies: written by a separate fully-coalesced pass after the scatter.  (Fusing them into the scatter saves a launch but
    // does 4 scattered 4-byte stores per entity: measured slower at every size — 69 vs 59 us per build at N = 1 M, 325 vs 205 us
    // at N = 10 M.)
    const bool fuse_phases = false;
    const uint32_t fused_stride = fuse_phases ? e->phase_stride : 0u;
    if (passes == 1 && part != 0) {
        if (part == 1) {
            st = sort_pass_fused(e, e->d_hist, e->site_hist, e->d_key, vals, n, n_ptr, per_block, nblocks, 0, bits0, nullptr, e->d_sorted_ent,
                                 ScatterExtras{0, nullptr, C, nullptr}, e->d_epoch + EP_BUILD, fap, 1);
            if (st != CHD_OK) return st;
            publish_cell_start_kernel<<<blocks_for((uint64_t)C + 2, 256), 256, 0, e->stream>>>(e->d_hist, nblocks, C, n, n_ptr, e->d_cell_start,
                                                                                                 &e->d_ctr->n_entities_in_world);
            KCHECK(e);
            return CHD_OK;
        }
        st = sort_pass_fused(e, e->d_hist, e->site_hist, e->d_key, vals, n, n_ptr, per_block, nblocks, 0, bits0, nullptr, e->d_sorted_ent,
                             ScatterExtras{fused_stride, nullptr, C, nullptr}, nullptr, nullptr, 2);
        if (st != CHD_OK) return st;
    } else if (passes == 1) {
        // single pass: digit == key, so the scatter also publishes the CSR offsets
        ScatterExtras ex{fused_stride, e->d_cell_start, C, &e->d_ctr->n_entities_in_world};
        st = sort_pass_fused(e, e->d_hist, e->site_hist, e->d_key, vals, n, n_ptr, per_block, nblocks, 0, bits0, nullptr, e->d_sorted_ent, ex,
                             e->d_epoch + EP_BUILD, fap);
        if (st != CHD_OK) return st;
    } else {
        st = sort_pass_fused(e, e->d_hist, e->site_hist, e->d_key, vals, n, n_ptr, per_block, nblocks, 0, bits0, e->d_tmp_key, e->d_tmp_val,
                             ScatterExtras{0, nullptr, 0, nullptr}, e->d_epoch + EP_BUILD, fap);
        if (st != CHD_OK) return st;
        ScatterExtras ex{fused_stride, nullptr, C, nullptr};
        st = chd_sort_pass_any(e, e->d_hist, e->site_hist_b, e->d_tmp_key, e->d_tmp_val, n, n_ptr, per_block, nblocks, bits0, bits1, e->d_sorted_key,
                           e->d_sorted_ent, ex);
        if (st != CHD_OK) return st;
        cell_bounds_kernel<<<blocks_for((uint64_t)n + 1, 256), 256, 0, e->stream>>>(e->d_sorted_key, n, n_ptr, C, e->d_cell_start,
                                                                                      &e->d_ctr->n_entities_in_world);
        KCHECK(e);
    }
    if (!fuse_phases && n) {
        replicate_phases_kernel<<<blocks_for(n, 256), 256, 0, e->stream>>>(e->d_sorted_ent, n, n_ptr, e->phase_stride, e->d_sorted4);
        KCHECK(e);
    }
    return CHD_OK;
}

chd_status chd_build(chd_engine* e) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    {
        chd_status gs_ = chd_fetch_guard(e);
        if (gs_ != CHD_OK) return gs_;
    }
    StageTimer timer(e, CHD_STAGE_BUILD);
    chd_status st = chd_epoch_tick(e, EP_BUILD);
    if (st != CHD_OK) return st;
    bool counts_recorded = false;
    if (!e->assigned && !e->halo_on_device) {
        // single-GPU flow: assign + sort as one replayable graph.  The key buffers swap every assignment
        // (handover detection compares against the previous keys), so there are two graph variants.
        uint32_t* target = e->have_prev_key ? e->d_prev_key : e->d_key;  // buffer the new keys will be written to
        const int slot = (target == e->d_key_a ? 0 : 1) + 2 * e->pos_buf;
        uint64_t key = mix_key(mix_key(mix_key(0x6275696c64ull, e->n_own), e->have_gid), e->have_prev_key);
        key = mix_key(mix_key(key, (uint64_t)(uintptr_t)target), (uint64_t)(uintptr_t)e->pos_x ^ ((uint64_t)(uintptr_t)e->pos_z << 1));
        // single-pass builds (<= 1023 cells) run as two replayable halves with an event in between: the cell CSR offsets are
        // final after the first (assignment + histogram + scan), so the emit preparation overlaps the scatter
        const bool split = e->g.cells + 1 <= BUILD_MAX_BINS && e->n_own > 0;
        st = run_stage(e, e->g_build[slot], key, [&]() { return build_enqueue(e, true, split ? 1 : 0); });
        if (st == CHD_OK && !e->assigned) {  // replayed graph: mirror the host-side bookkeeping of chd_assign_cells
            if (e->have_prev_key) {
                uint32_t* t = e->d_key;
                e->d_key = e->d_prev_key;
                e->d_prev_key = t;
            }
            if (e->n_own) e->have_prev_key = true;
            e->n_halo = 0;
            e->assigned = true;
        }
        if (st == CHD_OK && split) {
            CU(e, cudaEventRecord(e->ev_counts, e->stream));
            counts_recorded = true;
            st = run_stage(e, e->g_build_b[slot], mix_key(key, 0x62), [&]() { return build_enqueue(e, false, 2); });
        }
        if (st == CHD_OK) st = chd_note_pos_read(e);
    } else if (e->assigned && e->halo_on_device) {
        // multi-GPU flow: cells were assigned by chd_export_border and the halo appended on the device; the sort over
        // own + halo entities is sized by capacity (device-side length) and therefore replayable as well.
        const int slot = e->d_key == e->d_key_a ? 0 : 1;
        uint64_t key = mix_key(mix_key(mix_key(0x736f7274ull, e->lim.max_entities), e->have_gid), (uint64_t)(uintptr_t)e->d_key);
        st = run_stage(e, e->g_build[slot], key, [&]() { return build_enqueue(e, false); });
    } else {
        const bool with_assign = !e->assigned;
        st = build_enqueue(e, with_assign);
        if (st == CHD_OK && with_assign) st = chd_note_pos_read(e);
    }
    if (st != CHD_OK) return st;
    if (!counts_recorded) CU(e, cudaEventRecord(e->ev_counts, e->stream));  // (cell counts final = build done)
    e->n_sorted = e->n_own + e->n_halo;
    e->built = true;
    e->assigned_since_build = false;
    e->entities_dirty = false;
    return CHD_OK;
}
}  // extern "C"
