// chd_visdelta.cu — per-subscriber visibility deltas: chd_visible_delta_enable / chd_visible_delta / chd_get_visible_delta.
// Algorithm and semantics: chd_visdelta.cuh and include/chd_gpu.h.
#include "chd_engine.h"

#include "chd_visdelta.cuh"

// stable counting sort of the movers by one of their two keys (the build's radix passes, device-side length)
static chd_status vd_sort(chd_engine* e, const uint32_t* key_in, uint32_t* key_out, uint32_t* val_out, int site0) {
    chd_engine::VisDelta& V = e->vd;
    const uint32_t C = e->g.cells, N = e->lim.max_entities;
    uint32_t bits = 1;
    while ((1u << bits) < C + 1) bits++;  // keys are in [0, C]
    const uint32_t* n_ptr = &V.d_state->n_movers;
    if (bits <= 10)
        return chd_sort_pass_any(e, V.d_hist, V.site_h[site0], key_in, V.d_mv_ent, N, n_ptr, V.per_block, V.nb, 0, bits, key_out, val_out);
    const uint32_t bits0 = (bits + 1) / 2, bits1 = bits - bits0;
    chd_status st = chd_sort_pass_any(e, V.d_hist, V.site_h[site0], key_in, V.d_mv_ent, N, n_ptr, V.per_block, V.nb, 0, bits0, V.d_tmp_key,
                                      V.d_tmp_val);
    if (st != CHD_OK) return st;
    return chd_sort_pass_any(e, V.d_hist, V.site_h[site0 + 1], V.d_tmp_key, V.d_tmp_val, N, n_ptr, V.per_block, V.nb, bits0, bits1, key_out, val_out);
}

extern "C" {

chd_status chd_visible_delta_enable(chd_engine* e, uint64_t cap_entries) {
    if (!e) return CHD_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lk(e->mu);
    CU(e, cudaSetDevice(e->device));
    chd_engine::VisDelta& V = e->vd;
    const uint64_t N = e->lim.max_entities, S = e->lim.max_subscribers, P = e->lim.max_pairs, C = e->g.cells;
    if (!V.on) {
        V.nb = (uint32_t)std::min<uint64_t>((uint64_t)e->sm_count, (N + BUILD_TILE - 1) / BUILD_TILE);
        if (V.nb == 0) V.nb = 1;
        V.per_block = (uint32_t)(((N + V.nb - 1) / V.nb + BUILD_TILE - 1) / BUILD_TILE * BUILD_TILE);
        const uint64_t hist = (uint64_t)BUILD_MAX_BINS * V.nb;
        bool ok = dalloc(e, &V.d_state, 1) && dalloc(e, &V.d_base_key, N) && dalloc(e, &V.d_base_cs, C + 2) && dalloc(e, &V.d_base_sorted, N) &&
                  dalloc(e, &V.d_base_off, S + 1) && dalloc(e, &V.d_base_cell, P) && dalloc(e, &V.d_base_sub, P) && dalloc(e, &V.d_mv_ent, N) &&
                  dalloc(e, &V.d_mv_dkey, N) && dalloc(e, &V.d_mv_skey, N) && dalloc(e, &V.d_tmp_key, N) && dalloc(e, &V.d_tmp_val, N) &&
                  dalloc(e, &V.d_dst_key, N) && dalloc(e, &V.d_dst_ent, N) && dalloc(e, &V.d_src_key, N) && dalloc(e, &V.d_src_ent, N) &&
                  dalloc(e, &V.d_dst_start, C + 2) && dalloc(e, &V.d_src_start, C + 2) && dalloc(e, &V.d_hist, hist + 2) &&
                  dalloc(e, &V.d_ecnt, P) && dalloc(e, &V.d_lcnt, P) && dalloc(e, &V.d_epoff, P + 1) && dalloc(e, &V.d_lpoff, P + 1) &&
                  dalloc(e, &V.d_enter_off, S + 1) && dalloc(e, &V.d_leave_off, S + 1) && chd_make_site(e, V.site_mv, N, EP_DELTA) &&
                  chd_make_site(e, V.site_e, P + 1, EP_DELTA) && chd_make_site(e, V.site_l, P + 1, EP_DELTA);
        for (int i = 0; i < 4 && ok; i++) ok = chd_make_site(e, V.site_h[i], hist + 1, EP_DELTA);
        if (!ok) return CHD_ERR_CUDA;
        for (ScanSite* site : {&V.site_mv, &V.site_e, &V.site_l, &V.site_h[0], &V.site_h[1], &V.site_h[2], &V.site_h[3]}) site->error = &e->d_ctr->overflow;
        // the empty baseline: no entity, no slot, no pair
        CU(e, cudaMemsetAsync(V.d_state, 0, sizeof(VdState), e->stream));
        CU(e, cudaMemsetAsync(V.d_base_cs, 0, (C + 2) * 4, e->stream));
        CU(e, cudaMemsetAsync(V.d_base_off, 0, (S + 1) * 4, e->stream));
        CU(e, cudaMemsetAsync(V.d_enter_off, 0, (S + 1) * 8, e->stream));
        CU(e, cudaMemsetAsync(V.d_leave_off, 0, (S + 1) * 8, e->stream));
        V.on = true;
    }
    if (cap_entries > V.cap || !V.d_enter) {  // the output lists grow; the baseline is kept
        CU(e, cudaStreamSynchronize(e->stream));
        chd_dfree(e, V.d_enter);
        chd_dfree(e, V.d_leave);
        V.d_enter = V.d_leave = nullptr;
        const uint64_t cap = std::max<uint64_t>(cap_entries, V.cap);
        if (!dalloc(e, &V.d_enter, cap) || !dalloc(e, &V.d_leave, cap)) {
            V.cap = 0;
            return CHD_ERR_CUDA;
        }
        V.cap = cap;
    }
    return CHD_OK;
}

chd_status chd_visible_delta(chd_engine* e) {
    if (!e) return CHD_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lk(e->mu);
    chd_engine::VisDelta& V = e->vd;
    if (!V.on) {
        e->fail("chd_visible_delta: call chd_visible_delta_enable first");
        return CHD_ERR_STATE;
    }
    if (!e->built || e->assigned_since_build) {
        e->fail("chd_visible_delta: needs a chd_build of the current cell assignment");
        return CHD_ERR_STATE;
    }
    if (e->slab_set || e->comm || e->halo_on_device || e->n_halo || e->have_gid) {
        e->fail("chd_visible_delta: single-engine only (slab, communicator or global entity ids set)");
        return CHD_ERR_STATE;
    }
    if (e->interest_pending) {
        e->fail("chd_visible_delta: chd_begin_interest has not been joined by chd_tick yet");
        return CHD_ERR_STATE;
    }
    CU(e, cudaSetDevice(e->device));
    cudaStream_t s = e->stream;
    const uint32_t C = e->g.cells, S_now = e->n_slots, n_now = e->n_sorted;
    const uint32_t S_out = std::max(S_now, V.S_bound);
    V.n_bound = std::max(V.n_bound, n_now);
    PairBuf& cur = e->pairs[e->cur];
    VdState* st = V.d_state;
    chd_status r = chd_epoch_tick(e, EP_DELTA);
    if (r != CHD_OK) return r;
    vd_begin_kernel<<<1, 1, 0, s>>>(st, e->d_epoch + EP_DELTA, n_now, S_now, cur.off);
    KCHECK(e);
    // 1. movers: compaction in entity order, then two stable counting sorts (by destination / by source cell) + their CSR offsets
    const VdMoverFlag flag{e->d_key, V.d_base_key, st, C};
    SCAN(e, compact_1p(flag, VdMoverSink{flag, V.d_mv_ent, V.d_mv_dkey, V.d_mv_skey, &st->n_movers}, V.n_bound, V.site_mv, s));
    r = vd_sort(e, V.d_mv_dkey, V.d_dst_key, V.d_dst_ent, 0);
    if (r != CHD_OK) return r;
    r = vd_sort(e, V.d_mv_skey, V.d_src_key, V.d_src_ent, 2);
    if (r != CHD_OK) return r;
    vd_bounds_kernel<<<blocks_for((uint64_t)C + 2, 256), 256, 0, s>>>(V.d_dst_key, &st->n_movers, C, V.d_dst_start);
    KCHECK(e);
    vd_bounds_kernel<<<blocks_for((uint64_t)C + 2, 256), 256, 0, s>>>(V.d_src_key, &st->n_movers, C, V.d_src_start);
    KCHECK(e);
    // 2./3. enter over the current pairs, leave over the baseline pairs: count, scan, offsets + overflow decision, write
    const VdSide enter{cur.sub, cur.cell, &st->P_now, V.d_base_off, V.d_base_cell, &st->S_base, e->d_cell_start, e->d_sorted_ent,
                       V.d_dst_start, V.d_dst_ent, V.d_base_key, &st->n_base, C};
    const VdSide leave{V.d_base_sub, V.d_base_cell, &st->P_base, cur.off, cur.cell, &st->S_now, V.d_base_cs, V.d_base_sorted,
                       V.d_src_start, V.d_src_ent, e->d_key, &st->n_now, C};
    const unsigned grid = (unsigned)e->sm_count * 8;  // persistent: one warp per pair, strided
    vd_pairs_kernel<false><<<grid, 256, 0, s>>>(enter, st, V.d_ecnt, nullptr, nullptr);
    KCHECK(e);
    vd_pairs_kernel<false><<<grid, 256, 0, s>>>(leave, st, V.d_lcnt, nullptr, nullptr);
    KCHECK(e);
    const uint64_t P = e->lim.max_pairs;
    SCAN(e, exclusive_scan_1p<uint32_t, uint64_t>(V.d_ecnt, V.d_epoff, P, V.site_e, s, &st->P_now));
    SCAN(e, exclusive_scan_1p<uint32_t, uint64_t>(V.d_lcnt, V.d_lpoff, P, V.site_l, s, &st->P_base));
    auto* epoff = reinterpret_cast<unsigned long long*>(V.d_epoff);
    auto* lpoff = reinterpret_cast<unsigned long long*>(V.d_lpoff);
    vd_offsets_kernel<<<blocks_for((uint64_t)S_out + 1, 256), 256, 0, s>>>(st, S_out, cur.off, V.d_base_off, epoff, lpoff, V.cap,
                                                                           reinterpret_cast<unsigned long long*>(V.d_enter_off),
                                                                           reinterpret_cast<unsigned long long*>(V.d_leave_off));
    KCHECK(e);
    vd_pairs_kernel<true><<<grid, 256, 0, s>>>(enter, st, nullptr, epoff, V.d_enter);
    KCHECK(e);
    vd_pairs_kernel<true><<<grid, 256, 0, s>>>(leave, st, nullptr, lpoff, V.d_leave);
    KCHECK(e);
    // 4. the current state becomes the baseline (skipped on the device after an overflow)
    const VdSnap snap{e->d_key, e->d_cell_start, e->d_sorted_ent, cur.off, cur.cell, cur.sub,
                      V.d_base_key, V.d_base_cs, V.d_base_sorted, V.d_base_off, V.d_base_cell, V.d_base_sub, C};
    vd_snapshot_kernel<<<dim3((unsigned)e->sm_count, 6), 256, 0, s>>>(st, snap);
    KCHECK(e);
    V.S_out = S_out;
    V.S_call = S_now;
    V.S_bound = S_out;  // the baseline holds S_now slots after a success, its old count after an overflow
    V.called = true;
    return CHD_OK;
}

chd_status chd_get_visible_delta(chd_engine* e, uint64_t* enter_off, uint32_t* enter_entity, uint64_t enter_cap, uint64_t* leave_off,
                                 uint32_t* leave_entity, uint64_t leave_cap, uint64_t* n_enter, uint64_t* n_leave) {
    if (!e) return CHD_ERR_INVALID;
    chd_engine::VisDelta& V = e->vd;
    if (!V.called) {
        e->fail("chd_get_visible_delta: no chd_visible_delta has been enqueued");
        return CHD_ERR_STATE;
    }
    CU(e, cudaSetDevice(e->device));
    cudaStream_t s = e->stream;
    static_assert(sizeof(VdState) <= 64, "h_get holds 64 bytes");
    CU(e, cudaMemcpyAsync(e->h_get, V.d_state, sizeof(VdState), cudaMemcpyDeviceToHost, s));
    CU(e, cudaStreamSynchronize(s));
    VdState h;
    memcpy(&h, e->h_get, sizeof h);
    if (n_enter) *n_enter = h.n_enter;
    if (n_leave) *n_leave = h.n_leave;
    const uint64_t offs = (uint64_t)V.S_out + 1;
    if (enter_off) CU(e, cudaMemcpyAsync(enter_off, V.d_enter_off, 8 * offs, cudaMemcpyDefault, s));
    if (leave_off) CU(e, cudaMemcpyAsync(leave_off, V.d_leave_off, 8 * offs, cudaMemcpyDefault, s));
    chd_status ret = CHD_OK;
    if (h.ovf) {
        e->fail("chd_visible_delta: %llu enter / %llu leave entries > capacity %llu (baseline kept)", (unsigned long long)h.n_enter,
                (unsigned long long)h.n_leave, (unsigned long long)V.cap);
        ret = CHD_ERR_CAPACITY;
    } else {
        V.S_bound = V.S_call;  // the baseline advanced to the slot count of that call
        if ((enter_entity && h.n_enter > enter_cap) || (leave_entity && h.n_leave > leave_cap)) {
            e->fail("chd_get_visible_delta: %llu enter / %llu leave entries > caller capacity %llu / %llu", (unsigned long long)h.n_enter,
                    (unsigned long long)h.n_leave, (unsigned long long)enter_cap, (unsigned long long)leave_cap);
            ret = CHD_ERR_CAPACITY;
        } else {
            if (enter_entity) CU(e, cudaMemcpyAsync(enter_entity, V.d_enter, 4 * h.n_enter, cudaMemcpyDefault, s));
            if (leave_entity) CU(e, cudaMemcpyAsync(leave_entity, V.d_leave, 4 * h.n_leave, cudaMemcpyDefault, s));
        }
    }
    CU(e, cudaStreamSynchronize(s));
    return ret;
}

}  // extern "C"
