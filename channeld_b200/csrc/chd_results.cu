// chd_results.cu — results: getters, the one-call read-back of a tick (chd_fetch_results), device views.
#include "chd_engine.h"

#include "chd_misc.cuh"

// ---- asynchronous read-back (chd_fetch_results_async): result lists are written straight into the caller's PINNED host buffers by
// a copy kernel that knows the exact list lengths on the device (no host round trip to size a cudaMemcpy), so the host can
// enqueue the next tick before it looks at this one's results.
namespace {
struct PackSeg {
    const void* src;
    void* dst;
    const void* count_ptr;  // device address of the element count (nullptr: `fixed`)
    uint64_t fixed, cap;    // fixed count / capacity of dst in elements
    uint32_t elem_words;    // element size in 32-bit words
    uint32_t count_is_u64;
};
struct PackArgs {
    PackSeg seg[16];
    int n;
    uint32_t* truncated;  // pinned: set to 1 if a list did not fit its buffer
};
__global__ void __launch_bounds__(256) pack_kernel(PackArgs a) {
    const PackSeg sg = a.seg[blockIdx.y];
    uint64_t n = sg.fixed;
    if (sg.count_ptr) n = sg.count_is_u64 ? *reinterpret_cast<const unsigned long long*>(sg.count_ptr) : (uint64_t)*reinterpret_cast<const uint32_t*>(sg.count_ptr);
    if (n > sg.cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *a.truncated = 1;
        n = sg.cap;
    }
    const uint64_t words = n * sg.elem_words;
    const uint32_t* __restrict__ s = reinterpret_cast<const uint32_t*>(sg.src);
    uint32_t* __restrict__ d = reinterpret_cast<uint32_t*>(sg.dst);
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (uint64_t)gridDim.x * blockDim.x;
    if ((((uintptr_t)s | (uintptr_t)d) & 15) == 0) {  // 16-byte moves: full PCIe write bursts
        const uint64_t q = words / 4;
        const uint4* __restrict__ s4 = reinterpret_cast<const uint4*>(s);
        uint4* __restrict__ d4 = reinterpret_cast<uint4*>(d);
        for (uint64_t i = tid; i < q; i += nthr) d4[i] = s4[i];
        for (uint64_t i = q * 4 + tid; i < words; i += nthr) d[i] = s[i];
    } else {
        for (uint64_t i = tid; i < words; i += nthr) d[i] = s[i];
    }
}
bool is_pinned_host(const void* p) {
    if (!p) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}
}  // namespace

extern "C" {

chd_status chd_get_cells(chd_engine* e, uint32_t* cell_start, uint32_t* sorted_entity) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    const uint32_t C = e->g.cells;
    if (cell_start) CU(e, cudaMemcpyAsync(cell_start, e->d_cell_start, sizeof(uint32_t) * ((uint64_t)C + 1), cudaMemcpyDefault, e->stream));
    if (sorted_entity) {
        uint32_t nin = 0;
        chd_status st = chd_read_u32(e, e->d_cell_start + C, &nin);
        if (st != CHD_OK) return st;
        CU(e, cudaMemcpyAsync(sorted_entity, e->d_sorted_ent, sizeof(uint32_t) * nin, cudaMemcpyDefault, e->stream));
    }
    CU(e, cudaStreamSynchronize(e->stream));
    return CHD_OK;
}

chd_status chd_get_pairs(chd_engine* e, uint32_t* pair_off, uint32_t* channel_id, uint32_t* dist, uint32_t* interval_ms, uint8_t* flags,
                         int64_t* last_fanout_ns, uint64_t* last_message_index) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    PairBuf& pb = e->pairs[e->cur];
    const uint32_t S = e->n_slots;
    uint32_t P = 0;
    chd_status st = chd_read_u32(e, pb.off + S, &P);
    if (st != CHD_OK) return st;
    if (P > e->lim.max_pairs) return CHD_ERR_CAPACITY;
    cudaStream_t s = e->stream;
    if (pair_off) CU(e, cudaMemcpyAsync(pair_off, pb.off, sizeof(uint32_t) * ((uint64_t)S + 1), cudaMemcpyDefault, s));
    if (channel_id) {
        add_const_kernel<<<blocks_for(P ? P : 1, 256), 256, 0, s>>>(pb.cell, P, e->g.id_start, e->d_vcnt);
        KCHECK(e);
        CU(e, cudaMemcpyAsync(channel_id, e->d_vcnt, sizeof(uint32_t) * P, cudaMemcpyDefault, s));
    }
    if (dist) CU(e, cudaMemcpyAsync(dist, pb.dist, sizeof(uint32_t) * P, cudaMemcpyDefault, s));
    if (interval_ms) CU(e, cudaMemcpyAsync(interval_ms, pb.interval, sizeof(uint32_t) * P, cudaMemcpyDefault, s));
    if (flags) CU(e, cudaMemcpyAsync(flags, pb.flags, P, cudaMemcpyDefault, s));
    if (last_fanout_ns) CU(e, cudaMemcpyAsync(last_fanout_ns, pb.last, sizeof(int64_t) * P, cudaMemcpyDefault, s));
    if (last_message_index) CU(e, cudaMemcpyAsync(last_message_index, pb.last_index, sizeof(uint64_t) * P, cudaMemcpyDefault, s));
    CU(e, cudaStreamSynchronize(s));
    return CHD_OK;
}

chd_status chd_get_query_status(chd_engine* e, uint32_t* status, uint32_t n) {
    if (!e || !status) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    if (n > e->last_nq) n = e->last_nq;
    CU(e, cudaMemcpyAsync(status, e->d_status, sizeof(uint32_t) * n, cudaMemcpyDefault, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    return CHD_OK;
}

chd_status chd_get_diff(chd_engine* e, uint32_t* new_sub, uint32_t* new_channel, uint32_t* unsub_sub, uint32_t* unsub_channel) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaMemcpyAsync(e->h_ctr, e->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    const uint32_t nn = e->h_ctr->n_sub_new, nu = e->h_ctr->n_unsub;
    cudaStream_t s = e->stream;
    if (new_sub) CU(e, cudaMemcpyAsync(new_sub, e->d_new_sub, sizeof(uint32_t) * nn, cudaMemcpyDefault, s));
    if (new_channel) CU(e, cudaMemcpyAsync(new_channel, e->d_new_ch, sizeof(uint32_t) * nn, cudaMemcpyDefault, s));
    if (unsub_sub) CU(e, cudaMemcpyAsync(unsub_sub, e->d_gone_sub, sizeof(uint32_t) * nu, cudaMemcpyDefault, s));
    if (unsub_channel) CU(e, cudaMemcpyAsync(unsub_channel, e->d_gone_ch, sizeof(uint32_t) * nu, cudaMemcpyDefault, s));
    CU(e, cudaStreamSynchronize(s));
    return CHD_OK;
}

chd_status chd_get_visible(chd_engine* e, uint64_t* vis_off, uint32_t* vis_entity) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    const uint32_t S = e->n_slots;
    cudaStream_t s = e->stream;
    if (vis_off) CU(e, cudaMemcpyAsync(vis_off, e->d_vis_off, sizeof(uint64_t) * ((uint64_t)S + 1), cudaMemcpyDefault, s));
    if (vis_entity) {
        uint64_t* h64 = (uint64_t*)e->h_get;
        CU(e, cudaMemcpyAsync(h64, e->d_vis_off + S, 8, cudaMemcpyDeviceToHost, s));
        CU(e, cudaStreamSynchronize(s));
        const uint64_t V = *h64;
        if (V > e->lim.max_visible) return CHD_ERR_CAPACITY;
        CU(e, cudaMemcpyAsync(vis_entity, e->d_vis, sizeof(uint32_t) * V, cudaMemcpyDefault, s));
    }
    CU(e, cudaStreamSynchronize(s));
    return CHD_OK;
}

chd_status chd_get_visible_slot(chd_engine* e, uint32_t slot, uint32_t* out, uint64_t cap, uint64_t* count) {
    if (!e || !count || slot >= e->n_slots) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    uint64_t* h64 = (uint64_t*)e->h_get;
    CU(e, cudaMemcpyAsync(h64, e->d_vis_off + slot, 16, cudaMemcpyDeviceToHost, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    const uint64_t b = h64[0], n = h64[1] - h64[0];
    *count = n;
    if (h64[1] > e->lim.max_visible) return CHD_ERR_CAPACITY;
    const uint64_t m = n < cap ? n : cap;
    if (m && out) {
        CU(e, cudaMemcpyAsync(out, e->d_vis + b, sizeof(uint32_t) * m, cudaMemcpyDefault, e->stream));
        CU(e, cudaStreamSynchronize(e->stream));
    }
    return CHD_OK;
}

chd_status chd_get_due(chd_engine* e, chd_due* out, uint32_t cap) {
    if (!e || !out) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaMemcpyAsync(e->h_ctr, e->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    uint32_t n = e->h_ctr->n_due;
    if (n > e->lim.max_due) n = e->lim.max_due;  // the list overflowed (CHD_OVF_DUE): what fitted + CHD_DUE_VOID holes
    if (n > cap) n = cap;
    CU(e, cudaMemcpyAsync(out, e->d_due, sizeof(chd_due) * n, cudaMemcpyDefault, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    return CHD_OK;
}

chd_status chd_get_handover(chd_engine* e, uint32_t* entity, uint32_t* src_channel, uint32_t* dst_channel, uint32_t cap) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    uint32_t n = 0;
    chd_status st = chd_read_u32(e, &e->d_ctr->n_handover, &n);
    if (st != CHD_OK) return st;
    if (n > e->ho_cap) n = e->ho_cap;
    if (n > cap) n = cap;
    cudaStream_t s = e->stream;
    if (entity) CU(e, cudaMemcpyAsync(entity, e->d_ho_entity, sizeof(uint32_t) * n, cudaMemcpyDefault, s));
    if (src_channel) CU(e, cudaMemcpyAsync(src_channel, e->d_ho_src, sizeof(uint32_t) * n, cudaMemcpyDefault, s));
    if (dst_channel) CU(e, cudaMemcpyAsync(dst_channel, e->d_ho_dst, sizeof(uint32_t) * n, cudaMemcpyDefault, s));
    CU(e, cudaStreamSynchronize(s));
    return CHD_OK;
}

chd_status chd_fetch_results(chd_engine* e, const chd_result_buffers* b, chd_tick_summary* summary) {
    if (!e || !b || !summary) return CHD_ERR_INVALID;
    chd_status st;
    cudaStream_t s = e->stream;
    cudaStream_t main_stream = e->stream;
    const bool early = e->early_ready && e->dl_stream;
    // error exits: no copy into the caller's buffers may still be in flight when this returns
    auto drain = [&](chd_status r) {
        if (e->dl_stream) cudaStreamSynchronize(e->dl_stream);
        if (e->dl_stream_b) cudaStreamSynchronize(e->dl_stream_b);
        cudaStreamSynchronize(main_stream);
        return r;
    };
    Counters ca{};  // counters as of phase A
    if (early) {
        // The tick is probably still running.  Read back on a separate stream, in the order in which results become final:
        //   phase A  after the interest fill (ev_pairs) and the build: pairs, interest diff, query statuses, handover list, cell CSR
        //   phase B  after the aux chain (ev_join: fan-out) and the emit preparation (ev_prep_done): due list, visible offsets
        // while the emit kernel is still writing the expanded list.
        CU(e, cudaSetDevice(e->device));
        s = e->dl_stream;
        CU(e, cudaStreamWaitEvent(s, e->ev_pairs, 0));
        if (e->build_done_recorded) CU(e, cudaStreamWaitEvent(s, e->ev_build_done, 0));
        CU(e, cudaMemcpyAsync(e->h_ctr, e->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
        CU(e, cudaStreamSynchronize(s));  // sync A
        ca = *e->h_ctr;
        if (ca.overflow & CHD_OVF_PAIRS) {  // the pair arrays are incomplete: report through the full summary
            CU(e, cudaStreamSynchronize(main_stream));
            return chd_summary(e, summary);
        }
    } else {
        st = chd_summary(e, summary);  // sync #1 (also surfaces capacity overflows)
        if (st != CHD_OK) return st;
        ca.n_pairs = summary->n_pairs; ca.n_sub_new = summary->n_sub_new; ca.n_unsub = summary->n_unsub;
        ca.n_handover = summary->n_handover; ca.n_entities_in_world = summary->n_entities_in_world;
    }
    PairBuf& pb = e->pairs[e->cur];
    const uint32_t S = e->n_slots;
    const uint64_t P = ca.n_pairs;
    if ((b->pair_channel || b->pair_dist || b->pair_interval_ms) && P > b->pair_cap) {
        e->fail("chd_fetch_results: %llu pairs > pair_cap %llu", (unsigned long long)P, (unsigned long long)b->pair_cap);
        return drain(CHD_ERR_CAPACITY);
    }
    if (b->pair_off) CU(e, cudaMemcpyAsync(b->pair_off, pb.off, sizeof(uint32_t) * ((uint64_t)S + 1), cudaMemcpyDefault, s));
    if (b->pair_channel && e->pair_ch_valid) {
        CU(e, cudaMemcpyAsync(b->pair_channel, e->d_pair_ch, sizeof(uint32_t) * P, cudaMemcpyDefault, s));
    } else if (b->pair_channel) {
        add_const_kernel<<<blocks_for(P ? P : 1, 256), 256, 0, main_stream>>>(pb.cell, (uint32_t)P, e->g.id_start, e->d_vcnt);
        KCHECK(e);
        CU(e, cudaMemcpyAsync(b->pair_channel, e->d_vcnt, sizeof(uint32_t) * P, cudaMemcpyDefault, main_stream));
    }
    if (b->pair_dist) CU(e, cudaMemcpyAsync(b->pair_dist, pb.dist, sizeof(uint32_t) * P, cudaMemcpyDefault, s));
    if (b->pair_interval_ms) CU(e, cudaMemcpyAsync(b->pair_interval_ms, pb.interval, sizeof(uint32_t) * P, cudaMemcpyDefault, s));
    const uint64_t nn = ca.n_sub_new, nu = ca.n_unsub;
    if ((b->new_sub || b->new_channel) && nn > b->diff_cap) return drain(CHD_ERR_CAPACITY);
    if ((b->unsub_sub || b->unsub_channel) && nu > b->diff_cap) return drain(CHD_ERR_CAPACITY);
    if (b->new_sub) CU(e, cudaMemcpyAsync(b->new_sub, e->d_new_sub, sizeof(uint32_t) * nn, cudaMemcpyDefault, s));
    if (b->new_channel) CU(e, cudaMemcpyAsync(b->new_channel, e->d_new_ch, sizeof(uint32_t) * nn, cudaMemcpyDefault, s));
    if (b->unsub_sub) CU(e, cudaMemcpyAsync(b->unsub_sub, e->d_gone_sub, sizeof(uint32_t) * nu, cudaMemcpyDefault, s));
    if (b->unsub_channel) CU(e, cudaMemcpyAsync(b->unsub_channel, e->d_gone_ch, sizeof(uint32_t) * nu, cudaMemcpyDefault, s));
    if (b->handover_entity || b->handover_src || b->handover_dst) {
        uint32_t nh = ca.n_handover;
        if (nh > e->ho_cap) nh = e->ho_cap;
        if (nh > b->handover_cap) return drain(CHD_ERR_CAPACITY);
        if (b->handover_entity) CU(e, cudaMemcpyAsync(b->handover_entity, e->d_ho_entity, sizeof(uint32_t) * nh, cudaMemcpyDefault, s));
        if (b->handover_src) CU(e, cudaMemcpyAsync(b->handover_src, e->d_ho_src, sizeof(uint32_t) * nh, cudaMemcpyDefault, s));
        if (b->handover_dst) CU(e, cudaMemcpyAsync(b->handover_dst, e->d_ho_dst, sizeof(uint32_t) * nh, cudaMemcpyDefault, s));
    }
    if (b->query_status) {
        const uint32_t n = e->last_nq < b->status_cap ? e->last_nq : b->status_cap;
        CU(e, cudaMemcpyAsync(b->query_status, e->d_status, sizeof(uint32_t) * n, cudaMemcpyDefault, s));
    }
    if (b->cell_start) CU(e, cudaMemcpyAsync(b->cell_start, e->d_cell_start, sizeof(uint32_t) * ((uint64_t)e->g.cells + 1), cudaMemcpyDefault, s));
    if (b->sorted_entity) {
        if (ca.n_entities_in_world > b->entity_cap) return drain(CHD_ERR_CAPACITY);
        CU(e, cudaMemcpyAsync(b->sorted_entity, e->d_sorted_ent, sizeof(uint32_t) * (uint64_t)ca.n_entities_in_world, cudaMemcpyDefault, s));
    }
    cudaStream_t sa = s;  // stream carrying the phase-A copies
    if (early) {  // phase B, on its own stream: its counter read-back must not queue behind the phase-A copies
        s = e->dl_stream_b;
        CU(e, cudaStreamWaitEvent(s, e->ev_join, 0));
        CU(e, cudaStreamWaitEvent(s, e->ev_prep_done, 0));
        CU(e, cudaMemcpyAsync(e->h_ctr, e->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
        CU(e, cudaStreamSynchronize(s));  // sync B
        st = chd_decode_summary(e, summary);
        if (st != CHD_OK) return drain(st);
    }
    if (b->due) {
        if (summary->n_due > b->due_cap) return drain(CHD_ERR_CAPACITY);
        CU(e, cudaMemcpyAsync(b->due, e->d_due, sizeof(chd_due) * (uint64_t)summary->n_due, cudaMemcpyDefault, s));
    }
    if (b->vis_off) CU(e, cudaMemcpyAsync(b->vis_off, e->d_vis_off, sizeof(uint64_t) * ((uint64_t)S + 1), cudaMemcpyDefault, s));
    if (b->vis_entity) {
        if (summary->n_visible > b->vis_cap) return drain(CHD_ERR_CAPACITY);
        CU(e, cudaMemcpyAsync(b->vis_entity, e->d_vis, sizeof(uint32_t) * summary->n_visible, cudaMemcpyDefault, main_stream));
    }
    CU(e, cudaStreamSynchronize(s));  // last sync of the read-back stream(s)
    if (sa != s) CU(e, cudaStreamSynchronize(sa));
    if (s != main_stream) CU(e, cudaStreamSynchronize(main_stream));  // the tick itself (expanded list) has finished
    return CHD_OK;
}

chd_status chd_fetch_results_async(chd_engine* e, const chd_result_buffers* b, void* pinned_header) {
    if (!e || !b || !pinned_header) return CHD_ERR_INVALID;
    if (!e->early_ready || !e->dl_stream) {
        e->fail("chd_fetch_results_async needs a two-stream tick (chd_tick with emit, or chd_begin_interest + chd_tick) just before it");
        return CHD_ERR_STATE;
    }
    if (b->vis_entity) {
        e->fail("chd_fetch_results_async does not copy the expanded list (use chd_fetch_results / chd_get_visible)");
        return CHD_ERR_INVALID;
    }
    for (const void* p : {(const void*)b->pair_off, (const void*)b->pair_channel, (const void*)b->pair_dist, (const void*)b->pair_interval_ms, (const void*)b->new_sub,
                          (const void*)b->new_channel, (const void*)b->unsub_sub, (const void*)b->unsub_channel, (const void*)b->due, (const void*)b->handover_entity,
                          (const void*)b->handover_src, (const void*)b->handover_dst, (const void*)b->query_status, (const void*)b->vis_off,
                          (const void*)b->cell_start, (const void*)b->sorted_entity, (const void*)pinned_header})
        if (!is_pinned_host(p)) {
            e->fail("chd_fetch_results_async: every buffer must be pinned host memory (chd_alloc_pinned)");
            return CHD_ERR_INVALID;
        }
    CU(e, cudaSetDevice(e->device));
    if (e->fetch_issued - e->fetch_waited >= 2) {
        e->fail("chd_fetch_results_async: two fetches are already outstanding (call chd_fetch_wait)");
        return CHD_ERR_STATE;
    }
    const int fi = (int)(e->fetch_issued & 1);
    if (!e->ev_fetch_a[fi]) {
        CU(e, cudaEventCreateWithFlags(&e->ev_fetch_a[fi], cudaEventDisableTiming));
        CU(e, cudaEventCreateWithFlags(&e->ev_fetch_b[fi], cudaEventDisableTiming));
    }
    PairBuf& pb = e->pairs[e->cur];
    const uint32_t S = e->n_slots;
    Counters* ctr = e->d_ctr;
    uint32_t* hdr = reinterpret_cast<uint32_t*>(pinned_header);
    hdr[CHD_FETCH_HEADER_BYTES / 4 - 1] = 0;  // truncation flag (host write, ordered before the kernels are launched)
    auto seg = [](const void* src, void* dst, const void* cnt, uint64_t fixed, uint64_t cap, uint32_t words, uint32_t is64) {
        return PackSeg{src, dst, cnt, fixed, cap, words, is64};
    };
    // phase A: final once the interest fill and the build are done
    PackArgs A{};
    A.truncated = hdr + CHD_FETCH_HEADER_BYTES / 4 - 1;
    if (b->pair_off) A.seg[A.n++] = seg(pb.off, b->pair_off, nullptr, (uint64_t)S + 1, (uint64_t)S + 1, 1, 0);
    if (b->pair_channel) A.seg[A.n++] = seg(e->d_pair_ch, b->pair_channel, pb.off + S, 0, b->pair_cap, 1, 0);
    if (b->pair_dist) A.seg[A.n++] = seg(pb.dist, b->pair_dist, pb.off + S, 0, b->pair_cap, 1, 0);
    if (b->pair_interval_ms) A.seg[A.n++] = seg(pb.interval, b->pair_interval_ms, pb.off + S, 0, b->pair_cap, 1, 0);
    if (b->new_sub) A.seg[A.n++] = seg(e->d_new_sub, b->new_sub, &ctr->n_sub_new, 0, b->diff_cap, 1, 0);
    if (b->new_channel) A.seg[A.n++] = seg(e->d_new_ch, b->new_channel, &ctr->n_sub_new, 0, b->diff_cap, 1, 0);
    if (b->unsub_sub) A.seg[A.n++] = seg(e->d_gone_sub, b->unsub_sub, &ctr->n_unsub, 0, b->diff_cap, 1, 0);
    if (b->unsub_channel) A.seg[A.n++] = seg(e->d_gone_ch, b->unsub_channel, &ctr->n_unsub, 0, b->diff_cap, 1, 0);
    if (b->query_status) A.seg[A.n++] = seg(e->d_status, b->query_status, nullptr, std::min<uint64_t>(e->last_nq, b->status_cap), b->status_cap, 1, 0);
    if (b->cell_start) A.seg[A.n++] = seg(e->d_cell_start, b->cell_start, nullptr, (uint64_t)e->g.cells + 1, (uint64_t)e->g.cells + 1, 1, 0);
    if (b->sorted_entity) A.seg[A.n++] = seg(e->d_sorted_ent, b->sorted_entity, &ctr->n_entities_in_world, 0, b->entity_cap, 1, 0);
    PackArgs A2{};  // (the handover triple: a second launch keeps PackArgs small)
    A2.truncated = A.truncated;
    const uint64_t hcap = std::min<uint64_t>(b->handover_cap, e->ho_cap);
    if (b->handover_entity) A2.seg[A2.n++] = seg(e->d_ho_entity, b->handover_entity, &ctr->n_handover, 0, hcap, 1, 0);
    if (b->handover_src) A2.seg[A2.n++] = seg(e->d_ho_src, b->handover_src, &ctr->n_handover, 0, hcap, 1, 0);
    if (b->handover_dst) A2.seg[A2.n++] = seg(e->d_ho_dst, b->handover_dst, &ctr->n_handover, 0, hcap, 1, 0);
    // phase B: final after the fan-out pass and the emit preparation; the counters travel last
    PackArgs B{};
    B.truncated = A.truncated;
    if (b->due) B.seg[B.n++] = seg(e->d_due, b->due, &ctr->n_due, 0, std::min<uint64_t>(b->due_cap, e->lim.max_due), sizeof(chd_due) / 4, 0);
    if (b->vis_off) B.seg[B.n++] = seg(e->d_vis_off, b->vis_off, nullptr, (uint64_t)S + 1, (uint64_t)S + 1, 2, 0);
    B.seg[B.n++] = seg(ctr, pinned_header, nullptr, sizeof(Counters) / 4, sizeof(Counters) / 4, 1, 0);
    // ---- hop 1: snapshot into device staging (microseconds: the next tick is ordered after THIS, not after the PCIe transfer);
    //      hop 2: staging -> the caller's pinned buffers on a stream of its own, sized by the snapshot's own copy of the counts
    auto up16 = [](uint64_t v) { return (v + 15) & ~(uint64_t)15; };
    uint64_t need = 0;
    PackArgs* sets[3] = {&A, &A2, &B};
    for (PackArgs* pa : sets)
        for (int k = 0; k < pa->n; k++) need += up16(std::max<uint64_t>(pa->seg[k].cap, pa->seg[k].fixed) * pa->seg[k].elem_words * 4);
    need += 2 * up16(sizeof(Counters)) + 64;
    if (e->fetch_stage_bytes[fi] < need) {
        chd_dfree(e, e->d_fetch_stage[fi]);
        e->d_fetch_stage[fi] = nullptr;
        e->fetch_stage_bytes[fi] = 0;
        if (!dalloc(e, &e->d_fetch_stage[fi], need)) return CHD_ERR_CUDA;
        e->fetch_stage_bytes[fi] = need;
    }
    if (!e->dl_stream_c) {  // high priority like the other read-back streams: its CTAs must not queue behind the emit kernel's grid
        int lo_p = 0, hi_p = 0;
        CU(e, cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
        CU(e, cudaStreamCreateWithPriority(&e->dl_stream_c, cudaStreamNonBlocking, hi_p));
    }
    if (!e->ev_fetch_done[fi]) CU(e, cudaEventCreateWithFlags(&e->ev_fetch_done[fi], cudaEventDisableTiming));
    uint8_t* cursor = e->d_fetch_stage[fi];
    auto carve = [&](uint64_t bytes) {
        uint8_t* p = cursor;
        cursor += up16(bytes);
        return p;
    };
    Counters* ctr_a = reinterpret_cast<Counters*>(carve(sizeof(Counters)));  // the counts as they stand when phase A / B is final
    Counters* ctr_b = reinterpret_cast<Counters*>(carve(sizeof(Counters)));
    uint32_t* npairs_s = reinterpret_cast<uint32_t*>(carve(16));
    auto staged_count = [&](const void* cnt, Counters* snap) -> const void* {
        if (!cnt) return nullptr;
        if (cnt == (const void*)(pb.off + S)) return npairs_s;
        const uintptr_t o = (uintptr_t)cnt - (uintptr_t)ctr;
        return o < sizeof(Counters) ? (const void*)((const uint8_t*)snap + o) : cnt;
    };
    PackArgs H[3] = {};  // hop 2 of A, A2, B
    for (int j = 0; j < 3; j++) {
        PackArgs* pa = sets[j];
        H[j].truncated = pa->truncated;
        H[j].n = pa->n;
        for (int k = 0; k < pa->n; k++) {
            PackSeg& d1 = pa->seg[k];
            void* st = carve(std::max<uint64_t>(d1.cap, d1.fixed) * d1.elem_words * 4);
            H[j].seg[k] = d1;
            H[j].seg[k].src = st;
            H[j].seg[k].count_ptr = staged_count(d1.count_ptr, j == 2 ? ctr_b : ctr_a);
            d1.dst = st;  // hop 1 writes the snapshot
        }
    }
    // hop 1 also snapshots the counts themselves
    A.seg[A.n++] = seg(ctr, ctr_a, nullptr, sizeof(Counters) / 4, sizeof(Counters) / 4, 1, 0);
    A.seg[A.n++] = seg(pb.off + S, npairs_s, nullptr, 1, 1, 1, 0);
    B.seg[B.n++] = seg(ctr, ctr_b, nullptr, sizeof(Counters) / 4, sizeof(Counters) / 4, 1, 0);
    // (B's own copy of the counters to the pinned header reads the snapshot in hop 2)
    for (int k = 0; k < H[2].n; k++)
        if (H[2].seg[k].dst == pinned_header) H[2].seg[k].src = ctr_b;
    cudaStream_t sa = e->dl_stream, sb = e->dl_stream_b, sc = e->dl_stream_c;
    CU(e, cudaStreamWaitEvent(sa, e->ev_pairs, 0));
    if (e->build_done_recorded) CU(e, cudaStreamWaitEvent(sa, e->ev_build_done, 0));
    pack_kernel<<<dim3(24, (unsigned)A.n), 256, 0, sa>>>(A);
    KCHECK(e);
    if (A2.n) {
        pack_kernel<<<dim3(8, (unsigned)A2.n), 256, 0, sa>>>(A2);
        KCHECK(e);
    }
    CU(e, cudaEventRecord(e->ev_fetch_a[fi], sa));
    CU(e, cudaStreamWaitEvent(sc, e->ev_fetch_a[fi], 0));
    const bool prof = e->profiling == 1;
    if (prof) CU(e, cudaEventRecord(e->evt(CHD_STAGE_READBACK, e->stage_n[CHD_STAGE_READBACK], 0), sc));
    if (H[0].n) {
        pack_kernel<<<dim3(24, (unsigned)H[0].n), 256, 0, sc>>>(H[0]);
        KCHECK(e);
    }
    if (H[1].n) {
        pack_kernel<<<dim3(8, (unsigned)H[1].n), 256, 0, sc>>>(H[1]);
        KCHECK(e);
    }
    CU(e, cudaStreamWaitEvent(sb, e->ev_join, 0));
    CU(e, cudaStreamWaitEvent(sb, e->ev_prep_done, 0));
    pack_kernel<<<dim3(24, (unsigned)B.n), 256, 0, sb>>>(B);
    KCHECK(e);
    CU(e, cudaEventRecord(e->ev_fetch_b[fi], sb));
    CU(e, cudaStreamWaitEvent(sc, e->ev_fetch_b[fi], 0));
    pack_kernel<<<dim3(24, (unsigned)H[2].n), 256, 0, sc>>>(H[2]);
    KCHECK(e);
    CU(e, cudaEventRecord(e->ev_fetch_done[fi], sc));
    if (prof) {
        CU(e, cudaEventRecord(e->evt(CHD_STAGE_READBACK, e->stage_n[CHD_STAGE_READBACK], 1), sc));
        e->stage_n[CHD_STAGE_READBACK]++;
    }
    e->fetch_guard = true;  // the next tick's kernels are ordered after these copies (they overwrite the arrays being read)
    e->fetch_header[fi] = pinned_header;
    e->fetch_issued++;
    return CHD_OK;
}

chd_status chd_fetch_wait(chd_engine* e, chd_tick_summary* summary) {
    if (!e || !summary) return CHD_ERR_INVALID;
    if (e->fetch_issued == e->fetch_waited) {
        e->fail("chd_fetch_wait without a chd_fetch_results_async in flight");
        return CHD_ERR_STATE;
    }
    CU(e, cudaSetDevice(e->device));
    const int fi = (int)(e->fetch_waited & 1);  // the OLDEST outstanding fetch
    CU(e, cudaEventSynchronize(e->ev_fetch_done[fi]));
    e->fetch_waited++;
    static_assert(sizeof(Counters) + 4 <= CHD_FETCH_HEADER_BYTES, "CHD_FETCH_HEADER_BYTES too small");
    memcpy(e->h_ctr, e->fetch_header[fi], sizeof(Counters));
    const uint32_t truncated = reinterpret_cast<const uint32_t*>(e->fetch_header[fi])[CHD_FETCH_HEADER_BYTES / 4 - 1];
    chd_status st = chd_decode_summary(e, summary);
    if (st == CHD_OK && truncated) {
        e->fail("chd_fetch_results_async: a result list did not fit its buffer (truncated)");
        return CHD_ERR_CAPACITY;
    }
    return st;
}

chd_status chd_device_view(chd_engine* e, int which, void** d_ptr, uint64_t* count) {
    if (!e || !d_ptr) return CHD_ERR_INVALID;
    PairBuf& pb = e->pairs[e->cur];
    uint64_t c = 0;
    void* p = nullptr;
    switch (which) {
        case CHD_VIEW_CELL_START: p = e->d_cell_start; c = (uint64_t)e->g.cells + 2; break;
        case CHD_VIEW_SORTED_ENTITY: p = e->d_sorted_ent; c = e->n_sorted; break;
        case CHD_VIEW_ENT_CELL: p = e->d_key; c = e->n_own + e->n_halo; break;
        case CHD_VIEW_PAIR_OFF: p = pb.off; c = (uint64_t)e->n_slots + 1; break;
        case CHD_VIEW_PAIR_CHANNEL: p = pb.cell; c = e->lim.max_pairs; break;
        case CHD_VIEW_PAIR_DIST: p = pb.dist; c = e->lim.max_pairs; break;
        case CHD_VIEW_VIS_OFF: p = e->d_vis_off; c = (uint64_t)e->n_slots + 1; break;
        case CHD_VIEW_VIS_ENTITY: p = e->d_vis; c = e->lim.max_visible; break;
        case CHD_VIEW_DUE: p = e->d_due; c = e->lim.max_due; break;
        case CHD_VIEW_ENTER_OFF: p = e->vd.d_enter_off; c = (uint64_t)e->vd.S_out + 1; break;
        case CHD_VIEW_ENTER_ENTITY: p = e->vd.d_enter; c = e->vd.cap; break;
        case CHD_VIEW_LEAVE_OFF: p = e->vd.d_leave_off; c = (uint64_t)e->vd.S_out + 1; break;
        case CHD_VIEW_LEAVE_ENTITY: p = e->vd.d_leave; c = e->vd.cap; break;
        default: return CHD_ERR_INVALID;
    }
    if (which >= CHD_VIEW_ENTER_OFF && !e->vd.on) {
        e->fail("chd_device_view: the visibility delta is not enabled");
        return CHD_ERR_STATE;
    }
    *d_ptr = p;
    if (count) *count = c;
    return CHD_OK;
}
}  // extern "C"
