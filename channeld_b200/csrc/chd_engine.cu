// chd_engine.cu — engine object: create / destroy, streams, memory, look-back scan sites, instrumentation.
#include "chd_engine.h"

static thread_local std::string g_create_error;

// epochs start at 1 so that the zero-initialised descriptors (epoch 0) read as stale on first use
bool chd_init_epochs(chd_engine* e) {
    const unsigned long long ones[EP_COUNT] = {1, 1, 1, 1, 1, 1, 1, 1, 1};
    return cudaMemcpy(e->d_epoch, ones, sizeof ones, cudaMemcpyHostToDevice) == cudaSuccess;
}

bool chd_make_site(chd_engine* e, ScanSite& site, uint64_t n_max, int stage) {
    site.tiles = n_max == 0 ? 1 : (n_max + SCAN_TILE - 1) / SCAN_TILE;
    site.epoch = e->d_epoch + stage;
    site.error = e->d_ctr ? &e->d_ctr->overflow : nullptr;  // (sites made before d_ctr exists are patched in chd_create)
    site.stage = stage;
    if (std::find(e->sites.begin(), e->sites.end(), &site) == e->sites.end()) e->sites.push_back(&site);
    if (!dalloc(e, &site.desc, site.tiles)) return false;
    return cudaMemset(site.desc, 0, site.tiles * 8) == cudaSuccess;
}

// Zero-copy inputs: a pointer into this device's memory is consumed in place (no staging copy); the caller keeps it valid
// and unmodified until the work that reads it has finished (chd_summary / chd_sync / any chd_get_*).
bool chd_is_device_ptr(const chd_engine* e, const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice && a.device == e->device;
}

chd_status chd_epoch_tick(chd_engine* e, int stage) {
    if ((++e->stage_execs[stage] & ((1ull << 20) - 1)) != 0) return CHD_OK;
    for (ScanSite* site : e->sites)
        if (site->stage == stage && site->desc) CU(e, cudaMemsetAsync(site->desc, 0, site->tiles * 8, e->stream));
    return CHD_OK;
}

void chd_dfree(chd_engine* e, void* p) {
    if (!p) return;
    for (size_t i = 0; i < e->allocs.size(); i++)
        if (e->allocs[i] == p) {
            e->allocs.erase(e->allocs.begin() + (long)i);
            break;
        }
    cudaFree(p);
}

chd_status chd_ensure_upload_stream(chd_engine* e) {
    if (e->up_stream) return CHD_OK;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    CU(e, cudaStreamCreateWithPriority(&e->up_stream, cudaStreamNonBlocking, hi));
    CU(e, cudaEventCreateWithFlags(&e->ev_upload, cudaEventDisableTiming));
    CU(e, cudaEventCreateWithFlags(&e->ev_upload_q, cudaEventDisableTiming));
    CU(e, cudaEventCreateWithFlags(&e->ev_upload_rings, cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) {
        CU(e, cudaEventCreateWithFlags(&e->ev_q_read[i], cudaEventDisableTiming));
        CU(e, cudaEventCreateWithFlags(&e->ev_ring_read[i], cudaEventDisableTiming));
    }
    return CHD_OK;
}

chd_status chd_read_u32(chd_engine* e, const uint32_t* d, uint32_t* v) {
    CU(e, cudaMemcpyAsync(e->h_get, d, 4, cudaMemcpyDeviceToHost, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    *v = *e->h_get;
    return CHD_OK;
}

extern "C" {

uint32_t chd_abi_version(void) { return CHD_ABI_VERSION; }

uint32_t chd_damping_interval_ms(uint32_t dist, uint32_t default_ms) { return damping_interval_ms(dist, default_ms); }

void chd_default_limits(const chd_grid_cfg* cfg, uint32_t n_entities, uint32_t n_subscribers, chd_limits* lim) {
    memset(lim, 0, sizeof *lim);
    const uint64_t cells = (uint64_t)cfg->grid_cols * cfg->grid_rows;
    lim->max_entities = n_entities ? n_entities : 1;
    lim->max_subscribers = n_subscribers ? n_subscribers : 1;
    lim->max_queries = lim->max_subscribers;
    lim->max_spots = 1024;
    lim->max_pairs = (uint64_t)lim->max_subscribers * 16 + 1024;
    lim->max_window_cells = (uint64_t)lim->max_queries * 32 + 65536;
    const double per_cell = (double)n_entities / (double)(cells ? cells : 1);
    double v = (double)n_subscribers * 1.6 * per_cell * 1.5 + 1048576.0;
    if (v > 3.0e9) v = 3.0e9;
    lim->max_visible = (uint64_t)v;
    lim->max_ring_entries = (uint32_t)(cells * 64 < 1048576 ? 1048576 : (cells * 64 > 0x7fffffffull ? 0x7fffffffull : cells * 64));
    lim->max_due = (uint32_t)(lim->max_pairs * 2 > 0x7fffffffull ? 0x7fffffffull : lim->max_pairs * 2);
    lim->default_fanout_interval_ms = 20;  // GLOBAL defaults, settings.go:97-103
    lim->default_fanout_delay_ms = 0;
}

const char* chd_last_error(const chd_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

// NUMA node the GPU hangs off (sysfs), -1 if unknown: a host that runs its tick driver on that node's cores gets node-local
// pinned staging memory by first touch (measured: 37 GB/s -> > 50 GB/s H2D on the bench box when the staging memory is local)
int chd_device_numa_node(int device) {
    char bus[64] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    for (char* p = bus; *p; p++)
        if (*p >= 'A' && *p <= 'Z') *p = (char)(*p - 'A' + 'a');
    char path[160];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

void* chd_alloc_pinned(uint64_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void chd_free_pinned(void* p) {
    if (p) cudaFreeHost(p);
}

void chd_destroy(chd_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    chd_comm_destroy(e);
    if (e->up_stream) cudaStreamSynchronize(e->up_stream);
    for (void* p : e->allocs) cudaFree(p);
    for (auto* arr : {e->g_emit_prep, e->g_import})
        for (int i = 0; i < 2; i++)
            if (arr[i].exec) cudaGraphExecDestroy(arr[i].exec);
    for (auto* arr : {e->g_build, e->g_build_b, e->g_export, e->g_interest, e->g_interest_b, e->g_fanout})
        for (int i = 0; i < 4; i++)
            if (arr[i].exec) cudaGraphExecDestroy(arr[i].exec);
    for (cudaEvent_t ev : {e->ev_upload_q, e->ev_q_read[0], e->ev_q_read[1], e->ev_upload_rings, e->ev_ring_read[0], e->ev_ring_read[1]})
        if (ev) cudaEventDestroy(ev);
    if (e->up_stream) {
        cudaStreamSynchronize(e->up_stream);
        cudaStreamDestroy(e->up_stream);
    }
    if (e->ev_upload) cudaEventDestroy(e->ev_upload);
    for (int i = 0; i < 2; i++)
        if (e->ev_pos_read[i]) cudaEventDestroy(e->ev_pos_read[i]);
    if (e->ev) {
        for (size_t i = 0; i < (size_t)CHD_STAGE_COUNT * chd_engine::EV_RING * 2; i++)
            if (e->ev[i]) cudaEventDestroy(e->ev[i]);
        delete[] e->ev;
    }
    if (e->h_ctr) cudaFreeHost(e->h_ctr);
    if (e->h_u32) cudaFreeHost(e->h_u32);
    if (e->h_get) cudaFreeHost(e->h_get);
    if (e->aux_stream) cudaStreamDestroy(e->aux_stream);
    if (e->dl_stream) cudaStreamDestroy(e->dl_stream);
    if (e->dl_stream_b) cudaStreamDestroy(e->dl_stream_b);
    if (e->dl_stream_c) cudaStreamDestroy(e->dl_stream_c);
    for (int i = 0; i < 2; i++) {
        if (e->ev_fetch_a[i]) cudaEventDestroy(e->ev_fetch_a[i]);
        if (e->ev_fetch_b[i]) cudaEventDestroy(e->ev_fetch_b[i]);
        if (e->ev_fetch_done[i]) cudaEventDestroy(e->ev_fetch_done[i]);
    }
    if (e->ev_prep_done) cudaEventDestroy(e->ev_prep_done);
    if (e->ev_build_done) cudaEventDestroy(e->ev_build_done);
    if (e->ev_counts) cudaEventDestroy(e->ev_counts);
    if (e->prep_stream) cudaStreamDestroy(e->prep_stream);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    if (e->ev_interest) cudaEventDestroy(e->ev_interest);
    if (e->ev_pairs) cudaEventDestroy(e->ev_pairs);
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

static bool alloc_pairbuf(chd_engine* e, PairBuf& pb) {
    const uint64_t P = e->lim.max_pairs;
    return dalloc(e, &pb.off, (uint64_t)e->lim.max_subscribers + 1) && dalloc(e, &pb.sub, P) && dalloc(e, &pb.cell, P) &&
           dalloc(e, &pb.dist, P) && dalloc(e, &pb.interval, P) && dalloc(e, &pb.flags, P) && dalloc(e, &pb.last, P) &&
           dalloc(e, &pb.last_index, P);
}

chd_status chd_create(const chd_grid_cfg* cfg, const chd_limits* lim_in, int device, chd_engine** out) {
    if (!cfg || !out) {
        g_create_error = "null argument";
        return CHD_ERR_INVALID;
    }
    *out = nullptr;
    // LoadConfig validation (spatial.go:146-154); ServerInterestBorderSize == 0 tolerated (see header)
    if (!(cfg->grid_width > 0) || !(cfg->grid_height > 0)) {
        g_create_error = "GridWidth and GridHeight should be positive";
        return CHD_ERR_INVALID;
    }
    if (cfg->grid_cols == 0 || cfg->grid_rows == 0) {
        g_create_error = "GridCols and GridRows should be positive";
        return CHD_ERR_INVALID;
    }
    if (cfg->server_cols == 0 || cfg->server_rows == 0) {
        g_create_error = "ServerCols and ServerRows should be positive";
        return CHD_ERR_INVALID;
    }
    const uint64_t cells64 = (uint64_t)cfg->grid_cols * cfg->grid_rows;
    if (cells64 >= (1ull << 20)) {  // spatial id space is [0x10000, 0x80000) (settings.go:94-95): < 2^19 cells
        g_create_error = "too many cells (GridCols*GridRows must be < 2^20)";
        return CHD_ERR_INVALID;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        g_create_error = "no CUDA device: this engine has no CPU fallback";
        return CHD_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) {
        g_create_error = "bad device ordinal";
        return CHD_ERR_INVALID;
    }
    chd_engine* e = new (std::nothrow) chd_engine();
    if (!e) return CHD_ERR_INVALID;
    e->cfg = *cfg;
    if (lim_in)
        e->lim = *lim_in;
    else
        chd_default_limits(cfg, 1u << 20, 1u << 17, &e->lim);
    chd_limits& L = e->lim;
    if (!L.max_entities) L.max_entities = 1;
    if (!L.max_subscribers) L.max_subscribers = 1;
    if (!L.max_queries) L.max_queries = L.max_subscribers;
    if (!L.max_pairs) L.max_pairs = 1024;
    if (!L.max_window_cells) L.max_window_cells = 65536;
    if (!L.max_visible) L.max_visible = 1u << 20;
    if (!L.max_ring_entries) L.max_ring_entries = 1u << 16;
    if (!L.max_due) L.max_due = 1u << 16;
    if (L.max_pairs >= 0xFFFFFFF0ull || L.max_window_cells >= (1ull << 40) || L.max_entities >= (1u << 30)) {
        g_create_error = "limits too large (pairs are indexed with 32 bits)";
        delete e;
        return CHD_ERR_INVALID;
    }
    e->device = device;
#define CCU(call)                                                                       \
    do {                                                                                \
        cudaError_t _r = (call);                                                        \
        if (_r != cudaSuccess) {                                                        \
            g_create_error = std::string(#call " failed: ") + cudaGetErrorString(_r);   \
            chd_destroy(e);                                                             \
            return CHD_ERR_CUDA;                                                        \
        }                                                                               \
    } while (0)
    CCU(cudaSetDevice(device));
    CCU(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    e->own_stream = true;
    {
        // the aux stream carries short latency-bound kernels that should slot in ahead of the long emit kernel
        int lo_prio = 0, hi_prio = 0;
        CCU(cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio));
        CCU(cudaStreamCreateWithPriority(&e->aux_stream, cudaStreamNonBlocking, hi_prio));
    }
    CCU(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    CCU(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
    CCU(cudaEventCreateWithFlags(&e->ev_interest, cudaEventDisableTiming));
    CCU(cudaEventCreateWithFlags(&e->ev_pairs, cudaEventDisableTiming));
    CCU(cudaEventCreateWithFlags(&e->ev_prep_done, cudaEventDisableTiming));
    CCU(cudaEventCreateWithFlags(&e->ev_build_done, cudaEventDisableTiming));
    CCU(cudaEventCreateWithFlags(&e->ev_counts, cudaEventDisableTiming));
    {
        int lo_prio = 0, hi_prio2 = 0;
        CCU(cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio2));
        CCU(cudaStreamCreateWithPriority(&e->dl_stream, cudaStreamNonBlocking, hi_prio2));
        CCU(cudaStreamCreateWithPriority(&e->dl_stream_b, cudaStreamNonBlocking, hi_prio2));
        CCU(cudaStreamCreateWithPriority(&e->prep_stream, cudaStreamNonBlocking, hi_prio2));
    }
    CCU(cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, device));

    GridDev& g = e->g;
    g.off_x = cfg->world_offset_x; g.off_z = cfg->world_offset_z; g.w = cfg->grid_width; g.h = cfg->grid_height;
    g.grid_size = std::sqrt(g.w * g.w + g.h * g.h);                  // spatial.go:134-139
    g.world_x_hi = g.off_x + g.w * (double)cfg->grid_cols;           // spatial.go:126-132,287
    g.world_z_hi = g.off_z + g.h * (double)cfg->grid_rows;
    g.fcols = (double)cfg->grid_cols; g.frows = (double)cfg->grid_rows;
    g.cols = cfg->grid_cols; g.rows = cfg->grid_rows; g.cells = (uint32_t)cells64; g.id_start = cfg->channel_id_start;
    g.col_lo = 0; g.col_hi = g.cols; g.halo = 0;
    g.default_interval_ms = L.default_fanout_interval_ms; g.default_delay_ms = L.default_fanout_delay_ms;

    const uint64_t N = L.max_entities, S = L.max_subscribers, Q = L.max_queries, P = L.max_pairs, C = g.cells;
    e->build_blocks = (uint32_t)e->sm_count * 4;
    e->phase_stride = (uint32_t)(((N + 3) / 4) * 4 + 8);
    e->pc_blocks = (uint32_t)std::min<uint64_t>(4096, (P + BUILD_TILE - 1) / BUILD_TILE);
    if (e->pc_blocks == 0) e->pc_blocks = 1;
    e->ho_cap = L.max_entities;
    e->max_tiles = (L.max_visible + EMIT_WARP_TILE - 1) / EMIT_WARP_TILE + 1;  // (the smaller of the two tile sizes)
    uint64_t scan_n = (uint64_t)BUILD_MAX_BINS * e->build_blocks + 1;
    if (P + 1 > scan_n) scan_n = P + 1;
    if (Q + 1 > scan_n) scan_n = Q + 1;
    if (S + 1 > scan_n) scan_n = S + 1;
    if (N + 1 > scan_n) scan_n = N + 1;
    bool ok = true;
    ok = ok && dalloc(e, &e->d_x, N) && dalloc(e, &e->d_z, N) && (e->d_xb[0] = e->d_x, e->d_zb[0] = e->d_z, true) &&
         cudaEventCreateWithFlags(&e->ev_pos_read[0], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&e->ev_pos_read[1], cudaEventDisableTiming) == cudaSuccess && dalloc(e, &e->d_gid, N) && dalloc(e, &e->d_key, N) &&
         dalloc(e, &e->d_prev_key, N) && dalloc(e, &e->d_tmp_key, N) && dalloc(e, &e->d_tmp_val, N) &&
         dalloc(e, &e->d_sorted_key, N) && dalloc(e, &e->d_sorted4, 4 * (((N + 3) / 4) * 4 + 8)) && dalloc(e, &e->d_cell_start, C + 2) &&
         dalloc(e, &e->d_hist, (uint64_t)BUILD_MAX_BINS * e->build_blocks + 2) &&
         dalloc(e, &e->d_epoch, EP_COUNT) && chd_init_epochs(e) &&
         chd_make_site(e, e->site_hist, (uint64_t)BUILD_MAX_BINS * e->build_blocks + 1, EP_BUILD) &&
         chd_make_site(e, e->site_hist_b, (uint64_t)BUILD_MAX_BINS * e->build_blocks + 1, EP_BUILD) &&
         chd_make_site(e, e->site_qoff, Q + 1, EP_QUERY) && chd_make_site(e, e->site_slot, S + 1, EP_QUERY) &&
         chd_make_site(e, e->site_voff, P + 1, EP_EMIT) &&
         chd_make_site(e, e->site_border, N + 1, EP_BORDER) &&
         dalloc(e, &e->d_ho_entity, N) && dalloc(e, &e->d_ho_src, N) && dalloc(e, &e->d_ho_dst, N) &&
         dalloc(e, &e->d_bflag, N + 1) && dalloc(e, &e->d_boff, N + 2);
    e->d_sorted_ent = e->d_sorted4;  // phase copy 0 IS the plain sorted entity array
    e->d_key_a = e->d_key;
    ok = ok && dalloc(e, &e->d_conn, S) && dalloc(e, &e->d_slot_ctl, S) && dalloc(e, &e->d_slot_src, S) && dalloc(e, &e->d_lc_slot, S) &&
         dalloc(e, &e->d_lc_aux, S) && alloc_pairbuf(e, e->pairs[0]) && alloc_pairbuf(e, e->pairs[1]);
    ok = ok && dalloc(e, &e->dq.sub, Q) && dalloc(e, &e->dq.kind, Q) && dalloc(e, &e->dq.sph_cx, Q) && dalloc(e, &e->dq.sph_cz, Q) &&
         dalloc(e, &e->dq.sph_r, Q) && dalloc(e, &e->dq.box_cx, Q) && dalloc(e, &e->dq.box_cz, Q) && dalloc(e, &e->dq.box_ex, Q) &&
         dalloc(e, &e->dq.box_ez, Q) && dalloc(e, &e->dq.cone_cx, Q) && dalloc(e, &e->dq.cone_cz, Q) && dalloc(e, &e->dq.cone_dx, Q) &&
         dalloc(e, &e->dq.cone_dz, Q) && dalloc(e, &e->dq.cone_angle, Q) && dalloc(e, &e->dq.cone_r, Q) &&
         dalloc(e, &e->dq.spot_off, Q + 1) && dalloc(e, &e->dq.spot_ndist, Q) && dalloc(e, &e->dq.spot_x, (uint64_t)L.max_spots) &&
         dalloc(e, &e->dq.spot_z, (uint64_t)L.max_spots) && dalloc(e, &e->dq.spot_dist, (uint64_t)L.max_spots);
    ok = ok && dalloc(e, &e->d_bbox, Q) && dalloc(e, &e->d_win_off, Q + 1) && dalloc(e, &e->d_qstatus, Q) && dalloc(e, &e->d_win_cursor, 1) &&
         dalloc(e, &e->d_noff, S + 2) &&
         dalloc(e, &e->d_window, L.max_window_cells) && dalloc(e, &e->d_side_cell, (uint64_t)L.max_spots) &&
         dalloc(e, &e->d_side_dist, (uint64_t)L.max_spots) && dalloc(e, &e->d_side_cnt, Q) && dalloc(e, &e->d_status, Q) &&
         dalloc(e, &e->d_qcount, Q) && dalloc(e, &e->d_qoff, Q + 1) && dalloc(e, &e->d_qout_id, P) && dalloc(e, &e->d_qout_dist, P) &&
         dalloc(e, &e->d_slot_query, S);
    ok = ok && dalloc(e, &e->d_new_off, (Q > P ? Q : P) + 2) && dalloc(e, &e->d_new_sub, P) && dalloc(e, &e->d_new_ch, P) && dalloc(e, &e->d_gone_sub, P) &&
         dalloc(e, &e->d_gone_ch, P);
    ok = ok && dalloc(e, &e->d_pair_ch, P) && dalloc(e, &e->d_vcnt, P) && dalloc(e, &e->d_voff, P + 1) && dalloc(e, &e->d_first_pair, e->max_tiles + 8) && dalloc(e, &e->d_tile_desc, (L.max_visible + EMIT_TILE - 1) / EMIT_TILE + 8) &&
         dalloc(e, &e->d_general_tiles, (L.max_visible + EMIT_TILE - 1) / EMIT_TILE + 8) && dalloc(e, &e->d_n_general, 4) &&
         dalloc(e, &e->d_vis_off, S + 1) && dalloc(e, &e->d_vis, L.max_visible);
    ok = ok && dalloc(e, &e->d_cell_max_interval, C) && dalloc(e, &e->d_cell_start_ns, C) && dalloc(e, &e->d_rb_begin, C + 1) && dalloc(e, &e->d_rb_end, C + 1) &&
         dalloc(e, &e->d_ring_flat_off, C + 2) && dalloc(e, &e->d_upd_off, C + 1);
    ok = ok && dalloc(e, &e->d_ring_off, C + 1) && dalloc(e, &e->d_ring_arrival, (uint64_t)L.max_ring_entries) &&
         dalloc(e, &e->d_ring_sender, (uint64_t)L.max_ring_entries) && dalloc(e, &e->d_ring_index, (uint64_t)L.max_ring_entries) &&
         dalloc(e, &e->d_ch_msg_index, C) && dalloc(e, &e->d_by_cell, P) &&
         dalloc(e, &e->d_pc_hist, (uint64_t)BUILD_MAX_BINS * e->pc_blocks + 2) && dalloc(e, &e->d_pc_tmp_key, P) && dalloc(e, &e->d_pc_tmp_val, P) &&
         chd_make_site(e, e->site_pchist, (uint64_t)BUILD_MAX_BINS * e->pc_blocks + 1, EP_QUERY) &&
         chd_make_site(e, e->site_pchist_b, (uint64_t)BUILD_MAX_BINS * e->pc_blocks + 1, EP_QUERY) &&
         dalloc(e, &e->d_due, (uint64_t)L.max_due) && dalloc(e, &e->d_due_key, (uint64_t)L.max_due) && dalloc(e, &e->d_ctr, 1) && dalloc(e, &e->d_time, 2) &&
         dalloc(e, &e->d_ring_total, 1) && dalloc(e, &e->d_n_build, 1);
    if (!ok) {
        g_create_error = e->err;
        chd_destroy(e);
        return CHD_ERR_CUDA;
    }
    for (ScanSite* site : e->sites)
        site->error = &e->d_ctr->overflow;
    CCU(cudaHostAlloc((void**)&e->h_ctr, sizeof(Counters), cudaHostAllocDefault));
    CCU(cudaHostAlloc((void**)&e->h_u32, 64, cudaHostAllocDefault));
    CCU(cudaHostAlloc((void**)&e->h_get, 64, cudaHostAllocDefault));
    CCU(cudaMemsetAsync(e->d_ctr, 0, sizeof(Counters), e->stream));
    CCU(cudaMemsetAsync(e->d_win_cursor, 0, 8, e->stream));
    CCU(cudaMemsetAsync(e->d_n_general, 0, 16, e->stream));
    CCU(cudaMemsetAsync(e->d_slot_ctl, 0, S, e->stream));
    CCU(cudaMemsetAsync(e->d_cell_max_interval, 0, C * 4, e->stream));
    CCU(cudaMemsetAsync(e->d_cell_start_ns, 0, C * 8, e->stream));
    CCU(cudaMemsetAsync(e->d_ch_msg_index, 0, C * 8, e->stream));
    CCU(cudaMemsetAsync(e->d_conn, 0, S * 4, e->stream));
    CCU(cudaMemsetAsync(e->d_time, 0, 16, e->stream));
    CCU(cudaMemsetAsync(e->d_ring_total, 0, 4, e->stream));
    CCU(cudaMemsetAsync(e->pairs[0].off, 0, (S + 1) * 4, e->stream));
    CCU(cudaMemsetAsync(e->pairs[1].off, 0, (S + 1) * 4, e->stream));
    CCU(cudaMemsetAsync(e->d_ring_off, 0, (C + 1) * 4, e->stream));
    CCU(cudaMemsetAsync(e->d_cell_start, 0, (C + 2) * 4, e->stream));
    CCU(cudaMemsetAsync(e->d_vis_off, 0, (S + 1) * 8, e->stream));
    CCU(cudaStreamSynchronize(e->stream));
#undef CCU
    *out = e;
    return CHD_OK;
}

chd_status chd_set_stream(chd_engine* e, void* cuda_stream) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaStreamSynchronize(e->stream));
    if (e->own_stream) {
        cudaStreamDestroy(e->stream);
        e->own_stream = false;
    }
    e->stream = (cudaStream_t)cuda_stream;
    return CHD_OK;
}

chd_status chd_sync(chd_engine* e) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaStreamSynchronize(e->stream));
    return CHD_OK;
}

/* ------------------------------------------------------------------ instrumentation ---- */

uint64_t chd_launch_count(const chd_engine* e) { return e ? e->n_launch : 0; }

chd_status chd_enable_graphs(chd_engine* e, int on) {
    if (!e) return CHD_ERR_INVALID;
    e->use_graphs = on != 0;
    return CHD_OK;
}

uint64_t chd_graph_launch_count(const chd_engine* e) { return e ? e->graph_launches : 0; }

chd_status chd_profile_enable(chd_engine* e, int on) {
    if (!e) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    if (on && !e->ev) {
        const size_t n = (size_t)CHD_STAGE_COUNT * chd_engine::EV_RING * 2;
        e->ev = new cudaEvent_t[n]();
        for (size_t i = 0; i < n; i++) CU(e, cudaEventCreate(&e->ev[i]));
    }
    CU(e, cudaStreamSynchronize(e->stream));
    for (int s = 0; s < CHD_STAGE_COUNT; s++) e->stage_n[s] = 0;
    e->profiling = on == 2 ? 2 : (on != 0 ? 1 : 0);
    return CHD_OK;
}

chd_status chd_profile_timeline(chd_engine* e, int stage, double* start_ms, double* stop_ms) {
    if (!e || stage < 0 || stage >= CHD_STAGE_COUNT || !start_ms || !stop_ms || !e->ev) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaStreamSynchronize(e->stream));
    if (e->aux_stream) CU(e, cudaStreamSynchronize(e->aux_stream));
    if (!e->stage_n[CHD_STAGE_TICK] || !e->stage_n[stage]) return CHD_ERR_STATE;
    cudaEvent_t t0 = e->evt(CHD_STAGE_TICK, e->stage_n[CHD_STAGE_TICK] - 1, 0);
    float a = 0, b = 0;
    CU(e, cudaEventElapsedTime(&a, t0, e->evt(stage, e->stage_n[stage] - 1, 0)));
    CU(e, cudaEventElapsedTime(&b, t0, e->evt(stage, e->stage_n[stage] - 1, 1)));
    *start_ms = a;
    *stop_ms = b;
    return CHD_OK;
}

chd_status chd_profile_get(chd_engine* e, int stage, double* total_ms, uint64_t* samples) {
    if (!e || stage < 0 || stage >= CHD_STAGE_COUNT || !total_ms || !samples) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaStreamSynchronize(e->stream));
    const uint64_t n = e->stage_n[stage];
    const uint64_t m = n < (uint64_t)chd_engine::EV_RING ? n : (uint64_t)chd_engine::EV_RING;
    double tot = 0;
    for (uint64_t i = n - m; i < n; i++) {
        float ms = 0;
        CU(e, cudaEventElapsedTime(&ms, e->evt(stage, i, 0), e->evt(stage, i, 1)));
        tot += ms;
    }
    *total_ms = tot;
    *samples = m;
    return CHD_OK;
}
}  // extern "C"
