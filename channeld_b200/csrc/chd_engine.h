// chd_engine.h — internal: the engine object behind include/chd_gpu.h and the helpers its translation units share.
// Layout of the host code (all device buffers are allocated once in chd_create; the tick path allocates nothing and —
// apart from chd_summary / the chd_get_* copies — never synchronises with the host):
//   chd_engine.cu    create / destroy, streams, memory, CUDA-graph stage cache, instrumentation
//   chd_entities.cu  positions, cell assignment, spatial-hash build, radix sort passes
//   chd_interest.cu  subscribers (lifecycle), query batches, QueryChannelIds, interest update
//   chd_tick.cu      emit, rings, fan-out, the batched tick and its two-stream choreography, summary
//   chd_results.cu   getters, chd_fetch_results, device views
//   chd_shard.cu     multi-GPU X-slabs: border export, halo import, the NCCL exchange
//   chd_extras.cu    window classes, ADJACENT_CHANNELS broadcast sets, config-plane helpers
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "chd_scan.cuh"
#include "chd_types.cuh"

using namespace chd;

struct chd_engine {
    chd_grid_cfg cfg;
    chd_limits lim;
    GridDev g;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // Guards (a) the shared query scratch between the stateless query entry points and the tick driver and (b) the
    // temporary redirection of `stream` to aux_stream while the interest / fan-out chain is being enqueued.
    std::recursive_mutex mu;
    mutable std::string err;
    std::vector<void*> allocs;
    int sm_count = 148;
    uint64_t n_launch = 0;  // kernels launched by this engine (bench.py reports it as gpu_launches)
    // CUDA graphs: the launch-bound small-kernel stages are captured once per (shape, parity) and replayed.
    struct GraphSlot {
        cudaGraphExec_t exec = nullptr;
        uint64_t key = 0, pending_key = 0;
        uint64_t nodes = 0;
    };
    bool use_graphs = true;
    bool overlap_fanout = true;        // chd_tick runs interest + fan-out on aux_stream concurrently with build + emit
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_interest = nullptr, ev_pairs = nullptr;
    bool interest_pending = false, pending_fanout = false;  // chd_begin_interest issued, not yet joined by chd_tick
    GraphSlot g_build[4], g_build_b[4], g_interest[4], g_interest_b[4], g_emit_prep[2], g_fanout[4], g_export[8], g_import[4];  // build / export: [key buffer][position buffer]
    uint64_t graph_launches = 0, graph_captures = 0;
    uint32_t* d_key_a = nullptr;  // identity of the first key buffer (graph slot selection)
    int64_t* d_time = nullptr;      // [0] = now_ns of the last update_interest, [1] = t_ns of the last fanout_tick
    uint32_t* d_ring_total = nullptr;
    // optional per-stage CUDA-event timing (chd_profile_*): [stage][0=start,1=stop]
    int profiling = 0;  // 0 off, 1 every stage, 2 the emit kernel only
    static constexpr int EV_RING = 1024;
    cudaEvent_t* ev = nullptr;  // [CHD_STAGE_COUNT][EV_RING][2]
    uint64_t stage_n[CHD_STAGE_COUNT] = {};
    cudaEvent_t& evt(int stage, uint64_t i, int which) { return ev[((size_t)stage * EV_RING + (size_t)(i % EV_RING)) * 2 + which]; }

    // ---- entities
    uint32_t n_own = 0, n_halo = 0;  // entities with positions / appended halo records
    bool halo_on_device = false;     // multi-GPU: the build length (own + halo) lives in d_n_build
    uint32_t* d_n_build = nullptr;
    bool have_gid = false;
    double *d_x = nullptr, *d_z = nullptr;        // engine-owned staging for host inputs (the FRONT buffers)
    // chd_prefetch_entities: the BACK buffers receive the next tick's positions on `up_stream` while the current tick runs;
    // chd_adopt_prefetched swaps front and back.  ev_pos_read[b] = last assign_cells that read buffer pair b.
    double *d_xb[2] = {nullptr, nullptr}, *d_zb[2] = {nullptr, nullptr};
    uint32_t *d_general_tiles = nullptr, *d_n_general = nullptr;  // tiles with more than two segments: list, {length, consumer ticket}
    float* d_pos_f32[2] = {nullptr, nullptr};  // float staging of chd_set_entities_f32 [0] / chd_prefetch_entities_f32 [1]: x then z
    int pos_buf = 0;
    cudaStream_t up_stream = nullptr;
    cudaEvent_t ev_upload = nullptr, ev_pos_read[2] = {nullptr, nullptr};
    bool pos_read_recorded[2] = {false, false};
    bool staged = false;
    uint32_t staged_n = 0;
    const double *pos_x = nullptr, *pos_z = nullptr;  // what the kernels read: the staging buffers, or the caller's device arrays
    uint32_t *d_gid = nullptr;            // [max_entities] global ids (multi-GPU) of own + halo
    uint32_t *d_key = nullptr, *d_prev_key = nullptr;  // [max_entities] cell key per entity
    uint32_t *d_tmp_key = nullptr, *d_tmp_val = nullptr, *d_sorted_key = nullptr, *d_sorted_ent = nullptr;
    uint32_t *d_cell_start = nullptr;     // [C+2]
    uint32_t *d_sorted4 = nullptr;        // 4 phase-shifted copies of d_sorted_ent (chd_emit.cuh), stride = phase_stride
    uint32_t phase_stride = 0;
    uint32_t *d_hist = nullptr;           // [BUILD_MAX_BINS * nblocks + 1]
    // one look-back scan site per call site: stages run concurrently on two streams and must not share scan state
    unsigned long long* d_epoch = nullptr;  // [EP_COUNT] stage epochs for the look-back scans
    ScanSite site_hist_b{}, site_pchist_b{}, site_hist{}, site_qoff{}, site_slot{}, site_pchist{}, site_voff{}, site_border{};
    uint64_t stage_execs[9] = {};  // [EP_COUNT]
    std::vector<ScanSite*> sites;  // every scan site (chd_make_site registers them)
    uint32_t build_blocks = 0;
    bool assigned = false, built = false, have_prev_key = false, entities_dirty = false;
    uint32_t n_sorted = 0;
    // handover
    uint32_t *d_ho_entity = nullptr, *d_ho_src = nullptr, *d_ho_dst = nullptr;
    uint32_t ho_cap = 0;

    // ---- subscribers / pairs
    uint32_t n_slots = 0;
    uint32_t* d_conn = nullptr;
    // lifecycle: pending per-slot changes (SLOT_*), applied by the next interest update; source record of an immigrant;
    // staging for the slot / connection-id lists of chd_add_subscribers / chd_remove_subscribers / chd_migrate_*
    uint8_t* d_slot_ctl = nullptr;
    uint32_t *d_slot_src = nullptr, *d_lc_slot = nullptr, *d_lc_aux = nullptr;
    bool lifecycle_used = false;  // the interest kernels look at d_slot_ctl only once a lifecycle call has been made
    MigView mig{nullptr, 0, 0, 0};  // gathered migration blobs of this tick (chd_shard.cu)
    PairBuf pairs[2];
    int cur = 0;
    // ---- query scratch
    struct QStage {
        uint32_t *sub; uint8_t* kind;
        double *sph_cx, *sph_cz, *sph_r, *box_cx, *box_cz, *box_ex, *box_ez, *cone_cx, *cone_cz, *cone_dx, *cone_dz, *cone_angle, *cone_r;
        uint32_t *spot_off, *spot_ndist; double *spot_x, *spot_z; uint32_t* spot_dist;
    } dq{};
    // chd_prefetch_queries / chd_prefetch_rings: two dedicated staging sets each (allocated on first use), filled on
    // up_stream while a tick is in flight and handed to the next tick by chd_adopt_prefetched
    QStage dq_pf[2] = {};
    bool dq_pf_alloc[2] = {false, false};
    int q_next = 0;                       // set the next chd_prefetch_queries fills
    bool staged_q = false, have_adopted_q = false, wait_q = false;
    int staged_q_set = 0, adopted_q_set = 0;
    QueryDev staged_qd{}, adopted_qd{};
    cudaEvent_t ev_upload_q = nullptr, ev_q_read[2] = {nullptr, nullptr};
    bool q_read_recorded[2] = {false, false};
    struct RStage {
        uint32_t *off, *sender; int64_t* arrival; uint64_t *index, *cmi;
    } ring_pf[2] = {};
    bool ring_pf_alloc[2] = {false, false};
    int ring_next = 0, staged_ring_set = 0, ring_set = -1;  // ring_set: prefetch set the current ring pointers refer to (-1: none)
    bool staged_rings = false, staged_ring_cmi = false, wait_rings = false;
    uint32_t staged_ring_total = 0;
    cudaEvent_t ev_upload_rings = nullptr, ev_ring_read[2] = {nullptr, nullptr};
    bool ring_read_recorded[2] = {false, false};
    Bbox* d_bbox = nullptr;
    uint32_t *d_window = nullptr, *d_side_cell = nullptr, *d_side_dist = nullptr, *d_side_cnt = nullptr;
    uint64_t* d_win_off = nullptr;
    uint32_t *d_status = nullptr, *d_qcount = nullptr;
    uint32_t* d_qstatus = nullptr;              // statuses of the stateless query path (chd_query_channel_ids)
    unsigned long long* d_win_cursor = nullptr;  // bump cursor of the window scratch (zeroed by the stage's first kernel)
    uint32_t* d_noff = nullptr;                 // [S+1] new pair offsets, scanned into scratch: the interest update is transactional
    uint64_t* d_qoff = nullptr;  // stateless query CSR offsets
    uint32_t *d_qout_id = nullptr, *d_qout_dist = nullptr;
    int32_t* d_slot_query = nullptr;
    uint32_t last_nq = 0;
    // diff
    uint32_t *d_new_off = nullptr;  // scratch for u64 -> u32 offset narrowing (stateless query path)
    uint32_t *d_new_sub = nullptr, *d_new_ch = nullptr, *d_gone_sub = nullptr, *d_gone_ch = nullptr;
    // emit
    uint32_t *d_vcnt = nullptr, *d_first_pair = nullptr, *d_vis = nullptr;
    TileDesc* d_tile_desc = nullptr;  // per-tile copy descriptors (chd_emit.cuh)
    uint32_t* d_pair_ch = nullptr;  // channel id of every current pair (written by interest_fill_kernel)
    // ---- window classes of the due list (chd_due_classes): keys written by the fan-out kernel, scratch allocated on first use
    DueKey* d_due_key = nullptr;
    uint32_t *d_cls_table = nullptr, *d_cls_slot = nullptr, *d_cls_rep = nullptr, *d_cls_cnt = nullptr, *d_cls_flag = nullptr, *d_cls_rank = nullptr,
             *d_cls_of = nullptr, *d_cls_out_rep = nullptr, *d_cls_out_cnt = nullptr;
    uint32_t cls_table_size = 0;
    ScanSite site_class{};
    // ---- ADJACENT_CHANNELS broadcast sets (chd_adjacent_broadcast): scratch allocated on first use, grown on demand
    uint8_t* d_conn_type = nullptr;
    bool have_conn_type = false, by_cell_valid = false;
    uint32_t *d_bc_in = nullptr, *d_bc_cnt = nullptr, *d_bc_off = nullptr, *d_bc_msgoff = nullptr, *d_bc_out = nullptr;
    uint64_t bc_msg_cap = 0, bc_out_cap = 0;
    ScanSite site_bcast{};
    bool pair_ch_valid = false;
    // ---- payload assembly + framing (chd_payload.cu): optional stage, buffers grown on demand
    struct Payload {
        uint64_t *d_entry_off = nullptr, *d_full_off = nullptr, *d_cls_off = nullptr, *d_conn_off = nullptr;
        uint8_t *d_entry_bytes = nullptr, *d_full_bytes = nullptr, *d_url = nullptr, *d_blob = nullptr, *d_out = nullptr, *d_stage = nullptr, *d_comp = nullptr;
        uint32_t *d_cls_len = nullptr, *d_fc_cnt = nullptr, *d_fc_off = nullptr, *d_fc_cursor = nullptr, *d_fc_idx = nullptr, *d_conn_cap = nullptr,
                 *d_conn_len = nullptr, *d_conn_frames = nullptr, *d_ndrop = nullptr;
        uint64_t cap_entry_off = 0, cap_entry_bytes = 0, cap_full_off = 0, cap_full_bytes = 0, cap_url = 0, cap_cls = 0, cap_cls_off = 0, cap_blob = 0,
                 cap_fc = 0, cap_fc_off = 0, cap_fc_cur = 0, cap_fc_idx = 0, cap_conn_cap = 0, cap_conn_off = 0, cap_conn_len = 0, cap_conn_frames = 0,
                 cap_comp = 0, cap_ndrop = 0, cap_out = 0, cap_stage = 0, cap_site_cls = 0, cap_site_fc = 0, cap_site_conn = 0;
        ScanSite site_cls{}, site_fc{}, site_conn{};
        uint32_t url_len = 0, msg_type = 8, n_entries = 0, n_classes = 0;
        uint64_t blob_len = 0;
        bool have_input = false, assembled = false;
    } pl;
    // chd_fetch_results reads back on its own stream as soon as the aux chain (pairs, diff, due list) and the emit
    // preparation (visible offsets) are done, i.e. while the emit kernel is still streaming
    cudaStream_t dl_stream = nullptr, dl_stream_b = nullptr;  // phase A / phase B of the early read-back
    cudaEvent_t ev_prep_done = nullptr, ev_build_done = nullptr;
    // ev_counts: the cell CSR offsets of the build in flight are final (recorded between the two halves of a single-pass build);
    // prep_stream: where the emit preparation runs when it overlaps the build's scatter
    cudaEvent_t ev_counts = nullptr;
    cudaStream_t prep_stream = nullptr;
    bool build_done_recorded = false;  // this tick ran a build (its end is ev_build_done)
    // chd_fetch_results_async: completion events of the two copy phases; the next tick is ordered after them on the device
    // (two fetches may be outstanding: the host waits for tick k-1 after it has enqueued tick k and its fetch)
    cudaEvent_t ev_fetch_a[2] = {nullptr, nullptr}, ev_fetch_b[2] = {nullptr, nullptr};
    // chd_fetch_results_async is two hops: result arrays -> a device-side snapshot (ev_fetch_a/b: the next tick may overwrite the
    // arrays) -> pinned host memory at PCIe speed on its own stream (ev_fetch_done: chd_fetch_wait)
    cudaEvent_t ev_fetch_done[2] = {nullptr, nullptr};
    cudaStream_t dl_stream_c = nullptr;
    uint8_t* d_fetch_stage[2] = {nullptr, nullptr};
    uint64_t fetch_stage_bytes[2] = {0, 0};
    void* fetch_header[2] = {nullptr, nullptr};
    uint64_t fetch_issued = 0, fetch_waited = 0;
    bool fetch_guard = false;
    bool early_ready = false;  // ev_join + ev_prep_done of the last tick are recorded
    bool early_results_tick = false;  // CHD_TICK_EARLY_RESULTS of the tick being enqueued
    // CHD_TICK_EARLY_RESULTS: the expanded-list kernel starts after the aux chain (interest + fan-out), so every host-facing
    // result is final while it is still streaming (alternatives measured in round 1: profiles/README.md)
    cudaEvent_t wait_before_emit_kernel = nullptr;
    uint64_t *d_voff = nullptr, *d_vis_off = nullptr;
    uint64_t max_tiles = 0;
    uint64_t vis_estimate = 0;  // n_visible of the last summary the host decoded (0 = none yet): sizes the emit grid
    // fanout
    uint32_t *d_ring_off = nullptr, *d_ring_sender = nullptr;
    int64_t* d_ring_arrival = nullptr;
    uint64_t *d_ring_index = nullptr, *d_ch_msg_index = nullptr;
    bool have_ch_msg_index = false;
    // device-owned rings (chd_rings_init: ChannelData.OnUpdate on the GPU, data.go:149-173): per-cell begin / end cursors into
    // slabs of ring_cap entries inside d_ring_arrival / d_ring_sender / d_ring_index; d_ch_msg_index = ChannelData.msgIndex
    bool rings_owned = false;
    uint32_t ring_cap = 0;
    uint32_t *d_rb_begin = nullptr, *d_rb_end = nullptr, *d_upd_off = nullptr, *d_upd_sender = nullptr, *d_ring_flat_off = nullptr;
    int64_t* d_upd_arrival = nullptr;
    uint64_t upd_cap = 0;
    uint32_t* d_ring_scan_scratch = nullptr;
    uint32_t* d_cell_max_interval = nullptr;  // [C] ChannelData.maxFanOutIntervalMs (subscription.go:84-86)
    int64_t* d_cell_start_ns = nullptr;       // [C] per-channel ChannelTime origin (chd_set_channel_start_times) or nullptr
    bool have_cell_start = false;
    // what the fan-out kernel reads: the staging copies above or the caller's device arrays (zero-copy)
    const uint32_t *ring_off_p = nullptr, *ring_sender_p = nullptr;
    const int64_t* ring_arrival_p = nullptr;
    const uint64_t *ring_index_p = nullptr, *ch_msg_index_p = nullptr;

    uint32_t *d_by_cell = nullptr, *d_pc_hist = nullptr, *d_pc_tmp_key = nullptr, *d_pc_tmp_val = nullptr;  // pairs grouped by cell
    uint32_t pc_blocks = 0;
    chd_due* d_due = nullptr;
    // counters
    Counters* d_ctr = nullptr;
    Counters* h_ctr = nullptr;  // pinned
    // multi-GPU exchange (chd_comm_init): NCCL communicator (opaque here), engine-owned record buffers
    void* comm = nullptr;
    int comm_rank = 0, comm_world = 1;
    uint32_t border_cap = 0;
    uint32_t rec_per_rank = 0;        // border records per rank in the gathered buffer (0: plain contiguous records)
    uint64_t rec_stride_words = 0;    // words one rank contributes to the all-gather (border records + migration blob)
    uint32_t mig_subs = 0, mig_pairs = 0;  // migration blob capacities (0: no subscriber migration)
    bool mig_packed = false;          // chd_migrate_out was called for the coming tick
    uint32_t *d_rec_local = nullptr, *d_rec_all = nullptr;
    unsigned long long* assign_bump = nullptr;  // epoch the next assign_cells_kernel launch bumps for its caller (border export)
    // peer exchange (chd_shard.cuh): this rank's window, the peers' windows mapped with CUDA IPC, device-side sequence / counts
    bool peer_push = false, peer_mapped = false;
    uint32_t* d_peer_win = nullptr;
    void* peer_base[16] = {};
    unsigned long long* d_xchg_seq = nullptr;
    uint32_t *d_push_done = nullptr, *d_peer_count = nullptr;
    uint64_t xchg_seq = 0;  // host mirror of the device sequence (selects the window buffer a graph variant is captured for)
    uint64_t n_collectives = 0;
    // border export scratch
    uint32_t *d_bflag = nullptr, *d_boff = nullptr;
    uint32_t* h_u32 = nullptr;  // pinned scalar
    // scratch of the tick driver's getters (chd_get_visible*, export counts): separate from h_u32, which the stateless entry
    // points use under the engine mutex from other threads
    uint32_t* h_get = nullptr;
    // ---- per-subscriber visibility deltas (chd_visdelta.cu): allocated by chd_visible_delta_enable
    bool slab_set = false;              // chd_set_slab was called: entity indices are not stable across ticks
    bool assigned_since_build = false;  // d_key no longer holds the cell keys of the last build
    struct VisDelta {
        bool on = false, called = false;
        uint64_t cap = 0;                  // entries of each output list
        uint32_t S_out = 0, S_call = 0;    // slots in the output CSR / current slot count of the last call
        uint32_t S_bound = 0, n_bound = 0; // host upper bounds of the baseline's slot and entity counts
        uint32_t nb = 1, per_block = 0;    // mover sort geometry
        VdState* d_state = nullptr;
        uint32_t *d_base_key = nullptr, *d_base_cs = nullptr, *d_base_sorted = nullptr, *d_base_off = nullptr, *d_base_cell = nullptr,
                 *d_base_sub = nullptr;
        uint32_t *d_mv_ent = nullptr, *d_mv_dkey = nullptr, *d_mv_skey = nullptr, *d_tmp_key = nullptr, *d_tmp_val = nullptr,
                 *d_dst_key = nullptr, *d_dst_ent = nullptr, *d_src_key = nullptr, *d_src_ent = nullptr, *d_dst_start = nullptr,
                 *d_src_start = nullptr, *d_hist = nullptr;
        uint32_t *d_ecnt = nullptr, *d_lcnt = nullptr;
        uint64_t *d_epoff = nullptr, *d_lpoff = nullptr, *d_enter_off = nullptr, *d_leave_off = nullptr;
        uint32_t *d_enter = nullptr, *d_leave = nullptr;
        ScanSite site_mv{}, site_h[4]{}, site_e{}, site_l{};
    } vd;

    bool fail(const char* fmt, ...) const {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return false;
    }
};

#define CU(e, call)                                                                                  \
    do {                                                                                             \
        cudaError_t _r = (call);                                                                     \
        if (_r != cudaSuccess) {                                                                     \
            (e)->fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_r), __FILE__, __LINE__);   \
            return CHD_ERR_CUDA;                                                                     \
        }                                                                                            \
    } while (0)

// one kernel launch precedes every KCHECK; scans report their own launch count through SCAN()
#define KCHECK(e)                    \
    do {                             \
        (e)->n_launch++;             \
        CU(e, cudaGetLastError());   \
    } while (0)
#define SCAN(e, ...)                                  \
    do {                                              \
        (e)->n_launch += (uint64_t)(__VA_ARGS__);     \
        CU(e, cudaGetLastError());                    \
    } while (0)

struct StageTimer {  // records a CUDA-event pair around a stage on the engine stream when profiling is on
    chd_engine* e;
    int stage;
    bool on;
    StageTimer(chd_engine* e_, int stage_) : e(e_), stage(stage_), on(e_->profiling == 1 || (e_->profiling == 2 && stage_ == CHD_STAGE_EMIT_KERNEL)) {
        if (on) cudaEventRecord(e->evt(stage, e->stage_n[stage], 0), e->stream);
    }
    ~StageTimer() {
        if (on) {
            cudaEventRecord(e->evt(stage, e->stage_n[stage], 1), e->stream);
            e->stage_n[stage]++;
        }
    }
};

template <typename T>
static bool dalloc(chd_engine* e, T** p, uint64_t count) {
    void* q = nullptr;
    const uint64_t bytes = (count ? count : 1) * sizeof(T);
    cudaError_t r = cudaMalloc(&q, bytes);
    if (r != cudaSuccess) {
        e->fail("cudaMalloc(%llu bytes) failed: %s", (unsigned long long)bytes, cudaGetErrorString(r));
        return false;
    }
    e->allocs.push_back(q);
    *p = (T*)q;
    return true;
}

enum { EP_BUILD = 0, EP_QUERY, EP_EMIT, EP_FANOUT, EP_BORDER, EP_BCAST, EP_CLASS, EP_PAYLOAD, EP_DELTA, EP_COUNT };  // d_epoch has EP_COUNT slots
static_assert(sizeof(chd_engine::stage_execs) / sizeof(uint64_t) == EP_COUNT, "one execution counter per stage epoch");

// ---- helpers shared by the translation units (C linkage only so that definitions may sit inside their extern "C" blocks)
extern "C" {
// epochs start at 1 so that the zero-initialised descriptors (epoch 0) read as stale on first use
bool chd_init_epochs(chd_engine* e);
bool chd_make_site(chd_engine* e, ScanSite& site, uint64_t n_max, int stage);
// Zero-copy inputs: a pointer into this device's memory is consumed in place (no staging copy); the caller keeps it valid
// and unmodified until the work that reads it has finished (chd_summary / chd_sync / any chd_get_*).
bool chd_is_device_ptr(const chd_engine* e, const void* p);
void chd_dfree(chd_engine* e, void* p);
chd_status chd_ensure_upload_stream(chd_engine* e);
chd_status chd_read_u32(chd_engine* e, const uint32_t* d, uint32_t* v);
chd_status chd_decode_summary(chd_engine* e, chd_tick_summary* out);
chd_status chd_assign_cells_impl(chd_engine* e);
chd_status chd_note_pos_read(chd_engine* e);
// Called on the host wherever a stage's epoch is about to be bumped on the device: every 2^20 executions of a stage the
// descriptors of its scan sites are cleared, so no descriptor can survive until the 22-bit epoch repeats.
chd_status chd_epoch_tick(chd_engine* e, int stage);
// lifecycle / migration calls may name slots beyond the current count: extends the slot table (new slots hold no pairs)
chd_status chd_grow_slots(chd_engine* e, uint32_t new_n);
chd_status chd_fetch_guard(chd_engine* e);
// what the fan-out / payload kernels read: the host-owned CSR snapshot (staged or zero-copy) or the device-owned rings
RingDev chd_ring_view(const chd_engine* e);
// one stable LSD radix pass (histogram, look-back scan, scatter) over 32-bit keys; chd_entities.cu
chd_status chd_sort_pass_any(chd_engine* e, uint32_t* hist, const ScanSite& site, const uint32_t* key_in, const uint32_t* val_in, uint32_t n,
                             const uint32_t* n_ptr, uint32_t per_block, uint32_t nblocks, uint32_t shift, uint32_t bits, uint32_t* key_out,
                             uint32_t* val_out, ScatterExtras ex = ScatterExtras{0, nullptr, 0, nullptr}, unsigned long long* bump = nullptr);
}

static inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

static inline uint64_t mix_key(uint64_t h, uint64_t v) {
    h ^= v + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    return h;
}

// Runs `enqueue` (kernel launches + memsets only, no host sync) either directly or as a replayed CUDA graph.
// A graph is captured only after the same key was seen twice in a row, so workloads whose batch shape changes
// every tick simply run direct launches.
template <typename F>
static chd_status run_stage(chd_engine* e, chd_engine::GraphSlot& slot, uint64_t key, F&& enqueue) {
    key |= 1;  // never 0
    if (!e->use_graphs || e->stream == nullptr) return enqueue();
    if (slot.exec && slot.key == key) {
        CU(e, cudaGraphLaunch(slot.exec, e->stream));
        e->n_launch += slot.nodes;
        e->graph_launches++;
        return CHD_OK;
    }
    if (slot.pending_key != key) {  // first sighting: run direct, capture next time
        slot.pending_key = key;
        return enqueue();
    }
    if (slot.exec) {
        cudaGraphExecDestroy(slot.exec);
        slot.exec = nullptr;
    }
    const uint64_t l0 = e->n_launch;
    // Stateless entry points (chd_cell_of, chd_query_channel_ids) may be called from other threads and launch into the same
    // stream: they hold the engine mutex for their whole call, so taking it here keeps their work out of the capture.
    std::lock_guard<std::recursive_mutex> capture_lock(e->mu);
    CU(e, cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    chd_status st = enqueue();
    cudaGraph_t g = nullptr;
    cudaError_t r = cudaStreamEndCapture(e->stream, &g);
    if (st != CHD_OK || r != cudaSuccess || !g) {
        if (g) cudaGraphDestroy(g);
        if (st == CHD_OK) {
            e->fail("graph capture failed: %s", cudaGetErrorString(r));
            st = CHD_ERR_CUDA;
        }
        e->use_graphs = false;  // fall back to direct launches for the rest of this engine's life
        cudaGetLastError();
        e->n_launch = l0;
        return st == CHD_OK ? enqueue() : st;
    }
    r = cudaGraphInstantiate(&slot.exec, g, 0);
    cudaGraphDestroy(g);
    if (r != cudaSuccess) {
        slot.exec = nullptr;
        e->use_graphs = false;
        cudaGetLastError();
        e->n_launch = l0;
        return enqueue();
    }
    slot.nodes = e->n_launch - l0;
    e->n_launch = l0;
    slot.key = key;
    e->graph_captures++;
    CU(e, cudaGraphLaunch(slot.exec, e->stream));
    e->n_launch += slot.nodes;
    e->graph_launches++;
    return CHD_OK;
}
