// chd_shard.cu — multi-GPU X-slab sharding (SURVEY.md §8e): border export, halo import, and the per-tick exchange itself:
// ONE ncclAllGather of (entity id, cell) border records over NVLink / NVSwitch, issued by the library on the engine's
// stream (chd_tick_sharded), so a host needs no NCCL binding of its own.
//
// NCCL is loaded with dlopen on first use (libnccl.so.2; a copy already in the process, e.g. torch's, is reused): a
// single-GPU deployment needs no NCCL at all and the library keeps its link-time dependencies to libcudart.
#include "chd_engine.h"

#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only; every call goes through the table below

#include "chd_shard.cuh"

namespace {
struct NcclApi {
    void* lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    std::string err;
};
NcclApi* nccl_api() {
    static std::mutex mu;
    static NcclApi* api = nullptr;
    std::lock_guard<std::mutex> lk(mu);
    if (api && api->lib) return api;
    if (!api) api = new NcclApi();
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // a copy the process already loaded (torch bundles one)
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
        const char* m = dlerror();
        api->err = std::string("cannot load libnccl.so.2: ") + (m ? m : "?");
        return api;
    }
#define SYM(name)                                                          \
    api->name = (decltype(api->name))dlsym(h, "nccl" #name);              \
    if (!api->name) {                                                      \
        api->err = "libnccl.so.2 lacks nccl" #name;                        \
        return api;                                                        \
    }
    SYM(GetUniqueId) SYM(CommInitRank) SYM(CommDestroy) SYM(AllGather) SYM(GetErrorString) SYM(GetVersion)
#undef SYM
    api->lib = h;
    return api;
}
}  // namespace

#define NC(e, api, call)                                                                                         \
    do {                                                                                                         \
        ncclResult_t _r = (call);                                                                                \
        if (_r != ncclSuccess) {                                                                                 \
            (e)->fail("%s failed: %s (%s:%d)", #call, (api)->GetErrorString(_r), __FILE__, __LINE__);            \
            return CHD_ERR_CUDA;                                                                                 \
        }                                                                                                        \
    } while (0)

extern "C" {

chd_status chd_set_slab(chd_engine* e, uint32_t col_lo, uint32_t col_hi, uint32_t halo) {
    if (!e || col_lo >= col_hi || col_hi > e->g.cols) return CHD_ERR_INVALID;
    e->g.col_lo = col_lo;
    e->g.col_hi = col_hi;
    e->g.halo = halo;
    e->slab_set = true;
    e->halo_on_device = false;  // set again by chd_import_halo
    return CHD_OK;
}

chd_status chd_export_border(chd_engine* e, uint32_t* d_records, uint32_t cap_records, uint32_t* out_count) {
    if (!e || !d_records) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    {
        chd_status gs_ = chd_fetch_guard(e);
        if (gs_ != CHD_OK) return gs_;
    }
    cudaStream_t s = e->stream;
    const uint32_t n = e->n_own;
    // inside chd_tick_sharded with the peer exchange the records go straight into the peers' windows afterwards: no padding needed
    const bool to_peers = e->peer_push && d_records == e->d_rec_local;
    auto enqueue = [&]() -> chd_status {
        const bool bump_in_assign = !e->assigned && n;
        if (bump_in_assign) e->assign_bump = e->d_epoch + EP_BORDER;
        chd_status st = chd_assign_cells_impl(e);
        if (st != CHD_OK) return st;
        if (!bump_in_assign) {
            bump_epoch_kernel<<<1, 1, 0, s>>>(e->d_epoch + EP_BORDER);
            KCHECK(e);
        }
        if (!to_peers) CU(e, cudaMemsetAsync(d_records, 0xFF, 8ull * cap_records, s));  // unused records read as "no cell"
        SCAN(e, compact_1p(BorderFlag{e->g, e->d_key}, BorderSink{e->d_key, e->have_gid ? e->d_gid : nullptr, d_records, cap_records, e->d_boff + n, e->d_ctr},
                           n, e->site_border, s));
        if (to_peers) {
            PeerWindows pw{};
            for (int r = 0; r < e->comm_world; r++) pw.base[r] = (uint32_t*)e->peer_base[r];
            const uint64_t blob_words = e->rec_stride_words - 2ull * e->rec_per_rank;
            peer_push_kernel<<<(unsigned)std::min<uint64_t>((uint64_t)e->sm_count, 8 + (2ull * cap_records * e->comm_world) / 8192), 256, 0, s>>>(
                d_records, e->d_boff + n, cap_records, blob_words, e->rec_stride_words, pw, (uint32_t)e->comm_world, (uint32_t)e->comm_rank, e->d_xchg_seq,
                e->d_push_done, e->d_epoch + EP_BORDER);
            KCHECK(e);
        }
        return CHD_OK;
    };
    chd_status st = chd_epoch_tick(e, EP_BORDER);
    if (st != CHD_OK) return st;
    if (!e->assigned) {
        // replayable: cell assignment + border selection of one tick (two variants: the key buffers ping-pong)
        uint32_t* target = e->have_prev_key ? e->d_prev_key : e->d_key;
        const int slot = (target == e->d_key_a ? 0 : 1) + 2 * e->pos_buf;
        uint64_t key = mix_key(mix_key(mix_key(0x6578706full, n), e->have_gid), e->have_prev_key);
        key = mix_key(mix_key(key, (uint64_t)(uintptr_t)target), (uint64_t)(uintptr_t)e->pos_x ^ ((uint64_t)(uintptr_t)e->pos_z << 1));
        key = mix_key(mix_key(key, (uint64_t)(uintptr_t)d_records), cap_records);
        key = mix_key(mix_key(mix_key(key, e->g.col_lo), e->g.col_hi), e->g.halo);
        key = mix_key(key, to_peers ? 1 : 0);
        st = run_stage(e, e->g_export[slot + (to_peers ? 4 : 0)], key, enqueue);
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
        if (st == CHD_OK) st = chd_note_pos_read(e);
    } else {
        st = enqueue();
    }
    if (st != CHD_OK) return st;
    if (out_count) {
        st = chd_read_u32(e, e->d_boff + n, out_count);
        if (st != CHD_OK) return st;
        if (*out_count > cap_records) {
            e->fail("border export needs %u records > capacity %u", *out_count, cap_records);
            return CHD_ERR_CAPACITY;
        }
    }
    return CHD_OK;
}

chd_status chd_import_halo(chd_engine* e, const uint32_t* d_records, uint32_t n_records, uint32_t skip_first, uint32_t skip_count) {
    if (!e || (n_records && !d_records)) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    if (!e->assigned) {
        e->fail("chd_import_halo before chd_export_border / chd_assign_cells");
        return CHD_ERR_STATE;
    }
    if (!e->have_gid) {
        e->fail("chd_import_halo requires global entity ids (chd_set_entity_ids)");
        return CHD_ERR_STATE;
    }
    cudaStream_t s = e->stream;
    if (n_records > e->lim.max_entities) {
        e->fail("halo import of %u records > max_entities scratch %u", n_records, e->lim.max_entities);
        return CHD_ERR_CAPACITY;
    }
    {
        chd_status st0 = chd_epoch_tick(e, EP_BORDER);
        if (st0 != CHD_OK) return st0;
        const int slot = e->d_key == e->d_key_a ? 0 : 1;  // the halo keys are appended to the current key buffer
        // peer exchange: the records sit in this tick's buffer of the own window, the live counts come from the flags
        const bool from_peers = e->peer_push && d_records >= e->d_peer_win && d_records < e->d_peer_win + 2ull * e->comm_world * e->rec_stride_words;
        const int parity = from_peers && d_records != e->d_peer_win ? 1 : 0;
        uint64_t key = mix_key(mix_key(mix_key(0x696d706full, n_records), skip_first), skip_count);
        key = mix_key(mix_key(key, e->rec_per_rank), e->rec_stride_words);
        key = mix_key(mix_key(mix_key(key, (uint64_t)(uintptr_t)d_records), e->n_own), (uint64_t)(uintptr_t)e->d_key);
        key = mix_key(mix_key(mix_key(key, e->g.col_lo), e->g.col_hi), e->g.halo);
        key = mix_key(key, from_peers ? 1 : 0);
        chd_status st = run_stage(e, e->g_import[slot + 2 * parity], key, [&]() -> chd_status {
            const RecView rv{d_records, e->rec_per_rank ? e->rec_per_rank : (n_records ? n_records : 1u),
                             e->rec_per_rank ? e->rec_stride_words : 2ull * (n_records ? n_records : 1u)};
            if (from_peers) {  // (the push kernel of this tick has bumped the compaction site's epoch)
                peer_wait_kernel<<<1, 32, 0, s>>>(e->d_peer_win, e->rec_stride_words, (uint32_t)e->comm_world, e->d_xchg_seq, e->d_peer_count, e->d_ctr);
            } else {
                bump_epoch_kernel<<<1, 1, 0, s>>>(e->d_epoch + EP_BORDER);
            }
            KCHECK(e);
            // no host round trip: the kept count and the build length stay on the device (overflow -> CHD_OVF_BORDER)
            SCAN(e, compact_1p(HaloFlag{e->g, rv, from_peers ? e->d_peer_count : nullptr, skip_first, skip_count},
                               HaloSink{rv, e->n_own, e->lim.max_entities, e->d_key, e->d_gid, e->d_n_build, e->d_ctr}, n_records, e->site_border, s));
            return CHD_OK;
        });
        if (st != CHD_OK) return st;
    }
    e->halo_on_device = true;
    e->n_halo = 0;
    e->entities_dirty = true;
    return CHD_OK;
}

/* ------------------------------------------------------------------ the exchange behind the ABI ---- */

chd_status chd_comm_unique_id(void* out_id) {
    if (!out_id) return CHD_ERR_INVALID;
    NcclApi* api = nccl_api();
    if (!api->lib) return CHD_ERR_CUDA;
    ncclUniqueId id;
    if (api->GetUniqueId(&id) != ncclSuccess) return CHD_ERR_CUDA;
    static_assert(sizeof(ncclUniqueId) == CHD_COMM_ID_BYTES, "CHD_COMM_ID_BYTES must match ncclUniqueId");
    memcpy(out_id, &id, sizeof id);
    return CHD_OK;
}

chd_status chd_comm_init(chd_engine* e, const void* unique_id, int rank, int world, uint32_t halo_cols, uint32_t border_capacity,
                         uint32_t migrate_subscribers, uint32_t migrate_pairs) {
    if (!e || !unique_id || world < 1 || rank < 0 || rank >= world || border_capacity == 0) return CHD_ERR_INVALID;
    if (world >= 4096 || migrate_subscribers >= (1u << 20)) return CHD_ERR_INVALID;  // (slot_src packs rank:12 | record:20)
    if (e->comm) {
        e->fail("chd_comm_init: already initialised");
        return CHD_ERR_STATE;
    }
    if ((uint32_t)world > e->g.cols) {
        e->fail("chd_comm_init: %d ranks > %u grid columns (a slab is at least one column)", world, e->g.cols);
        return CHD_ERR_INVALID;
    }
    CU(e, cudaSetDevice(e->device));
    NcclApi* api = nccl_api();
    if (!api->lib) {
        e->fail("%s", api->err.c_str());
        return CHD_ERR_CUDA;
    }
    if ((uint64_t)border_capacity * (uint64_t)world + 1 > e->lim.max_entities) {
        e->fail("chd_comm_init: border_capacity %u x %d ranks does not fit the halo scratch (max_entities %u)", border_capacity, world,
                e->lim.max_entities);
        return CHD_ERR_CAPACITY;
    }
    ncclUniqueId id;
    memcpy(&id, unique_id, sizeof id);
    ncclComm_t comm = nullptr;
    NC(e, api, api->CommInitRank(&comm, world, id, rank));
    e->comm = comm;
    e->comm_rank = rank;
    e->comm_world = world;
    border_capacity = (border_capacity + 1u) & ~1u;  // (16-byte alignment of everything that follows the records)
    e->border_cap = border_capacity;
    // one contribution per rank and tick = its border records followed by its migration blob (subscriber state in flight)
    e->mig_subs = (migrate_subscribers + 1u) & ~1u;
    e->mig_pairs = (migrate_pairs + 1u) & ~1u;
    if (e->mig_subs && !e->mig_pairs) e->mig_pairs = 16 * e->mig_subs;
    const uint64_t blob_words = e->mig_subs ? ((MigView::words(e->mig_subs, e->mig_pairs) + 3ull) & ~3ull) : 0ull;
    e->rec_per_rank = border_capacity;
    e->rec_stride_words = 2ull * border_capacity + blob_words;
    if (!dalloc(e, &e->d_rec_local, e->rec_stride_words) || !dalloc(e, &e->d_rec_all, e->rec_stride_words * (uint64_t)world)) return CHD_ERR_CUDA;
    CU(e, cudaMemsetAsync(e->d_rec_local, 0, e->rec_stride_words * 4, e->stream));
    CU(e, cudaMemsetAsync(e->d_rec_all, 0, e->rec_stride_words * 4 * (uint64_t)world, e->stream));
    // ---- peer exchange: every rank's receive window is mapped into every other rank (CUDA IPC); the tick then moves the border
    // records with plain stores over NVLink and 64-bit flags (chd_shard.cuh).  NCCL carries the handles once, here.  If any rank
    // cannot map a peer (no P2P path, more ranks than CHD_MAX_PEERS) ALL ranks keep the ncclAllGather exchange.
    {
        const uint64_t win_words = 2ull * world * e->rec_stride_words + 4ull * world + 8;
        uint32_t* hbuf = nullptr;
        if (!dalloc(e, &e->d_peer_win, win_words) || !dalloc(e, &e->d_xchg_seq, 1) || !dalloc(e, &e->d_push_done, 4) ||
            !dalloc(e, &e->d_peer_count, CHD_MAX_PEERS) || !dalloc(e, &hbuf, 32ull * (uint64_t)world))
            return CHD_ERR_CUDA;
        CU(e, cudaMemsetAsync(e->d_peer_win, 0, win_words * 4, e->stream));
        CU(e, cudaMemsetAsync(e->d_xchg_seq, 0, 8, e->stream));
        CU(e, cudaMemsetAsync(e->d_push_done, 0, 16, e->stream));
        CU(e, cudaMemsetAsync(e->d_peer_count, 0, 4 * CHD_MAX_PEERS, e->stream));
        CU(e, cudaStreamSynchronize(e->stream));  // the window is clean before any peer can learn its address
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
        struct Slot { cudaIpcMemHandle_t h; uint32_t ok, pad[15]; } mine{};  // 128 bytes per rank
        mine.ok = (world <= CHD_MAX_PEERS && cudaIpcGetMemHandle(&mine.h, e->d_peer_win) == cudaSuccess) ? 1u : 0u;
        cudaGetLastError();
        std::vector<Slot> all((size_t)world);
        auto gather = [&]() -> chd_status {  // all-gather of one Slot per rank through hbuf
            CU(e, cudaMemcpyAsync(hbuf + 32ull * rank, &mine, sizeof mine, cudaMemcpyHostToDevice, e->stream));
            NC(e, api, api->AllGather(hbuf + 32ull * rank, hbuf, 32, ncclUint32, comm, e->stream));
            CU(e, cudaMemcpyAsync(all.data(), hbuf, sizeof(Slot) * (size_t)world, cudaMemcpyDeviceToHost, e->stream));
            CU(e, cudaStreamSynchronize(e->stream));
            return CHD_OK;
        };
        chd_status gs = gather();
        if (gs != CHD_OK) return gs;
        bool ok = true;
        for (int r = 0; r < world; r++) ok = ok && all[(size_t)r].ok;
        if (ok) {
            for (int r = 0; r < world && ok; r++) {
                if (r == rank) {
                    e->peer_base[r] = e->d_peer_win;
                    continue;
                }
                void* p = nullptr;
                if (cudaIpcOpenMemHandle(&p, all[(size_t)r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                    cudaGetLastError();
                    ok = false;
                } else {
                    e->peer_base[r] = p;
                }
            }
        }
        mine.ok = ok ? 1u : 0u;  // second round: did EVERY rank map every peer?
        gs = gather();
        if (gs != CHD_OK) return gs;
        for (int r = 0; r < world; r++) ok = ok && all[(size_t)r].ok;
        if (!ok)
            for (int r = 0; r < world; r++) {
                if (r != rank && e->peer_base[r]) cudaIpcCloseMemHandle(e->peer_base[r]);
                e->peer_base[r] = nullptr;
            }
        e->peer_mapped = ok;
        e->peer_push = ok;
        e->xchg_seq = 0;
        chd_dfree(e, hbuf);
    }
    // X-slabs by grid column (SURVEY.md §8e): rank g of G owns columns [floor(g*cols/G), floor((g+1)*cols/G))
    const uint32_t lo = (uint32_t)(((uint64_t)rank * e->g.cols) / (uint64_t)world), hi = (uint32_t)(((uint64_t)(rank + 1) * e->g.cols) / (uint64_t)world);
    return chd_set_slab(e, lo, hi, halo_cols);
}

chd_status chd_comm_info(const chd_engine* e, int* rank, int* world, uint32_t* col_lo, uint32_t* col_hi, uint32_t* halo_cols, int* nccl_version) {
    if (!e) return CHD_ERR_INVALID;
    if (rank) *rank = e->comm ? e->comm_rank : 0;
    if (world) *world = e->comm ? e->comm_world : 1;
    if (col_lo) *col_lo = e->g.col_lo;
    if (col_hi) *col_hi = e->g.col_hi;
    if (halo_cols) *halo_cols = e->g.halo;
    if (nccl_version) {
        *nccl_version = 0;
        NcclApi* api = nccl_api();
        if (api->lib) api->GetVersion(nccl_version);
    }
    return CHD_OK;
}

chd_status chd_comm_destroy(chd_engine* e) {
    if (!e) return CHD_ERR_INVALID;
    if (!e->comm) return CHD_OK;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaStreamSynchronize(e->stream));
    for (int r = 0; r < e->comm_world && r < CHD_MAX_PEERS; r++) {
        if (r != e->comm_rank && e->peer_base[r]) cudaIpcCloseMemHandle(e->peer_base[r]);
        e->peer_base[r] = nullptr;
    }
    e->peer_push = e->peer_mapped = false;
    NcclApi* api = nccl_api();
    if (api->lib) api->CommDestroy((ncclComm_t)e->comm);
    e->comm = nullptr;
    return CHD_OK;
}

// One sharded tick: interest + fan-out start on the second stream (they do not need positions), this rank's border records
// are selected, ONE all-gather moves every rank's records over NVLink, the records this slab needs are appended as halo
// entities, then build + emit run over own + halo entities and the streams join.  Nothing synchronises with the host.
chd_status chd_tick_sharded(chd_engine* e, const chd_query_batch* q, int64_t t_ns, uint32_t flags, chd_tick_summary* out) {
    if (!e) return CHD_ERR_INVALID;
    if (!e->comm) {
        e->fail("chd_tick_sharded before chd_comm_init");
        return CHD_ERR_STATE;
    }
    {
        chd_status gs_ = chd_fetch_guard(e);
        if (gs_ != CHD_OK) return gs_;
    }
    chd_status st;
    const bool has_batch = q || e->have_adopted_q;
    // Without subscriber migration the interest update does not depend on the exchange: it starts first and overlaps it.
    // With migration the immigrants' previous state arrives in the all-gather, so the update starts right after it.
    if (has_batch && !e->mig_subs) {
        st = chd_begin_interest(e, q, t_ns, (flags & CHD_TICK_FANOUT) ? 1 : 0);
        if (st != CHD_OK) return st;
    }
    const uint32_t cap = e->border_cap;
    if (e->mig_subs && !e->mig_packed) CU(e, cudaMemsetAsync(e->d_rec_local + 2ull * cap, 0, 16, e->stream));  // empty blob header
    e->mig_packed = false;
    {
        StageTimer tm(e, CHD_STAGE_EXPORT);  // (with the peer exchange: assignment + border selection + the push into the peers' windows)
        st = chd_export_border(e, e->d_rec_local, cap, nullptr);
    }
    if (st != CHD_OK) return st;
    const uint32_t* gathered = e->d_rec_all;
    if (e->peer_push) {
        e->xchg_seq++;
        gathered = e->d_peer_win + (e->xchg_seq & 1ull) * (uint64_t)e->comm_world * e->rec_stride_words;
    } else {
        NcclApi* api = nccl_api();
        StageTimer tm(e, CHD_STAGE_EXCHANGE);
        NC(e, api, api->AllGather(e->d_rec_local, e->d_rec_all, e->rec_stride_words, ncclUint32, (ncclComm_t)e->comm, e->stream));
        e->n_collectives++;
    }
    {
        // the halo import comes first: with the peer exchange its first kernel is the one that waits for the peers' records, and the
        // immigrants' state (read by the interest update below) sits in the same window
        StageTimer tm(e, CHD_STAGE_IMPORT);
        st = chd_import_halo(e, gathered, cap * (uint32_t)e->comm_world, (uint32_t)e->comm_rank * cap, cap);
    }
    if (st != CHD_OK) return st;
    if (e->mig_subs) {
        e->mig = MigView{const_cast<uint32_t*>(gathered) + 2ull * cap, e->rec_stride_words, e->mig_subs, e->mig_pairs};
        if (has_batch) {
            st = chd_begin_interest(e, q, t_ns, (flags & CHD_TICK_FANOUT) ? 1 : 0);
            if (st != CHD_OK) return st;
        }
    }
    if (st != CHD_OK) return st;
    return chd_tick(e, nullptr, t_ns, flags, out);
}

/* ---- subscriber migration between ranks (state travels in the tick's all-gather) */

chd_status chd_migrate_out(chd_engine* e, const uint32_t* slot, uint32_t n) {
    if (!e || (n && !slot)) return CHD_ERR_INVALID;
    if (!e->comm || !e->mig_subs) {
        e->fail("chd_migrate_out: chd_comm_init was not given a migration capacity");
        return CHD_ERR_STATE;
    }
    if (n > e->mig_subs) {
        e->fail("chd_migrate_out: %u subscribers > migration capacity %u", n, e->mig_subs);
        return CHD_ERR_CAPACITY;
    }
    if (e->mig_packed) {
        e->fail("chd_migrate_out: one call per tick (pass every emigrant at once)");
        return CHD_ERR_STATE;
    }
    std::lock_guard<std::recursive_mutex> lk(e->mu);
    CU(e, cudaSetDevice(e->device));
    for (uint32_t i = 0; i < n; i++)
        if (slot[i] >= e->n_slots) {
            e->fail("chd_migrate_out: slot %u is not in use (%u slots)", slot[i], e->n_slots);
            return CHD_ERR_INVALID;
        }
    CU(e, cudaMemcpyAsync(e->d_lc_slot, slot, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    uint32_t* blob = e->d_rec_local + 2ull * e->border_cap;
    const MigView lay{blob, e->rec_stride_words, e->mig_subs, e->mig_pairs};
    mig_pack_kernel<<<1, 256, 0, e->stream>>>(e->d_lc_slot, n, e->pairs[e->cur], e->d_conn, blob, lay, e->d_ctr);
    KCHECK(e);
    if (n) {
        slot_ctl_mark_kernel<<<blocks_for(n, 256), 256, 0, e->stream>>>(e->d_lc_slot, n, (uint8_t)SLOT_DROP, e->d_slot_ctl);
        KCHECK(e);
    }
    e->mig_packed = true;
    e->lifecycle_used = true;
    return CHD_OK;
}

chd_status chd_migrate_in(chd_engine* e, uint32_t src_rank, uint32_t first_index, const uint32_t* slot, const uint32_t* conn_id, uint32_t n) {
    if (!e || (n && (!slot || !conn_id))) return CHD_ERR_INVALID;
    if (!e->comm || !e->mig_subs) {
        e->fail("chd_migrate_in: chd_comm_init was not given a migration capacity");
        return CHD_ERR_STATE;
    }
    if ((int)src_rank >= e->comm_world || (uint64_t)first_index + n > e->mig_subs) return CHD_ERR_INVALID;
    if (n == 0) return CHD_OK;
    std::lock_guard<std::recursive_mutex> lk(e->mu);
    CU(e, cudaSetDevice(e->device));
    uint32_t max_slot = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (slot[i] >= e->lim.max_subscribers) return CHD_ERR_INVALID;
        if (slot[i] > max_slot) max_slot = slot[i];
    }
    CU(e, cudaMemcpyAsync(e->d_lc_slot, slot, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, e->stream));
    CU(e, cudaMemcpyAsync(e->d_lc_aux, conn_id, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    slot_import_mark_kernel<<<blocks_for(n, 256), 256, 0, e->stream>>>(e->d_lc_slot, e->d_lc_aux, n, src_rank, first_index, e->d_slot_ctl, e->d_slot_src,
                                                                      e->d_conn);
    KCHECK(e);
    chd_status st = chd_grow_slots(e, max_slot + 1);
    if (st != CHD_OK) return st;
    e->lifecycle_used = true;
    return CHD_OK;
}

chd_status chd_get_rehome(chd_engine* e, uint32_t* global_id, uint32_t* dst_rank, uint32_t cap, uint32_t* count) {
    if (!e || !count) return CHD_ERR_INVALID;
    CU(e, cudaSetDevice(e->device));
    if (!e->assigned) {
        e->fail("chd_get_rehome before the tick's cell assignment");
        return CHD_ERR_STATE;
    }
    cudaStream_t s = e->stream;
    const uint32_t n = e->n_own, world = e->comm ? (uint32_t)e->comm_world : 1u;
    // scratch: the radix sort's temporaries are free between builds
    CU(e, cudaMemsetAsync(e->d_boff, 0, 4, s));
    if (n) {
        rehome_kernel<<<blocks_for(n, 256), 256, 0, s>>>(e->g, e->d_key, e->have_gid ? e->d_gid : nullptr, n, world, e->d_tmp_key, e->d_tmp_val,
                                                         e->lim.max_entities, e->d_boff);
        KCHECK(e);
    }
    chd_status st = chd_read_u32(e, e->d_boff, count);
    if (st != CHD_OK) return st;
    const uint32_t m = *count < cap ? *count : cap;
    if (m && global_id) CU(e, cudaMemcpyAsync(global_id, e->d_tmp_key, 4ull * m, cudaMemcpyDefault, s));
    if (m && dst_rank) CU(e, cudaMemcpyAsync(dst_rank, e->d_tmp_val, 4ull * m, cudaMemcpyDefault, s));
    CU(e, cudaStreamSynchronize(s));
    return CHD_OK;
}

uint64_t chd_collective_count(const chd_engine* e) { return e ? e->n_collectives : 0; }

int chd_comm_exchange_mode(const chd_engine* e) { return !e || !e->comm ? 0 : (e->peer_push ? 2 : 1); }

chd_status chd_comm_use_collective(chd_engine* e, int on) {
    if (!e) return CHD_ERR_INVALID;
    if (!e->comm) {
        e->fail("chd_comm_use_collective before chd_comm_init");
        return CHD_ERR_STATE;
    }
    e->peer_push = !on && e->peer_mapped;
    return CHD_OK;
}

}  // extern "C"
