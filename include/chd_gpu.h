/*
 * chd_gpu.h — C ABI of the B200-native spatial interest-management + fan-out engine (libchd_b200.so).
 *
 * This is the drop-in boundary behind channeld's SpatialController plugin surface
 * (reference: channeldorg/channeld @ 61fa8add, pkg/channeld/spatial.go:17-35).  A cgo shim binds exactly
 * these entry points (INTEGRATION.md, go/gpucontroller.go).  Plain pointers and sizes only; no C++/torch
 * types; integer status codes; no exceptions cross the ABI.  Pointer retention: the synchronous entry points (chd_cell_of,
 * chd_query_channel_ids, chd_adjacent_broadcast, chd_get_*, chd_fetch_results, chd_summary) are done with every caller pointer
 * when they return; the stream-ordered ones (chd_set_*, chd_prefetch_*, chd_tick, chd_update_interest with HOST arrays) read
 * caller memory asynchronously until the next synchronising call — such buffers must be C memory (chd_alloc_pinned), never
 * Go-managed memory (cgo pointer rules, INTEGRATION.md).  Pointer arguments may be host (pageable or pinned) or device pointers unless
 * stated otherwise.  HOST inputs are copied (cudaMemcpyAsync on the engine's stream; pinned memory makes that
 * asynchronous) and may be reused once the call that consumes them has been followed by chd_summary / chd_sync /
 * a chd_get_* call.  DEVICE inputs of the tick path (chd_set_entities, chd_set_rings, the arrays of a
 * chd_query_batch) that live on the engine's GPU are consumed IN PLACE (zero copy): the producer keeps them valid
 * and unmodified until the tick that reads them has finished.
 *
 * Threading: one tick driver per engine handle (thread-compatible).  chd_cell_of / chd_query_channel_ids
 * take an internal mutex and may be called from any thread (the reference calls GetChannelId /
 * QueryChannelIds concurrently from channel goroutines, spatial.go:20-29).
 *
 * There is NO CPU fallback: every compute entry point runs sm_100a kernels and returns CHD_ERR_CUDA if no
 * device is usable.
 */
#ifndef CHD_GPU_H
#define CHD_GPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define CHD_ABI_VERSION 1

typedef struct chd_engine chd_engine;

typedef enum chd_status {
    CHD_OK = 0,
    CHD_ERR_INVALID = 1,  /* bad argument / config (LoadConfig validation, spatial.go:146-157) */
    CHD_ERR_CUDA = 2,     /* CUDA runtime failure or no device; see chd_last_error */
    CHD_ERR_CAPACITY = 3, /* an output or scratch capacity in chd_limits was exceeded; summary.required_* says by how much */
    CHD_ERR_STATE = 4     /* call order violated (e.g. emit before build) */
} chd_status;

/* Grid constants.  Replaces StaticGrid2DSpatialController's config fields (spatial.go:89-124, JSON in
 * config/spatial_static_*.json) + GlobalSettings.SpatialChannelIdStart (settings.go:94). */
typedef struct chd_grid_cfg {
    double   world_offset_x, world_offset_z;
    double   grid_width, grid_height;
    uint32_t grid_cols, grid_rows;
    uint32_t server_cols, server_rows;
    uint32_t server_interest_border_size;
    uint32_t channel_id_start; /* 0x10000 */
} chd_grid_cfg;

/* Capacities (device allocations are made once in chd_create; nothing allocates on the tick path). */
typedef struct chd_limits {
    uint32_t max_entities;
    uint32_t max_subscribers;
    uint32_t max_queries;       /* per chd_update_interest / chd_query_channel_ids batch */
    uint32_t max_spots;         /* total SpotsAOI spots per batch */
    uint64_t max_pairs;         /* (subscriber, cell) subscriptions alive at once */
    uint64_t max_window_cells;  /* query scratch: sum over the batch of each query's cell bounding box */
    uint64_t max_visible;       /* expanded visible-entity list entries per tick */
    uint32_t max_ring_entries;  /* total update-ring entries over all cells */
    uint32_t max_due;           /* fan-out decisions per tick */
    /* SPATIAL channel-type settings the reference reads from GlobalSettings.ChannelSettings
     * (settings.go:97-103,237-243; subscription.go:21-31): */
    uint32_t default_fanout_interval_ms; /* used when dist matches no damping row (message_spatial.go:68-72) */
    int32_t  default_fanout_delay_ms;
} chd_limits;

/* Fills `lim` with capacities sized for n_entities / n_subscribers (helper; edit before chd_create). */
void chd_default_limits(const chd_grid_cfg* cfg, uint32_t n_entities, uint32_t n_subscribers, chd_limits* lim);

/* Replaces InitSpatialController + LoadConfig (spatial.go:40-74,141-159).  Validates like LoadConfig except
 * that ServerInterestBorderSize == 0 is accepted: the reference discards that error (spatial.go:68) and both
 * benchmark configs rely on it.  `device` = CUDA ordinal. */
chd_status chd_create(const chd_grid_cfg* cfg, const chd_limits* lim, int device, chd_engine** out);
void chd_destroy(chd_engine* e);
/* Last error text of this engine (or of chd_create when e == NULL).  Valid until the next call. */
const char* chd_last_error(const chd_engine* e);
/* Run all work on this cudaStream_t (default: a private non-blocking stream).  torch passes its current stream. */
chd_status chd_set_stream(chd_engine* e, void* cuda_stream);
/* Blocks until all work queued on the engine stream has finished. */
chd_status chd_sync(chd_engine* e);

/* Pinned host memory for the per-tick staging buffers (plain C memory, legal to hold from Go). */
void* chd_alloc_pinned(uint64_t bytes);
/* NUMA node of the GPU (from sysfs; -1 = unknown).  Pinned memory is placed by first touch: run the tick driver (the thread that
 * calls chd_alloc_pinned) on that node's cores and the per-tick uploads cross no socket interconnect. */
int chd_device_numa_node(int device);
void chd_free_pinned(void* p);

/* ---- GetChannelId, batched (spatial.go:161-180; the batch form is handleQuerySpatialChannel,
 * message_spatial.go:335-370).  out_channel_id[i] = channel id, or 0 where the reference returns an error
 * (outside [0,cols) x [0,rows), NaN, +-Inf, huge).  Synchronous. */
chd_status chd_cell_of(chd_engine* e, const double* x, const double* z, uint32_t n, uint32_t* out_channel_id);
/* The same with an explicit validity flag per position (out_valid[i] = 1 / 0; may be NULL): needed when
 * channel_id_start == 0, where channel id 0 is a real cell and cannot double as the error value. */
chd_status chd_cell_of_valid(chd_engine* e, const double* x, const double* z, uint32_t n, uint32_t* out_channel_id, uint8_t* out_valid);

/* ---- entity positions (SoA).  Replaces the per-cell entity maps the reference keeps in
 * SpatialChannelData.Entities (pkg/unrealpb/extension.go:38-62) fed by AddEntity/RemoveEntity
 * (spatial.go:606-609,702-736).  Entity i has id i (the host maps it to EntityChannelIdStart + i). */
chd_status chd_set_entities(chd_engine* e, const double* x, const double* z, uint32_t n);
/* Double-buffered upload for pipelined hosts: chd_prefetch_entities starts copying the NEXT tick's host positions
 * into the engine's second pair of position buffers on a dedicated upload stream and returns immediately; it may be
 * called while a tick is in flight (the H2D transfer then overlaps that tick's kernels).  x / z must stay valid until
 * chd_adopt_prefetched has been followed by chd_summary / chd_sync / chd_fetch_results.  chd_adopt_prefetched makes the
 * prefetched positions the current ones (replaces chd_set_entities for that tick; CHD_ERR_STATE if nothing was
 * prefetched).  The second buffer pair is allocated on the first prefetch. */
chd_status chd_prefetch_entities(chd_engine* e, const double* x, const double* z, uint32_t n);
/* The same two calls for positions that ARE floats at the source: channeld's entities move as unrealpb.FVector (three floats,
 * pkg/unrealpb/unreal_common.proto:55-59) and only become SpatialInfo doubles by float64(*vec.X) (pkg/unrealpb/extension.go:10-24;
 * x = FVector.X, z = FVector.Y).  The widening is exact and is done on the device behind the copy, so a snapshot costs 8 instead of
 * 16 bytes per entity on PCIe and every result is bit-identical to chd_set_entities fed with the widened values.  Device-resident
 * float arrays (16-byte aligned) are widened in place of the copy. */
chd_status chd_set_entities_f32(chd_engine* e, const float* x, const float* z, uint32_t n);
chd_status chd_prefetch_entities_f32(chd_engine* e, const float* x, const float* z, uint32_t n);
/* (chd_prefetch_queries / chd_prefetch_rings, declared after chd_set_rings, do the same for the other per-tick inputs.) */
chd_status chd_adopt_prefetched(chd_engine* e);
/* Device pointers of the resident position arrays, for producers that write positions on the GPU. */
chd_status chd_entity_buffers(chd_engine* e, double** d_x, double** d_z, uint32_t* n);

/* Declares that the resident position arrays hold n entities (after writing them through chd_entity_buffers). */
chd_status chd_set_entity_count(chd_engine* e, uint32_t n);

/* GetChannelId for every resident entity (the first half of chd_build; idempotent until positions change).
 * Also runs handover detection against the previous assignment. */
chd_status chd_assign_cells(chd_engine* e);

/* Spatial-hash build: cell id per entity (GetChannelId), stable counting sort into the cell CSR
 * (cell asc, entity id asc), and — when a previous build exists — handover detection, the prefix of
 * Notify (spatial.go:612-626): entities whose cell changed since the previous build. */
chd_status chd_build(chd_engine* e);

/* ---- subscribers: slot s in [0,n) <-> connection id (Connection.Id(), used for SkipSelfUpdateFanOut,
 * data.go:240).  Resets all subscriptions. */
chd_status chd_set_subscribers(chd_engine* e, const uint32_t* conn_id, uint32_t n);

/* ---- subscriber lifecycle: slots are managed by the HOST (it owns the connection table, connection.go).  Neither call
 * disturbs any other slot's subscriptions or fan-out state (lastFanOutTime, hadFirstFanOut, lastMessageIndex).
 *   chd_add_subscribers    slot[i] (free: never used, or removed before) becomes connection conn_id[i]; it has no subscriptions
 *                          until its first query (SubscribeToChannel then starts it like any new pair, subscription.go:60-87)
 *   chd_remove_subscribers UnsubscribeFromChannel for every spatial channel of the slot (subscription.go:104-125; also what
 *                          tickConnections does for a closed connection, channel.go:414-475): applied by the NEXT
 *                          chd_update_interest / chd_tick with a batch (an empty batch will do) — the slot's subscriptions appear
 *                          in that update's unsub list, a query for the slot in the same batch is ignored, the slot is free
 *                          afterwards.
 * slot / conn_id are HOST arrays (copied before the call returns).  Slots may exceed the count given to chd_set_subscribers
 * (up to chd_limits.max_subscribers). */
chd_status chd_add_subscribers(chd_engine* e, const uint32_t* slot, const uint32_t* conn_id, uint32_t n);
chd_status chd_remove_subscribers(chd_engine* e, const uint32_t* slot, uint32_t n);

enum { CHD_AOI_SPOTS = 1, CHD_AOI_BOX = 2, CHD_AOI_SPHERE = 4, CHD_AOI_CONE = 8 };

/* A batch of SpatialInterestQuery (channeld.proto:436-469), SoA.  Arrays of kinds no query uses may be
 * NULL.  Y components are not carried: the 2-D grid never reads them (spatial.go:205,237,272).
 * At most one query per subscriber slot per batch (the host coalesces; the reference would apply them
 * in arrival order and only the last one's subscriptions survive). */
typedef struct chd_query_batch {
    uint32_t        n;
    const uint32_t* sub;   /* [n] subscriber slot (UpdateSpatialInterestMessage.connId -> slot), or NULL = identity (query i is
                              subscriber slot i, n <= subscribers); ignored by chd_query_channel_ids */
    const uint8_t*  kind;  /* [n] CHD_AOI_* mask, or NULL = all CHD_AOI_SPHERE */
    const double *sph_cx, *sph_cz, *sph_r;
    const double *box_cx, *box_cz, *box_ex, *box_ez;
    const double *cone_cx, *cone_cz, *cone_dx, *cone_dz, *cone_angle, *cone_r;
    const uint32_t* spot_off;    /* [n+1] CSR into spot_* (NULL when no query has spots) */
    const uint32_t* spot_ndist;  /* [n] how many leading spots of query i carry an explicit dist (len(Dists)) */
    const double *  spot_x, *spot_z;
    const uint32_t* spot_dist;   /* [spot_off[n]]; 0xFFFFFFFF is reserved */
} chd_query_batch;

/* Per-query status (the reference's error returns, spatial.go:208-215,228-231,...). */
enum {
    CHD_Q_OK = 0,
    CHD_Q_ERR_OUT_OF_WORLD = 1, /* centre of a box/sphere/cone outside the world: (nil, err) */
    CHD_Q_ERR_BAD_STEP = 2,     /* radius / extent <= 0 */
    CHD_Q_ERR_ITER_BOUND = 5,   /* step absorbed by a huge coordinate (v + step == v: the reference would loop forever), or a
                                   lattice walk of more than 2^24 samples (cut off: a documented deviation) */
    CHD_Q_ERR_ANGLE_RANGE = 6,  /* |cone angle| >= 2^29: Go switches to Payne-Hanek reduction, not reproduced */
    CHD_Q_ERR_CAPACITY = 7,     /* the query's cell window did not fit chd_limits.max_window_cells (CHD_OVF_WINDOW is raised):
                                   like every failed query it leaves the subscriber's subscriptions untouched */
    CHD_Q_ERR_MISSING_ARRAY = 8 /* a kind bit is set but that kind's arrays were not supplied in the batch */
};

/* ---- QueryChannelIds, batched and stateless (spatial.go:182-317).  CSR output, entries of one query sorted
 * by channel id ascending (the reference returns a Go map: order is unspecified, parity is on keys+dists).
 * out_off[n+1], out_status[n]; out_channel_id/out_dist sized `cap`.  Synchronous. */
chd_status chd_query_channel_ids(chd_engine* e, const chd_query_batch* q, uint32_t* out_status, uint32_t* out_off,
                                 uint32_t* out_channel_id, uint32_t* out_dist, uint64_t cap);

/* ---- handleUpdateSpatialInterest, batched (message_spatial.go:41-129): query -> damping
 * (message_spatial.go:16-38) -> diff against the subscriber's current spatial subscriptions (util.go:105-113)
 * -> SubscribeToChannel / UnsubscribeFromChannel state changes (subscription.go:34-125): new pairs start with
 * lastFanOutTime = now_ns + delay, hadFirstFanOut = false; kept pairs keep their fan-out state and take the
 * new interval; a query that errors leaves that subscriber's subscriptions untouched (message_spatial.go:60-63).
 * Asynchronous (stream-ordered). */
chd_status chd_update_interest(chd_engine* e, const chd_query_batch* q, int64_t now_ns);

/* ---- expanded per-subscriber visible-entity lists: for each subscriber the concatenation, in channel-id
 * order, of the entity lists of its subscribed cells (SURVEY.md §8 a14).  Asynchronous. */
chd_status chd_emit_visible(chd_engine* e);

/* ---- update rings: the per-channel updateMsgBuffer metadata (data.go:46-51) in insertion order, CSR by cell
 * index (channel id - channel_id_start): ring_off[cells+1], n_entries = ring_off[cells].  channel_msg_index[cells] = ChannelData.msgIndex
 * (data.go:25,158) or NULL for zeros.  The host owns OnUpdate/eviction (data.go:149-173): payload merging is
 * opaque protobuf work. */
chd_status chd_set_rings(chd_engine* e, const uint32_t* ring_off, uint32_t n_entries, const int64_t* arrival_ns,
                         const uint32_t* sender_conn_id, const uint64_t* message_index, const uint64_t* channel_msg_index);
/* The same for the other per-tick inputs: the query batch (consumed by the next chd_begin_interest / chd_update_interest
 * called with q == NULL) and the update rings (arguments as chd_set_rings).  Each kind has two staging sets; a set is
 * refilled only after the tick that read it.  chd_adopt_prefetched hands over everything prefetched since the last
 * adoption (any subset of positions / queries / rings). */
chd_status chd_prefetch_queries(chd_engine* e, const chd_query_batch* q);
chd_status chd_prefetch_rings(chd_engine* e, const uint32_t* ring_off, uint32_t n_entries, const int64_t* arrival, const uint32_t* sender,
                              const uint64_t* index, const uint64_t* ch_msg_index);


/* ---- device-owned rings: the buffer half of ChannelData.OnUpdate (data.go:149-173) on the GPU, for every channel at once.
 * chd_rings_init switches the engine from host-owned ring snapshots (chd_set_rings every tick: 20 bytes x every live entry) to rings
 * that live in HBM: capacity_per_cell (> 512) entries per cell, cells x capacity_per_cell <= chd_limits.max_ring_entries.
 * chd_rings_append applies a tick's updates: CSR by cell (upd_off[cells + 1]) in arrival order per cell; for each one
 * msgIndex++, push (arrival, sender, msgIndex), and — if the buffer holds more than 512 entries and its OLDEST is older than the
 * channel's maxFanOutIntervalMs (tracked on the device: it grows when a subscription with a longer interval is created,
 * subscription.go:84-86) — pop that one.  Merging the update into the channel's data message (opaque protobuf) stays with the
 * host.  chd_get_rings reads the live rings back as the CSR chd_set_rings takes (tests, recovery).  Stream-ordered except
 * chd_get_rings. */
chd_status chd_rings_init(chd_engine* e, uint32_t capacity_per_cell);
chd_status chd_rings_append(chd_engine* e, const uint32_t* upd_off, uint32_t n_updates, const int64_t* arrival_ns, const uint32_t* sender_conn_id);
chd_status chd_get_rings(chd_engine* e, uint32_t* ring_off, int64_t* arrival_ns, uint32_t* sender_conn_id, uint64_t* message_index,
                         uint64_t* channel_msg_index, uint32_t cap_entries);
/* ChannelTime origin per channel (channel.go:28-37,178: every channel counts nanoseconds from its own creation): start_ns[cells]
 * in the clock of the t_ns / now_ns arguments; channel c then sees time t - start_ns[c] (subscription times, fan-out windows; ring
 * arrival times are channel times already).  NULL = one shared origin (the default). */
chd_status chd_set_channel_start_times(chd_engine* e, const int64_t* start_ns);

/* One fan-out decision = one fanOutDataUpdate call of the reference (data.go:221,263). */
#define CHD_DUE_VOID 0xFFFFFFFFu
typedef struct chd_due {
    uint32_t sub;          /* subscriber slot */
    uint32_t channel_id;   /* spatial channel */
    uint32_t kind;         /* 0 = FULL channel data (first fan-out, data.go:218-224), 1 = accumulated UPDATE,
                              CHD_DUE_VOID = not a decision (only in a list that overflowed, see CHD_OVF_DUE) */
    uint32_t n_selected;   /* UPDATE: ring entries merged (data.go:246-256) */
    uint32_t first_sel, last_sel; /* ring positions (0-based within the cell's ring) of the first/last merged entry */
    uint64_t sel_hash;     /* sum of merged entries' messageIndex mod 2^64 (lets the host verify its own selection) */
    uint64_t last_message_index; /* foc.lastMessageIndex after the step */
    int64_t  window_hi;    /* nextFanOutTime of the step: entries with lastUpdateTime <= arrival <= window_hi */
} chd_due;

/* ---- Channel.tickData for every spatial channel in one launch (data.go:175-291; replaces the per-channel
 * goroutine loop channel.go:358-387).  Per (subscriber, cell) pair: while t >= lastFanOutTime + interval
 * { first time: FULL, last = t; else select ring entries in [max(last,prev picked), last+interval] skipping
 * own updates, last += interval }.  All cells share one time origin (documented deviation: the reference
 * gives each channel its own startTime, channel.go:178).  Asynchronous. */
chd_status chd_fanout_tick(chd_engine* e, int64_t t_ns);

/* Counters of the work queued since the last summary; read back with ONE small device->host copy. */
typedef struct chd_tick_summary {
    uint64_t n_pairs;          /* live (subscriber, cell) subscriptions */
    uint64_t n_visible;        /* entries of the expanded visible list */
    uint32_t n_entities_in_world;
    uint32_t n_query_errors;
    uint32_t n_sub_new, n_unsub, n_kept;
    uint32_t n_due;
    uint32_t n_handover;
    uint32_t overflow;         /* bitmask of CHD_OVF_* (see below for what each one leaves behind) */
    uint64_t required_pairs, required_window_cells, required_visible;
    uint32_t required_due;
    uint32_t reserved;
} chd_tick_summary;
/* Capacities are fixed at chd_create, so an overflow cannot be retried with the same engine; what matters is that it never
 * corrupts state:
 *   CHD_OVF_PAIRS   the interest update was NOT applied: every subscriber keeps its previous subscriptions and fan-out state,
 *                   the diff lists are empty; required_pairs = the total the update would have needed
 *   CHD_OVF_WINDOW  the queries whose cell windows did not fit got CHD_Q_ERR_CAPACITY and, like any failed query, left their
 *                   subscribers untouched; the rest of the batch was applied; required_window_cells = scratch needed
 *   CHD_OVF_VISIBLE the expanded visible list was not written (offsets are valid); required_visible = entries needed
 *   CHD_OVF_DUE     the pairs whose decisions did not fit were left untouched (still due: they catch up at the next
 *                   chd_fanout_tick); the list holds the decisions that did fit plus CHD_DUE_VOID holes; required_due
 *   CHD_OVF_BORDER  multi-GPU border / halo capacity exceeded: this tick's halo is incomplete */
enum { CHD_OVF_PAIRS = 1, CHD_OVF_WINDOW = 2, CHD_OVF_VISIBLE = 4, CHD_OVF_DUE = 8, CHD_OVF_BORDER = 16,
       CHD_OVF_RING = 32 /* a device-owned ring slab was full of live entries: its oldest entry was dropped */ };
/* bit 31: a device-side wait timed out (results invalid, please report).  A macro, not an enumerator: ISO C enumerators
 * must fit an int. */
#define CHD_OVF_INTERNAL 0x80000000u

/* Synchronises the stream and returns the counters.  CHD_ERR_CAPACITY if any overflow bit is set. */
chd_status chd_summary(chd_engine* e, chd_tick_summary* out);

/* ---- Channel.Tick for all spatial channels (channel.go:358-387), batched: build (if entities changed) ->
 * update_interest(q) (if q != NULL) -> emit_visible (flags & CHD_TICK_EMIT) -> fanout_tick(t_ns)
 * (flags & CHD_TICK_FANOUT) -> summary.  One stream, no intermediate host sync. */
enum {
    CHD_TICK_BUILD = 1, CHD_TICK_EMIT = 2, CHD_TICK_FANOUT = 4, CHD_TICK_ALL = 7,
    /* The host will read this tick's results back (chd_fetch_results): start the expanded-list kernel only after the
     * fan-out pass (it would otherwise starve it of SM slots), so that every host-facing result is final, and is copied
     * to the host, while that kernel is still running.  Costs ~0.06 ms of device time per tick; results are identical. */
    CHD_TICK_EARLY_RESULTS = 8
};
/* Optional early start: the interest update (and the fan-out pass when with_fanout != 0) do not depend on the entity
 * positions, so a host can start them as soon as the tick's queries and rings are known — on the engine's second
 * stream — and then upload / exchange positions; the following chd_tick(e, NULL, t_ns, flags, ..) runs build + emit
 * and joins.  Used by the multi-GPU driver to overlap the border exchange with the interest stage.
 * q == NULL (here and in chd_update_interest) = the batch uploaded by chd_prefetch_queries and handed over by
 * chd_adopt_prefetched; CHD_ERR_STATE if there is none. */
chd_status chd_begin_interest(chd_engine* e, const chd_query_batch* q, int64_t t_ns, int with_fanout);
chd_status chd_tick(chd_engine* e, const chd_query_batch* q, int64_t t_ns, uint32_t flags, chd_tick_summary* out);

/* ---- results.  Each copies to caller memory (host or device) on the engine stream and synchronises.
 * Pass NULL for arrays you do not need.  Counts come from chd_summary. */
/* cell CSR: cell_start[cells+1], sorted_entity[n_entities_in_world] */
chd_status chd_get_cells(chd_engine* e, uint32_t* cell_start, uint32_t* sorted_entity);
/* subscriptions CSR by subscriber slot: pair_off[n_subscribers+1]; per pair channel id, dist, interval ms,
 * flags (bit0 hadFirstFanOut, bit1 subscribed by the last update_interest, bit2 skipSelf), lastFanOutTime */
chd_status chd_get_pairs(chd_engine* e, uint32_t* pair_off, uint32_t* channel_id, uint32_t* dist, uint32_t* interval_ms,
                         uint8_t* flags, int64_t* last_fanout_ns, uint64_t* last_message_index);
/* status per query of the last chd_update_interest batch */
chd_status chd_get_query_status(chd_engine* e, uint32_t* status, uint32_t n);
/* interest diff of the last update: (subscriber slot, channel id) lists.  They are SETS: the order is unspecified
 * (the reference issues these messages in Go map order); sort on the host if a canonical order is needed. */
chd_status chd_get_diff(chd_engine* e, uint32_t* new_sub, uint32_t* new_channel, uint32_t* unsub_sub, uint32_t* unsub_channel);
/* visible lists: vis_off[n_subscribers+1] (u64), vis_entity[n_visible] */
chd_status chd_get_visible(chd_engine* e, uint64_t* vis_off, uint32_t* vis_entity);
/* one subscriber's visible list: copies min(count, cap) entries, *count = its full length */
chd_status chd_get_visible_slot(chd_engine* e, uint32_t slot, uint32_t* out, uint64_t cap, uint64_t* count);
/* fan-out decisions of the last chd_fanout_tick.  A SET: the decisions of one (subscriber, channel) pair are contiguous
 * and in step order, the order across pairs is unspecified (the reference sends from independent channel goroutines). */
chd_status chd_get_due(chd_engine* e, chd_due* out, uint32_t cap);
/* handover candidates of the last build: entity, src channel id, dst channel id (0 = left/entered the world) */
chd_status chd_get_handover(chd_engine* e, uint32_t* entity, uint32_t* src_channel, uint32_t* dst_channel, uint32_t cap);

/* ---- all host-facing results of a tick in ONE call instead of one or two synchronisations per getter.  After a
 * two-stream tick (chd_tick with emit, or chd_begin_interest + chd_tick) the lists are copied in the order they become
 * final, on the engine's read-back streams, while the expanded-list kernel may still be running: first the pairs /
 * sub-unsub lists / query statuses / handover list / cell CSR (after the interest fill and the build), then the due list
 * and the visible offsets (after the fan-out pass and the emit preparation; see CHD_TICK_EARLY_RESULTS); the call returns
 * when the tick has finished.  Otherwise: waits for the tick, reads the summary, enqueues every copy, waits once.
 * Exact sizes come from the device counters.  Any pointer may be NULL (skipped).  Capacities are in elements; CHD_ERR_CAPACITY if a requested list does not
 * fit (nothing is truncated silently).  This is what a channeld host calls once per tick. */
typedef struct chd_result_buffers {
    uint32_t *pair_off, *pair_channel, *pair_dist, *pair_interval_ms; /* pair_off[n_subscribers+1]; others [pair_cap] */
    uint64_t pair_cap;
    uint32_t *new_sub, *new_channel, *unsub_sub, *unsub_channel;      /* [diff_cap] each */
    uint64_t diff_cap;
    chd_due* due;                                                     /* [due_cap] */
    uint32_t due_cap;
    uint32_t *handover_entity, *handover_src, *handover_dst;          /* [handover_cap] */
    uint32_t handover_cap;
    uint32_t* query_status;                                           /* [status_cap] */
    uint32_t status_cap;
    uint64_t* vis_off;                                                /* [n_subscribers+1] */
    uint32_t* vis_entity;                                             /* [vis_cap] (the big one: usually NULL) */
    uint64_t vis_cap;
    uint32_t *cell_start, *sorted_entity;                             /* [cells+1], [entity_cap] */
    uint32_t entity_cap;
} chd_result_buffers;
chd_status chd_fetch_results(chd_engine* e, const chd_result_buffers* bufs, chd_tick_summary* summary);

/* ---- the same read-back WITHOUT blocking: copy kernels that know the exact lengths on the device first snapshot the lists into a
 * staging area in HBM (microseconds; the next tick's kernels are ordered after THIS, not after the PCIe transfer), then write the
 * snapshot into the caller's PINNED host buffers (chd_alloc_pinned) on a stream of their own; the call returns at once, so the host
 * can enqueue the NEXT tick before looking at this one.
 * pinned_header: CHD_FETCH_HEADER_BYTES of pinned memory the engine uses for the counters.  Up to two fetches may be outstanding
 * (use two sets of buffers); chd_fetch_wait blocks until the copies of the OLDEST outstanding chd_fetch_results_async are
 * complete and returns that tick's summary (CHD_ERR_CAPACITY if a list did not fit its
 * buffer: it was truncated to the capacity).  vis_entity is not supported here (the expanded list stays in HBM).
 * Loop of a pipelined host:  prefetch(k+1) ... adopt, chd_begin_interest, chd_tick(k) ; chd_fetch_results_async(k) ;
 * [enqueue tick k+1 the same way] ; chd_fetch_wait -> results of tick k while tick k+1 runs. */
#define CHD_FETCH_HEADER_BYTES 256
chd_status chd_fetch_results_async(chd_engine* e, const chd_result_buffers* bufs, void* pinned_header);
chd_status chd_fetch_wait(chd_engine* e, chd_tick_summary* summary);

/* Device-resident views (valid until the next call that rewrites them) for consumers that stay on the GPU. */
enum {
    CHD_VIEW_CELL_START = 0, CHD_VIEW_SORTED_ENTITY, CHD_VIEW_ENT_CELL, CHD_VIEW_PAIR_OFF, CHD_VIEW_PAIR_CHANNEL,
    CHD_VIEW_PAIR_DIST, CHD_VIEW_VIS_OFF, CHD_VIEW_VIS_ENTITY, CHD_VIEW_DUE,
    /* the lists of the last chd_visible_delta (CHD_ERR_STATE before chd_visible_delta_enable): offsets count = S + 1, entity
     * lists count = cap_entries */
    CHD_VIEW_ENTER_OFF, CHD_VIEW_ENTER_ENTITY, CHD_VIEW_LEAVE_OFF, CHD_VIEW_LEAVE_ENTITY
};
chd_status chd_device_view(chd_engine* e, int which, void** d_ptr, uint64_t* count);

/* ---- per-subscriber visibility deltas: the entities that entered and left each subscriber's view since the last call, without
 * the expanded visible list (a channeld host spawns / despawns and subscribes / unsubscribes entity channels from them; the
 * reference does this bookkeeping by hand in Notify, spatial.go:776-857).
 *   V(s)  = { e : cell(e) in C(s) } for subscriber slot s, where cell(e) is the cell of entity e in the last chd_build (entities out
 *           of the world and entities with id >= n are in no cell) and C(s) the slot's spatial subscriptions after the last interest
 *           update (the pairs of chd_get_pairs): exactly the list chd_emit_visible writes for s.
 *   The engine keeps a BASELINE: cell(e) and C(s) as they stood at the last successful chd_visible_delta (before the first call:
 *   empty, no entity is visible to anyone).  chd_visible_delta computes for every slot
 *           enter(s) = V_now(s) \ V_base(s)        leave(s) = V_base(s) \ V_now(s)
 *   and makes "now" the baseline.  The delta spans everything since the previous call however many ticks that is: an entity
 *   that left and came back in between is in neither list.
 *   Output: two CSRs by slot, enter_off[S+1] (u64) / enter_entity[] and leave_off[S+1] / leave_entity[], S = the current slot
 *   count (or the baseline's, if chd_set_subscribers made it smaller since: those slots' views leave too).  Fixed order: enter
 *   entries by (current cell asc, entity id asc), leave entries by (baseline cell asc, entity id asc) within a slot.
 *   Slots are the unit: chd_remove_subscribers / chd_set_subscribers make a slot's whole view leave, a query that errors keeps
 *   the slot's subscriptions and so gives it no delta from them; a slot recycled between two calls (removed, then added for
 *   another connection) shows ONE merged delta of the old and the new view.
 *   Independent of CHD_TICK_EMIT: a tick without the expanded list gives the same delta.
 *   Single engine only: CHD_ERR_STATE after chd_set_slab / chd_comm_init / chd_set_entity_ids (entity indices are not stable
 *   across ticks there), also while a chd_begin_interest is pending and when cells were assigned after the last chd_build.
 * Overflow is transactional: if either list needs more than cap_entries, the offsets are valid, the entity lists are not written
 * and the baseline is NOT advanced (decided on the device, in stream order); chd_visible_delta_enable with the required size and
 * another chd_visible_delta give the whole delta since the old baseline.  Nothing here touches chd_tick_summary. */
/* allocates the baseline + output buffers (cap_entries each for enter and leave); may be called again to grow them, the baseline
 * is kept.  Nothing is allocated on the delta path afterwards. */
chd_status chd_visible_delta_enable(chd_engine* e, uint64_t cap_entries);
/* stream-ordered, no host synchronisation; CHD_ERR_STATE before enable / before a build / on a sharded engine */
chd_status chd_visible_delta(chd_engine* e);
/* synchronous getter in the style of chd_get_visible; any pointer may be NULL; *n_enter / *n_leave = exact totals.
 * CHD_ERR_CAPACITY if the last chd_visible_delta did not fit cap_entries or the caller's caps. */
chd_status chd_get_visible_delta(chd_engine* e, uint64_t* enter_off, uint32_t* enter_entity, uint64_t enter_cap,
                                 uint64_t* leave_off, uint32_t* leave_entity, uint64_t leave_cap,
                                 uint64_t* n_enter, uint64_t* n_leave);

/* ---- multi-GPU X-slab sharding (SURVEY.md §8e).  The engine owns grid columns [col_lo, col_hi) and serves
 * queries whose cells lie in [col_lo-halo, col_hi+halo).  After chd_build, chd_export_border writes the
 * (entity id, cell index) records of the entities in this rank's outermost `halo` columns on each side into a
 * caller-provided DEVICE buffer (2 x u32 per record; the unused tail is padded with 0xFFFFFFFF) for the all-gather;
 * chd_import_halo takes the gathered records of all ranks (records [skip_first, skip_first+skip_count) are this
 * rank's own and ignored), keeps those whose column lies in [col_lo-halo, col_hi+halo) and appends them as
 * position-less halo entities; the following chd_build sorts own + halo entities into the cell CSR.
 * Call order per tick: chd_set_entities -> chd_export_border (runs chd_assign_cells) -> all-gather ->
 * chd_import_halo -> chd_build.  Entity ids are global: set with chd_set_entity_ids. */
chd_status chd_set_slab(chd_engine* e, uint32_t col_lo, uint32_t col_hi, uint32_t halo);
chd_status chd_set_entity_ids(chd_engine* e, const uint32_t* global_id, uint32_t n);
/* out_count may be NULL: then nothing synchronises with the host (an overflow of cap_records or of the entity capacity
 * surfaces as CHD_OVF_BORDER in the next chd_summary). */
chd_status chd_export_border(chd_engine* e, uint32_t* d_records, uint32_t cap_records, uint32_t* out_count);
chd_status chd_import_halo(chd_engine* e, const uint32_t* d_records, uint32_t n_records, uint32_t skip_first, uint32_t skip_count);

/* ---- the exchange behind the ABI: NCCL over NVLink / NVSwitch, one process per GPU.  libnccl.so.2 is loaded on first use
 * (a copy the process already holds is reused); a host needs no NCCL binding of its own.
 *   rank 0:      chd_comm_unique_id(id)            -> the host distributes the 128 bytes by any means (TCP, a file, MPI, ...)
 *   every rank:  chd_comm_init(e, id, rank, world, halo_cols, border_capacity, migrate_subscribers, migrate_pairs)   (collective;
 *                also sets this rank's slab: columns [floor(rank*cols/world), floor((rank+1)*cols/world)), halo_cols =
 *                ceil(max radius / grid_width); migrate_* = capacity of the per-tick subscriber migration blob, 0 = none)
 *   every tick:  chd_set_rings / chd_set_entities (this rank's entities, global ids via chd_set_entity_ids) ...
 *                chd_tick_sharded(e, q, t_ns, flags, summary) = chd_begin_interest + chd_export_border + ONE ncclAllGather of
 *                (entity id, cell) records (border_capacity records per rank, padded) + chd_import_halo + chd_tick: collective,
 *                stream-ordered, no host synchronisation unless summary != NULL.
 * border_capacity bounds the records ONE rank exports per tick (entities in its outermost halo_cols columns on each side
 * plus entities that left its slab); border_capacity * world must fit chd_limits.max_entities together with the own
 * entities.  Exceeding it raises CHD_OVF_BORDER. */
#define CHD_COMM_ID_BYTES 128
chd_status chd_comm_unique_id(void* out_id);
chd_status chd_comm_init(chd_engine* e, const void* unique_id, int rank, int world, uint32_t halo_cols, uint32_t border_capacity,
                         uint32_t migrate_subscribers, uint32_t migrate_pairs);
chd_status chd_comm_info(const chd_engine* e, int* rank, int* world, uint32_t* col_lo, uint32_t* col_hi, uint32_t* halo_cols, int* nccl_version);
chd_status chd_comm_destroy(chd_engine* e);
chd_status chd_tick_sharded(chd_engine* e, const chd_query_batch* q, int64_t t_ns, uint32_t flags, chd_tick_summary* out);
uint64_t chd_collective_count(const chd_engine* e); /* NCCL collectives issued so far */
/* How chd_tick_sharded moves the border records: 2 = PEER WINDOWS (default when every rank could map every other rank's receive
 * window with CUDA IPC at chd_comm_init: the export kernel's successor stores the live records straight into the peers' memory over
 * NVLink and publishes a 64-bit flag; the import's first kernel polls the local flags — no collective call on the tick path),
 * 1 = one ncclAllGather per tick (ranks without a P2P path, more than 16 ranks), 0 = no communicator.
 * chd_comm_use_collective(e, 1) selects the NCCL exchange even when peer windows are mapped (every rank must make the same choice,
 * between ticks); (e, 0) returns to the peer windows. */
int chd_comm_exchange_mode(const chd_engine* e);
chd_status chd_comm_use_collective(chd_engine* e, int on);

/* ---- re-homing.  ENTITIES: an entity that leaves its owner's slab is still exported by that owner and adopted, for this tick, by
 * every rank that needs it (visibility stays exact whatever the ownership); chd_get_rehome lists the own entities whose column
 * now belongs to another rank (global id, destination rank) so the host can re-route their position feed — the sender drops
 * them from its next chd_set_entities, the receiver includes them (the reference moves an entity between spatial channels the
 * same way, spatial.go:683-736).
 * SUBSCRIBERS live on the rank that owns their centre's column (the host routes each query there).  When that owner changes
 * from rank A to rank B the subscriber's subscriptions and fan-out state (lastFanOutTime, hadFirstFanOut, lastMessageIndex per
 * channel) travel INSIDE the tick's all-gather, so nothing is reset and nobody is re-sent FULL channel data:
 *   on A, before chd_tick_sharded:  chd_migrate_out(eA, slot[], n)          record i of A's blob = state of slot[i]; A's slots are
 *                                                                           freed by this tick's interest update (no unsub entries)
 *   on B, before chd_tick_sharded:  chd_migrate_in(eB, A, first_index, slot[], conn_id[], n)
 *                                   B's slot[i] becomes connection conn_id[i] with the state of record first_index + i of A's blob;
 *                                   its query in this tick's batch is diffed against that state.
 * Both ranks pass a query batch (an empty one will do) to the same chd_tick_sharded.  One chd_migrate_out per tick and rank;
 * any number of chd_migrate_in.  Capacities: chd_comm_init's migrate_* (overflow: CHD_OVF_BORDER, the cut-off subscribers arrive
 * without state).  slot / conn_id are HOST arrays. */
chd_status chd_migrate_out(chd_engine* e, const uint32_t* slot, uint32_t n);
chd_status chd_migrate_in(chd_engine* e, uint32_t src_rank, uint32_t first_index, const uint32_t* slot, const uint32_t* conn_id, uint32_t n);
/* own entities (of the last cell assignment) whose column lies outside this rank's slab: global id + the rank that owns the
 * column now.  Synchronous.  *count = how many there are (copies min(count, cap)). */
chd_status chd_get_rehome(chd_engine* e, uint32_t* global_id, uint32_t* dst_rank, uint32_t cap, uint32_t* count);

/* ---- window classes of the last fan-out pass (SURVEY.md §8f rank 1: payload assembly).  The reference merges the selected
 * update window afresh for every subscriber (data.go:248-252); decisions of one channel whose merged payload is
 * necessarily identical are grouped so the host merges / frames each distinct payload once:
 *   - all FULL decisions (kind 0) of a channel form one class (they all send ch.data.msg, data.go:219-224);
 *   - UPDATE decisions (kind 1) of a channel with the same lastFanOutTime at the start of the step, the same window_hi and
 *     no own update left out by SkipSelfUpdateFanOut form one class (the selection loop data.go:226-256 is then a
 *     function of the channel's buffer and these two times only);
 *   - an UPDATE decision whose subscriber had own updates inside the window is a class of its own.
 * out_class_of[i] = class of due record i (index into the list chd_get_due / chd_fetch_results return, same order),
 * out_class_rep[k] = lowest due index of class k (classes are numbered by it), out_class_count[k] = its size.
 * Any output may be NULL.  CHD_ERR_CAPACITY if there are more than cap_classes classes.  Synchronous. */
chd_status chd_due_classes(chd_engine* e, uint32_t* out_class_of, uint32_t* out_class_rep, uint32_t* out_class_count,
                           uint32_t cap_classes, uint32_t* out_n_classes);

/* ---- the BYTE half of the fan-out (SURVEY.md §8f rank 1 and 4): per window class the wire bytes of its CHANNEL_DATA_UPDATE
 * message are assembled ONCE on the device (the reference re-merges and marshals three times per subscriber: data.go:246-256,
 * :295, connection.go:58, :671), then every connection's packets are laid out framed — 'C' 'H' size_hi size_lo compressionType
 * + marshalled Packet, optionally snappy-compressed (connection.go:626-714) — ready for conn.Write.
 *   chd_set_payload_bytes   per-tick input next to chd_set_rings: serialized updateMsg of every ring entry (CSR entry_off[n_entries+1]
 *                           in the ring order of chd_set_rings) and serialized full data message of every channel (full_off[cells+1]),
 *                           the Any type URL of the channel data type and the message type (MessageType_CHANNEL_DATA_UPDATE = 8).
 *   chd_assemble_payloads   after chd_fanout_tick / chd_tick: window classes (chd_due_classes) + for class k the bytes
 *                           blob[class_off[k] .. class_off[k+1]) = one Packet.messages entry (0x0A len MessagePack{channelId,
 *                           msgType, msgBody = ChannelDataUpdateMessage{data = Any{type_url, value}}}) where value = the
 *                           concatenation of the selected ring entries' bytes (= proto.Merge of them, by the protobuf encoding
 *                           rules) or the channel's full data for a FULL send.  Outputs may be NULL (results stay on the GPU).
 *   chd_frame_packets       per connection (subscriber slot s): bytes out[conn_off[s] .. conn_off[s] + conn_len[s]) = its packets
 *                           back to back, each 5-byte tag + body; a packet holds as many of the connection's messages as fit
 *                           MaxPacketSize (0xffff), a single message >= MaxPacketSize - 5 is dropped (connection.go:73-77; counted
 *                           in *n_dropped); compression[s] = 1 -> snappy block format (decodes with any snappy decoder; the bytes
 *                           differ from Go's encoder).  conn_off is spaced for the worst case; conn_frames[s] = packets written.
 * Valid for channel data types merged by the default reflection merge without ChannelDataMergeOptions (data.go:326-388);
 * types with a custom Merge stay on the host.  Synchronous; buffers of this stage grow on demand. */
chd_status chd_set_payload_bytes(chd_engine* e, const uint64_t* entry_off, uint32_t n_entries, const uint8_t* entry_bytes, const uint64_t* full_off,
                                 const uint8_t* full_bytes, const char* type_url, uint32_t msg_type);
chd_status chd_assemble_payloads(chd_engine* e, uint32_t* n_classes, uint64_t* class_off, uint32_t cap_classes, uint8_t* blob, uint64_t blob_cap,
                                 uint64_t* blob_len);
chd_status chd_frame_packets(chd_engine* e, const uint8_t* compression, uint64_t* conn_off, uint32_t* conn_len, uint32_t* conn_frames, uint8_t* out,
                             uint64_t out_cap, uint64_t* out_len, uint32_t* n_dropped);

/* ---- BroadcastType_ADJACENT_CHANNELS recipient sets, batched (message.go:188-239; SURVEY.md §8f rank 3).
 * For message m sent to spatial channel channel_id[m] with BroadcastType mask broadcast[m] (channeld.proto: ALL_BUT_SENDER 4,
 * ALL_BUT_OWNER 8, ALL_BUT_CLIENT 16, ALL_BUT_SERVER 32; the ADJACENT_CHANNELS bit itself is implied): the recipients are
 * the subscribers (slots of chd_set_subscribers, per the CURRENT spatial subscriptions = last chd_update_interest) of the
 * channel's 3x3 neighbours (spatial.go:358-381) and — unless ALL_BUT_OWNER — of the channel itself, each slot once
 * (the reference's adjacentConns map), minus the slot whose connection id equals sender_conn_id[m] when ALL_BUT_SENDER
 * is set, the clients / servers when ALL_BUT_CLIENT / ALL_BUT_SERVER are set (chd_set_subscriber_types), and the slot
 * whose connection id equals client_conn_id[m] (ServerForwardMessage.ClientConnId; 0 = none).
 * Output: CSR out_off[n + 1] / out_slot[] (a SET per message: the reference iterates a Go map), out_status[m] =
 * CHD_BC_OK or CHD_BC_ERR_NOT_A_CELL (channel id outside this grid: the reference cannot reach this, the channel must
 * exist; such a message gets no recipients).  Synchronous; CHD_ERR_CAPACITY if the lists need more than cap entries.
 * sender_conn_id / client_conn_id may be NULL (= all 0). */
typedef struct chd_broadcast_batch {
    uint32_t n;
    const uint32_t* channel_id;
    const uint32_t* broadcast;
    const uint32_t* sender_conn_id;
    const uint32_t* client_conn_id;
} chd_broadcast_batch;
enum { CHD_BC_OK = 0, CHD_BC_ERR_NOT_A_CELL = 1 };
enum { CHD_CONN_SERVER = 1, CHD_CONN_CLIENT = 2 }; /* channeldpb.ConnectionType */
/* ConnectionType per subscriber slot (NULL = unknown: the ALL_BUT_CLIENT / ALL_BUT_SERVER filters then remove nobody). */
chd_status chd_set_subscriber_types(chd_engine* e, const uint8_t* conn_type, uint32_t n);
chd_status chd_adjacent_broadcast(chd_engine* e, const chd_broadcast_batch* b, uint32_t* out_status, uint32_t* out_off,
                                  uint32_t* out_slot, uint64_t cap);

/* ---- control-plane helpers kept for interface completeness (pure integer/config math on the host; not part
 * of the data-parallel path): GetAdjacentChannels (spatial.go:358-381) and GetRegions (spatial.go:319-356). */
uint32_t chd_get_adjacent_channels(const chd_grid_cfg* cfg, uint32_t channel_id, uint32_t* out8);
chd_status chd_get_regions(const chd_grid_cfg* cfg, double* min_x, double* min_z, double* max_x, double* max_z,
                           uint32_t* channel_id, uint32_t* server_index);
/* dist -> FanOutIntervalMs (message_spatial.go:16-38); the same table the kernels use. */
uint32_t chd_damping_interval_ms(uint32_t dist, uint32_t default_ms);

/* ---- instrumentation.  chd_launch_count: kernels launched by this engine so far.  chd_profile_enable(1)
 * makes every stage record a CUDA-event pair on the engine stream (the last 1024 samples are kept);
 * chd_profile_get synchronises and returns the summed device time of a stage.  CHD_STAGE_EMIT_KERNEL brackets
 * exactly the emit_visible kernel (the dominant HBM term; bench.py's roofline uses it); chd_profile_enable(2) records that
 * pair only (two events per tick instead of about twenty: what bench.py leaves on inside its timed region). */
enum { CHD_STAGE_BUILD = 0, CHD_STAGE_INTEREST, CHD_STAGE_EMIT, CHD_STAGE_EMIT_KERNEL, CHD_STAGE_FANOUT, CHD_STAGE_TICK,
       CHD_STAGE_EXPORT, CHD_STAGE_EXCHANGE, CHD_STAGE_IMPORT, /* the three steps of chd_tick_sharded before the tick proper */
       CHD_STAGE_READBACK,                                     /* chd_fetch_results_async: the PCIe hop (snapshot -> pinned host) */
       CHD_STAGE_COUNT };
uint64_t chd_launch_count(const chd_engine* e);
/* The launch-bound stages (build, interest update, emit preparation, fan-out) are replayed as CUDA graphs once
 * their shape (entity / query / subscriber counts) has been stable for two ticks.  chd_enable_graphs(e, 0) forces
 * direct launches; chd_graph_launch_count reports how many stage executions were graph replays. */
chd_status chd_enable_graphs(chd_engine* e, int on);
uint64_t chd_graph_launch_count(const chd_engine* e);
chd_status chd_profile_enable(chd_engine* e, int on);
chd_status chd_profile_get(chd_engine* e, int stage, double* total_ms, uint64_t* samples);
/* Timeline of the most recent chd_tick: start / stop of a stage in ms after the tick started (CHD_STAGE_TICK start). */
chd_status chd_profile_timeline(chd_engine* e, int stage, double* start_ms, double* stop_ms);

uint32_t chd_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif
