// chd_types.cuh — plain structs shared between the kernels (csrc/*.cuh) and the host-side launch code (csrc/*.cu).
#pragma once
#include "chd_device.cuh"

namespace chd {

// tile geometry the host-side sizing code shares with the kernels
constexpr int BUILD_THREADS = 256;
constexpr int BUILD_WARPS = BUILD_THREADS / 32;
constexpr int BUILD_ROUNDS = 8;
constexpr int BUILD_TILE = BUILD_THREADS * BUILD_ROUNDS;  // 2048 entities per tile
constexpr int BUILD_MAX_BINS = 1024;
constexpr int EMIT_THREADS = 256;
#ifndef CHD_EMIT_ROWS
#define CHD_EMIT_ROWS 4
#endif
#ifndef CHD_EMIT_MIN_BLOCKS
#define CHD_EMIT_MIN_BLOCKS 8
#endif
// Dynamic shared memory the two-segment emit kernel asks for WITHOUT using it: 0 lets 8 CTAs (every warp slot and the whole
// register file of an SM) be emit CTAs; 30 KB caps them at 7 per SM, which keeps one slot (256 threads, 8 K registers, 18 KB)
// free for the latency-bound kernels of the second stream (fan-out pass) that run next to it.
#ifndef CHD_EMIT_DYN_SMEM
#define CHD_EMIT_DYN_SMEM 0
#endif
#ifndef CHD_EMIT_TILES_PER_CTA
#define CHD_EMIT_TILES_PER_CTA 1
#endif
constexpr int EMIT_TILES_PER_CTA = CHD_EMIT_TILES_PER_CTA;  // tiles one CTA copies (their descriptor loads overlap)
constexpr int EMIT_ROWS = CHD_EMIT_ROWS;                    // 16-byte chunks per thread per tile
constexpr int EMIT_TILE = EMIT_THREADS * 4 * EMIT_ROWS;     // 4096 entries = 16 KB of output per CTA
constexpr int EMIT_SMEM_PAIRS = 256;                        // pairs per tile staged in shared memory (one per thread)
// the general (warp-tile) kernel: 8 x 16 bytes per lane = 4 KB of output per warp tile
constexpr int EMIT_WARP_WARPS = EMIT_THREADS / 32;
constexpr int EMIT_WARP_CHUNKS = 8;
constexpr int EMIT_WARP_TILE = 32 * EMIT_WARP_CHUNKS * 4;   // 1024 entries
constexpr int EMIT_WARP_SMEM_PAIRS = 64;

// Per-tile copy descriptor written by the partition pass: the emit kernel needs ONE 16-byte load (broadcast to the CTA)
// before it can issue its data loads, instead of a chain of three dependent index loads (first pair -> offsets / cell ->
// cell start).  A tile is "simple" if at most two pairs' lists intersect it (always the case when cells hold more entities
// than a tile: 4 444 vs 4 096 on the benchmark config); other tiles take the general path (segment table in shared memory).
struct TileDesc {
    uint32_t src0;  // phase-adjusted base of the first segment: slot o of the tile <- sorted4[src0 + o]
    uint32_t src1;  // the same for the second segment (slots o >= end0)
    uint32_t ends;  // end0 | end1 << 16 (relative to the tile base, <= EMIT_TILE); bit 31 = not simple
    uint32_t p0;    // the pair that owns the tile's first slot (general path)
};
static_assert(EMIT_TILE <= 0x7FFF, "segment ends are packed into 15 bits");

struct QueryDev {
    uint32_t n;
    const uint32_t* sub;
    const uint8_t* kind;
    const double *sph_cx, *sph_cz, *sph_r;
    const double *box_cx, *box_cz, *box_ex, *box_ez;
    const double *cone_cx, *cone_cz, *cone_dx, *cone_dz, *cone_angle, *cone_r;
    const uint32_t *spot_off, *spot_ndist;
    const double *spot_x, *spot_z;
    const uint32_t* spot_dist;
};

struct Bbox {
    uint32_t gx0, gy0, bw, bh;  // bw == 0 => empty
};

struct PairBuf {
    uint32_t* off;         // [S+1]
    uint32_t* sub;         // [P] owning subscriber slot
    uint32_t* cell;        // [P] cell index
    uint32_t* dist;        // [P]
    uint32_t* interval;    // [P] FanOutIntervalMs
    uint8_t* flags;        // [P]
    int64_t* last;         // [P] lastFanOutTime (ns)
    uint64_t* last_index;  // [P] lastMessageIndex
};
enum : uint8_t { PF_HAD_FIRST = 1, PF_NEW = 2, PF_SKIP_SELF = 4 };

struct Counters {  // device mirror of chd_tick_summary's counters
    unsigned long long n_pairs, n_visible;
    uint32_t n_entities_in_world, n_query_errors, n_sub_new, n_unsub, n_kept, n_due, n_handover, overflow;
    unsigned long long required_pairs, required_window_cells, required_visible;
    uint32_t required_due, reserved;
};

// Pending lifecycle change of a subscriber slot, applied by the next interest update (chd_interest.cuh):
enum : uint8_t {
    SLOT_NORMAL = 0,
    SLOT_REMOVE = 1,  // chd_remove_subscribers: every subscription of the slot is reported as unsubscribed, the slot is freed
    SLOT_DROP = 2,    // chd_migrate_out: the slot's state was packed for another rank; its run vanishes without unsub entries
    SLOT_IMPORT = 3   // chd_migrate_in: the slot's previous run comes out of the gathered migration blob (MigView)
};

// Subscriber state in flight between ranks: every rank contributes one fixed-size blob to the tick's all-gather (after its
// border records).  Word layout of a blob (u32 words; Ms = max_subs, Mp = max_pairs, both even):
//   [0] n_sub  [1] n_pairs  [2..3] pad | off[Ms+2] | conn[Ms] | cell[Mp] | dist[Mp] | interval[Mp] | flags[Mp] |
//   last[Mp] (i64) | last_index[Mp] (u64)
struct MigView {
    const uint32_t* base;   // nullptr: no migration data this tick
    uint64_t stride_words;  // distance between the blobs of consecutive ranks
    uint32_t max_subs, max_pairs;
    __host__ __device__ static uint64_t words(uint32_t ms, uint32_t mp) { return 4ull + (ms + 2ull) + ms + 4ull * mp + 4ull * mp; }
    __host__ __device__ uint64_t o_off() const { return 4; }
    __host__ __device__ uint64_t o_conn() const { return o_off() + max_subs + 2ull; }
    __host__ __device__ uint64_t o_cell() const { return o_conn() + max_subs; }
    __host__ __device__ uint64_t o_dist() const { return o_cell() + max_pairs; }
    __host__ __device__ uint64_t o_interval() const { return o_dist() + max_pairs; }
    __host__ __device__ uint64_t o_flags() const { return o_interval() + max_pairs; }
    __host__ __device__ uint64_t o_last() const { return o_flags() + max_pairs; }
    __host__ __device__ uint64_t o_lidx() const { return o_last() + 2ull * max_pairs; }
};

struct DiffOut {  // the two interest-diff lists of a tick: (subscriber slot, channel id)
    uint32_t *new_sub, *new_ch, *gone_sub, *gone_ch;
};

struct RingDev {
    const uint32_t* off;        // ring of cell c = entries [off[c], end[c]): host-owned rings are a CSR (end = off + 1),
    const uint32_t* end;        // device-owned rings (chd_rings_init) keep begin / end cursors per cell
    const int64_t* arrival;     // insertion order per cell
    const uint32_t* sender;
    const uint64_t* index;
    const uint64_t* channel_msg_index;  // [C] or nullptr
    const uint32_t* total;              // entries uploaded (device scalar): offsets are clamped to it
    const int64_t* start;               // [C] ChannelTime origin of each channel (channel.go:28-37,178) or nullptr = one shared origin
};

// Payload identity of a decision (window classes, chd_classes.cuh): two decisions of one channel carry the same merged
// payload if they are both FULL, or if they start from the same lastFanOutTime (`lo`), end at the same nextFanOutTime
// (the record's window_hi) and neither subscriber had an own update left out of that window; a decision with
// self-skipped updates is its own class.  word = cell << 34 | kind << 33 | skipped << 32 | (skipped ? subscriber slot : 0).
struct DueKey {
    int64_t lo;
    uint64_t word;
};

struct HandoverOut {
    uint32_t* entity;
    uint32_t* src_cell;
    uint32_t* dst_cell;
    uint32_t* count;  // device counter (may exceed cap: required size)
    uint32_t cap;
};

// Extras of the FINAL pass of the entity build, fused into the scatter:
//   phase_stride != 0 : also write the three phase-shifted copies of the payload (chd_emit.cuh)
//   cell_start != null: single-pass sorts only (digit == key): block 0 publishes the cell CSR offsets straight from
//                       the scanned histogram (cell_start[c] = #keys < c), replacing a separate boundaries kernel
struct ScatterExtras {
    uint32_t phase_stride;
    uint32_t* cell_start;
    uint32_t cells;
    uint32_t* n_in_world;
};

// device-side state of the visibility-delta stage (chd_visdelta.cuh), one per engine
struct VdState {
    uint32_t n_now, S_now, P_now;     // this call: entities of the last build, subscriber slots, live pairs
    uint32_t n_base, S_base, P_base;  // the baseline
    uint32_t n_movers;                // entities whose cell key differs between the two states
    uint32_t ovf;                     // the delta did not fit the output capacity: nothing written, baseline kept
    unsigned long long n_enter, n_leave;
};

struct BcastDev {
    uint32_t n;
    const uint32_t *channel, *flags, *sender, *client;
};

}  // namespace chd
