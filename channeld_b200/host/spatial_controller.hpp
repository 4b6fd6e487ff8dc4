// spatial_controller.hpp — header-only C++17 host mirror of channeld's SpatialController plugin surface
// (pkg/channeld/spatial.go:17-35) on top of the C ABI (include/chd_gpu.h).  Method names, argument meaning and
// error behaviour follow the Go interface: Go's `(value, error)` becomes `value` + SpatialError thrown.
// No hot-path arithmetic lives here: every position -> cell, query and fan-out decision is a libchd_b200.so call.
#pragma once
#include <cstdint>
#include <map>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/chd_gpu.h"

namespace channeld {

struct SpatialError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

struct SpatialInfo {  // pkg/common/common.go:20-24
    double X = 0, Y = 0, Z = 0;
};

struct SpatialInterestQuery {  // channeld.proto:436-469
    struct Spots { std::vector<SpatialInfo> spots; std::vector<uint32_t> dists; };
    struct Box { SpatialInfo center, extent; };
    struct Sphere { SpatialInfo center; double radius = 0; };
    struct Cone { SpatialInfo center, direction; double angle = 0, radius = 0; };
    std::optional<Spots> spotsAOI;
    std::optional<Box> boxAOI;
    std::optional<Sphere> sphereAOI;
    std::optional<Cone> coneAOI;
};

struct SpatialRegion {  // channeld.proto:419-424
    SpatialInfo min, max;
    uint32_t channelId = 0, serverIndex = 0;
};

class GpuStaticGrid2DSpatialController {
   public:
    GpuStaticGrid2DSpatialController() = default;
    GpuStaticGrid2DSpatialController(const GpuStaticGrid2DSpatialController&) = delete;
    GpuStaticGrid2DSpatialController& operator=(const GpuStaticGrid2DSpatialController&) = delete;
    ~GpuStaticGrid2DSpatialController() { chd_destroy(engine_); }

    // LoadConfig (spatial.go:141-159) with the fields already parsed from the -scc JSON.
    void LoadConfig(const chd_grid_cfg& cfg, uint32_t max_entities, uint32_t max_subscribers, int device = 0) {
        cfg_ = cfg;
        chd_limits lim;
        chd_default_limits(&cfg_, max_entities, max_subscribers, &lim);
        chd_destroy(engine_);
        engine_ = nullptr;
        if (chd_create(&cfg_, &lim, device, &engine_) != CHD_OK) throw SpatialError(chd_last_error(nullptr));
    }

    // GetChannelId (spatial.go:161-163)
    uint32_t GetChannelId(const SpatialInfo& info) {
        uint32_t id = 0;
        uint8_t ok = 0;  // explicit validity: with SpatialChannelIdStart == 0 the id 0 is a real cell
        check(chd_cell_of_valid(engine_, &info.X, &info.Z, 1, &id, &ok));
        if (!ok) throw SpatialError("position is outside the grid");
        return id;
    }
    // batched form (handleQuerySpatialChannel, message_spatial.go:335-370); 0 marks an error
    std::vector<uint32_t> GetChannelIds(const std::vector<double>& x, const std::vector<double>& z) {
        std::vector<uint32_t> out(x.size());
        check(chd_cell_of(engine_, x.data(), z.data(), (uint32_t)x.size(), out.data()));
        return out;
    }

    // QueryChannelIds (spatial.go:182-317)
    std::map<uint32_t, uint32_t> QueryChannelIds(const SpatialInterestQuery& q) {
        chd_query_batch b{};
        b.n = 1;
        uint8_t kind = 0;
        double sph[3] = {}, box[4] = {}, cone[6] = {};
        uint32_t spot_off[2] = {0, 0}, spot_nd = 0;
        std::vector<double> sx, sz;
        std::vector<uint32_t> sd;
        if (q.spotsAOI) {
            kind |= CHD_AOI_SPOTS;
            for (size_t i = 0; i < q.spotsAOI->spots.size(); i++) {
                sx.push_back(q.spotsAOI->spots[i].X);
                sz.push_back(q.spotsAOI->spots[i].Z);
                sd.push_back(i < q.spotsAOI->dists.size() ? q.spotsAOI->dists[i] : 0u);
            }
            spot_off[1] = (uint32_t)sx.size();
            spot_nd = (uint32_t)std::min(q.spotsAOI->dists.size(), q.spotsAOI->spots.size());
        }
        if (q.boxAOI) {
            kind |= CHD_AOI_BOX;
            box[0] = q.boxAOI->center.X; box[1] = q.boxAOI->center.Z; box[2] = q.boxAOI->extent.X; box[3] = q.boxAOI->extent.Z;
        }
        if (q.sphereAOI) {
            kind |= CHD_AOI_SPHERE;
            sph[0] = q.sphereAOI->center.X; sph[1] = q.sphereAOI->center.Z; sph[2] = q.sphereAOI->radius;
        }
        if (q.coneAOI) {
            kind |= CHD_AOI_CONE;
            cone[0] = q.coneAOI->center.X; cone[1] = q.coneAOI->center.Z; cone[2] = q.coneAOI->direction.X;
            cone[3] = q.coneAOI->direction.Z; cone[4] = q.coneAOI->angle; cone[5] = q.coneAOI->radius;
        }
        b.kind = &kind;
        b.sph_cx = &sph[0]; b.sph_cz = &sph[1]; b.sph_r = &sph[2];
        b.box_cx = &box[0]; b.box_cz = &box[1]; b.box_ex = &box[2]; b.box_ez = &box[3];
        b.cone_cx = &cone[0]; b.cone_cz = &cone[1]; b.cone_dx = &cone[2]; b.cone_dz = &cone[3]; b.cone_angle = &cone[4]; b.cone_r = &cone[5];
        if (!sx.empty()) {
            b.spot_off = spot_off; b.spot_ndist = &spot_nd; b.spot_x = sx.data(); b.spot_z = sz.data(); b.spot_dist = sd.data();
        }
        std::vector<uint32_t> ids(1 << 16), dists(1 << 16);
        uint32_t status = 0, off[2] = {0, 0};
        check(chd_query_channel_ids(engine_, &b, &status, off, ids.data(), dists.data(), ids.size()));
        if (status != CHD_Q_OK) throw SpatialError("spatial query failed with status " + std::to_string(status));
        std::map<uint32_t, uint32_t> res;
        for (uint32_t i = 0; i < off[1]; i++) res[ids[i]] = dists[i];
        return res;
    }

    // GetRegions (spatial.go:319-356); Y bounds are the reference's MinY/MaxY constants (spatial.go:80-83)
    std::vector<SpatialRegion> GetRegions() const {
        const size_t n = (size_t)cfg_.grid_cols * cfg_.grid_rows;
        std::vector<double> a(n), b(n), c(n), d(n);
        std::vector<uint32_t> id(n), srv(n);
        if (chd_get_regions(&cfg_, a.data(), b.data(), c.data(), d.data(), id.data(), srv.data()) != CHD_OK)
            throw SpatialError("GetRegions failed");
        std::vector<SpatialRegion> out(n);
        for (size_t i = 0; i < n; i++)
            out[i] = SpatialRegion{{a[i], -3.40282347e+38 / 2, b[i]}, {c[i], 3.40282347e+38 / 2, d[i]}, id[i], srv[i]};
        return out;
    }

    // GetAdjacentChannels (spatial.go:358-381)
    std::vector<uint32_t> GetAdjacentChannels(uint32_t spatialChannelId) const {
        uint32_t out8[8];
        const uint32_t n = chd_get_adjacent_channels(&cfg_, spatialChannelId, out8);
        return std::vector<uint32_t>(out8, out8 + n);
    }

    // Tick (channel.go:358-387 for every spatial channel): see include/chd_gpu.h for the result getters.
    chd_tick_summary Tick(const chd_query_batch* batch, int64_t t_ns, uint32_t flags = CHD_TICK_ALL) {
        chd_tick_summary s{};
        check(chd_tick(engine_, batch, t_ns, flags, &s));
        return s;
    }

    // Pipelined host loop (include/chd_gpu.h): the inputs of tick k+1 go up while tick k runs, tick k+1 starts with
    // AdoptPrefetched() + BeginInterest(nullptr, ...) and Tick(nullptr, t, CHD_TICK_ALL | CHD_TICK_EARLY_RESULTS).
    void PrefetchEntities(const double* x, const double* z, uint32_t n) { check(chd_prefetch_entities(engine_, x, z, n)); }
    void PrefetchQueries(const chd_query_batch& batch) { check(chd_prefetch_queries(engine_, &batch)); }
    void PrefetchRings(const uint32_t* ring_off, uint32_t n_entries, const int64_t* arrival, const uint32_t* sender, const uint64_t* index,
                       const uint64_t* ch_msg_index) {
        check(chd_prefetch_rings(engine_, ring_off, n_entries, arrival, sender, index, ch_msg_index));
    }
    void AdoptPrefetched() { check(chd_adopt_prefetched(engine_)); }
    void BeginInterest(const chd_query_batch* batch, int64_t t_ns, bool with_fanout = true) {
        check(chd_begin_interest(engine_, batch, t_ns, with_fanout ? 1 : 0));
    }
    void FetchResults(const chd_result_buffers& buffers, chd_tick_summary* summary) { check(chd_fetch_results(engine_, &buffers, summary)); }

    // Non-blocking read-back: FetchResultsAsync(k) right after Tick(k), enqueue tick k+1, then FetchWait() = results of tick k.
    // `pinned_header` is CHD_FETCH_HEADER_BYTES of pinned host memory that stays valid until the matching FetchWait.
    void FetchResultsAsync(const chd_result_buffers& buffers, void* pinned_header) { check(chd_fetch_results_async(engine_, &buffers, pinned_header)); }
    chd_tick_summary FetchWait() {
        chd_tick_summary s{};
        check(chd_fetch_wait(engine_, &s));
        return s;
    }

    // Subscriber lifecycle (subscription.go:34-125): AddConnection = a fresh subscriber in a free slot; RemoveConnection =
    // UnsubscribeFromChannel on every spatial channel of the slot (what connection close does, channel.go:414-475).
    void AddConnections(const std::vector<uint32_t>& slot, const std::vector<uint32_t>& conn_id) {
        if (slot.size() != conn_id.size()) throw SpatialError("AddConnections: array sizes differ");
        check(chd_add_subscribers(engine_, slot.data(), conn_id.data(), (uint32_t)slot.size()));
    }
    void RemoveConnections(const std::vector<uint32_t>& slot) { check(chd_remove_subscribers(engine_, slot.data(), (uint32_t)slot.size())); }

    // ChannelData.OnUpdate's buffer kept on the device (data.go:149-173): append a tick's updates (CSR by cell, arrival order).
    void InitUpdateBuffers(uint32_t capacity_per_cell) { check(chd_rings_init(engine_, capacity_per_cell)); }
    void OnUpdates(const std::vector<uint32_t>& upd_off, const std::vector<int64_t>& arrival_ns, const std::vector<uint32_t>& sender_conn_id) {
        if (arrival_ns.size() != sender_conn_id.size()) throw SpatialError("OnUpdates: array sizes differ");
        check(chd_rings_append(engine_, upd_off.data(), (uint32_t)arrival_ns.size(), arrival_ns.data(), sender_conn_id.data()));
    }
    // Channel.startTime of every spatial channel (channel.go:178): ChannelTime = t - start.
    void SetChannelStartTimes(const std::vector<int64_t>& start_ns) {
        if (start_ns.size() != (size_t)cfg_.grid_cols * cfg_.grid_rows) throw SpatialError("SetChannelStartTimes: one entry per cell");
        check(chd_set_channel_start_times(engine_, start_ns.data()));
    }

    // N GPUs, one process per GPU: X-slab of this rank + ONE all-gather of border records per tick inside TickSharded.
    static std::vector<uint8_t> CommUniqueId() {
        std::vector<uint8_t> id(128);
        if (chd_comm_unique_id(id.data()) != CHD_OK) throw SpatialError(chd_last_error(nullptr));
        return id;
    }
    void CommInit(const std::vector<uint8_t>& unique_id, int rank, int world, uint32_t halo_cols, uint32_t border_capacity,
                  uint32_t migrate_subscribers = 0, uint32_t migrate_pairs = 0) {
        if (unique_id.size() != 128) throw SpatialError("CommInit: the id is 128 bytes");
        check(chd_comm_init(engine_, unique_id.data(), rank, world, halo_cols, border_capacity, migrate_subscribers, migrate_pairs));
    }
    chd_tick_summary TickSharded(const chd_query_batch* batch, int64_t t_ns, uint32_t flags = CHD_TICK_ALL) {
        chd_tick_summary s{};
        check(chd_tick_sharded(engine_, batch, t_ns, flags, &s));
        return s;
    }
    void MigrateOut(const std::vector<uint32_t>& slot) { check(chd_migrate_out(engine_, slot.data(), (uint32_t)slot.size())); }
    void MigrateIn(uint32_t src_rank, uint32_t first_index, const std::vector<uint32_t>& slot, const std::vector<uint32_t>& conn_id) {
        if (slot.size() != conn_id.size()) throw SpatialError("MigrateIn: array sizes differ");
        check(chd_migrate_in(engine_, src_rank, first_index, slot.data(), conn_id.data(), (uint32_t)slot.size()));
    }
    // own entities whose column now belongs to another rank: (global id, new owner)
    std::vector<std::pair<uint32_t, uint32_t>> GetRehome(uint32_t cap) {
        std::vector<uint32_t> id(cap ? cap : 1), dst(cap ? cap : 1);
        uint32_t n = 0;
        check(chd_get_rehome(engine_, id.data(), dst.data(), cap, &n));
        std::vector<std::pair<uint32_t, uint32_t>> r;
        for (uint32_t i = 0; i < n && i < cap; i++) r.emplace_back(id[i], dst[i]);
        return r;
    }

    // Recipients of BroadcastType_ADJACENT_CHANNELS messages (message.go:188-239), batched: CSR of subscriber slots.
    struct BroadcastSets {
        std::vector<uint32_t> status, off, slot;
    };
    BroadcastSets AdjacentBroadcast(const std::vector<uint32_t>& channel_id, const std::vector<uint32_t>& broadcast,
                                    const std::vector<uint32_t>& sender_conn_id, const std::vector<uint32_t>& client_conn_id, uint64_t cap) {
        const uint32_t n = (uint32_t)channel_id.size();
        if (broadcast.size() != n || (!sender_conn_id.empty() && sender_conn_id.size() != n) ||
            (!client_conn_id.empty() && client_conn_id.size() != n))
            throw SpatialError("AdjacentBroadcast: array sizes differ");
        chd_broadcast_batch b{n, channel_id.data(), broadcast.data(), sender_conn_id.empty() ? nullptr : sender_conn_id.data(),
                              client_conn_id.empty() ? nullptr : client_conn_id.data()};
        BroadcastSets r;
        r.status.resize(n);
        r.off.resize((size_t)n + 1);
        r.slot.resize(cap);
        check(chd_adjacent_broadcast(engine_, &b, r.status.data(), r.off.data(), r.slot.data(), cap));
        r.slot.resize(r.off[n]);
        return r;
    }

    // Window classes of the last fan-out pass (data.go:248-252: which decisions share one merged payload).
    struct DueClasses {
        std::vector<uint32_t> class_of, rep, count;
    };
    DueClasses GetDueClasses(uint32_t n_due) {
        DueClasses r;
        r.class_of.resize(n_due);
        r.rep.resize(n_due ? n_due : 1);
        r.count.resize(n_due ? n_due : 1);
        uint32_t n = 0;
        check(chd_due_classes(engine_, r.class_of.data(), r.rep.data(), r.count.data(), (uint32_t)r.rep.size(), &n));
        r.rep.resize(n);
        r.count.resize(n);
        return r;
    }

    // Per-subscriber visibility deltas (chd_visible_delta): the entities that entered / left each slot's view since the last
    // call, CSR by slot.  The host spawns + subscribes the entity channels of `enter` and despawns + unsubscribes those of
    // `leave` (spatial.go:797-857).
    struct VisibleDelta {
        std::vector<uint64_t> enter_off, leave_off;
        std::vector<uint32_t> enter, leave;
    };
    void EnableVisibleDelta(uint64_t cap_entries) { check(chd_visible_delta_enable(engine_, cap_entries)); }
    void VisibleDeltaAsync() { check(chd_visible_delta(engine_)); }
    VisibleDelta GetVisibleDelta() {
        void* p = nullptr;
        uint64_t n_off = 0, ne = 0, nl = 0;
        check(chd_device_view(engine_, CHD_VIEW_ENTER_OFF, &p, &n_off));
        VisibleDelta r;
        r.enter_off.resize(n_off);
        r.leave_off.resize(n_off);
        check(chd_get_visible_delta(engine_, r.enter_off.data(), nullptr, 0, r.leave_off.data(), nullptr, 0, &ne, &nl));
        r.enter.resize(ne);
        r.leave.resize(nl);
        check(chd_get_visible_delta(engine_, nullptr, r.enter.data(), ne, nullptr, r.leave.data(), nl, nullptr, nullptr));
        return r;
    }

    chd_engine* engine() { return engine_; }

   private:
    void check(chd_status st) const {
        if (st != CHD_OK) throw SpatialError(chd_last_error(engine_));
    }
    chd_grid_cfg cfg_{};
    chd_engine* engine_ = nullptr;
};

}  // namespace channeld
