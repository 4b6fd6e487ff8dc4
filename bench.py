#!/usr/bin/env python
"""bench.py — subscriber-AOI-queries/s of the spatial hot path (BASELINE.json metric) on N B200s.

A step = one batched tick over one synthetic snapshot: spatial-hash build of all entities (positions change
every step, so the hash is rebuilt and handover candidates detected) -> AOI query + interest diff for every
subscriber -> expanded visible-entity lists -> fan-out decisions over the update rings.

  value : whole-job queries/s, inputs already resident in HBM, device time (CUDA events), max over ranks
  e2e   : same tick through the C ABI with HOST (pinned) inputs: H2D of positions/queries/rings and D2H of the
          results a channeld host consumes, inside the timed region (wall clock, max over ranks)
  --impl reference : the CPU restatement of the reference's Go path (oracle/), all host cores, same config

N>1: X-slab sharding of the SAME world (strong scaling, BASELINE config #4), one NCCL all-gather of border
entity records per tick.  Launch: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "subscriber-AOI-queries/s"
TICK_NS = 33_333_333  # 30 Hz


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="benchmark", choices=["2x2", "benchmark", "10m", "handover"])
    ap.add_argument("--entities", type=int, default=0)
    ap.add_argument("--subscribers", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 30)")
    ap.add_argument("--expanded-steps", type=int, default=2, help="extra e2e steps that also copy the expanded list to the host")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gate", action="store_true")
    ap.add_argument("--trace-e2e", action="store_true", help="diagnostics: host-side phase times of the pipelined e2e step on stderr")
    ap.add_argument("--no-early", action="store_true", help="e2e ticks without CHD_TICK_EARLY_RESULTS")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: border exchange through the peer windows (stores over NVLink + flags) or one ncclAllGather per tick")
    ap.add_argument("--positions", default="f32", choices=["f32", "f64"],
                    help="e2e upload format of the (float32-valued) entity positions: the floats (chd_prefetch_entities_f32) or doubles")
    ap.add_argument("--updates-per-cell", type=int, default=8)
    ap.add_argument("--ring-len", type=int, default=64)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N>1: strong = the named config sharded over N GPUs (BASELINE config #4); weak = the world, the entities and "
                         "the subscribers grow N-fold in X (per-GPU work fixed)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (the results a caller of the tick receives) as DIR/<name>.npy, "
                         "float64, at most 60 MB in all: lists the library returns as sets in sorted row order, larger arrays as a fixed, seeded "
                         "sample of rows.  N>1: one set of files per rank (rank<r>_<name>.npy)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm only counts queries, it keeps no results")
    return args


def world_config(args):
    from channeld_b200 import synth

    wc = synth.CONFIGS[args.config]
    if args.entities or args.subscribers:
        wc = synth.scaled(wc, args.entities or wc.n_entities, args.subscribers or wc.n_subscribers)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.scaling == "weak" and world > 1:
        import copy

        wc = copy.copy(wc)
        wc.name += " x%d in X (weak scaling)" % world
        wc.cols *= world
        wc.n_entities *= world
        wc.n_subscribers *= world
    return wc


def config_dict(wc, world, scaling):
    """The workload description both arms print (identical dicts: the driver compares them)."""
    return {"workload": wc.name, "entities": wc.n_entities, "subscribers": wc.n_subscribers, "radius": wc.radius,
            "grid": "%dx%d" % (wc.cols, wc.rows), "parallelism": "xslab%d" % world if world > 1 else "single",
            "scaling": scaling if world > 1 else "strong",
            "tick": "build+query+interest-diff+emit-visible+fanout, positions change every step",
            "positions": "float32-valued (unrealpb.FVector widened by float64(), pkg/unrealpb/extension.go:10-24), computed on as float64",
            "l2": "inputs larger than L2 in effect: every step streams the expanded visible list (4 bytes x V, about 1.95 GB on the "
                  "1M/100K workload) through the 126 MB L2, evicting the step's inputs; no explicit flush"}


def oracle_grid(wc):
    from tests import _oracle

    return _oracle.make_grid(wc.offx, wc.offz, wc.w, wc.h, wc.cols, wc.rows, wc.server_cols, wc.server_rows)


def make_snapshots(wc):
    """Two position snapshots (A, B): B = A displaced by up to 60 units per axis (SURVEY §8d #3 velocity).  Entity positions are
    float32-VALUED doubles: in channeld they arrive as unrealpb.FVector floats and are widened by float64(*vec.X)
    (pkg/unrealpb/extension.go:10-24).  Both arms compute on the same doubles; the e2e leg of the GPU arm uploads the floats."""
    from channeld_b200 import synth

    def f32v(a):
        return a.astype(np.float32).astype(np.float64)

    ax, az = synth.entities(wc)
    ax, az = f32v(ax), f32v(az)
    bx, bz = synth.move_entities(wc, ax, az, 1, 60.0)
    bx, bz = f32v(bx), f32v(bz)
    snaps = []
    for x, z in ((ax, az), (bx, bz)):
        conn, cx, cz, r = synth.subscribers(wc, x, z)
        snaps.append(dict(x=x, z=z, cx=cx, cz=cz, r=r))
    return conn, snaps


# ----------------------------------------------------------------------------------------- reference arm

def run_reference(args):
    """The reference's CPU implementation of the path = oracle/ (C++ restatement of channeld's Go path; the Go
    toolchain is absent, see DESIGN.md).  Each step = one full tick of the same config: build of the per-cell
    entity lists + QueryChannelIds per subscriber (per-call hash map, per-sample GetChannelId) + materialising
    every subscriber's visible list, over all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tests import _oracle

    orc = _oracle.load()
    wc = world_config(args)
    conn, snaps = make_snapshots(wc)
    g = oracle_grid(wc)
    cores = os.cpu_count() or 1
    S = wc.n_subscribers
    # bounded sample: cap a step at ~1.5 s of CPU work by sub-sampling subscribers if a full tick is slower
    a = snaps[0]
    t0 = time.perf_counter()
    orc.baseline_run(g, a["x"], a["z"], a["cx"], a["cz"], a["r"], 0, min(S, 20000), cores, True)
    probe = time.perf_counter() - t0
    per_q = probe / min(S, 20000)
    q_per_step = S if per_q * S < 1.5 else max(1000, int(1.5 / per_q))
    for i in range(args.warmup):
        s = snaps[i % 2]
        orc.baseline_run(g, s["x"], s["z"], s["cx"], s["cz"], s["r"], 0, q_per_step, cores, True)
    t0 = time.perf_counter()
    for i in range(args.steps):
        s = snaps[i % 2]
        orc.baseline_run(g, s["x"], s["z"], s["cx"], s["cz"], s["r"], 0, q_per_step, cores, True)
    dt = time.perf_counter() - t0
    val = q_per_step * args.steps / dt
    # round 1's arm rebuilt the cell lists on ONE thread (Amdahl-bound): printed once for comparison
    t0 = time.perf_counter()
    for i in range(3):
        s = snaps[i % 2]
        orc.baseline_run(g, s["x"], s["z"], s["cx"], s["cz"], s["r"], 0, q_per_step, cores, 2)
    serial = {"value": q_per_step * 3 / (time.perf_counter() - t0), "note": "same run with the round-1 single-threaded build"}
    sample = "%d of %d subscribers per step (full build of %d entities every step), %d steps" % (q_per_step, S, wc.n_entities, args.steps)
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": args.scaling if int(os.environ.get("WORLD_SIZE", "1")) > 1 else "strong",
        "vs_baseline": None, "dtype": "f64+u32", "data": "synthetic",
        "config": config_dict(wc, int(os.environ.get("WORLD_SIZE", "1")), args.scaling),
        "cpu_baseline": {"value": val, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": sample + "; C++ restatement of channeld's Go path (no Go toolchain in the image), persistent thread "
                                            "pool, per-cell entity lists rebuilt in parallel every step",
                         "serial_build_variant": serial},
        "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit_line(_OUT_FD, json.dumps(out))


# ----------------------------------------------------------------------------------------- clocks

class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin, t_end):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            f = [v.strip() for v in line.split(",")]
            if len(f) < 9:
                continue
            try:
                mx = float(f[2])
                if t_begin - 0.05 <= ts <= t_end + 0.15:
                    sm.append(float(f[1]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------- our arm

def pinned(shape, dtype):
    import torch

    t = torch.empty(shape, dtype=dtype, pin_memory=True)
    return t, t.numpy()


DUMP_BYTES = 60_000_000  # --dump-outputs, all files of all ranks (under 64 MB with room to spare)


def _fair_caps(sizes, budget):
    """Per-array value caps within `budget`: equal shares, and what a smaller array leaves of its share goes to the larger ones."""
    caps, left = {}, budget
    for i, (k, n) in enumerate(sorted(sizes.items(), key=lambda kv: kv[1])):
        caps[k] = min(n, left // (len(sizes) - i))
        left -= caps[k]
    return caps


def _sample_rows(n, k):
    """The fixed, seeded sample of k of n rows, in row order: the same rows in every run with the same n."""
    return np.arange(n) if k >= n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def _sorted_rows(a):
    return a[np.lexsort(a.T[::-1])]


class _DeviceArray:
    """A device array of the library, for torch.as_tensor."""

    def __init__(self, address, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (address, False), "version": 2}


def dump_outputs(e, dirname, S, sm, dev, prefix, budget_bytes):
    """--dump-outputs: the results of the engine's last tick as float64 .npy files, for comparing two builds output for output.
    Everything chd_fetch_results returns, plus the expanded visible list (vis_entity) that stays in HBM.  All values are integers
    below 2^53, so float64 holds them exactly; a due record is its twelve 32-bit words (64-bit fields as low, high).  The interest
    diff, the due list and the handover list are sets (include/chd_gpu.h) and are written in sorted row order.  An array larger
    than its share of the budget is a fixed, seeded sample of its rows (_sample_rows)."""
    import torch

    from channeld_b200 import capi

    def u32(n):
        return np.zeros(int(n), np.uint32)

    P, D, H = int(sm.n_pairs), max(int(sm.n_sub_new), int(sm.n_unsub)), int(sm.n_handover)
    b = dict(pair_off=u32(S + 1), pair_channel=u32(P), pair_dist=u32(P), pair_interval_ms=u32(P), new_sub=u32(D), new_channel=u32(D),
             unsub_sub=u32(D), unsub_channel=u32(D), due=np.zeros(int(sm.n_due), capi.DUE_DTYPE), handover_entity=u32(H),
             handover_src=u32(H), handover_dst=u32(H), query_status=u32(S), vis_off=np.zeros(S + 1, np.uint64),
             cell_start=u32(e.n_cells + 1), sorted_entity=u32(sm.n_entities_in_world))
    rb = capi.ResultBuffers()
    for k, a in b.items():
        setattr(rb, k, capi.ptr(a))
    rb.pair_cap, rb.diff_cap, rb.due_cap, rb.handover_cap, rb.status_cap, rb.entity_cap = P, D, int(sm.n_due), H, S, int(sm.n_entities_in_world)
    got = capi.TickSummary()
    e._ck(e.L.chd_fetch_results(e.h, C.byref(rb), C.byref(got)))
    nn, nu = int(got.n_sub_new), int(got.n_unsub)
    out = {
        "summary": np.array(list(got.as_dict().values()), np.uint64),  # chd_tick_summary, in field order
        "query_status": b["query_status"],
        "pair_off": b["pair_off"],
        "pairs": np.stack([b["pair_channel"], b["pair_dist"], b["pair_interval_ms"]], 1),
        "sub_new": _sorted_rows(np.stack([b["new_sub"][:nn], b["new_channel"][:nn]], 1)),
        "unsub": _sorted_rows(np.stack([b["unsub_sub"][:nu], b["unsub_channel"][:nu]], 1)),
        "due": _sorted_rows(b["due"].view(np.uint32).reshape(-1, 12)),
        "handover": _sorted_rows(np.stack([b["handover_entity"], b["handover_src"], b["handover_dst"]], 1)),
        "vis_off": b["vis_off"],
        "cell_start": b["cell_start"],
        "sorted_entity": b["sorted_entity"],
    }
    V = int(got.n_visible)
    sizes = dict({k: a.size for k, a in out.items()}, vis_entity=V)
    caps = _fair_caps(sizes, budget_bytes // 8 - 16 * len(sizes))  # 128 bytes of .npy header per file
    out["vis_entity"] = u32(0)
    if V:
        vis = torch.as_tensor(_DeviceArray(e.device_view(capi.VIEW_VIS_ENTITY)[0], V, "<i4"), device=dev)
        rows = torch.from_numpy(_sample_rows(V, caps["vis_entity"])).to(dev)
        out["vis_entity"] = vis[rows].cpu().numpy().view(np.uint32)
    os.makedirs(dirname, exist_ok=True)
    for k, a in out.items():
        if a.size > caps[k]:
            a = a[_sample_rows(len(a), caps[k] // (a.size // len(a)))]
        np.save(os.path.join(dirname, prefix + k + ".npy"), a.astype(np.float64))
    sampled = ["%s %d of %d" % (k, caps[k], n) for k, n in sizes.items() if n > caps[k]]
    print("[bench] outputs of the last timed step in %s (sampled values: %s)" % (dirname, ", ".join(sampled) or "none"), file=sys.stderr)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from channeld_b200 import capi, engine, sharding, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # run the tick driver on the GPU's socket: pinned staging memory is then node-local by first touch (what `numactl
    # --cpunodebind` does for a production host); the CPU baseline leg gets the full mask back
    full_mask, numa = os.sched_getaffinity(0), None
    try:
        node = capi.lib().chd_device_numa_node(local)
        if node >= 0:
            cpus = set()
            for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
                a, _, b = part.partition("-")
                cpus |= set(range(int(a), int(b or a) + 1))
            cpus &= full_mask
            if cpus:
                os.sched_setaffinity(0, cpus)
                numa = {"gpu_numa_node": node, "driver_cpus": len(cpus)}
    except Exception as ex_:  # noqa: BLE001
        print("numa binding skipped: %r" % (ex_,), file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=dev)
    wc = world_config(args)
    conn_all, snaps = make_snapshots(wc)
    S_total, N_total = wc.n_subscribers, wc.n_entities

    # ---- shard (X-slabs by grid column; identity at world == 1)
    halo = sharding.halo_columns(wc.radius, wc.w)
    col_lo, col_hi = sharding.slab_columns(wc.cols, world, rank)
    ent_col = sharding.column_of(snaps[0]["x"], wc.offx, wc.w, wc.cols)
    sub_col = sharding.column_of(snaps[0]["cx"], wc.offx, wc.w, wc.cols)
    # out-of-world items (column -1) go to rank 0
    ent_mine = np.nonzero(((ent_col >= col_lo) & (ent_col < col_hi)) | ((ent_col < 0) & (rank == 0)))[0]
    sub_mine = np.nonzero(((sub_col >= col_lo) & (sub_col < col_hi)) | ((sub_col < 0) & (rank == 0)))[0]
    n_own, S = len(ent_mine), len(sub_mine)
    gid = ent_mine.astype(np.uint32)
    conn = conn_all[sub_mine]

    per_cell = N_total / wc.cells
    border_cap = int(min(N_total, (2 * halo * wc.rows * per_cell) * 1.5 + 65536)) if world > 1 else 1
    max_ent = n_own + (border_cap * world if world > 1 else 0) + 1024
    # visible-list capacity from the oracle-free estimate: pairs ~ S*E[K]; each pair ~ per_cell entries
    stream = torch.cuda.Stream(device=dev)
    e = engine.Engine(wc.cfg(), max_ent, max(S, 1), device=local,
                      max_visible=int(max(S, 1) * 1.3 * max(per_cell, 1.0) * (1.0 + 4.0 * (wc.radius / wc.w) ** 1) + (1 << 22)),
                      max_ring_entries=wc.cells * args.ring_len + 1024, max_due=int(max(S, 1) * 8 + 4096))
    e.set_stream(stream.cuda_stream)
    if world > 1:
        # the exchange lives behind the C ABI (chd_comm_init / chd_tick_sharded: NCCL inside libchd_b200.so); torch.distributed
        # only carries the 128-byte bootstrap id and the timing reductions
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(engine.Engine.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        e.comm_init(bytes(uid.cpu().numpy().tobytes()), rank, world, halo, border_cap)
        if args.exchange == "nccl":
            e.use_collective(True)
        info = e.comm_info()
        assert (info["col_lo"], info["col_hi"]) == (col_lo, col_hi), (info, col_lo, col_hi)
        e.set_entity_ids(gid)
    e.set_subscribers(conn if S else np.zeros(0, np.uint32))
    sub_idx = np.arange(S, dtype=np.uint32)

    # ---- inputs: device-resident (value) and pinned host (e2e) copies of both snapshots
    dev_in, host_in = [], []
    for sn in snaps:
        h = {}
        for k, src in (("x", sn["x"][ent_mine]), ("z", sn["z"][ent_mine]), ("cx", sn["cx"][sub_mine]), ("cz", sn["cz"][sub_mine]),
                       ("r", sn["r"][sub_mine])):
            t, a = pinned((len(src),), torch.float64)
            a[:] = src
            h[k] = t
        dev_in.append({k: v.to(dev) for k, v in h.items()})
        for k in ("x", "z"):  # the same positions as the floats they are at the source (e2e upload: 8 bytes per entity)
            t, a = pinned((len(h[k]),), torch.float32)
            a[:] = h[k].numpy()
            assert np.array_equal(a.astype(np.float64), h[k].numpy()), "bench positions must be float32-valued"
            h[k + "f"] = t
        host_in.append(h)
    t_sub, a_sub = pinned((S,), torch.int32)
    a_sub[:] = sub_idx.view(np.int32)
    d_sub = t_sub.to(dev)

    n_e2e = args.e2e_steps or min(args.steps, 30)
    n_prof = min(args.steps, 20)  # steps of the instrumented pass after the timed region
    n_steps_total = 1 + args.warmup + args.steps + n_prof + 5 * (2 + n_e2e) + 4 + args.expanded_steps + 2
    # one ring snapshot per step (arrival times follow the tick clock); bound the staging memory for huge grids
    ring_len, upc = args.ring_len, args.updates_per_cell
    while wc.cells * ring_len * 20 * n_steps_total > (768 << 20) and ring_len > 4:
        ring_len //= 2
        upc = max(1, upc // 2)
    ring_state = None
    rings_host, rings_dev = [], []
    for i in range(n_steps_total):
        ring_state, off, arr, snd, idx, cmi = synth.update_rings(wc, i, (i + 1) * TICK_NS, TICK_NS, upc, S_total,
                                                                 ring_len=ring_len, state=ring_state)
        hh = {}
        for k, a_, dt in (("off", off.view(np.int32), torch.int32), ("arr", arr, torch.int64), ("snd", snd.view(np.int32), torch.int32),
                          ("idx", idx.view(np.int64), torch.int64), ("cmi", cmi.view(np.int64), torch.int64)):
            t, a = pinned((len(a_),), dt)
            a[:] = a_
            hh[k] = t
        hh["n"] = int(off[-1])
        rings_host.append(hh)
        rings_dev.append({k: (v.to(dev) if k != "n" else v) for k, v in hh.items()})

    keep = []

    def batch_of(src):
        b, k = engine.make_batch(S, sub=d_sub if src is dev_in else t_sub, sphere=None)
        return b

    def make_batches(inputs, sub_t):
        out = []
        for d in inputs:
            # every subscriber queries every tick, query i <-> slot i: the identity batch (sub = NULL)
            b, k = engine.make_batch(S, sub=None, sphere=(d["cx"], d["cz"], d["r"]))
            keep.append(k)
            out.append(b)
        return out

    batches_dev = make_batches(dev_in, d_sub)
    batches_host = make_batches(host_in, t_sub)
    L = e.L

    def ck(st):
        if st != capi.OK:
            raise capi.ChdError(st, L.chd_last_error(e.h).decode())

    def step(i, inputs, batches, rings):
        """One tick, enqueue only (no host sync at world == 1)."""
        d = inputs[i % 2]
        rg = rings[i]
        t_ns = (i + 1) * TICK_NS
        ck(L.chd_set_rings(e.h, capi.ptr(rg["off"]), rg["n"], capi.ptr(rg["arr"]), capi.ptr(rg["snd"]), capi.ptr(rg["idx"]), capi.ptr(rg["cmi"])))
        if world > 1:
            # one library call: interest + fan-out start on the engine's second stream, border records are selected, ONE
            # ncclAllGather over NVLink, halo import, build + emit, join (chd_tick_sharded)
            ck(L.chd_set_entities(e.h, capi.ptr(d["x"]), capi.ptr(d["z"]), n_own))
            ck(L.chd_tick_sharded(e.h, C.byref(batches[i % 2]), t_ns, capi.TICK_ALL, None))
        else:
            ck(L.chd_set_entities(e.h, capi.ptr(d["x"]), capi.ptr(d["z"]), n_own))
            ck(L.chd_tick(e.h, C.byref(batches[i % 2]), t_ns, capi.TICK_ALL, None))

    def barrier():
        if world > 1:
            dist.barrier()

    with torch.cuda.stream(stream):
        # ---- correctness gate before timing (rank-local 1 % sample against the oracle; world == 1 only)
        gate = None
        step(0, dev_in, batches_dev, rings_dev)
        s0 = e.summary()
        if not args.no_gate:
            # every rank checks a 1 % sample of ITS subscribers against the oracle run over the FULL snapshot: (cell, dist) pairs
            # bit-identical, visible lists identical as sets of global entity ids (per subscriber; within a cell the order of
            # halo entities depends on the exchange, the canonical order is defined on one GPU only)
            from tests import _oracle

            orc = _oracle.load()
            m = max(1, S // 100) if S else 0
            sel = np.linspace(0, S - 1, m).astype(np.int64) if S else np.zeros(0, np.int64)
            a = snaps[0]
            gsel = sub_mine[sel]
            want = orc.sphere_tick(oracle_grid(wc), a["x"], a["z"], a["cx"][gsel], a["cz"][gsel], a["r"][gsel])
            pairs = e.get_pairs(s0.n_pairs)
            bad = 0
            for k, j in enumerate(sel):
                sl = slice(pairs["off"][j], pairs["off"][j + 1])
                ok = np.array_equal(pairs["channel"][sl], want["pair_cell"][want["pair_off"][k]:want["pair_off"][k + 1]])
                ok &= np.array_equal(pairs["dist"][sl], want["pair_dist"][want["pair_off"][k]:want["pair_off"][k + 1]])
                got_vis = e.get_visible_slot(int(j))
                want_vis = want["vis_entity"][want["vis_off"][k]:want["vis_off"][k + 1]]
                ok &= np.array_equal(got_vis, want_vis) if world == 1 else np.array_equal(np.sort(got_vis), np.sort(want_vis))
                bad += 0 if ok else 1
            counts = torch.tensor([float(m), float(bad)], dtype=torch.float64, device=dev)
            per_rank = [counts.clone() for _ in range(world)]
            if world > 1:
                dist.all_gather(per_rank, counts)
            per_rank = [[int(v[0]), int(v[1])] for v in per_rank]
            if sum(v[1] for v in per_rank):
                raise SystemExit("parity gate FAILED: GPU results differ from the oracle (checked, mismatches per rank: %r)" % per_rank)
            gate = {"checked_per_rank": [v[0] for v in per_rank], "mismatches": 0,
                    "what": "(cell,dist) pairs bit-identical and visible lists identical (exact order on 1 GPU, as sets of global ids "
                            "per subscriber on N GPUs) to the oracle run over the full snapshot"}

        # ---- value: device-resident inputs, device time
        barrier()  # (the gate's CPU work takes a different time on every rank: start the ticks together)
        for i in range(1, args.warmup + 1):
            step(i, dev_in, batches_dev, rings_dev)
        e.summary()
        # inside the timed region only the emit kernel is bracketed by CUDA events (the roofline's denominator): two event records per
        # step; the per-stage times and the timeline come from a separate instrumented pass right after it
        e.profile_enable(2)
        launches0 = e.launch_count()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
            time.sleep(0.25)
        barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tb = time.perf_counter()
        ev0.record(stream)
        for i in range(args.steps):
            step(args.warmup + 1 + i, dev_in, batches_dev, rings_dev)
        ev1.record(stream)
        t_enq = time.perf_counter()  # the host has ENQUEUED every step (no sync inside the loop)
        torch.cuda.synchronize()
        te = time.perf_counter()
        host_enqueue_ms = (t_enq - tb) * 1e3 / args.steps
        barrier()
        ms = ev0.elapsed_time(ev1)
        launches = e.launch_count() - launches0
        clocks = sampler.stop(tb, te) if rank == 0 else None
        sm = e.summary()  # raises on any capacity overflow during the timed steps
        ek_tot, ek_n = e.profile_get(capi.STAGE_EMIT_KERNEL)
        emit_kernel_ms_timed = ek_tot / max(ek_n, 1)
        if args.dump_outputs:  # before the passes below overwrite the last timed step's results
            dump_outputs(e, args.dump_outputs, S, sm, dev, "rank%d_" % rank if world > 1 else "", DUMP_BYTES // world)
        e.profile_enable(True)  # instrumented pass (not timed): every stage, same inputs
        for i in range(n_prof):
            step(args.warmup + 1 + args.steps + i, dev_in, batches_dev, rings_dev)
        sm = e.summary()  # (the last tick's counts: the calls below size their buffers from them)
        # window classes of the last tick's due list (outside the timed region): distinct payloads a host has to merge
        n_classes, classes_ms = None, None
        try:
            tc0 = time.perf_counter()
            _, cls_rep, _ = e.due_classes(int(sm.n_due))
            classes_ms = (time.perf_counter() - tc0) * 1e3
            n_classes = int(len(cls_rep))
        except Exception as ex_:  # noqa: BLE001
            print("due_classes failed: %r" % (ex_,), file=sys.stderr)
        # write-only stream of the same size as the visible list (torch fill): the DRAM-side ceiling of the emit kernel
        wp = None
        try:
            nfill = int(min(max(int(sm.n_visible), 1 << 26), 1 << 30))
            buf = torch.empty(nfill, dtype=torch.int32, device=dev)
            best = 1e9
            for _ in range(6):
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record(stream)
                buf.fill_(7)
                a1.record(stream)
                a1.synchronize()
                best = min(best, a0.elapsed_time(a1))
            wp = 4.0 * nfill / (best * 1e-3) / 1e9
            del buf
        except Exception:
            pass
        stage = {}
        for name, sid in (("build", capi.STAGE_BUILD), ("interest", capi.STAGE_INTEREST), ("emit", capi.STAGE_EMIT),
                          ("emit_kernel", capi.STAGE_EMIT_KERNEL), ("fanout", capi.STAGE_FANOUT)) + (
                (("export", capi.STAGE_EXPORT), ("exchange", capi.STAGE_EXCHANGE), ("import", capi.STAGE_IMPORT)) if world > 1 else ()):
            tot, n = e.profile_get(sid)
            stage[name] = tot / max(n, 1)
        stage["emit_kernel_instrumented_pass"] = stage["emit_kernel"]
        stage["emit_kernel"] = emit_kernel_ms_timed  # the timed region's own measurement
        timeline = {}
        for name, sid in (("tick", capi.STAGE_TICK), ("build", capi.STAGE_BUILD), ("interest", capi.STAGE_INTEREST), ("emit", capi.STAGE_EMIT),
                          ("emit_kernel", capi.STAGE_EMIT_KERNEL), ("fanout", capi.STAGE_FANOUT)):
            try:
                a, b = e.profile_timeline(sid)
                timeline[name] = [round(a, 4), round(b, 4)]
            except Exception:
                pass
        e.profile_enable(False)

        # ---- e2e: host inputs, H2D + tick + D2H of the host-facing results, wall clock
        P_cap = int(sm.n_pairs * 1.25) + 1024

        def make_result_set():
            """One set of pinned host result buffers (chd_result_buffers) + the tensors that keep them alive."""
            keep_ = dict(off=pinned((S + 1,), torch.int32)[0], ch=pinned((P_cap,), torch.int32)[0], dist=pinned((P_cap,), torch.int32)[0],
                         iv=pinned((P_cap,), torch.int32)[0], diff=[pinned((P_cap,), torch.int32)[0] for _ in range(4)],
                         due=pinned((2 * P_cap, 12), torch.int32)[0], ho=[pinned((max_ent,), torch.int32)[0] for _ in range(3)],
                         status=pinned((max(S, 1),), torch.int32)[0], voff=pinned((S + 1,), torch.int64)[0],
                         cs=pinned((wc.cells + 1,), torch.int32)[0], se=pinned((max_ent,), torch.int32)[0], hdr=pinned((64,), torch.int32)[0])
            r = capi.ResultBuffers()
            r.pair_off, r.pair_channel, r.pair_dist, r.pair_interval_ms, r.pair_cap = (capi.ptr(keep_["off"]), capi.ptr(keep_["ch"]), capi.ptr(keep_["dist"]),
                                                                                    capi.ptr(keep_["iv"]), P_cap)
            r.new_sub, r.new_channel, r.unsub_sub, r.unsub_channel, r.diff_cap = (*[capi.ptr(t) for t in keep_["diff"]], P_cap)
            r.due, r.due_cap = capi.ptr(keep_["due"]), 2 * P_cap
            r.handover_entity, r.handover_src, r.handover_dst, r.handover_cap = (*[capi.ptr(t) for t in keep_["ho"]], max_ent)
            r.query_status, r.status_cap = capi.ptr(keep_["status"]), S
            r.vis_off = capi.ptr(keep_["voff"])
            # the cell CSR makes the host result LOSSLESS: visible(s) = concatenation over the subscriber's pairs (ascending channel
            # id) of sorted_entity[cell_start[c] : cell_start[c + 1]] — the expanded list itself (1.95 GB) stays in HBM
            r.cell_start, r.sorted_entity, r.entity_cap = capi.ptr(keep_["cs"]), capi.ptr(keep_["se"]), max_ent
            return r, keep_

        rb, rb_keep = make_result_set()
        rb2, rb2_keep = make_result_set()
        summ = capi.TickSummary()
        r_vis_keep = []

        phase_acc = {}

        pos_f32 = [args.positions == "f32"]

        def prefetch_inputs(i):
            dn, rn = host_in[i % 2], rings_host[i]
            ck(L.chd_prefetch_rings(e.h, capi.ptr(rn["off"]), rn["n"], capi.ptr(rn["arr"]), capi.ptr(rn["snd"]), capi.ptr(rn["idx"]), capi.ptr(rn["cmi"])))
            ck(L.chd_prefetch_queries(e.h, C.byref(batches_host[i % 2])))
            if pos_f32[0]:
                ck(L.chd_prefetch_entities_f32(e.h, capi.ptr(dn["xf"]), capi.ptr(dn["zf"]), n_own))
            else:
                ck(L.chd_prefetch_entities(e.h, capi.ptr(dn["x"]), capi.ptr(dn["z"]), n_own))

        def e2e_step(i, expanded=False, pipelined=False, early=not args.no_early):
            """Host inputs -> H2D -> one batched tick -> D2H of everything a channeld host consumes (chd_fetch_results).
            pipelined: the positions of step i were uploaded with chd_prefetch_entities while step i-1 ran, and this step
            uploads those of step i+1 behind its own kernels (double-buffered staging: one 16 B/entity upload per step,
            inside the timed region, like the serial form)."""
            d = host_in[i % 2]
            rg = rings_host[i]
            t_ns = (i + 1) * TICK_NS
            tp0 = time.perf_counter()
            if pipelined:
                ck(L.chd_adopt_prefetched(e.h))  # rings + queries + positions of this step went up during the previous one
                if world == 1:
                    ck(L.chd_begin_interest(e.h, None, t_ns, 1))  # (chd_tick_sharded starts the adopted batch itself)
            else:
                ck(L.chd_set_rings(e.h, capi.ptr(rg["off"]), rg["n"], capi.ptr(rg["arr"]), capi.ptr(rg["snd"]), capi.ptr(rg["idx"]), capi.ptr(rg["cmi"])))
                # queries + rings go up first and the interest / fan-out stages start on the second stream while the
                # (much larger) position upload is still in flight
                ck(L.chd_begin_interest(e.h, C.byref(batches_host[i % 2]), t_ns, 1))
                if pos_f32[0]:
                    ck(L.chd_set_entities_f32(e.h, capi.ptr(d["xf"]), capi.ptr(d["zf"]), n_own))
                else:
                    ck(L.chd_set_entities(e.h, capi.ptr(d["x"]), capi.ptr(d["z"]), n_own))
            tick_flags = capi.TICK_ALL | (capi.TICK_EARLY_RESULTS if early else 0)
            if world > 1:
                ck(L.chd_tick_sharded(e.h, None, t_ns, tick_flags, None))
            else:
                ck(L.chd_tick(e.h, None, t_ns, tick_flags, None))
            tp1 = time.perf_counter()
            if pipelined:  # the next step's inputs go up while this tick's kernels run
                prefetch_inputs(i + 1)
            tp2 = time.perf_counter()
            if expanded:
                rb.vis_entity, rb.vis_cap = capi.ptr(r_vis_keep[0]), r_vis_keep[0].numel()
            else:
                rb.vis_entity, rb.vis_cap = None, 0
            ck(L.chd_fetch_results(e.h, C.byref(rb), C.byref(summ)))
            tp3 = time.perf_counter()
            for k_, v_ in (("launch", tp1 - tp0), ("prefetch", tp2 - tp1), ("fetch", tp3 - tp2)):
                phase_acc[k_] = phase_acc.get(k_, 0.0) + v_
            phase_acc["n"] = phase_acc.get("n", 0) + 1
            h2d = (8 if pos_f32[0] else 16) * n_own + 24 * S + (wc.cells + 1) * 4 + rg["n"] * 20 + wc.cells * 8
            d2h = (C.sizeof(capi.TickSummary) + (S + 1) * 4 + 12 * int(summ.n_pairs) + 8 * (int(summ.n_sub_new) + int(summ.n_unsub))
                   + 48 * int(summ.n_due) + 12 * int(summ.n_handover) + 4 * S + (S + 1) * 8 + (wc.cells + 1) * 4 + 4 * int(summ.n_entities_in_world)
                   + (4 * int(summ.n_visible) if expanded else 0))
            return h2d, d2h

        base = args.warmup + 1 + args.steps + n_prof
        for i in range(2):
            e2e_step(base + i)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(n_e2e):
            h2d, d2h = e2e_step(base + 2 + i)
        torch.cuda.synchronize()
        barrier()
        e2e_serial_dt = time.perf_counter() - t0
        # pipelined form: same work per step, the position upload of step i+1 overlaps the kernels of step i
        base += 2 + n_e2e
        prefetch_inputs(base)
        for i in range(2):
            e2e_step(base + i, pipelined=True)
        barrier()
        torch.cuda.synchronize()
        phase_acc.clear()
        if args.trace_e2e:
            e.profile_enable(False)  # also resets the CHD_TRACE_FETCH accumulators
        t0 = time.perf_counter()
        for i in range(n_e2e):
            h2d, d2h = e2e_step(base + 2 + i, pipelined=True)
        torch.cuda.synchronize()
        barrier()
        e2e_dt = time.perf_counter() - t0
        # asynchronous form: the host never waits for a tick before it has enqueued the next one (chd_fetch_results_async writes the
        # results into pinned memory with device-side sizes; chd_fetch_wait returns the PREVIOUS tick's results while the current
        # one runs).  Same bytes up and down per step, all inside the timed region.
        base += 2 + n_e2e
        sets = [(rb, rb_keep), (rb2, rb2_keep)]

        host_acc = {"tick": 0.0, "prefetch": 0.0, "fetch_async": 0.0, "fetch_wait": 0.0, "n": 0}

        def async_enqueue(i):
            t_ns = (i + 1) * TICK_NS
            h0 = time.perf_counter()
            ck(L.chd_adopt_prefetched(e.h))
            if world > 1:
                ck(L.chd_tick_sharded(e.h, None, t_ns, capi.TICK_ALL, None))
            else:
                ck(L.chd_begin_interest(e.h, None, t_ns, 1))
                ck(L.chd_tick(e.h, None, t_ns, capi.TICK_ALL, None))
            h1 = time.perf_counter()
            prefetch_inputs(i + 1)
            h2 = time.perf_counter()
            r_, k_ = sets[i % 2]
            ck(L.chd_fetch_results_async(e.h, C.byref(r_), capi.ptr(k_["hdr"])))
            h3 = time.perf_counter()
            host_acc["tick"] += h1 - h0
            host_acc["prefetch"] += h2 - h1
            host_acc["fetch_async"] += h3 - h2
            host_acc["n"] += 1

        def async_run(first, n):
            got = []
            async_enqueue(first)
            for i in range(first + 1, first + n):
                async_enqueue(i)
                h0 = time.perf_counter()
                ck(L.chd_fetch_wait(e.h, C.byref(summ)))  # results of step i - 1, while step i runs
                host_acc["fetch_wait"] += time.perf_counter() - h0
                got.append((int(summ.n_pairs), int(summ.n_due), int(summ.n_sub_new), int(summ.n_unsub), int(summ.n_handover), int(summ.n_entities_in_world)))
            ck(L.chd_fetch_wait(e.h, C.byref(summ)))
            got.append((int(summ.n_pairs), int(summ.n_due), int(summ.n_sub_new), int(summ.n_unsub), int(summ.n_handover), int(summ.n_entities_in_world)))
            return got

        prefetch_inputs(base)
        async_run(base, 2)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if args.trace_e2e:  # diagnostics: device-side stage times of the asynchronous loop itself (instrumented: not the reported run)
            e.profile_enable(True)
            async_run(base + 2, n_e2e)
            torch.cuda.synchronize()
            tr = {}
            for name, sid in (("tick", capi.STAGE_TICK), ("build", capi.STAGE_BUILD), ("interest", capi.STAGE_INTEREST), ("emit", capi.STAGE_EMIT),
                              ("emit_kernel", capi.STAGE_EMIT_KERNEL), ("fanout", capi.STAGE_FANOUT), ("readback_pcie_hop", capi.STAGE_READBACK)):
                tot, n_ = e.profile_get(sid)
                tr[name] = round(tot / max(n_, 1), 4)
            e.profile_enable(False)
            print("[bench] async e2e loop, device stage ms: %r" % (tr,), file=sys.stderr)
            base += n_e2e
            prefetch_inputs(base)
            async_run(base, 2)
            torch.cuda.synchronize()
        for k_ in host_acc:
            host_acc[k_] = 0
        got_async = async_run(base + 2, n_e2e)
        torch.cuda.synchronize()
        barrier()
        e2e_async_dt = time.perf_counter() - t0
        host_phases = {k_: round(v_ / max(host_acc["n"], 1) * 1e3, 4) for k_, v_ in host_acc.items() if k_ != "n"}
        e2e_async_f64_dt = None
        if pos_f32[0]:  # the same loop uploading the positions as doubles (16 bytes per entity), for comparison
            pos_f32[0] = False
            base2 = base + 2 + n_e2e
            prefetch_inputs(base2)
            async_run(base2, 2)
            barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got_async = async_run(base2 + 2, n_e2e)
            torch.cuda.synchronize()
            barrier()
            e2e_async_f64_dt = time.perf_counter() - t0
            pos_f32[0] = True
            base = base2
        npairs_, ndue_, nnew_, nun_, nho_, nin_ = got_async[-1]
        d2h_async = (256 + (S + 1) * 4 + 12 * npairs_ + 8 * (nnew_ + nun_) + 48 * ndue_ + 12 * nho_ + 4 * S + (S + 1) * 8 + (wc.cells + 1) * 4 + 4 * nin_)
        # the asynchronously fetched lists are the same lists: check the last step against a synchronous fetch of the same state
        rchk, rchk_keep = make_result_set()
        ck(L.chd_fetch_results(e.h, C.byref(rchk), C.byref(summ)))
        last_keep = sets[(base + 2 + n_e2e - 1) % 2][1]
        npr = int(summ.n_pairs)
        async_ok = (torch.equal(last_keep["off"], rchk_keep["off"]) and torch.equal(last_keep["ch"][:npr], rchk_keep["ch"][:npr])
                    and torch.equal(last_keep["voff"], rchk_keep["voff"]) and torch.equal(last_keep["cs"], rchk_keep["cs"])
                    and torch.equal(last_keep["se"][:int(summ.n_entities_in_world)], rchk_keep["se"][:int(summ.n_entities_in_world)])
                    and torch.equal(last_keep["due"][:int(summ.n_due)], rchk_keep["due"][:int(summ.n_due)]))
        if not async_ok:
            raise SystemExit("asynchronous read-back differs from the synchronous one")
        if args.trace_e2e and rank == 0:
            n_ = max(phase_acc.get("n", 1), 1)
            print("[bench] pipelined e2e step, host view (us): " + ", ".join("%s %.1f" % (k_, phase_acc[k_] / n_ * 1e6)
                                                                              for k_ in ("launch", "prefetch", "fetch")), file=sys.stderr)
        e2e_exp = None
        if args.expanded_steps > 0 and world == 1:
            r_vis_keep.append(pinned((int(sm.n_visible) + (1 << 20),), torch.int32)[0])
            e2e_step(base + 2 + n_e2e, True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(args.expanded_steps):
                _, d2h_x = e2e_step(base + 3 + n_e2e + i, True)
            torch.cuda.synchronize()
            dtx = time.perf_counter() - t0
            e2e_exp = {"value": S * args.expanded_steps / dtx, "unit": "queries/s", "d2h_bytes_per_step": int(d2h_x),
                       "note": "also copies the expanded visible list to pinned host memory"}

    # ---- reductions over ranks
    stage_all, host_enq_all = [dict(stage, visible=float(sm.n_visible))], [round(host_enqueue_ms, 4)]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, (stage_all[0], host_enq_all[0]))
        stage_all, host_enq_all = [g[0] for g in gathered], [g[1] for g in gathered]
    if world > 1:
        t = torch.tensor([ms, e2e_dt, e2e_serial_dt, e2e_async_dt, e2e_async_f64_dt or 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_dt, e2e_serial_dt, e2e_async_dt = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        e2e_async_f64_dt = float(t[4]) or None
        d2h = d2h_async
        c = torch.tensor([float(sm.n_pairs), float(sm.n_visible), float(sm.n_due), float(launches), float(h2d), float(d2h)],
                         dtype=torch.float64, device=dev)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        tot_pairs, tot_vis, tot_due, launches, h2d, d2h = [float(v) for v in c]
    else:
        tot_pairs, tot_vis, tot_due = float(sm.n_pairs), float(sm.n_visible), float(sm.n_due)

    if rank == 0:
        peaks, peak_src = None, "fallback"
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            peak, peak_src = float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            peak = 6650.0
            peak_src = "fallback 6.65 TB/s (B200_PROFILING.md)"
        ms_step = ms / args.steps
        value = S_total * args.steps / (ms * 1e-3)
        # Roofline of the dominant kernel (emit_visible), DRAM basis.  Algorithmic DRAM bytes per launch = 4 V (every visible
        # entry written once) + 4 N (the cell CSR payload read once; its re-reads are L2 hits by design: 16 MB of phase copies
        # against a 126 MB L2).  SURVEY §8d's 8 V counts the L2-side re-reads as well: reported as l2_side_gbs, not as the
        # fraction.  `traffic` = dram__bytes_read.sum + dram__bytes_write.sum of one launch from an `ncu --set full` pass over
        # this tree (profiles/r2_emit_traffic.json names the commit it was taken on), null if that file is absent.
        v_rank = float(sm.n_visible)
        n_sorted = float(sm.n_entities_in_world)
        ek_ms = stage["emit_kernel"]
        dram_bytes = 4.0 * v_rank + 4.0 * n_sorted
        achieved = (dram_bytes / (ek_ms * 1e-3)) / 1e9 if ek_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_emit_traffic.json")))
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling if world > 1 else "strong", "vs_baseline": None,
            "dtype": "f64+u32",
            "data": "synthetic",
            "config": config_dict(wc, world, args.scaling),
            "clocks": clocks,
            "e2e": {"value": S_total * n_e2e / e2e_async_dt, "unit": "queries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h if world > 1 else d2h_async),
                    "ms_per_step": e2e_async_dt / n_e2e * 1e3,
                    "host_ms_per_step": host_phases,
                    "pipeline": "double-buffered inputs AND results through the C ABI: chd_prefetch_{rings,queries,entities} upload the inputs of step "
                                "i+1 (pinned host memory) while the kernels of step i run; chd_fetch_results_async writes the results of step i "
                                "into pinned host buffers (device-side sizes) while step i+1 — already enqueued — runs; chd_fetch_wait hands the "
                                "host step i's results.  Every step uploads one full position snapshot + its queries + rings and reads back its "
                                "results inside the timed region; checked equal to a synchronous chd_fetch_results",
                    "positions": ("uploaded as the float32 values they are at the source (unrealpb.FVector), 8 bytes per entity, widened exactly "
                                  "on the device (chd_prefetch_entities_f32)") if args.positions == "f32" else "uploaded as float64, 16 bytes per entity",
                    "f64_upload": ({"value": S_total * n_e2e / e2e_async_f64_dt, "ms_per_step": e2e_async_f64_dt / n_e2e * 1e3,
                                    "h2d_bytes_per_step": int(h2d) + 8 * int(N_total if world > 1 else n_own),
                                    "note": "same loop with chd_prefetch_entities (16 bytes per entity on PCIe)"} if e2e_async_f64_dt else None),
                    "sync_fetch": {"value": S_total * n_e2e / e2e_dt, "ms_per_step": e2e_dt / n_e2e * 1e3,
                                   "note": "same pipeline with the blocking chd_fetch_results + CHD_TICK_EARLY_RESULTS (round-1 form): the host waits "
                                           "for step i before it enqueues step i+1"},
                    "serial": {"value": S_total * n_e2e / e2e_serial_dt, "ms_per_step": e2e_serial_dt / n_e2e * 1e3,
                               "note": "no overlap between steps: upload -> tick -> read-back, one after the other (per-tick latency)"},
                    "result": "chd_fetch_results: summary + (cell,dist,interval) pairs + sub/unsub lists + fan-out due list + handover "
                              "list + query statuses + visible offsets + the cell CSR (cell_start, sorted_entity): LOSSLESS — every "
                              "visible list is the concatenation of its pairs' cell lists; the 4-bytes-per-entry expansion itself stays in "
                              "HBM for GPU-side consumers (e2e_expanded copies it as well)"},
            "e2e_expanded": e2e_exp,
            "gpu_launches": int(launches),
            "collectives": {"exchange": {0: None, 1: "one ncclAllGather per tick", 2: "peer windows: stores over NVLink into CUDA-IPC-mapped receive buffers + 64-bit flags, no collective call on the tick path"}[e.exchange_mode()],
                            "nccl_all_gathers_issued_by_the_library_rank0": e.collective_count(), "where": "chd_tick_sharded (libchd_b200.so)"} if world > 1 else None,
            "roofline": {"bound": "hbm", "kernel": "emit_visible_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_dram_bytes_per_launch": dram_bytes, "algorithmic_dram_bytes": "4*V + 4*N (writes + one read of the CSR)",
                         "kernel_ms": ek_ms, "l2_side_gbs": (8.0 * v_rank / (ek_ms * 1e-3)) / 1e9 if ek_ms > 0 else None,
                         "write_only_peak_gbs_this_run": wp,
                         "frac_of_write_only_peak": (achieved / wp) if wp else None,
                         "note": "DRAM basis; the kernel is a write stream on the DRAM side, so the tighter ceiling is the write-only "
                                 "one measured in this run (torch fill_ of the same size, best of 6)"},
            "stage_ms": stage,
            "stage_ms_per_rank": stage_all,
            "host_enqueue_ms_per_step": host_enq_all,
            "last_tick_timeline_ms": timeline,
            "per_tick": {"pairs": tot_pairs, "visible": tot_vis, "fanout_decisions": tot_due, "handover": int(sm.n_handover),
                         "fanout_msgs_per_s": tot_due / (ms_step * 1e-3),
                         "window_classes_rank0": n_classes, "window_classes_call_ms": classes_ms},
            "parity_gate": gate,
        }
        out["host"] = numa
        os.sched_setaffinity(0, full_mask)  # the CPU legs use every host thread
        if world == 1 and not args.no_cpu_baseline:
            from tests import _oracle

            orc = _oracle.load()
            cores = os.cpu_count() or 1
            a = snaps[0]
            g = oracle_grid(wc)
            t0 = time.perf_counter()
            orc.baseline_run(g, a["x"], a["z"], a["cx"], a["cz"], a["r"], 0, min(S_total, 20000), cores, True)
            probe = (time.perf_counter() - t0) / min(S_total, 20000)
            qn = S_total if probe * S_total < 2.0 else max(1000, int(2.0 / probe))
            reps = max(1, min(20, int(10.0 / max(probe * qn, 1e-3))))
            t0 = time.perf_counter()
            for k in range(reps):
                s_ = snaps[k % 2]
                orc.baseline_run(g, s_["x"], s_["z"], s_["cx"], s_["cz"], s_["r"], 0, qn, cores, True)
            dtc = time.perf_counter() - t0
            # the same restatement on ONE host thread (SURVEY.md §8d asks for both)
            reps1, single = 3, None
            try:
                t0 = time.perf_counter()
                for k in range(reps1):
                    s_ = snaps[k % 2]
                    orc.baseline_run(g, s_["x"], s_["z"], s_["cx"], s_["cz"], s_["r"], 0, qn, 1, True)
                dt1 = time.perf_counter() - t0
                single = {"value": qn * reps1 / dt1, "cores": 1, "sample": "%d ticks x %d subscribers, build included" % (reps1, qn)}
            except Exception as ex_:  # noqa: BLE001  (never lose the result line over the extra baseline)
                print("single-thread baseline failed: %r" % (ex_,), file=sys.stderr)
            serial = None
            try:  # round 1's arm rebuilt the cell lists on ONE thread: printed for comparison
                t0 = time.perf_counter()
                for k in range(3):
                    s_ = snaps[k % 2]
                    orc.baseline_run(g, s_["x"], s_["z"], s_["cx"], s_["cz"], s_["r"], 0, qn, cores, 2)
                serial = {"value": qn * 3 / (time.perf_counter() - t0), "note": "same threads, round-1 single-threaded build"}
            except Exception as ex_:  # noqa: BLE001
                print("serial-build baseline failed: %r" % (ex_,), file=sys.stderr)
            out["cpu_baseline"] = {"value": qn * reps / dtc, "unit": "queries/s", "cores": cores, "kind": "port",
                                   "sample": "%d ticks x %d of %d subscribers (parallel build of %d entities included each tick); C++ "
                                             "restatement of channeld's Go path, persistent pool over all host threads" % (reps, qn, S_total, N_total),
                                   "single_thread": single, "serial_build_variant": serial}
        _emit_line(_OUT_FD, json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def _protect_stdout():
    """rank 0 must print exactly ONE JSON line: route everything libraries write to fd 1 (e.g. NCCL's version banner)
    to stderr and keep the real stdout for the result line."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit_line(saved_fd, text):
    os.write(saved_fd, (text + "\n").encode())


if __name__ == "__main__":
    a = parse()
    _OUT_FD = _protect_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
