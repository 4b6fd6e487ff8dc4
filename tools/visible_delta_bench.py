"""Cost of chd_visible_delta against the expanded visible list it replaces, on the bench's own inputs.

For config #2 ("benchmark", full size) and the "handover" config at bench.py's default size: the A/B position snapshots of
bench.py (B = A moved by up to 60 units, queries on the subscribers' pawns) are ping-ponged, every tick is BUILD | EMIT | FANOUT,
and after each tick chd_visible_delta runs on the engine stream (torch's stream via chd_set_stream).  Timed per call:
  delta_ms        CUDA events around chd_visible_delta alone
  emit_kernel_ms  the expanded-list kernel of the same ticks (CHD_STAGE_EMIT_KERNEL)
  get_delta_ms    host clock of a synchronous chd_get_visible_delta (offsets + both lists to pageable host memory)
  get_visible_ms  host clock of chd_get_visible (offsets + the whole expanded list), for comparison
Bytes are what the delta must move at least, computed from the counts: mover detection reads both key arrays (8 N), the movers
are compacted and sorted (about 40 bytes each), every enter/leave candidate is read, its other-state key gathered and each
kept entry written (count pass + write pass), and the baseline snapshot copies 8 N + 4 C + 4 S + 8 P bytes.
Prints one JSON line (also written to --out).  Run from the repository root on the GPU box.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBPS = 7.7  # HGX B200 data sheet, one GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def run(name, calls, warmup):
    import torch

    import bench
    from channeld_b200 import capi, engine, synth

    wc = synth.CONFIGS[name]
    N, S = wc.n_entities, wc.n_subscribers
    conn, snaps = bench.make_snapshots(wc)
    per_cell = N / wc.cells
    e = engine.Engine(wc.cfg(), N, S, max_visible=int(S * 1.15 * per_cell * (1.0 + 4.0 * wc.radius / wc.w) + (1 << 22)))
    stream = torch.cuda.current_stream()
    e.set_stream(stream.cuda_stream)
    e.set_subscribers(conn)
    batches = [engine.make_batch(S, sub=None, sphere=(s["cx"], s["cz"], s["r"])) for s in snaps]
    e.enable_visible_delta(e.lim.max_visible)  # a delta never exceeds two full views
    flags = capi.TICK_BUILD | capi.TICK_EMIT | capi.TICK_FANOUT
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def tick(k):
        s = snaps[k & 1]
        e.set_entities(s["x"], s["z"])
        e.tick(batches[k & 1][0], (k + 1) * 33_000_000, flags, want_summary=False)

    tick(0)  # first call: the whole view enters; not part of the steady state
    e.visible_delta()
    e.get_visible_delta()
    for k in range(1, warmup + 1):
        tick(k)
        e.visible_delta()
    torch.cuda.synchronize()
    e.profile_enable(2)
    delta_ms, n_enter, n_leave = [], [], []
    k0 = warmup + 1
    for k in range(k0, k0 + calls):
        tick(k)
        ev0.record(stream)
        e.visible_delta()
        ev1.record(stream)
        ev1.synchronize()
        delta_ms.append(ev0.elapsed_time(ev1))
        ne, nl = C.c_uint64(), C.c_uint64()
        e._ck(e.L.chd_get_visible_delta(e.h, None, None, 0, None, None, 0, C.byref(ne), C.byref(nl)))
        n_enter.append(ne.value)
        n_leave.append(nl.value)
    emit_total, emit_n = e.profile_get(capi.STAGE_EMIT_KERNEL)
    e.profile_enable(0)
    s = e.summary()
    t = time.perf_counter()
    e.get_visible_delta()
    get_delta_ms = (time.perf_counter() - t) * 1e3
    t = time.perf_counter()
    voff, vis = e.get_visible()
    get_visible_ms = (time.perf_counter() - t) * 1e3
    # movers between the two snapshots (what the delta sorts every call)
    ca, cb = e.cell_of(snaps[0]["x"], snaps[0]["z"]), e.cell_of(snaps[1]["x"], snaps[1]["z"])
    M = int((ca != cb).sum())
    e.close()
    ent = float(np.mean(n_enter)) + float(np.mean(n_leave))
    P, Cc = int(s.n_pairs), wc.cells
    # candidates: every enter/leave entry is a candidate; kept cells add their movers (bounded by entries + M per subscriber cell)
    bytes_min = 8 * N + 40 * M + 2 * (12 * ent) + (8 * N + 4 * Cc + 4 * S + 8 * P) * 2 + 2 * 2 * 8 * P
    d = float(np.median(delta_ms))
    return dict(config=name, entities=N, subscribers=S, pairs=P, visible_per_tick=int(s.n_visible), movers=M,
                enter_per_call=float(np.mean(n_enter)), leave_per_call=float(np.mean(n_leave)), calls=calls, warmup=warmup,
                delta_ms_median=d, delta_ms_mean=float(np.mean(delta_ms)), delta_ms_p90=float(np.percentile(delta_ms, 90)),
                emit_kernel_ms=emit_total / max(emit_n, 1), emit_samples=emit_n,
                delta_bytes_min=int(bytes_min), delta_share_of_hbm_bound=bytes_min / (HBM_TBPS * 1e12) / (d * 1e-3),
                get_delta_ms=get_delta_ms, get_delta_bytes=int(8 * 2 * (S + 1) + 4 * (n_enter[-1] + n_leave[-1])),
                get_visible_ms=get_visible_ms, get_visible_bytes=int(8 * (S + 1) + 4 * len(vis)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="benchmark,handover")
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(gpu=gpu_info(), hbm_bound_tbps=HBM_TBPS, runs=[run(n, a.calls, a.warmup) for n in a.configs.split(",")])
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
