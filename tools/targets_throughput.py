#!/usr/bin/env python
"""What the Targets of many maps cost: one bflk_targets_batch_dev launch against one synchronous bflk_targets call per
host map, and bflk_session_targets against bflk_stream_power_maps followed by one bflk_targets per frame.

Device batches: cfg3 (32 x 32 grid) with 592 maps, bench.py's step; cfg5 (256 x 256 grid) with 31 maps and max_targets 8
and 256.  The maps are real power maps of synthetic sources, computed once; they stay in the device buffer the maps call
wrote, 2.4 MB (cfg3) or 8.1 MB (cfg5), within the 126 MB of L2, as the maps of the step just before are when a caller takes
their Targets.  The device call is timed with CUDA events on the caller's stream around CALLS calls back to back (a window
of milliseconds, not one launch of a few microseconds); the per-map host calls (which copy one map up and the records back
each) with a host clock.
Session backlog: a cfg3 session holding 592 ready frames, taken by one call; pushing the samples is not timed.  Every leg
also checks that both paths give the same records.

Writes the report (with the card's name and power limit, read in the same run) to --out."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "beamforming-lk_b200"), os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402
import bflk  # noqa: E402
from bflk import synth  # noqa: E402
import cases  # noqa: E402

B3 = 592
CALLS = 100   # device calls per timed window


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"
    return q


def worker(name):
    c = cases.CONFIGS[name]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"], frame_len=c["N"], history=c["H"],
                        window_len=c["W"])
    return w, c


def stream(c, B):
    T = (B - 1) * c["N"] + c["W"]
    s = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), T)
    s *= np.linspace(0.5, 1.5, T, dtype=np.float32)[None, :]
    return np.ascontiguousarray(s), T


def host_targets(w, maps, max_targets, min_rel):
    """one bflk_targets per host map: (records per map as bytes, seconds)"""
    L, h = w._L, w._h
    out = (bflk.Target * max_targets)()
    n = C.c_int32()
    got = []
    t0 = time.perf_counter()
    for m in maps:
        rc = L.bflk_targets(h, C.c_void_p(m.ctypes.data), max_targets, min_rel, out, C.byref(n))
        if rc:
            raise bflk.BflkError(rc, L.bflk_last_error(h).decode())
        got.append(bytes(out)[:n.value * 40])
    return got, time.perf_counter() - t0


def device_batch(name, B, max_targets, min_rel, reps, lines):
    w, c = worker(name)
    s, T = stream(c, B)
    D = c["rows"] * c["cols"]
    x = torch.from_numpy(s).cuda()
    p = torch.empty((B, D), dtype=torch.float32, device="cuda")
    w.power_map_batch_dev(x.data_ptr(), T, B, p.data_ptr())
    torch.cuda.synchronize()
    del x
    maps = [np.ascontiguousarray(m) for m in p.cpu().numpy()]
    raw = torch.empty((B, max_targets * 40), dtype=torch.uint8, device="cuda")
    cnt = torch.empty(B, dtype=torch.int32, device="cuda")
    st = torch.cuda.Stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dev_ms, host_ms = [], []
    for i in range(reps + 1):
        e0.record(st)
        for _ in range(CALLS):
            w.targets_batch_dev(p.data_ptr(), B, raw.data_ptr(), cnt.data_ptr(), max_targets, min_rel, st.cuda_stream)
        e1.record(st)
        e1.synchronize()
        got, sec = host_targets(w, maps, max_targets, min_rel)
        if i:                                   # the first round warms both paths up
            dev_ms.append(e0.elapsed_time(e1) / CALLS)
            host_ms.append(sec * 1e3)
    n = cnt.cpu().numpy()
    r = raw.cpu().numpy()
    assert all(r[b, :n[b] * 40].tobytes() == got[b] for b in range(B)), "device and host records differ"
    d, hst = np.median(dev_ms), np.median(host_ms)
    lines.append(f"{name} ({c['rows']} x {c['cols']}) {B} maps, max_targets {max_targets}, min_rel {min_rel} "
                 f"({int(n.sum())} targets, {int(n.min())}..{int(n.max())} per map; {reps} rounds, medians):")
    lines.append(f"  bflk_targets_batch_dev, one launch (CUDA events, {CALLS} calls a window) {d:9.3f} ms  = {d * 1e3 / B:8.2f} us per map")
    lines.append(f"  {B} x bflk_targets on host maps (host clock)                  {hst:9.3f} ms  = {hst * 1e3 / B:8.2f} us per map")
    lines.append(f"  ratio {hst / d:.1f} x")
    w.close()


def session_backlog(reps, max_targets, min_rel, lines):
    w, c = worker("cfg3")
    L, h = w._L, w._h
    s, _ = stream(c, B3)
    D = c["rows"] * c["cols"]
    power = np.zeros((B3, D), np.float32)
    recs = (bflk.Target * (B3 * max_targets))()
    counts = np.zeros(B3, np.int32)
    first, got = C.c_int64(), C.c_int32()

    tn = (B3 - 1) * c["N"] + c["N"] + c["H"] + 1         # what the last frame reads: the ring of B3 frames holds it

    def fill():
        w.stream_open(B3)
        w.stream_push(s[:, :tn // 2])
        w.stream_push(s[:, tn // 2:tn])
        assert w.stream_status()[2] == B3

    times = {True: [], False: []}
    for i in range(reps + 1):
        for with_targets in (True, False):
            fill()
            t0 = time.perf_counter()
            if with_targets:
                rc = L.bflk_session_targets(h, B3, max_targets, min_rel, power.ctypes.data, recs, counts.ctypes.data,
                                            C.byref(first), C.byref(got))
                if rc:
                    raise bflk.BflkError(rc, L.bflk_last_error(h).decode())
                assert got.value == B3
            else:
                rc = L.bflk_stream_power_maps(h, B3, power.ctypes.data, C.byref(first), C.byref(got))
                if rc:
                    raise bflk.BflkError(rc, L.bflk_last_error(h).decode())
                host, _ = host_targets(w, power, max_targets, min_rel)
            if i:
                times[with_targets].append((time.perf_counter() - t0) * 1e3)
    sess = bytes(recs)
    assert all(sess[b * max_targets * 40:(b * max_targets + counts[b]) * 40] == host[b] for b in range(B3)), "records differ"
    a, b = np.median(times[True]), np.median(times[False])
    lines.append(f"cfg3 session backlog of {B3} ready frames, max_targets {max_targets}, min_rel {min_rel} "
                 f"({int(counts.sum())} targets; {reps} rounds, medians, host clock, pageable outputs):")
    lines.append(f"  bflk_session_targets({B3})                                  {a:9.3f} ms")
    lines.append(f"  bflk_stream_power_maps({B3}) + {B3} x bflk_targets            {b:9.3f} ms")
    lines.append(f"  ratio {b / a:.2f} x")
    w.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = [f"card (name, power limit, maximum SM clock): {card()}",
             "Targets of many maps in one launch against one bflk_targets call per map (tools/targets_throughput.py)"]
    device_batch("cfg3", B3, 8, 0.05, a.reps, lines)
    device_batch("cfg5", 31, 8, 0.05, a.reps, lines)
    device_batch("cfg5", 31, 256, 0.0, a.reps, lines)   # min_rel 0: every local maximum of the map competes for the slots
    session_backlog(a.reps, 8, 0.05, lines)
    print("\n".join(lines), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
