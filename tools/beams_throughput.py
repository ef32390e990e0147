#!/usr/bin/env python
"""What returning the beams costs: bflk_beams_batch_dev against bflk_power_map_batch_dev, and bflk_session_beams against
bflk_stream_power_maps, in one process, the two paths alternating.

Batch (cfg3, 592 frames = bench.py's step: 312 MB of input, larger than L2; kernels 4 and 2): ms per call from CUDA events
on the caller's stream, the delay-and-sum and pack kernels' own time from bflk_kernel_time_ms, and the bytes each call
writes (power [B][D], beams [B][D][N]).  Single frame (cfg3, kernel 4): one block pushed, then a one-frame maps or beams
call into pinned host buffers; the calls are synchronous, so a host clock around them measures them.

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

N, H, W = 256, 256, 1024
B = 592


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"
    return q


def cfg3_worker(kernel):
    c = cases.CONFIGS["cfg3"]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
    w.set_kernel(kernel)
    return w, c["rows"] * c["cols"]


def check(L, h, rc):
    if rc != 0:
        raise bflk.BflkError(rc, L.bflk_last_error(h).decode())


def batch(kernel, reps, warm, out):
    w, D = cfg3_worker(kernel)
    L, h = w._L, w._h
    T = (B - 1) * N + W
    x = torch.from_numpy(synth.make_stream(synth.tile_geometry(cases.origins(4, 2)), T)).cuda()
    power = torch.empty((B, D), dtype=torch.float32, device="cuda")
    beams = torch.empty((B, D, N), dtype=torch.float32, device="cuda")
    st = torch.cuda.Stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def call(with_beams):
        if with_beams:
            rc = L.bflk_beams_batch_dev(h, C.c_void_p(x.data_ptr()), T, B, C.c_void_p(beams.data_ptr()),
                                        C.c_void_p(power.data_ptr()), C.c_void_p(st.cuda_stream))
        else:
            rc = L.bflk_power_map_batch_dev(h, C.c_void_p(x.data_ptr()), T, B, C.c_void_p(power.data_ptr()),
                                            C.c_void_p(st.cuda_stream))
        check(L, h, rc)

    torch.cuda.synchronize()
    for _ in range(warm):
        call(False)
        call(True)
    torch.cuda.synchronize()
    w.enable_timing(True)
    w.kernel_time_ms()
    res = {False: [], True: []}
    for _ in range(reps):
        for with_beams in (False, True):
            e0.record(st)
            call(with_beams)
            e1.record(st)
            e1.synchronize()
            das, nd, pack, npk = w.kernel_time_ms()
            res[with_beams].append((e0.elapsed_time(e1), das / max(nd, 1), pack / max(npk, 1)))
    assert w.kernel_info()[0] == kernel
    lines = [f"cfg3 B = {B} kernel {kernel} ({reps} calls of each, alternating; medians):"]
    for with_beams in (False, True):
        a = np.asarray(res[with_beams])
        written = B * D * 4 + (B * D * N * 4 if with_beams else 0)
        name = "bflk_beams_batch_dev    " if with_beams else "bflk_power_map_batch_dev"
        lines.append(f"  {name} call {np.median(a[:, 0]):7.3f} ms (p95 {np.percentile(a[:, 0], 95):7.3f})  "
                     f"delay-and-sum kernel {np.median(a[:, 1]):7.3f} ms  pack {np.median(a[:, 2]):6.3f} ms  "
                     f"writes {written / 1e6:7.1f} MB  = {B / np.median(a[:, 0]) * 1e3:8.0f} maps/s")
    p, b = np.median(np.asarray(res[False]), 0), np.median(np.asarray(res[True]), 0)
    lines.append(f"  beams - power only: call {b[0] - p[0]:+.3f} ms ({(b[0] / p[0] - 1) * 100:+.1f} %), "
                 f"kernel {b[1] - p[1]:+.3f} ms ({(b[1] / p[1] - 1) * 100:+.1f} %)")
    for line in lines:
        print(line, flush=True)
        out.append(line)
    w.close()


def single_frame(n, warm, out):
    w, D = cfg3_worker(4)
    L, h = w._L, w._h
    K = 16
    stream = synth.make_stream(synth.tile_geometry(cases.origins(4, 2)), 2 * K * N + W)
    blocks = torch.from_numpy(np.stack([stream[:, k * N:(k + 1) * N] for k in range(2 * K)])).pin_memory()
    p_out = torch.zeros(D, dtype=torch.float32).pin_memory()
    b_out = torch.zeros((D, N), dtype=torch.float32).pin_memory()
    first, got = C.c_int64(), C.c_int32()
    w.stream_open(4)
    w.stream_push(np.ascontiguousarray(stream[:, :H + 1]))   # from here on each block completes one frame
    t = {False: [], True: []}
    for i in range(warm + n):
        for with_beams in (False, True):
            k = (2 * i + with_beams) % (2 * K)
            check(L, h, L.bflk_stream_push(h, C.c_void_p(blocks[k].data_ptr()), N))
            t0 = time.perf_counter()
            if with_beams:
                rc = L.bflk_session_beams(h, 1, C.c_void_p(b_out.data_ptr()), C.c_void_p(p_out.data_ptr()), C.byref(first),
                                          C.byref(got))
            else:
                rc = L.bflk_stream_power_maps(h, 1, C.c_void_p(p_out.data_ptr()), C.byref(first), C.byref(got))
            t1 = time.perf_counter()
            check(L, h, rc)
            assert got.value == 1
            if i >= warm:
                t[with_beams].append((t1 - t0) * 1e6)
    lines = [f"cfg3 single frame, kernel 4 ({n} frames of each after {warm} warm-up, alternating; host clock, pinned outputs):"]
    for with_beams in (False, True):
        a = np.asarray(t[with_beams])
        name = "bflk_session_beams(1)    " if with_beams else "bflk_stream_power_maps(1)"
        lines.append(f"  {name} p50 {np.median(a):7.1f} us  p95 {np.percentile(a, 95):7.1f} us  "
                     f"(returns {D * 4 + (D * N * 4 if with_beams else 0)} bytes)")
    for line in lines:
        print(line, flush=True)
        out.append(line)
    w.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_beams.txt"))
    ap.add_argument("--reps", type=int, default=40, help="timed batch calls of each kind per kernel")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=1000, help="timed single frames of each kind")
    args = ap.parse_args()
    out = [f"card: {card()}",
           "beams with the power map against the power map alone (bflk_beams_batch_dev / bflk_session_beams)"]
    print("\n".join(out), flush=True)
    for kernel in (4, 2):
        batch(kernel, args.reps, args.warmup, out)
    single_frame(args.frames, 100, out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
