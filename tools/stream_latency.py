#!/usr/bin/env python
"""Streaming session against the single-frame and batch entry points, in one process, the two paths alternating.

Per frame (cfg1 / cfg2 / cfg3; kernel 4, kernel 4 with the channel split, kernel 2): bflk_stream_push of one block
[C][256] + bflk_stream_power_maps(1), against bflk_power_map of a pinned window [C][1024].  Both read pinned host memory
and write a pinned map; every call is synchronous, so a host clock around it measures it.
Catch-up (cfg3): the 592 frames of a bench.py step pushed block by block into a session of 592 frames, then ONE maps call,
against bflk_power_map_batch over the same pinned stream.

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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"
    return q


def pinned(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


def check(L, h, rc):
    if rc != 0:
        raise bflk.BflkError(rc, L.bflk_last_error(h).decode())


def us(t):
    t = np.asarray(t) * 1e6
    return f"p50 {np.median(t):7.1f} us  p95 {np.percentile(t, 95):7.1f} us"


def per_frame(name, kernel, split, n, warm, out):
    c = cases.CONFIGS[name]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
    w.set_kernel(kernel)
    w.set_channel_split(split)
    L, h = w._L, w._h
    Cn, D = w.n_channels, c["rows"] * c["cols"]
    K = 16                                                   # distinct blocks / windows, reused cyclically
    stream = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), K * N + W)
    blocks = pinned(np.stack([stream[:, k * N:(k + 1) * N] for k in range(K)]))
    windows = pinned(np.stack([stream[:, k * N:k * N + W] for k in range(K)]))
    p_sess, p_win = pinned(np.zeros(D, np.float32)), pinned(np.zeros(D, np.float32))
    first, got = C.c_int64(), C.c_int32()
    w.stream_open(4)
    w.stream_push(np.ascontiguousarray(stream[:, :H + 1]))   # from here on each block completes one frame
    t_push, t_maps, t_sess, t_win = [], [], [], []
    for i in range(warm + n):
        k = i % K
        t0 = time.perf_counter()
        check(L, h, L.bflk_stream_push(h, C.c_void_p(blocks[k].data_ptr()), N))
        t1 = time.perf_counter()
        check(L, h, L.bflk_stream_power_maps(h, 1, C.c_void_p(p_sess.data_ptr()), C.byref(first), C.byref(got)))
        t2 = time.perf_counter()
        assert got.value == 1
        check(L, h, L.bflk_power_map(h, C.c_void_p(windows[k].data_ptr()), C.c_void_p(p_win.data_ptr())))
        t3 = time.perf_counter()
        if i >= warm:
            t_push.append(t1 - t0)
            t_maps.append(t2 - t1)
            t_sess.append(t2 - t0)
            t_win.append(t3 - t2)
    label = f"{name} kernel {kernel}{' + channel split' if split else ''}"
    lines = [f"{label:28s} session push+maps(1): {us(t_sess)}   bflk_power_map (pinned window): {us(t_win)}",
             f"{'':28s}   of which push: {us(t_push)}   maps(1): {us(t_maps)}"]
    for line in lines:
        print(line, flush=True)
        out.append(line)
    w.close()


def catch_up(reps, out):
    c = cases.CONFIGS["cfg3"]
    B = 592
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
    L, h = w._L, w._h
    D = c["rows"] * c["cols"]
    T = (B - 1) * N + W
    stream = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), T)
    p_stream = pinned(stream)
    first_push = pinned(stream[:, :H + 1])
    blocks = pinned(np.stack([stream[:, H + 1 + k * N:H + 1 + (k + 1) * N] for k in range(B)]))
    p_sess, p_batch = pinned(np.zeros((B, D), np.float32)), pinned(np.zeros((B, D), np.float32))
    first, got = C.c_int64(), C.c_int32()
    t_push, t_maps, t_batch = [], [], []
    for r in range(reps + 1):                                # rep 0 warms up both shapes
        w.stream_open(B)
        t0 = time.perf_counter()
        check(L, h, L.bflk_stream_push(h, C.c_void_p(first_push.data_ptr()), H + 1))
        for k in range(B):
            check(L, h, L.bflk_stream_push(h, C.c_void_p(blocks[k].data_ptr()), N))
        t1 = time.perf_counter()
        check(L, h, L.bflk_stream_power_maps(h, B, C.c_void_p(p_sess.data_ptr()), C.byref(first), C.byref(got)))
        t2 = time.perf_counter()
        assert (first.value, got.value) == (0, B)
        check(L, h, L.bflk_power_map_batch(h, C.c_void_p(p_stream.data_ptr()), T, B, C.c_void_p(p_batch.data_ptr())))
        t3 = time.perf_counter()
        if r:
            t_push.append(t1 - t0)
            t_maps.append(t2 - t1)
            t_batch.append(t3 - t2)
    same = torch.equal(p_sess, p_batch)
    lines = [f"cfg3 catch-up, {B} frames ({reps} repetitions, medians):",
             f"  session: {B} pushes of [512][256] {np.median(t_push) * 1e3:7.2f} ms, then ONE maps({B}) call "
             f"{np.median(t_maps) * 1e3:7.2f} ms = {B / np.median(t_maps):9.0f} maps/s",
             f"  bflk_power_map_batch over the same pinned stream: {np.median(t_batch) * 1e3:7.2f} ms = {B / np.median(t_batch):9.0f} maps/s",
             f"  maps bit-identical: {same}"]
    for line in lines:
        print(line, flush=True)
        out.append(line)
    w.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_stream_latency.txt"))
    ap.add_argument("--frames", type=int, default=1000, help="timed frames per configuration")
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5, help="timed catch-up repetitions")
    args = ap.parse_args()
    out = [f"card: {card()}",
           f"streaming session vs single-frame / batch entry points; {args.frames} timed frames per row after {args.warmup} "
           "warm-up frames, the two paths alternating frame by frame; host clock around synchronous calls"]
    print("\n".join(out), flush=True)
    for name in ("cfg1", "cfg2", "cfg3"):
        for kernel, split in ((4, False), (4, True), (2, False)):
            per_frame(name, kernel, split, args.frames, args.warmup, out)
    catch_up(args.reps, out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
