#!/usr/bin/env python
"""What focusing the grid at the source's distance (bflk_set_focus) gains, and what it costs.

Geometries: 2 x 4 tiles (cfg3/4/5: 0.64 m x 0.32 m) and 8 tiles in a row (1.28 m), each with cfg3's 32 x 32 grid over
180 degrees, N = H = 256.  Source: one point source (synth.point_source_stream, noise sigma 1e-3) on the grid node nearest
theta 20 deg, phi 30 deg, at 3, 5, 10 and 20 m, at 3 kHz and 9 kHz, amplitude 1e-2.  For each case the report gives the
power at the source's cell of the far-field map and of the map focused at the source's distance, their ratio, the argmax
cell of each map, and the kernel and tile_span (bflk_get_kernel) each map ran on.

Rate: maps/s of a 592-frame cfg3 batch as bench.py measures it on one GPU -- a device-resident stream, consecutive steps in
continuous operation (bflk_power_map_batch_dev_submit / _join on a caller's stream, two output buffers), CUDA events around
STEPS steps after WARMUP warm-up steps -- for the far-field grid and the grid focused at 3 m and 20 m, in alternating rounds
in the same process; medians.  The focused maps of the timed steps are checked against the same call on a fresh handle.

Writes the report (with the card's name and power limit, read in the same run) to --out."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "beamforming-lk_b200"), os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402
import bflk  # noqa: E402
from bflk import synth  # noqa: E402
import cases  # noqa: E402

KERNELS = {1: "generic", 2: "tiled exact", 3: "lane-broadcast", 4: "tiled two-FMA"}
GEOMETRIES = {"2 x 4 tiles (cfg3)": (4, 2), "8 tiles in a row": (8, 1)}
B = 592
STEPS, WARMUP = 20, 5


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"


def worker(nx, ny, focus=0.0):
    c = cases.CONFIGS["cfg3"]
    w = bflk.MIMOWorker(cases.origins(nx, ny), c["rows"], c["cols"], c["fov"], frame_len=c["N"], history=c["H"],
                        window_len=c["W"])
    if focus:
        w.set_focus(focus)
    return w, c


def gain(lines):
    lines.append("Power at the source's cell, far-field grid against the grid focused at the source's distance")
    lines.append(f"{'geometry':<20} {'f kHz':>5} {'r m':>4} {'cell':>5} {'far':>10} {'focused':>10} {'far/foc':>8} "
                 f"{'argmax far':>10} {'argmax foc':>10}  kernel, tile_span far | focused")
    for gname, (nx, ny) in GEOMETRIES.items():
        xyz = synth.tile_geometry(cases.origins(nx, ny))
        far_w, c = worker(nx, ny)
        th, ph = far_w.grid()
        src = synth.nearest_direction(th, ph, np.deg2rad(20.0), np.deg2rad(30.0))
        for f in (3000.0, 9000.0):
            for r in (3.0, 5.0, 10.0, 20.0):
                window = synth.point_source_stream(xyz, c["W"], [(th[src], ph[src], r, f, 1e-2)])
                pf = far_w.update(window)
                kf = far_w.kernel_info()
                near_w, _ = worker(nx, ny, r)
                pn = near_w.update(window)
                kn = near_w.kernel_info()
                near_w.close()
                lines.append(f"{gname:<20} {f / 1e3:5.0f} {r:4.0f} {src:5d} {pf[src]:10.4e} {pn[src]:10.4e} "
                             f"{pf[src] / pn[src]:8.3f} {int(np.argmax(pf)):10d} {int(np.argmax(pn)):10d}  "
                             f"{KERNELS.get(kf[0], kf[0])}, {kf[1]} | {KERNELS.get(kn[0], kn[0])}, {kn[1]}")
        far_w.close()


def rate(reps, lines):
    c = cases.CONFIGS["cfg3"]
    T = (B - 1) * c["N"] + c["W"]
    x = torch.from_numpy(synth.make_stream(synth.tile_geometry(cases.origins(4, 2)), T)).cuda()
    D = c["rows"] * c["cols"]
    st = torch.cuda.Stream()
    cs = st.cuda_stream
    legs = {"far field": 0.0, "focused at 3 m": 3.0, "focused at 20 m": 20.0}
    handles = {k: worker(4, 2, r)[0] for k, r in legs.items()}
    outs = {k: [torch.empty((B, D), device="cuda") for _ in range(2)] for k in legs}
    times = {k: [] for k in legs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def steps(k, n):
        w = handles[k]
        for i in range(n):
            w.power_map_batch_dev_submit(x.data_ptr(), T, B, outs[k][i & 1].data_ptr(), cs)
        w.power_map_batch_dev_join(cs)

    for i in range(reps + 1):
        for k in legs:
            steps(k, WARMUP)
            e0.record(st)
            steps(k, STEPS)
            e1.record(st)
            e1.synchronize()
            if i:
                times[k].append(e0.elapsed_time(e1))
    lines.append(f"cfg3 batch of {B} frames, device-resident, continuous operation, {STEPS} steps a window after {WARMUP} "
                 f"warm-up steps, {reps} rounds alternating the legs, medians:")
    for k, r in legs.items():
        ms = float(np.median(times[k]))
        ki = handles[k].kernel_info()
        check, _ = worker(4, 2, r)
        ref = torch.empty((B, D), device="cuda")
        check.power_map_batch_dev(x.data_ptr(), T, B, ref.data_ptr(), cs)
        st.synchronize()
        same = torch.equal(ref, outs[k][(STEPS - 1) & 1])
        check.close()
        lines.append(f"  {k:<16} {B * STEPS / (ms / 1e3) / 1e3:9.2f} k maps/s  ({ms / STEPS:.3f} ms a step; kernel "
                     f"{KERNELS.get(ki[0], ki[0])}, tile_span {ki[1]}, window chunks {ki[2]}; maps equal a fresh handle's: {same})")
    for w in handles.values():
        w.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = [f"card (name, power limit, maximum SM clock): {card()}",
             "Near-field steering: gain and rate of a focused grid (tools/focus_gain.py)"]
    gain(lines)
    rate(a.reps, lines)
    print("\n".join(lines), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
