#!/usr/bin/env python
"""bench.py -- full-grid delay-and-sum power maps per second on B200 (BASELINE.json's metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg3] [--frames B] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of B synthetic frames (C channels x (B+3)*N samples, larger than
L2) for every direction of the grid.  N = 1 runs the configuration the target is quoted on (cfg3: 512 microphones x
32x32 = 1024 directions x 256-sample frames).  N > 1 (torchrun, one rank per GPU): every rank attaches its handle to a
multi-GPU job INSIDE the library (bflk_comm_init_rank; the NCCL id is the only thing exchanged through
torch.distributed) and a step is one bflk_power_map_batch_sharded_dev call -- the library shards the grid x the frames
(default 2 direction groups x N/2 frame groups; --dir-groups N = the pure grid sharding, also measured and reported as
`grid_shard`), all-gathers the slices with NCCL and leaves the complete [B][D] maps on every rank.  Total work is fixed
("strong" scaling).

The K timed steps run in CONTINUOUS OPERATION, as a live system would: at N = 1 consecutive steps alternate between the
handle's two compute streams (bflk_power_map_batch_dev_submit; the pack pre-pass of step i + 1 under the kernel of step i),
at N > 1 the all-gather + assembly of step i run on the communicator's stream under the kernels of step i + 1
(bflk_power_map_batch_sharded_dev_submit); the join that makes the last maps visible is inside the timed region, and every
step computes and delivers its own complete maps.  `synchronous_call_value`: the same with one synchronous call per step
(--no-overlap makes that the headline).  The dominant kernel's OWN launch duration (`roofline.achieved`, the shares of a
step) is timed in a pass of synchronous calls -- overlapping launches would stretch the event pairs around them.

One JSON line on rank 0.  `value`: maps/s with inputs resident in HBM (automatic kernel = two-FMA form);
`bit_identical`: the same with the kernel whose delayed sums equal the reference's delay() bit for bit.  `e2e`: through
the host-buffer C-ABI call (H2D of the batch + D2H of the maps inside the timed region).  `roofline`: the dominant
kernel against the FP32-FMA roofline (nominal, and against an in-job packed-FMA saturation run), `roofline_hbm` against
the measured copy bandwidth.  `sustained`: >= 2 s of back-to-back steps with clocks and board power.  `other_configs`:
cfg1 / cfg2 / cfg5 (and cfg4 MISO latency) in the same run.  `cpu_baseline`: the compiled reference delay() loop
(oracle/_ref) on the host.  --config cfg4 benchmarks the dynamic-steering (MISO) path on its own.

--dump-outputs DIR writes what the timed path delivered in its last timed step (power-map configurations: the [B][D]
maps as DIR/power_maps.npy; cfg4: DIR/audio.npy and DIR/power.npy) so that two builds can be compared output for output:
the input is synthesised from a fixed seed, so the same arguments give the same input on every run.  The benchmark
writes nothing into the source tree (it may be read-only); DIR is the caller's.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

sys.dont_write_bytecode = True      # no __pycache__ in the source tree
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "beamforming-lk_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

import cases  # noqa: E402

METRIC = "power_maps_per_sec"
UNIT = "maps/s"
FP32_LANES_PER_SM = 128
KERNEL_NAMES = {1: "das_generic", 2: "das_tile", 3: "das_bcast", 4: "das_tile_fma2"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300, help="timed steps (default: ~2.4 s at cfg3 on one B200)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg3", choices=list(cases.CONFIGS) + ["cfg4"])
    ap.add_argument("--frames", type=int, default=0, help="frames per step (default: sized so the input exceeds L2)")
    ap.add_argument("--kernel", type=int, default=0, help="0 auto, 1 generic, 2 register-tiled (bit-identical sums), 3 lane-broadcast, 4 register-tiled two-FMA form")
    ap.add_argument("--dir-groups", type=int, default=0,
                    help="N > 1: direction groups G_d (ranks = G_d x frame groups); 0 = 2 when N is even; N = pure grid sharding")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: synchronous bflk_power_map_batch_sharded_dev per step instead of _dev_submit / _join")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip bit_identical / sustained / other_configs / latency / grid_shard")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step delivered as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs is defined for --impl ours")
    return args


def default_frames(c):
    # input stream = C x (B + 3) x N floats, at least 256 MB (L2 is 126 MB).  The kernel works on pairs of 256-sample
    # blocks, one CTA per (16 direction tiles, block pair): B is rounded up so that the number of block pairs is a
    # multiple of the 148 SMs -- the CTAs then fill whole waves at 1, 2, 4 and 8 GPUs (cfg3: B = 592, 310 MB)
    C = 64 * c["nx"] * c["ny"]
    per_frame = C * c["N"] * 4
    B = max(2, int(np.ceil(256e6 / per_frame)))
    if c["N"] == 256:
        pairs = -(-B // 2)
        B = 2 * (-(-pairs // 148) * 148)
    return B


def workload(c, name, B):
    C = 64 * c["nx"] * c["ny"]
    D = c["rows"] * c["cols"]
    T = (B - 1) * c["N"] + c["W"]
    T += T & 1
    return dict(workload=f"{name}: {C} mics x {c['rows']}x{c['cols']}={D} directions x {c['N']}-sample frames",
                channels=C, directions=D, frame_len=c["N"], frames_per_step=B, samples_per_channel=T,
                input_mb=round(C * T * 4 / 1e6, 1), l2="inputs larger than L2 (126 MB); no flush needed",
                frames_rule="256 MB of input, block pairs rounded up to a multiple of 148 SMs (whole CTA waves at 1-8 GPUs)")


def flops_per_map(C, D, N):
    return D * N * (4 * C + 6)          # SURVEY.md 8d: 4 FLOP per (dir, ch, sample) + 6 per (dir, sample)


DUMP_BYTES = 60_000_000      # stays under 64 MB with the .npy headers


def dump_outputs(path, **arrays):
    """--dump-outputs: each array (a torch tensor [rows][...] on the device) as path/<name>.npy in float32.  When the arrays
    together exceed DUMP_BYTES, each keeps a fixed, seeded, sorted sample of its rows (frames)."""
    import torch
    os.makedirs(path, exist_ok=True)
    total = sum(a.numel() * 4 for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, int(a.shape[0] * DUMP_BYTES / total))
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))
            a = a.index_select(0, torch.from_numpy(rows).to(a.device))
        np.save(os.path.join(path, f"{name}.npy"), a.float().cpu().numpy())


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """Samples SM clock, board power and throttle reasons of one GPU through NVML while a timed region runs."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.stop = index, [], set(), threading.Event()
        self.max_mhz = None
        self.thread = None
        self.t0 = self.t1 = None     # the timed region; only samples inside it are reported

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            while not self.stop.is_set():
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(h) / 1e3
                except Exception:
                    watts = None
                self.samples.append((time.perf_counter(), mhz, r, names, watts))
                time.sleep(0.005)
        except Exception as e:  # NVML unavailable: report that rather than fail the bench
            self.reasons.add(f"nvml_error:{type(e).__name__}")

    def __enter__(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join(timeout=2)

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def summary(self, t0=None, t1=None):
        t0 = self.t0 if t0 is None else t0
        t1 = (self.t1 or 1e30) if t1 is None else t1
        inside = [s for s in self.samples if t0 is not None and t0 <= s[0] <= t1]
        reasons = set(self.reasons)
        for _, _, r, names, _ in inside:
            for bit, nm in names.items():
                if r & bit:
                    reasons.add(nm)
        watts = [s[4] for s in inside if s[4] is not None]
        return {"sm_mhz": statistics.median([s[1] for s in inside]) if inside else None, "sm_max_mhz": self.max_mhz,
                "samples": len(inside), "reasons": sorted(reasons), "power_w_max": max(watts) if watts else None,
                "power_w_median": statistics.median(watts) if watts else None}


def make_input(c, T):
    from bflk import synth
    xyz = synth.tile_geometry(cases.origins(c["nx"], c["ny"]))
    # tones are cheap, white noise for 512 x 132k samples is not: tile a 16-frame noise block
    base = synth.make_stream(xyz, T, sigma=0.0)
    rng = np.random.Generator(np.random.Philox(synth.SEED))
    blk = (1e-3 * rng.standard_normal((xyz.shape[0], 16 * c["N"]))).astype(np.float32)
    reps = int(np.ceil(T / blk.shape[1]))
    base += np.tile(blk, (1, reps))[:, :T]
    return np.ascontiguousarray(base, np.float32)


# ---- the reference's CPU path (oracle/_ref: the unmodified delay.cpp) -----------------------------------------------
def cpu_tables(c):
    from oracle import oracle as O
    if O.ref() is None:
        raise RuntimeError("oracle/_ref/libref.so is missing")
    xyz = O.create_tiled_antenna(cases.origins(c["nx"], c["ny"]))
    return O.mimo_lut(xyz, c["rows"], c["cols"], c["fov"], c["H"])


def cpu_reference_rate(c, stream, n_threads, budget_s, frames=None, tables=None):
    """maps/s of the compiled reference delay() loop (oracle/_ref) over all directions, n_threads threads."""
    from oracle import oracle as O
    off, fr = tables if tables is not None else cpu_tables(c)
    D = off.shape[0]
    sub = 1
    est_units = D * off.shape[1] * c["N"]
    if est_units / (1.5e9 * n_threads) > budget_s / 3:      # cfg5: time a direction subset and scale
        sub = int(np.ceil(est_units / (1.5e9 * n_threads) / (budget_s / 3)))
        off, fr = np.ascontiguousarray(off[::sub]), np.ascontiguousarray(fr[::sub])
    n_avail = max(1, (stream.shape[1] - c["W"]) // c["N"] + 1)
    window = np.ascontiguousarray(stream[:, :c["W"]])
    O.ref_mimo_update(window, off, fr, n=c["N"], n_threads=n_threads)      # warm-up
    done, t0 = 0, time.perf_counter()
    while True:
        b = done % n_avail
        window = np.ascontiguousarray(stream[:, b * c["N"]: b * c["N"] + c["W"]])
        O.ref_mimo_update(window, off, fr, n=c["N"], n_threads=n_threads)
        done += 1
        el = time.perf_counter() - t0
        if (frames and done >= frames) or (not frames and el > budget_s):
            break
    rate = done / el / sub
    sample = f"{done} frames x {off.shape[0]} of {D} directions in {el:.2f} s" + (f" (1/{sub} direction subset, scaled)" if sub > 1 else "")
    return rate, sample


def run_reference(args, c, name):
    """The reference arm: every step is the SAME step as the GPU arm's -- all B frames of the batch, every direction --
    through the compiled, unmodified reference delay() (oracle/_ref) on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = args.frames or default_frames(c)
    n_threads = os.cpu_count() or 1
    T = 15 * c["N"] + c["W"]                       # 16 distinct frames, cycled: the arithmetic per frame is what is timed
    stream = make_input(c, T)
    tables = cpu_tables(c)
    for _ in range(min(args.warmup, 2)):
        cpu_reference_rate(c, stream, n_threads, 1e9, frames=8, tables=tables)
    t0 = time.perf_counter()
    rates, sample = [], ""
    for _ in range(args.steps):
        r, sample = cpu_reference_rate(c, stream, n_threads, 1e9, frames=B, tables=tables)
        rates.append(r)
    el = time.perf_counter() - t0
    value = B * args.steps / el
    cfg = workload(c, name, B)
    cfg["parallelism"] = f"{n_threads} host threads over directions"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / max(1, args.steps), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_threads, "kind": "reference",
                             "sample": f"each step = all {B} frames of the workload (16 distinct frames cycled); last step: {sample}"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "dir_samples_per_sec": value * cfg["directions"] * c["N"]}
    print(json.dumps(line))


# ---- helpers of the GPU arm ----------------------------------------------------------------------------------------
class Timer:
    def __init__(self, torch, dist, world, dev):
        self.torch, self.dist, self.world, self.dev = torch, dist, world, dev

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup):
        """ms for `steps` calls of fn, CUDA events on the current stream, max over ranks.  fn.finish (if any) runs after
        the last call, inside the timed region: a step that leaves work on another stream joins it there."""
        torch = self.torch
        finish = getattr(fn, "finish", None)
        for _ in range(warmup):
            fn()
        if finish:
            finish()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish:
            finish()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item())


def measure_resident(w, tm, step, steps, flops_launch):
    """maps-independent numbers of a timed region: (ms, launches, das_ms, das_n, pack_ms, pack_n)."""
    tm.barrier()
    w.enable_timing(True)
    w.kernel_time_ms()
    l0 = w.launch_count()
    ms = tm.timed(step, steps, 0)
    launches = w.launch_count() - l0
    das_ms, das_n, pack_ms, pack_n = w.kernel_time_ms()
    w.enable_timing(False)
    return ms, launches, das_ms, das_n, pack_ms, pack_n


def small_config_run(bflk, torch, name, dev, local, steps=8, warmup=3, kernel=0):
    """cfg1 / cfg2 / cfg5 on one GPU: maps/s resident + the dominant kernel's fraction of the FP32 peak."""
    c = cases.CONFIGS[name]
    B = default_frames(c)
    cfg = workload(c, name, B)
    C, D, N, T = cfg["channels"], cfg["directions"], c["N"], cfg["samples_per_channel"]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"], device=local,
                        frame_len=N, history=c["H"], window_len=c["W"])
    w.set_kernel(kernel)
    x = torch.from_numpy(make_input(c, T)).to(dev)
    out = torch.empty((B, D), dtype=torch.float32, device=dev)
    cs = torch.cuda.current_stream().cuda_stream

    def step():
        w.power_map_batch_dev(x.data_ptr(), T, B, out.data_ptr(), cs)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    w.enable_timing(True)
    w.kernel_time_ms()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    das_ms, das_n, _, _ = w.kernel_time_ms()
    w.enable_timing(False)
    k = w.kernel_info()
    res = {"workload": cfg["workload"], "frames_per_step": B, "value": B * steps / (ms / 1e3), "unit": UNIT, "steps": steps,
           "kernel": KERNEL_NAMES.get(k[0], "?"), "tflops_kernel": flops_per_map(C, D, N) * B / (das_ms / 1e3 / max(1, das_n)) / 1e12 if das_n else None}
    w.close()
    del x, out
    return res


def miso_bench(bflk, torch, dev, local, calls=300, steps=None, warmup=20, dump=None):
    """cfg4: 16 tracked targets x 512 microphones, enhanced audio + beam power per frame.  Latency of the host call on a
    window kept on the device (what a tracker iterating on one frame pays) and of the call that uploads the frame first,
    sampled over `calls` calls each; the device-side throughput of `steps` (default `calls`) timed back-to-back
    asynchronous calls after `warmup` untimed ones (the last call's audio and power go to `dump`, if given)."""
    import ctypes as C
    from bflk import synth
    c = cases.CFG4
    m = bflk.MISOWorker(cases.origins(c["nx"], c["ny"]), device=local)
    th, ph = cases.cfg4_targets()
    win = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), c["W"])
    T, N, Cn = c["T"], c["N"], 64 * c["nx"] * c["ny"]

    def lat(fn, n):
        for _ in range(20):
            fn()
        t = []
        for _ in range(n):
            t0 = time.perf_counter()
            fn()
            t.append((time.perf_counter() - t0) * 1e6)
        return {"p50_us": float(np.percentile(t, 50)), "p95_us": float(np.percentile(t, 95))}

    upload = lat(lambda: m.miso(th, ph, win), calls)
    m.set_window(win)
    resident = lat(lambda: m.miso(th, ph), calls)
    P = 26
    rng = np.random.default_rng(5)
    pth, pph = rng.random(P) * np.deg2rad(70.0), rng.random(P) * 2 * np.pi
    mono = lat(lambda: m.monopulse(pth, pph, None, np.deg2rad(4.0), np.deg2rad(80.0), 3e-4), calls)
    # device-side rate: asynchronous calls back to back on one stream
    wd = torch.from_numpy(win).to(dev)
    audio = torch.zeros((T, N), device=dev)
    power = torch.zeros(T, device=dev)
    st = torch.cuda.Stream(device=dev)
    tt, pp = np.ascontiguousarray(th, np.float64), np.ascontiguousarray(ph, np.float64)

    def call():
        rc = m._L.bflk_miso_dev(m._h, tt.ctypes.data_as(C.c_void_p), pp.ctypes.data_as(C.c_void_p), T, C.c_void_p(wd.data_ptr()),
                                C.c_void_p(audio.data_ptr()), C.c_void_p(power.data_ptr()), C.c_void_p(st.cuda_stream))
        assert rc == 0
    steps = steps or calls
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        call()
    e1.record(st)
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / steps
    if dump:
        dump_outputs(dump, audio=audio, power=power)
    flop = T * N * 4 * Cn
    # CPU: Particle::das + beam for the same targets = the reference delay() loop over T directions
    cpu = None
    try:
        from oracle import oracle as O
        xyz = O.create_tiled_antenna(cases.origins(c["nx"], c["ny"]))
        off, fr = O.steer_tables(xyz, th, ph)
        O.ref_mimo_update(win, off, fr, want_das=True)
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < 1.0:
            O.ref_mimo_update(win, off, fr, want_das=True)
            n += 1
        cpu = {"us_per_frame": (time.perf_counter() - t0) / n * 1e6, "cores": 1, "kind": "reference",
               "sample": f"{n} frames x {T} targets, compiled reference delay() loop, one thread (the reference's MISO worker is one thread)"}
    except Exception as e:
        cpu = {"us_per_frame": None, "sample": f"failed: {e}"}
    m.close()
    return {"workload": f"cfg4: {Cn} mics x {T} tracked targets x {N}-sample frames (audio + beam power per target)",
            "latency_resident_window": resident, "latency_with_upload": upload, "latency_monopulse_26_particles": mono,
            "device_us_per_call": us, "target_samples_per_sec": T * N / (us * 1e-6),
            "roofline": {"bound": "latency (512 dependent adds per output sample; 8.4 MFLOP per call)", "flop_per_call": flop,
                         "achieved_tflops": flop / (us * 1e-6) / 1e12},
            "realtime_budget_us": 5243, "cpu_baseline": cpu}


def single_frame_latency(bflk, name, local, calls=200):
    """One live frame through bflk_power_map (what a Worker adapter calls once per 5.24 ms): host window in, host map out.
    The window is page-locked like the adapters' snapshot buffer (`auto_pageable`: an ordinary numpy array instead)."""
    import ctypes as C
    import torch
    from bflk import synth
    c = cases.CONFIGS[name]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"], device=local)
    win = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), c["W"])
    pin = torch.from_numpy(win).pin_memory()
    res = torch.empty(c["rows"] * c["cols"], dtype=torch.float32).pin_memory()
    out = {}
    # auto = two-FMA form; channel_split = the same with bflk_set_channel_split (a thread-block cluster splits the channels
    # of the frame: deterministic, within the 1e-4 bar, but not the bits a large batch gives); bit_identical = kernel 2
    for kernel, split, src, label in ((0, False, pin.data_ptr(), "auto"), (0, True, pin.data_ptr(), "channel_split"),
                                      (2, False, pin.data_ptr(), "bit_identical"), (0, False, win.ctypes.data, "auto_pageable")):
        w.set_kernel(kernel)
        w.set_channel_split(split)

        def call():
            rc = w._L.bflk_power_map(w._h, C.c_void_p(src), C.c_void_p(res.data_ptr()))
            assert rc == 0
        for _ in range(20):
            call()
        t = []
        for _ in range(calls):
            t0 = time.perf_counter()
            call()
            t.append((time.perf_counter() - t0) * 1e6)
        out[label] = {"p50_us": float(np.percentile(t, 50)), "p95_us": float(np.percentile(t, 95))}
    w.close()
    return out


def run_miso_only(args):
    import torch
    import bflk
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    with ClockSampler(local) as clk:
        clk.begin()
        # latency percentiles want at least 100 samples; the timed throughput region runs exactly --steps calls
        r = miso_bench(bflk, torch, dev, local, calls=max(100, args.steps), steps=args.steps, warmup=args.warmup,
                       dump=args.dump_outputs)
        clk.end()
    c = cases.CFG4
    line = {"metric": "miso_target_samples_per_sec", "value": r["target_samples_per_sec"], "unit": "target-samples/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["device_us_per_call"] / 1e3, "higher_is_better": True,
            "scaling": "replicas only", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": r["workload"], "targets": c["T"], "channels": 64 * c["nx"] * c["ny"], "frame_len": c["N"]},
            "clocks": clk.summary(), "e2e": {"value": c["T"] * c["N"] / (r["latency_with_upload"]["p50_us"] * 1e-6), "unit": "target-samples/s",
                                            "h2d_bytes_per_step": 64 * c["nx"] * c["ny"] * c["W"] * 4, "d2h_bytes_per_step": c["T"] * (c["N"] + 1) * 4 + 4,
                                            "path": "bflk_miso (host window uploaded per call)"},
            "gpu_launches": 1, "miso": r, "roofline": r["roofline"], "cpu_baseline": r["cpu_baseline"]}
    print(json.dumps(line))


def run_ours(args, c, name):
    import torch
    import torch.distributed as dist
    import bflk

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # stdout carries the one JSON line and nothing else
        dist.init_process_group("nccl", device_id=dev)
    tm = Timer(torch, dist, world, dev)

    B = args.frames or default_frames(c)
    C, D, N = 64 * c["nx"] * c["ny"], c["rows"] * c["cols"], c["N"]
    cfg = workload(c, name, B)
    T = cfg["samples_per_channel"]

    def make_worker(dir_groups):
        w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"], device=local,
                            frame_len=N, history=c["H"], window_len=c["W"])
        w.set_kernel(args.kernel)
        if world > 1:
            # the only thing torch.distributed carries: the 128-byte NCCL id of the library's own communicator
            box = [bflk.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            w.comm_init_rank(box[0], world, rank, dir_groups)
        return w

    w = make_worker(args.dir_groups)
    gd, gf = (w.comm_info()[2], w.comm_info()[3]) if world > 1 else (1, 1)
    d_first, d_count, f_first, f_count = bflk.shard_plan(D, B, world, rank, gd) if world > 1 else (0, D, 0, B)

    host_in = torch.from_numpy(make_input(c, T)).pin_memory()
    stream_dev = host_in.to(dev, non_blocking=True)
    out_all = torch.zeros((B, D), dtype=torch.float32, device=dev)
    out_alt = torch.zeros((B, D), dtype=torch.float32, device=dev) if world == 1 else None
    host_out = torch.empty((B, D), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()
    # a real (non-null) stream: kernels, NCCL and the timing events all go on it
    work_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(work_stream)
    cs = work_stream.cuda_stream
    assert cs != 0

    def step_with(worker, overlap=True):
        overlap = overlap and not args.no_overlap
        if world > 1 and overlap:
            # continuous operation: the all-gather + assembly of step i run on the communicator's stream under the kernels of
            # step i + 1 (bflk_power_map_batch_sharded_dev_submit); the join after the last step is inside the timed region
            def fn():
                worker.power_map_batch_sharded_dev_submit(stream_dev.data_ptr(), T, B, out_all.data_ptr(), cs)
            fn.finish = lambda: worker.power_map_batch_sharded_dev_join(cs)
            return fn
        if world > 1:
            return lambda: worker.power_map_batch_sharded_dev(stream_dev.data_ptr(), T, B, out_all.data_ptr(), cs)
        if overlap:
            # continuous operation on one GPU: consecutive steps alternate between the handle's two compute streams (each with its
            # own scratch and its own output buffer): the pack pre-pass of step i + 1 runs under the kernel of step i and its
            # CTAs fill the SMs the last CTAs of step i leave idle (bflk_power_map_batch_dev_submit); join inside the timed region
            state = {"k": 0}

            def fn1():
                o = out_all if state["k"] & 1 == 0 else out_alt
                state["k"] += 1
                worker.power_map_batch_dev_submit(stream_dev.data_ptr(), T, B, o.data_ptr(), cs)

            def fin1():
                worker.power_map_batch_dev_join(cs)
                if state["k"] & 1 == 0 and state["k"]:       # the last step wrote out_alt: out_all must hold the latest maps
                    out_all.copy_(out_alt)
            fn1.finish = fin1
            return fn1
        return lambda: worker.power_map_batch_dev(stream_dev.data_ptr(), T, B, out_all.data_ptr(), cs)

    step = step_with(w)
    fl_launch = flops_per_map(C, d_count, N) * f_count          # algorithmic FLOPs of one das launch on this rank

    # ---- device-resident throughput, dominant-kernel time and clocks over the timed region ----
    with ClockSampler(local) as clk:       # NVML start-up overlaps the warm-up; samples are filtered to the timed region
        for _ in range(args.warmup):
            step()
        clk.begin()
        ms, launches, das_ms, das_n, pack_ms, pack_n = measure_resident(w, tm, step, args.steps, fl_launch)
        clk.end()
        value = B * args.steps / (ms / 1e3)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, power_maps=out_all)     # the complete [B][D] maps of the last timed step
        # the dominant kernel's OWN launch duration (roofline.achieved) is timed with one synchronous call per step: in
        # continuous operation consecutive launches overlap, and an event pair around a launch then also spans its wait
        # for the SMs the previous launch still holds
        ms_sync = None
        if not args.no_overlap:
            sync_step = step_with(w, overlap=False)
            n_sync = max(5, min(args.steps, 40))
            for _ in range(2):
                sync_step()
            ms_sync_total, _, das_ms, das_n, pack_ms, pack_n = measure_resident(w, tm, sync_step, n_sync, fl_launch)
            ms_sync = ms_sync_total / n_sync
        kinfo = w.kernel_info()
        clocks = clk.summary()
        ref_maps = out_all.clone()

        # ---- >= 2 s of back-to-back steps: clocks and board power under sustained load ----
        sustained = None
        if not args.no_extras:
            n_sus = max(args.steps, int(np.ceil(2.2e3 / (ms / args.steps))))
            t0 = time.perf_counter()
            sms = tm.timed(step, n_sus, 0)
            t1 = time.perf_counter()
            s = clk.summary(t0, t1)
            sustained = {"seconds": sms / 1e3, "steps": n_sus, "value": B * n_sus / (sms / 1e3), "unit": UNIT, "sm_mhz": s["sm_mhz"],
                         "power_w_max": s["power_w_max"], "power_w_median": s["power_w_median"], "reasons": s["reasons"]}

    # ---- the kernel whose delayed sums are bit-identical to the reference's delay() ----
    bit_identical = None
    if not args.no_extras and args.kernel == 0:
        w.set_kernel(2)
        for _ in range(3):
            step()
        n_bi = min(args.steps, 20)
        bms, _, bdas_ms, bdas_n, _, _ = measure_resident(w, tm, step, n_bi, fl_launch)
        if not args.no_overlap:      # the kernel's own launch duration: synchronous calls (see above)
            _, _, bdas_ms, bdas_n, _, _ = measure_resident(w, tm, step_with(w, overlap=False), n_bi, fl_launch)
        bk = w.kernel_info()
        bit_identical = {"value": B * n_bi / (bms / 1e3), "unit": UNIT, "steps": n_bi, "kernel": KERNEL_NAMES.get(bk[0], "?"),
                         "tflops_kernel": fl_launch / (bdas_ms / 1e3 / max(1, bdas_n)) / 1e12 if bdas_n else None,
                         "max_rel_diff_vs_automatic_kernel": float(((out_all - ref_maps).abs() / ref_maps).max().item())}
        w.set_kernel(args.kernel)
        step()

    # ---- end to end: host buffers through the C ABI ----
    e2e = None
    if not args.no_e2e:
        if world == 1:
            def e2e_step():
                w.power_map_batch_ptr(host_in.data_ptr(), T, B, host_out.data_ptr())
        else:
            # host batches want chunks of whole CTA waves that are as short as possible (upload of chunk k+1 under the kernels of
            # chunk k): with 4 direction groups a wave of a rank's 64 tiles is 37 block pairs, so an 8-rank job cuts its frame
            # slices into four one-wave chunks instead of two two-wave chunks (the resident path prefers 2 groups: less pack)
            e2e_gd = 4 if (world % 4 == 0 and world >= 8 and args.dir_groups == 0) else args.dir_groups
            we = make_worker(e2e_gd) if e2e_gd != args.dir_groups else w
            out_ptr = host_out.data_ptr() if rank == 0 else 0      # the maps are read back where they are consumed: rank 0

            def e2e_step():
                we.power_map_batch_sharded_ptr(host_in.data_ptr(), T, B, out_ptr)
        e2e_steps = max(3, min(args.steps, 40) // 2)

        def wall(fn_all):
            """ms of fn_all() between barriers, host wall clock, max over ranks (the host API returns after the D2H copy)"""
            tm.barrier()
            t0 = time.perf_counter()
            fn_all()
            tm.barrier()
            v = torch.tensor([1e3 * (time.perf_counter() - t0)], device=dev)
            if world > 1:
                dist.all_reduce(v, op=dist.ReduceOp.MAX)
            return float(v.item())

        e2e_step()
        ems_sync = wall(lambda: [e2e_step() for _ in range(e2e_steps)])
        ems = ems_sync
        pipelined = False
        if world == 1:
            # continuous operation: bflk_power_map_batch_submit / _wait, two batches in flight -- the upload of step i + 1 runs
            # under the kernels of step i; every step still uploads its own input and reads back its own maps
            host_out2 = torch.empty((B, D), dtype=torch.float32).pin_memory()
            outs = [host_out, host_out2]

            def pipelined_steps():
                for i in range(e2e_steps):
                    w.power_map_batch_submit_ptr(host_in.data_ptr(), T, B, outs[i & 1].data_ptr())
                for _ in range(2):
                    w.power_map_batch_wait()
            pipelined_steps()
            ems = wall(pipelined_steps)
            pipelined = True
            assert torch.equal(host_out, host_out2)
        else:
            def pipelined_steps():
                for i in range(e2e_steps):
                    we.power_map_batch_sharded_submit_ptr(host_in.data_ptr(), T, B, out_ptr)
                    if i & 1:
                        we.power_map_batch_sharded_wait()      # at most two batches in flight
                we.power_map_batch_sharded_wait()
            pipelined_steps()
            ems = wall(pipelined_steps)
            pipelined = True
        # what the PCIe links deliver when every rank uploads at once (the e2e path moves C*T*4 bytes per step in total)
        probe_bytes = min(host_in.numel() * 4, 64 << 20)
        probe_dev = torch.empty(probe_bytes // 4, dtype=torch.float32, device=dev)
        probe_src = host_in.view(-1)[:probe_bytes // 4]
        probe_dev.copy_(probe_src, non_blocking=True)
        tm.barrier()
        tp = time.perf_counter()
        for _ in range(8):
            probe_dev.copy_(probe_src, non_blocking=True)
        tm.barrier()
        h2d_gbs = torch.tensor([8 * probe_bytes / (time.perf_counter() - tp) / 1e9], device=dev)
        if world > 1:
            dist.all_reduce(h2d_gbs, op=dist.ReduceOp.MIN)
        del probe_dev
        e2e = {"value": B * e2e_steps / (ems / 1e3), "unit": UNIT, "h2d_gbs_per_rank_all_ranks_uploading": float(h2d_gbs.item()), "h2d_bytes_per_step": C * T * 4 if world == 1 else
               C * (B * N + gf * (c["W"] - N)) * 4, "d2h_bytes_per_step": B * D * 4, "steps": e2e_steps,
               "synchronous_call_value": B * e2e_steps / (ems_sync / 1e3), "pipelined": pipelined,
               "path": "bflk_power_map_batch_submit / _wait, two batches in flight (host buffers; synchronous_call_value = bflk_power_map_batch, one call at a time)" if world == 1 else
               "bflk_power_map_batch_sharded_submit / _wait (two batches in flight; synchronous_call_value = one call at a time): per frame chunk each rank uploads C/G_d channel rows over its own PCIe link, NCCL all-gather "
               "inside the frame group (copy stream) overlapping the kernels of the previous chunk, NCCL all-gather of the maps, D2H of "
               "[B][D] on rank 0; h2d bytes summed over the ranks" + (f"; {we.comm_info()[2]} direction groups x {we.comm_info()[3]} frame groups" if world > 1 else ""),
               "same_maps_as_resident_path": bool(torch.equal(host_out, ref_maps.cpu())) if rank == 0 else None}
        if world > 1 and we is not w:
            we.close()

    # ---- the other split (pure grid sharding, the north_star's) in the same run ----
    grid_shard = None
    if world > 1 and not args.no_extras and args.dir_groups == 0 and gd != world:
        wg = make_worker(world)
        gstep = step_with(wg)
        for _ in range(3):
            gstep()
        gms, _, gdas_ms, gdas_n, gpack_ms, gpack_n = measure_resident(wg, tm, gstep, args.steps, 0)
        gms_step = gms / args.steps
        if not args.no_overlap:
            n_g = max(5, min(args.steps, 20))
            gms_sync, _, gdas_ms, gdas_n, gpack_ms, gpack_n = measure_resident(wg, tm, step_with(wg, overlap=False), n_g, 0)
            gms_step = gms_sync / n_g
        g_first, g_count, _, _ = bflk.shard_plan(D, B, world, rank, world)
        grid_shard = {"parallelism": f"{world} direction groups x 1 frame group", "value": B * args.steps / (gms / 1e3), "unit": UNIT,
                      "tflops_kernel": flops_per_map(C, g_count, N) * B / (gdas_ms / 1e3 / max(1, gdas_n)) / 1e12 if gdas_n else None,
                      "pack_share_of_step": gpack_ms / max(1, gpack_n) / gms_step, "same_maps": bool(torch.equal(out_all, ref_maps))}
        wg.close()

    # ---- cfg5 (256x256 grid x 4096-sample frames) on all N GPUs, grid sharded N ways, same run ----
    cfg5_multi = None
    if world > 1 and not args.no_extras and name == "cfg3":
        del stream_dev, out_all, ref_maps
        torch.cuda.empty_cache()
        c5 = cases.CONFIGS["cfg5"]
        B5 = default_frames(c5)
        w5cfg = workload(c5, "cfg5", B5)
        T5, D5, C5 = w5cfg["samples_per_channel"], w5cfg["directions"], w5cfg["channels"]
        w5 = bflk.MIMOWorker(cases.origins(c5["nx"], c5["ny"]), c5["rows"], c5["cols"], c5["fov"], device=local,
                             frame_len=c5["N"], history=c5["H"], window_len=c5["W"])
        box = [bflk.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        w5.comm_init_rank(box[0], world, rank, world)
        x5 = torch.from_numpy(make_input(c5, T5)).to(dev)
        o5 = torch.empty((B5, D5), dtype=torch.float32, device=dev)

        def step5():
            w5.power_map_batch_sharded_dev(x5.data_ptr(), T5, B5, o5.data_ptr(), cs)
        for _ in range(2):
            step5()
        n5 = 4
        ms5, _, das5, dn5, _, _ = measure_resident(w5, tm, step5, n5, 0)
        _, cnt5, _, _ = bflk.shard_plan(D5, B5, world, rank, world)
        cfg5_multi = {"workload": w5cfg["workload"], "frames_per_step": B5, "parallelism": f"{world} direction groups x 1 frame group",
                      "value": B5 * n5 / (ms5 / 1e3), "unit": UNIT, "steps": n5,
                      "tflops_kernel_rank0": flops_per_map(C5, cnt5, c5["N"]) * B5 / (das5 / 1e3 / max(1, dn5)) / 1e12 if dn5 else None}
        w5.close()
        del x5, o5

    # ---- rank 0: derived numbers, the other configurations, CPU baseline ----
    if rank == 0:
        pk, pk_kind = peaks()
        sm_count = torch.cuda.get_device_properties(local).multi_processor_count
        max_mhz = pk.get("sm_max_mhz") or clocks["sm_max_mhz"] or 1965.0
        peak_tf = sm_count * FP32_LANES_PER_SM * 2 * max_mhz * 1e6 / 1e12
        das_avg_s = das_ms / 1e3 / max(1, das_n)
        achieved_tf = fl_launch / das_avg_s / 1e12 if das_n else None
        alg_bytes = 4 * C * ((f_count - 1) * N + c["W"]) + 4 * f_count * d_count
        ubench_tf = None
        try:
            ubench_tf = w.fp32_peak_tflops()
        except Exception:
            pass
        roof = {"bound": "fp32", "kernel": KERNEL_NAMES.get(kinfo[0], "?"), "achieved": achieved_tf,
                "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf if achieved_tf else None,
                "peak_source": f"{sm_count} SMs x 128 FP32 lanes x 2 x sm_max_mhz {max_mhz:.0f} ({pk_kind} MEASURED_PEAKS.json clock)",
                "frac_at_sampled_clock": (achieved_tf / (peak_tf * clocks["sm_mhz"] / max_mhz)) if achieved_tf and clocks["sm_mhz"] else None,
                "ffma_ubench_tflops": ubench_tf, "frac_vs_ffma_ubench": achieved_tf / ubench_tf if achieved_tf and ubench_tf else None,
                "flop_per_launch": fl_launch, "avg_launch_ms": das_avg_s * 1e3, "launches_timed": das_n,
                "kernel_share_of_step": das_ms / max(1, das_n) / (ms_sync if ms_sync else ms / args.steps),
                "pack_share_of_step": pack_ms / max(1, pack_n) / (ms_sync if ms_sync else ms / args.steps), "traffic": None}
        if ms_sync:
            roof["timed_with"] = "one synchronous call per step (kernel and pack durations, shares); `value` is continuous operation"
        if bit_identical and bit_identical["tflops_kernel"]:
            bit_identical["roofline_frac"] = bit_identical["tflops_kernel"] / peak_tf
        if grid_shard and grid_shard["tflops_kernel"]:
            grid_shard["roofline_frac"] = grid_shard["tflops_kernel"] / peak_tf
        try:        # DRAM bytes per launch from the committed ncu capture of this exact command, if there is one
            t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(name)
            if t and t["frames_per_step"] == B and t["kernel"] == roof["kernel"] and t["n_gpus"] == world:
                roof["traffic"] = t["dram_bytes_per_launch"]
                roof["traffic_source"] = t["source"]
        except Exception:
            pass
        roof_hbm = {"bound": "hbm", "achieved": alg_bytes / das_avg_s / 1e9 if das_n else None, "peak": pk["hbm_gbs"],
                    "unit": "GB/s", "frac": alg_bytes / das_avg_s / 1e9 / pk["hbm_gbs"] if das_n else None,
                    "bytes_per_launch": alg_bytes, "peak_source": pk_kind}
        cfg.update(parallelism=(f"{gd} direction groups x {gf} frame groups, sharded and gathered inside libbflk (NCCL)" +
                                ("" if args.no_overlap else "; continuous operation: the all-gather of step i runs under the kernels of step i + 1 (bflk_power_map_batch_sharded_dev_submit / _join)"))
                   if world > 1 else ("single GPU" if args.no_overlap else "single GPU; continuous operation: consecutive steps alternate between the handle's two compute streams (bflk_power_map_batch_dev_submit / _join)"),
                   directions_per_gpu=d_count, frames_per_gpu=f_count, kernel=roof["kernel"], tile_span=kinfo[1], window_chunks=kinfo[2])
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks, "e2e": e2e,
                "gpu_launches": launches, "roofline": roof, "roofline_hbm": roof_hbm,
                "dir_samples_per_sec": value * D * N, "tflops_whole_job": value * flops_per_map(C, D, N) / 1e12}
        if ms_sync:
            line["synchronous_call_value"] = B / (ms_sync / 1e3)     # one bflk_power_map_batch(_sharded)_dev call per step, nothing overlapped
        if world > 1:
            line["comm"] = dict(zip(("n_ranks", "rank", "dir_groups", "frame_groups", "collectives"), w.comm_info()))
        if bit_identical:
            line["bit_identical"] = bit_identical
        if sustained:
            line["sustained"] = sustained
        if grid_shard:
            line["grid_shard"] = grid_shard
        if cfg5_multi:
            if cfg5_multi["tflops_kernel_rank0"]:
                cfg5_multi["roofline_frac_rank0"] = cfg5_multi["tflops_kernel_rank0"] / peak_tf
            line["other_configs"] = {"cfg5": cfg5_multi}
        if not args.no_extras and world == 1 and name == "cfg3":
            del stream_dev, out_all, ref_maps
            torch.cuda.empty_cache()
            others = {}
            for other in ("cfg1", "cfg2", "cfg5"):
                try:
                    r = small_config_run(bflk, torch, other, dev, local)
                    r["roofline_frac"] = r["tflops_kernel"] / peak_tf if r["tflops_kernel"] else None
                    others[other] = r
                except Exception as e:
                    others[other] = {"error": str(e)}
            try:
                others["cfg4"] = miso_bench(bflk, torch, dev, local, calls=200)
            except Exception as e:
                others["cfg4"] = {"error": str(e)}
            line["other_configs"] = others
            try:
                line["latency_single_frame_us"] = {k: single_frame_latency(bflk, k, local) for k in ("cfg1", "cfg3")}
            except Exception as e:
                line["latency_single_frame_us"] = {"error": str(e)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                n_threads = os.cpu_count() or 1
                sub = host_in.numpy()[:, :16 * N + c["W"]]
                tables = cpu_tables(c)
                rate, sample = cpu_reference_rate(c, sub, n_threads, budget_s=5.0, tables=tables)
                rate1, sample1 = cpu_reference_rate(c, sub, 1, budget_s=3.0, tables=tables)
                line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": n_threads, "kind": "reference",
                                        "sample": sample, "single_thread_value": rate1, "single_thread_sample": sample1}
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        w.close()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.config == "cfg4":
        if args.impl == "reference":
            raise SystemExit("--impl reference is defined for the power-map configurations")
        return run_miso_only(args)
    c = cases.CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, c, args.config)
    else:
        run_ours(args, c, args.config)


if __name__ == "__main__":
    main()
