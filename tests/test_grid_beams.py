"""Beams of the grid kernels (bflk_beams_batch_dev, bflk_session_beams): the delayed sum out[i] of every direction of the
range, for every frame, next to the power map that squares it (MIMOWorker::update, src/dsp/mimo.cpp:121-137).

Bars, per the accuracy contract of the kernels:
  * kernels 1, 2 and 3 (the reference's exact triple): bit-identical to oracle.mimo_das, itself pinned against the
    compiled delay() through golden["snapshot"]["das"];
  * kernel 4 (two-FMA form) and the channel split: |beam - mimo_das| <= 6 usable 2^-24 S_i on every sample, with
    S_i = sum over the summed channels of |x[o + i]| + |x[o + i + 1]| (float64).  Each form rounds at most three times
    per channel and no rounded value exceeds S_i, so each rounding costs at most 2^-24 S_i; a sample shift or a wrong
    channel misses this by orders of magnitude;
  * the power of a beams call: the bits of the power-only call on the same input, and (seeded white noise) within 1e-5 of
    the float64 high-pass and mean square of the returned beams -- which ties every beam sample to the map, including
    which block of a multi-block frame wrote it."""
import ctypes as C

import numpy as np
import pytest

import cases
from test_tile_variants import CASES as VARIANT_CASES, dir_range, make_beamformer, variant_lut

BFLK_ERR_INVALID, BFLK_ERR_STATE = -1, -2
POWER_RTOL = 1e-5
EPS32 = 2.0 ** -24
B = 7                        # frames per batch: an odd count leaves the last block pair half empty


# ---- no GPU ----------------------------------------------------------------------------------------------------------
def test_null_handle_is_invalid():
    import bflk
    L = bflk.load_library()
    buf = np.zeros(4096, np.float32)
    i64, i32 = C.c_int64(), C.c_int32()
    assert L.bflk_beams_batch_dev(None, buf.ctypes.data, 1024, 1, buf.ctypes.data, buf.ctypes.data, None) == BFLK_ERR_INVALID
    assert L.bflk_session_beams(None, 1, buf.ctypes.data, buf.ctypes.data, C.byref(i64), C.byref(i32)) == BFLK_ERR_INVALID


# ---- references --------------------------------------------------------------------------------------------------------
def das_ref(oracle, x, off, frac, index, N, b):
    """oracle.mimo_das of frame b of the host stream x [C][T]: [D][N] float32"""
    return oracle.mimo_das(np.ascontiguousarray(x[:, b * N:]), off, frac, index, N)


def abs_taps(x, off, index, N, b):
    """S [D][N] (float64): sum over the summed channels of |x[o + i]| + |x[o + i + 1]| of frame b (gathered on the device:
    a cfg5 frame on 600 directions is 1.3 G taps)"""
    import torch
    idx = np.arange(x.shape[0]) if index is None else np.asarray(index, np.int64)
    ax = torch.from_numpy(np.abs(np.asarray(x)[idx].astype(np.float64))).cuda()
    pair = ax[:, :-1] + ax[:, 1:]                                           # [usable][T - 1]
    o = torch.from_numpy(off[:, idx].astype(np.int64)).cuda()[:, :, None] + b * N
    rows = torch.arange(len(idx), device="cuda")[None, :, None]
    ar = torch.arange(N, device="cuda")
    S = torch.empty((off.shape[0], N), dtype=torch.float64, device="cuda")
    step = max(1, (1 << 24) // (len(idx) * N))
    for d0 in range(0, off.shape[0], step):
        S[d0:d0 + step] = pair[rows, o[d0:d0 + step] + ar].sum(dim=1)
    return S.cpu().numpy()


def assert_within_bound(beam, ref, S, usable, what):
    err = np.abs(beam.astype(np.float64) - ref.astype(np.float64))
    bar = 6 * usable * EPS32 * S
    assert np.all(np.isfinite(beam)) and np.all(err <= bar), (what, float(np.max(err / np.maximum(bar, 1e-300))))


def assert_bits(beam, ref, what):
    assert beam.shape == ref.shape and np.array_equal(beam.view(np.uint32), ref.view(np.uint32)), (
        what, int(np.sum(beam.view(np.uint32) != ref.view(np.uint32))))


def power_of(beams, usable):
    """float64 power [..][D] of beams [..][D][N]: 3-tap high-pass (mimo.cpp:133-134), mean square over N * usable"""
    o = beams.astype(np.float64)
    ma = 0.5 * o[..., 1:-1] - 0.25 * (o[..., :-2] + o[..., 2:])
    return (ma * ma).sum(-1) / (o.shape[-1] * usable)


def assert_power_of_beams(power, beams, usable, what):
    ref = power_of(beams, usable)
    rel = float(np.max(np.abs(power.astype(np.float64) - ref) / ref))
    assert rel <= POWER_RTOL, (what, rel)


# ---- calls -------------------------------------------------------------------------------------------------------------
def beams_dev(w, x, nf):
    """bflk_beams_batch_dev of nf frames of the device stream x [C][T] -> device (beams [nf][count][N], power [nf][count]).
    Both outputs start as NaN: a sample no kernel writes fails every comparison, whatever an earlier call left in memory."""
    import torch
    count, N = w.n_directions()[2], w.cfg.frame_len
    beams = torch.full((nf, count, N), float("nan"), dtype=torch.float32, device=x.device)
    power = torch.full((nf, count), float("nan"), dtype=torch.float32, device=x.device)
    torch.cuda.synchronize()
    w.beams_batch_dev(x.data_ptr(), x.shape[1], nf, beams.data_ptr(), power.data_ptr())
    torch.cuda.synchronize()
    return beams, power


def beams_host(w, x, nf):
    beams, power = beams_dev(w, x, nf)
    beams, power = beams.cpu().numpy(), power.cpu().numpy()
    assert np.all(np.isfinite(beams)) and np.all(np.isfinite(power)), "a beam sample or a map entry was not written"
    return beams, power


def maps_host(w, x, nf):
    import torch
    out = torch.empty((nf, w.n_directions()[2]), dtype=torch.float32, device=x.device)
    torch.cuda.synchronize()
    w.power_map_batch_dev(x.data_ptr(), x.shape[1], nf, out.data_ptr())
    torch.cuda.synchronize()
    return out.cpu().numpy()


def white_noise(C_, T, seed):
    """[C][T] float32 white noise, T rounded up to even (the tiled kernels read float rows of even length); host, device"""
    import torch
    T += T & 1
    x = np.random.default_rng(seed).standard_normal((C_, T)).astype(np.float32)
    return x, torch.from_numpy(x).cuda()


# ---- the golden snapshot -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [1, 2, 3, 4, 0])
def test_snapshot_beams(oracle, golden, kernel):
    """The snapshot window as a one-frame stream of 1024 samples, 64 microphones, 16 x 16 directions over 180 degrees."""
    import bflk
    import torch
    g = golden["snapshot"]
    window = np.ascontiguousarray(g["window"])
    x = torch.from_numpy(window).cuda()
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    w.set_kernel(kernel)
    off, fr = w.tables()
    for index in (None, g["mask"]):
        w.set_channel_mask(index)
        beams, power = beams_host(w, x, 1)
        assert w.kernel_info()[0] == (kernel or 4)
        assert np.array_equal(power, maps_host(w, x, 1))
        das = oracle.mimo_das(window, off, fr, index)
        usable = 64 if index is None else len(index)
        if kernel in (1, 2, 3):
            assert_bits(beams[0], das, (kernel, index is None))
            if index is None:
                assert_bits(beams[0][g["das_sel"]], g["das"], (kernel, "compiled delay()"))
        else:
            assert_within_bound(beams[0], das, abs_taps(window, off, index, 256, 0), usable, kernel)
        assert_power_of_beams(power, beams, usable, kernel)
    w.close()


# ---- batches -------------------------------------------------------------------------------------------------------------
def check_batch(oracle, w, x_host, x, nf, kernels, frames, index, what):
    """kernels on nf frames: kernel_info, beams against the oracle on `frames`, power against the power-only call and
    against the beams"""
    total, first, count = w.n_directions()
    N = w.cfg.frame_len
    usable = x_host.shape[0] if index is None else len(index)
    off, fr = w.tables()
    off, fr = off[first:first + count], fr[first:first + count]
    refs = {b: das_ref(oracle, x_host, off, fr, index, N, b) for b in frames}
    bounds = {}
    for kernel in kernels:
        w.set_kernel(kernel)
        beams, power = beams_host(w, x, nf)
        assert w.kernel_info()[0] == kernel, (what, kernel)
        assert beams.shape == (nf, count, N)
        assert np.array_equal(power, maps_host(w, x, nf)), (what, kernel)
        assert_power_of_beams(power, beams, usable, (what, kernel))
        for b in frames:
            if kernel == 4:
                if b not in bounds:
                    bounds[b] = abs_taps(x_host, off, index, N, b)
                assert_within_bound(beams[b], refs[b], bounds[b], usable, (what, kernel, b))
            else:
                assert_bits(beams[b], refs[b], (what, kernel, b))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3"])
def test_config_batches(oracle, name):
    import bflk
    c = cases.CONFIGS[name]
    N, H = c["N"], c["H"]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
    x_host, x = white_noise(64 * c["nx"] * c["ny"], (B - 1) * N + H + N + 1, seed=3)
    check_batch(oracle, w, x_host, x, B, (1, 2, 3, 4), (0, B - 1), None, name)
    w.close()


def small_grid(N, H):
    import bflk
    return bflk.MIMOWorker(cases.origins(1, 1), 12, 10, 150.0, frame_len=N, history=H, window_len=H + N + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [64, 255, 256])
@pytest.mark.parametrize("N", [256, 258, 300, 512])
def test_frame_lengths_and_histories(oracle, N, H):
    """One to three blocks per frame, with heavily overlapping blocks at 258 and an odd history (staging parity)."""
    w = small_grid(N, H)
    x_host, x = white_noise(64, (B - 1) * N + H + N + 1, seed=N + H)
    check_batch(oracle, w, x_host, x, B, (1, 2, 3, 4), range(B), None, (N, H))
    w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["mask", "range", "mask+range"])
def test_mask_and_range(oracle, variant):
    """A ragged channel mask, and a direction range that starts inside a row of direction tiles (row 1, column 3)."""
    N, H = 300, 255
    w = small_grid(N, H)
    index = None
    if "mask" in variant:
        index = np.array([i for i in range(64) if i % 7 != 3], np.int32)[::-1].copy()   # ragged, and not in order
        w.set_channel_mask(index)
    if "range" in variant:
        w.set_direction_range(13, 71)
    x_host, x = white_noise(64, (B - 1) * N + H + N + 1, seed=11)
    check_batch(oracle, w, x_host, x, B, (1, 2, 3, 4), range(B), index, variant)
    w.close()


@pytest.mark.gpu
def test_cfg5_frame_on_a_few_tiles(oracle):
    """cfg5 (4096 samples = 17 blocks a frame, 512 microphones): one frame, directions 25 637 .. 26 236 of the 256 x 256
    grid (a range that starts inside a tile row)."""
    import bflk
    c = cases.CONFIGS["cfg5"]
    N, H = c["N"], c["H"]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"], frame_len=N, history=H,
                        window_len=c["W"])
    w.set_direction_range(100 * 256 + 37, 600)
    x_host, x = white_noise(512, N + H + 1, seed=5)
    check_batch(oracle, w, x_host, x, 1, (1, 2, 3, 4), (0,), None, "cfg5")
    w.close()


# ---- every compiled variant of the register-tiled kernel --------------------------------------------------------------------
def max_warps(case):
    return 12 if case.kernel == 2 and case.mode != 0 and case.nch == 7 else 16


@pytest.mark.gpu
@pytest.mark.parametrize("case", VARIANT_CASES, ids=lambda c: c.name)
def test_tile_variant_beams(oracle, case, monkeypatch):
    """test_tile_variants' LUT for each compiled variant: the latency shape (automatic for 7 frames) and the throughput
    shape (forced warps per CTA) give the same beams, bit-exact (kernel 2) or within the bound (kernel 4); kernel 4 also on
    single frames with the channels split across clusters of 2 and 4 CTAs: deterministic and within the bound."""
    import torch
    off, frac, index = variant_lut(case)
    first, count = dir_range(case)
    off_r, frac_r = off[first:first + count], frac[first:first + count]
    x_host, x = white_noise(case.C, (B - 1) * case.N + case.H + case.N + 1, seed=1)
    refs = [das_ref(oracle, x_host, off_r, frac_r, index, case.N, b) for b in range(B)]
    S = [abs_taps(x_host, off_r, index, case.N, b) for b in range(B)] if case.kernel == 4 else None
    usable = len(index)

    def check(beams, bs, what):
        for i, b in enumerate(bs):
            if case.kernel == 2:
                assert_bits(beams[i], refs[b], (case.name, what, b))
            else:
                assert_within_bound(beams[i], refs[b], S[b], usable, (case.name, what, b))

    got = {}
    for shape, env in (("latency", {}), ("throughput", {"BFLK_TILE_WARPS": max_warps(case)})):
        w = make_beamformer(case, off, frac, index, monkeypatch, env)
        beams, power = beams_host(w, x, B)
        assert w.kernel_info() == (case.kernel, case.spans[case.mode], case.nch), shape
        assert np.array_equal(power, maps_host(w, x, B)), shape
        assert_power_of_beams(power, beams, usable, (case.name, shape))
        check(beams, range(B), shape)
        got[shape] = beams
        w.close()
    assert np.array_equal(got["latency"], got["throughput"])

    if case.kernel == 4:
        for split in (2, 4):
            w = make_beamformer(case, off, frac, index, monkeypatch, {"BFLK_LAT_SPLIT": split})
            w.set_channel_split(True)
            for b in (0, B - 1):
                xb = x[:, b * case.N:].contiguous()
                b0, p0 = beams_host(w, xb, 1)
                b1, p1 = beams_host(w, xb, 1)
                assert np.array_equal(b0, b1) and np.array_equal(p0, p1), (case.name, split, b)
                assert np.array_equal(p0, maps_host(w, xb, 1)), (case.name, split, b)
                check(b0, [b], ("split", split))
            w.close()
    del x
    torch.cuda.empty_cache()


# ---- FIR interpolation ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 1])
def test_fir_beams(golden, kernel):
    """With the reference's 101 x 8 FIR table the generic kernel's FIR sums come back, and they square to its map."""
    import bflk
    coeffs = golden["fir"]["coeffs"]
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    w.set_kernel(kernel)
    w.set_fir(coeffs)
    N, H = 256, 256
    x_host, x = white_noise(64, (B - 1) * N + H + N + 1 + coeffs.shape[1] - 2, seed=7)
    beams, power = beams_host(w, x, B)
    assert w.kernel_info()[0] == 1
    assert np.array_equal(power, maps_host(w, x, B))
    assert_power_of_beams(power, beams, 64, kernel)
    w.set_fir(None)
    plain, _ = beams_host(w, x, B)
    assert not np.array_equal(plain, beams)                 # the FIR sums are not the 2-tap ones
    w.close()


# ---- past the grid limits ------------------------------------------------------------------------------------------------------
B_BIG = 2 * 32768 + 35
SLICE = 16384
LINE = np.array([[0.02 * (k - 3.5), 0.0, 0.0] for k in range(8)], np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("N,kernels", [(256, (1, 2, 3, 4)), (512, (1, 2, 3, 4))])
def test_large_batch_equals_sliced_calls(N, kernels):
    """65 571 frames on an 8-microphone line array: past the 32 768-pair slabs of the staged kernels and the 65 535-frame
    slabs of the generic kernel, beams and power carry the bits of calls of at most 16 384 frames."""
    import bflk
    import torch
    H = 256
    T = (B_BIG - 1) * N + H + N + 1
    T += T & 1
    g = torch.Generator(device="cuda").manual_seed(N)
    x = torch.randn((8, T), generator=g, device="cuda", dtype=torch.float32)
    for kernel in kernels:
        w = bflk.Beamformer(n_channels=8, frame_len=N, history=H, window_len=H + N + 1)
        w.set_geometry(LINE)
        w.set_grid_fov(6, 6, 120.0)
        w.set_kernel(kernel)
        beams, power = beams_dev(w, x, B_BIG)
        assert w.kernel_info()[0] == kernel
        assert bool(torch.isfinite(beams).all()) and bool(torch.isfinite(power).all()), kernel
        for b0 in range(0, B_BIG, SLICE):
            nb = min(SLICE, B_BIG - b0)
            t1 = b0 * N + (nb - 1) * N + H + N + 1
            xs = x[:, b0 * N:t1 + ((t1 - b0 * N) & 1)].contiguous()
            sb, sp = beams_dev(w, xs, nb)
            assert torch.equal(sb, beams[b0:b0 + nb]) and torch.equal(sp, power[b0:b0 + nb]), (kernel, b0)
            del xs, sb, sp
        pw = power[:64].cpu().numpy()
        assert_power_of_beams(pw, beams[:64].cpu().numpy(), 8, kernel)
        del beams, power
        w.close()
        torch.cuda.empty_cache()
    del x
    torch.cuda.empty_cache()


# ---- streaming sessions ----------------------------------------------------------------------------------------------------------
N_S, H_S, W_S = 256, 256, 1024
B_S = 40


def session_stream(n_samples, seed):
    from bflk import synth
    s = synth.make_stream(synth.tile_geometry(cases.origins(1, 1)), n_samples, seed=seed)
    s *= np.linspace(0.5, 1.5, n_samples, dtype=np.float32)[None, :]          # no two frames alike
    return np.ascontiguousarray(s)


def quantised(stream):
    """the floats the wire rows of stream carry (int32 / 2^23 is exact)"""
    return (np.rint(stream.astype(np.float64) * 8388608.0) / 8388608.0).astype(np.float32)


def run_session(w, wire, data, n_samples, rng, max_frames=4):
    """Pushes samples [0, n_samples) in random pieces (1 sample to more than a frame) into a session of max_frames frames
    and takes the ready frames through randomly interleaved stream_beams and stream_power_maps calls; returns, per frame
    in the order the calls returned them, (frame, beams or None, power)."""
    w.stream_open(max_frames)
    got = []

    def take(k):
        if rng.random() < 0.5:
            f, bm, p = w.stream_beams(k)
            got.extend((f + i, bm[i], p[i]) for i in range(len(p)))
        else:
            f, p = w.stream_power_maps(k)
            got.extend((f + i, None, p[i]) for i in range(len(p)))

    t = 0
    while t < n_samples:
        while w.stream_status()[2] > 1:
            take(int(rng.integers(1, max_frames + 1)))
        n = int(rng.choice([rng.integers(1, 8), rng.integers(8, N_S), rng.integers(N_S, 2 * N_S + 80)]))
        n = min(n, n_samples - t)
        if wire:
            w.stream_push_i32(data[t:t + n])
        else:
            w.stream_push(data[:, t:t + n])
        t += n
        if rng.random() < 0.5:
            take(int(rng.integers(1, max_frames + 1)))
    while w.stream_status()[2] > 0:
        take(int(rng.integers(1, max_frames + 1)))
    assert w.stream_status() == (n_samples, B_S, 0, 0)
    w.stream_close()
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["float", "wire"])
@pytest.mark.parametrize("kernel", [0, 1, 2, 3, 4])
def test_session_beams_equal_the_batch(source, kernel):
    """40 frames pushed in random pieces into a session of 4 frames (the ring wraps about seven times; backlogs, single
    frames and frames across the wrap), taken by interleaved beams and maps calls: frames 0..39 in order, the beams carry
    the bits of bflk_beams_batch_dev over the same samples, the power those of the power-only batch."""
    import bflk
    import torch
    from bflk import synth
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    w.set_kernel(kernel)
    T = (B_S - 1) * N_S + N_S + H_S + 1
    stream = session_stream((B_S - 1) * N_S + W_S, seed=21)
    if source == "wire":
        data = synth.to_wire_i32(stream)
        stream = quantised(stream)
    else:
        data = stream
    x = torch.from_numpy(stream).cuda()
    want_beams, want_power = beams_host(w, x, B_S)
    assert np.array_equal(want_power, maps_host(w, x, B_S))
    got = run_session(w, source == "wire", data, T, np.random.default_rng(77 + kernel), 4)
    assert [f for f, _, _ in got] == list(range(B_S))
    n_beams = 0
    for f, bm, p in got:
        assert np.array_equal(p, want_power[f]), f
        if bm is not None:
            assert np.array_equal(bm, want_beams[f]), f
            n_beams += 1
    assert 0 < n_beams < B_S
    if kernel:
        assert w.kernel_info()[0] == kernel
    w.close()


@pytest.mark.gpu
def test_session_beams_overrun_and_targets():
    """Frames overwritten before they were taken are skipped and counted as by the maps calls; after a one-frame beams call
    bflk_targets with a NULL map uses that frame's map, after a three-frame call it has none."""
    import bflk
    import torch
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    T = 10 * N_S
    stream = session_stream(T + W_S, seed=5)
    want_beams, want_power = beams_host(w, torch.from_numpy(stream).cuda(), 12)
    status = []
    for beams in (False, True):
        w.stream_open(4)
        for t in range(0, T, N_S):
            w.stream_push(stream[:, t:t + N_S])
        status.append(w.stream_status())
        next_frame = status[-1][1]
        if beams:
            f, bm, p = w.stream_beams(2)
            assert f == next_frame and np.array_equal(bm, want_beams[f:f + 2]) and np.array_equal(p, want_power[f:f + 2])
        else:
            f, p = w.stream_power_maps(2)
            assert f == next_frame and np.array_equal(p, want_power[f:f + 2])
        status.append(w.stream_status())
    assert status[0] == status[2] and status[1] == status[3] and status[0][3] > 0

    def targets(power=None):
        out = (bflk.Target * 16)()
        k = C.c_int32()
        src = None if power is None else np.ascontiguousarray(power, np.float32)
        w._check(w._L.bflk_targets(w._h, None if src is None else src.ctypes.data, 16, 0.05, out, C.byref(k)))
        return [(t.direction, t.power, t.probability) for t in out[:k.value]]

    w.stream_open(8)
    w.stream_push(stream[:, :N_S + H_S + 1])
    f, bm, p = w.stream_beams(4)
    assert (f, len(p)) == (0, 1) and np.array_equal(bm[0], want_beams[0])
    assert targets() == targets(p[0])
    w.stream_push(stream[:, N_S + H_S + 1:4 * N_S + H_S + 1])
    f, bm, p = w.stream_beams(4)
    assert (f, len(p)) == (1, 3)
    with pytest.raises(bflk.BflkError) as e:
        targets()
    assert e.value.code == BFLK_ERR_STATE
    w.close()


TOLERANCE = 64 << 20      # as in test_handle_lifetime: far below what a cycle allocates, not derived from a measurement


def _free():
    import torch
    torch.cuda.synchronize(0)
    return torch.cuda.mem_get_info(0)[0]


@pytest.mark.gpu
def test_session_beams_return_their_memory():
    """Three open / push / beams / close cycles on one handle, and three handles destroyed with a session open after a beams
    call, each give their device memory back."""
    import bflk
    c = cases.CONFIGS["cfg3"]
    from bflk import synth
    stream = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), 3 * N_S + H_S + 1)
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])

    def open_push_beams(h):
        h.stream_open(1024)
        h.stream_push(stream)
        assert len(h.stream_beams(8)[2]) == 3
        return _free()

    def close_cycle():
        used = open_push_beams(w)
        w.stream_close()
        return used

    def destroy_cycle():
        h = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
        used = open_push_beams(h)
        h.close()
        return used

    for cycle in (close_cycle, destroy_cycle):
        after = []
        for _ in range(3):
            before = _free()
            used = cycle()
            assert before - used > 1 << 30, "the cycle must allocate over 1 GiB"
            after.append(_free())
        drift = [after[0] - a for a in after[1:]]
        assert all(d <= TOLERANCE for d in drift), (cycle.__name__, drift)
    w.close()


@pytest.mark.gpu
def test_beams_argument_checks():
    """Null or misaligned beams, and the power-only call's own checks, return BFLK_ERR_INVALID; a session call without a
    session BFLK_ERR_STATE."""
    import bflk
    import torch
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    x = torch.zeros((64, 1024), dtype=torch.float32, device="cuda")
    buf = torch.zeros(256 * 256 + 2, dtype=torch.float32, device="cuda")
    p = torch.zeros(256, dtype=torch.float32, device="cuda")
    for beams_ptr, n_samples, nf in ((0, 1024, 1), (buf.data_ptr() + 4, 1024, 1), (buf.data_ptr(), 512, 1),
                                     (buf.data_ptr(), 1024, 0)):
        with pytest.raises(bflk.BflkError) as e:
            w.beams_batch_dev(x.data_ptr(), n_samples, nf, beams_ptr, p.data_ptr())
        assert e.value.code == BFLK_ERR_INVALID
    with pytest.raises(bflk.BflkError) as e:
        w.beams_batch_dev(x.data_ptr(), 1024, 1, buf.data_ptr(), 0)
    assert e.value.code == BFLK_ERR_INVALID
    with pytest.raises(bflk.BflkError) as e:
        w.stream_beams(1)
    assert e.value.code == BFLK_ERR_STATE
    w.close()
