"""Streaming sessions (bflk_stream_*): samples pushed as they arrive into a device-resident history, a power map for every
frame.  Frame b of a session is frame b of bflk_power_map_batch over everything pushed since bflk_stream_open, so every
map a session returns must carry the bits of that batch, however the samples were cut into pushes and however the frames
were grouped into maps calls."""
import ctypes as C

import numpy as np
import pytest

import cases

N, H, W = 256, 256, 1024
BFLK_ERR_INVALID, BFLK_ERR_STATE = -1, -2


def test_null_handle_is_invalid():
    import bflk
    L = bflk.load_library()
    buf = np.zeros(4096, np.float32)
    i64, i32 = C.c_int64(), C.c_int32()
    calls = {
        "bflk_stream_open": (None, 4),
        "bflk_stream_close": (None,),
        "bflk_stream_push": (None, buf.ctypes.data, 1),
        "bflk_stream_push_i32": (None, buf.ctypes.data, 1),
        "bflk_stream_power_maps": (None, 1, buf.ctypes.data, C.byref(i64), C.byref(i32)),
        "bflk_stream_discard": (None, 0),
        "bflk_stream_status": (None, C.byref(i64), C.byref(i64), C.byref(i32), C.byref(i64)),
        "bflk_stream_window": (None, 0),
    }
    assert sorted(calls) == sorted(s for s in bflk.SYMBOLS if s.startswith("bflk_stream_"))
    for name, args in calls.items():
        assert getattr(L, name)(*args) == BFLK_ERR_INVALID, name


# ---- helpers --------------------------------------------------------------------------------------------------------
def _tail(w):
    """samples a frame reads beyond its own N"""
    return H + 1 + (w.fir_taps - 2 if getattr(w, "fir_taps", 0) else 0)


def _stream(C_, n_samples, seed=0):
    from bflk import synth
    xyz = synth.tile_geometry(cases.origins(1, 1) if C_ == 64 else cases.origins(4, 2))
    s = synth.make_stream(xyz, n_samples, seed=seed)
    s *= np.linspace(0.5, 1.5, n_samples, dtype=np.float32)[None, :]          # no two frames alike
    return np.ascontiguousarray(s)


def _quantised(stream):
    """the floats the wire rows of stream carry (int32 / 2^23 is exact)"""
    return (np.rint(stream.astype(np.float64) * 8388608.0) / 8388608.0).astype(np.float32)


def _push(w, source, data, t0, t1):
    if source == "wire":
        w.stream_push_i32(data[t0:t1])
    else:
        w.stream_push(data[:, t0:t1])


def _run_session(w, source, data, n_samples, rng, max_frames):
    """Pushes samples [0, n_samples) in random pieces (1 sample to more than a frame) and maps between the pushes with
    random max_frames, never letting a frame be overwritten unmapped; returns the first frames and the maps, in order."""
    w.stream_open(max_frames)
    firsts, maps = [], []

    def maps_call(k):
        f, m = w.stream_power_maps(k)
        if len(m):
            firsts.extend(range(f, f + len(m)))
            maps.append(m)

    t = 0
    while t < n_samples:
        # at most one ready frame left unmapped before a push: the unmapped samples then fit the ring of 4 frames
        while w.stream_status()[2] > 1:
            maps_call(int(rng.integers(1, max_frames + 1)))
        n = int(rng.choice([rng.integers(1, 8), rng.integers(8, N), rng.integers(N, 2 * N + 80)]))
        n = min(n, n_samples - t)
        _push(w, source, data, t, t + n)
        t += n
        if rng.random() < 0.5:
            maps_call(int(rng.integers(1, max_frames + 1)))
    while w.stream_status()[2] > 0:
        maps_call(int(rng.integers(1, max_frames + 1)))
    pushed, next_frame, ready, skipped = w.stream_status()
    assert (pushed, ready, skipped) == (n_samples, 0, 0)
    return firsts, np.concatenate(maps)


def _worker(kernel, variant, golden):
    import bflk
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    w.set_kernel(kernel)
    if variant == "range":
        w.set_direction_range(37, 150)
    elif variant == "mask":
        w.set_channel_mask(np.sort(np.random.default_rng(11).choice(64, 48, replace=False)))
    elif variant == "fir":
        coeffs = golden["fir"]["coeffs"]
        w.set_fir(coeffs)
        w.fir_taps = coeffs.shape[1]
    return w


B = 40
CASES = [(k, v) for v in ("plain", "range", "mask") for k in (0, 1, 2, 3, 4)] + [(0, "fir"), (1, "fir")]


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["float", "wire"])
@pytest.mark.parametrize("kernel,variant", CASES)
def test_session_maps_equal_the_batch(golden, source, kernel, variant):
    """40 frames pushed in random pieces into a session of 4 frames (the ring wraps about seven times), mapped by random
    maps calls: the maps run 0..39 without a gap and carry the bits of one batch over the whole stream.  Wire pushes
    give the bits of the wire batch and of a float session over the floats the wire rows carry."""
    from bflk import synth
    w = _worker(kernel, variant, golden)
    T = (B - 1) * N + N + _tail(w)                       # what the session is given: the samples of B frames
    stream = _stream(64, (B - 1) * N + W)                # the batch's rows: an even length, as the tiled kernels need
    rng = np.random.default_rng(1000 + 10 * kernel + len(variant))
    if source == "wire":
        wire = synth.to_wire_i32(stream)
        want = w.power_map_batch_i32(wire, B)
        firsts, got = _run_session(w, "wire", wire, T, rng, 4)
        _, got_float = _run_session(w, "float", _quantised(stream), T, rng, 4)
        assert np.array_equal(got_float, want)
    else:
        want = w.power_map_batch(stream, B)
        firsts, got = _run_session(w, "float", stream, T, rng, 4)
    assert firsts == list(range(B))
    assert got.shape == want.shape and np.all(np.isfinite(got)) and got.min() > 0
    assert np.array_equal(got, want)
    if kernel:
        assert w.kernel_info()[0] == kernel
    w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [4, 2])
def test_cfg3_single_frames_and_catch_up(kernel):
    """cfg3 (512 channels, 32 x 32 directions): one frame per call (latency shape) and a 64-frame backlog in one call
    (throughput shape) carry the bits of the batch.  With the channel split on, the bits depend on the call's size, so
    each maps call is compared with a batch of the same frames."""
    import bflk
    c = cases.CONFIGS["cfg3"]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
    w.set_kernel(kernel)
    n_single, n_catch = 8, 64
    nf = n_single + n_catch
    T = (nf - 1) * N + N + H + 1                        # pushed: the samples of nf frames
    stream = _stream(512, (nf - 1) * N + W, seed=3)     # the batches' rows: an even length, as the tiled kernels need
    want = w.power_map_batch(stream, nf)
    for split in (False, True):
        w.set_channel_split(split)
        w.stream_open(n_catch)
        got = []
        t = 0
        for b in range(n_single):
            t1 = b * N + N + H + 1
            w.stream_push(stream[:, t:t1])
            t = t1
            f, m = w.stream_power_maps(4)
            assert (f, len(m)) == (b, 1)
            got.append(m)
        while t < T:
            t1 = min(T, t + 3 * N)
            w.stream_push(stream[:, t:t1])
            t = t1
        assert w.stream_status() == (T, n_single, n_catch, 0)
        f, m = w.stream_power_maps(n_catch)
        assert (f, len(m)) == (n_single, n_catch)
        got.append(m)
        if not split:
            assert np.array_equal(np.concatenate(got), want)
        else:
            for f0, g in zip(list(range(n_single)) + [n_single], got):
                k = len(g)
                assert np.array_equal(g, w.power_map_batch(stream[:, f0 * N:f0 * N + (k - 1) * N + W], k)), f0
        w.stream_close()
    w.close()


@pytest.mark.gpu
def test_overrun_skips_frames_and_never_blocks():
    import bflk
    w = _worker(0, "plain", None)
    cap = -(-(4 * N + H + 1) // N) * N                  # max_frames = 4: room for 4 frames and the last one's tail
    T = 10 * N
    stream = _stream(64, T + W, seed=5)
    want = w.power_map_batch(stream, 12)
    w.stream_open(4)
    with pytest.raises(bflk.BflkError) as e:
        w.stream_push(stream[:, :cap + 1])                # more than the ring holds
    assert e.value.code == BFLK_ERR_INVALID
    for t in range(0, T, N):
        w.stream_push(stream[:, t:t + N])
    next_frame = -(-(T - cap) // N)
    ready = (T - N - H - 1) // N + 1 - next_frame
    assert w.stream_status() == (T, next_frame, ready, next_frame)
    with pytest.raises(bflk.BflkError) as e:
        w.stream_window(next_frame - 1)                   # skipped: no longer in the ring
    assert e.value.code == BFLK_ERR_STATE
    with pytest.raises(bflk.BflkError) as e:
        w.stream_window(next_frame + ready)               # not fully pushed
    assert e.value.code == BFLK_ERR_STATE
    f, m = w.stream_power_maps(2)
    assert f == next_frame and np.array_equal(m, want[f:f + 2])
    w.stream_discard(1)
    assert w.stream_status() == (T, next_frame + ready - 1, 1, next_frame + ready - 3)
    f, m = w.stream_power_maps(4)
    assert f == next_frame + ready - 1 and np.array_equal(m, want[f:f + 1])
    assert w.stream_power_maps(4)[1].shape[0] == 0
    w.close()


def _miso_case(w, stream, b, th, ph):
    win = np.ascontiguousarray(stream[:, b * N:b * N + W])
    a0, p0 = w.miso(th, ph, win)
    a1, p1 = w.miso(th, ph, None)
    assert np.array_equal(a0, a1) and np.array_equal(p0, p1)
    pth, pph = th[:3], ph[:3]
    m0 = w.monopulse(pth, pph, win, spread=0.05, theta_limit=1.2)
    m1 = w.monopulse(pth, pph, None, spread=0.05, theta_limit=1.2)
    for x, y in zip(m0, m1):
        assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("fir", [False, True])
def test_miso_and_monopulse_on_a_session_frame(golden, fir):
    """After stream_window(b), MISO and monopulse with window=None read frame b in the ring (here across the ring's wrap)
    with the bits of the same calls on stream[:, bN : bN + W].  Once the frame is overwritten they have no window."""
    import bflk
    w = _worker(0, "fir" if fir else "plain", golden)
    th, ph = np.deg2rad([20.0, 45.0, 0.0, 63.0, 30.0]), np.deg2rad([30.0, 200.0, 0.0, 310.0, 90.0])
    stream = _stream(64, 16 * N + W, seed=7)
    w.stream_open(4)
    for t in range(0, 8 * N, N):
        w.stream_push(stream[:, t:t + N])
    b = 5                                                # the ring holds samples from 512 on: frame 5 crosses its wrap
    w.stream_window(b)
    _miso_case(w, stream, b, th, ph)
    w.stream_push(stream[:, 8 * N:9 * N])              # frame 5 is still held
    _miso_case(w, stream, b, th, ph)
    for t in range(9 * N, 12 * N, N):                  # ... and now overwritten
        w.stream_push(stream[:, t:t + N])
    with pytest.raises(bflk.BflkError) as e:
        w.miso(th, ph, None)
    assert e.value.code == BFLK_ERR_INVALID
    w.set_window(np.ascontiguousarray(stream[:, 2 * N:2 * N + W]))
    assert np.array_equal(w.miso(th, ph, None)[0], w.miso(th, ph, np.ascontiguousarray(stream[:, 2 * N:2 * N + W]))[0])
    w.stream_window(9)                                   # the session window replaces it; close forgets it
    _miso_case(w, stream, 9, th, ph)
    w.stream_close()
    with pytest.raises(bflk.BflkError) as e:
        w.miso(th, ph, None)
    assert e.value.code == BFLK_ERR_INVALID
    w.close()


def _targets(w, power=None):
    """bflk_targets; power None: the map left on the device"""
    import bflk
    out = (bflk.Target * 16)()
    k = C.c_int32()
    src = None if power is None else np.ascontiguousarray(power, np.float32)
    w._check(w._L.bflk_targets(w._h, None if src is None else src.ctypes.data, 16, 0.05, out, C.byref(k)))
    return [(t.direction, t.power, t.probability) for t in out[:k.value]]


def _heatmap(w, power=None):
    """bflk_heatmap; power None: the map left on the device"""
    n = w.n_directions()[2]
    heat = np.zeros(n, np.uint8)
    arg, mx = C.c_int32(), C.c_float()
    src = None if power is None else np.ascontiguousarray(power, np.float32)
    w._check(w._L.bflk_heatmap(w._h, None if src is None else src.ctypes.data, n, heat.ctypes.data, C.byref(arg), C.byref(mx)))
    return heat.tobytes(), arg.value, mx.value


@pytest.mark.gpu
def test_single_frame_map_stays_on_the_device():
    import bflk
    w = _worker(0, "plain", None)
    stream = _stream(64, 8 * N + W, seed=9)
    w.stream_open(8)
    w.stream_push(stream[:, :N + H + 1])
    f, m = w.stream_power_maps(4)
    assert (f, len(m)) == (0, 1)
    assert _targets(w) == _targets(w, m[0]) and _heatmap(w) == _heatmap(w, m[0])
    w.stream_push(stream[:, N + H + 1:4 * N + H + 1])
    f, m = w.stream_power_maps(4)
    assert (f, len(m)) == (1, 3)
    with pytest.raises(bflk.BflkError) as e:
        _targets(w)
    assert e.value.code == BFLK_ERR_STATE
    with pytest.raises(bflk.BflkError) as e:
        _heatmap(w)
    assert e.value.code == BFLK_ERR_INVALID              # bflk_heatmap's code for "no map of that size left"
    w.close()


@pytest.mark.gpu
def test_session_interleaved_with_other_calls():
    """Session calls between host batches, a submitted host batch (in flight across a push and a maps call), an overlapped
    device batch and MISO on one handle give the results of the same calls on separate handles."""
    import torch
    th, ph = np.deg2rad([20.0, 45.0, 63.0]), np.deg2rad([30.0, 200.0, 310.0])
    live = _stream(64, 24 * N + W, seed=13)
    other = _stream(64, 15 * N + W, seed=17)
    pinned = torch.from_numpy(other).pin_memory()
    dev = torch.from_numpy(other).cuda()
    torch.cuda.synchronize()
    cuts = [0, 700, 1500, 2600, 3300, 4400, 5500, 6400]

    def session_step(w, k):
        w.stream_push(live[:, cuts[k]:cuts[k + 1]])
        return w.stream_power_maps(1 + k % 3)

    class Others:
        def __init__(self, w):
            self.w, self.pending = w, None

        def step(self, k):
            w = self.w
            if k == 0:
                return w.power_map_batch(other, 16)
            if k == 1:
                self.pending = torch.zeros((16, 256), dtype=torch.float32).pin_memory()
                w.power_map_batch_submit_ptr(pinned.data_ptr(), pinned.shape[1], 16, self.pending.data_ptr())
                return None
            if k == 2:
                w.power_map_batch_wait()
                st = torch.cuda.Stream()                 # a caller's stream (0 would name the handle's own)
                with torch.cuda.stream(st):
                    res = torch.zeros((16, 256), dtype=torch.float32, device="cuda")
                    w.power_map_batch_dev_submit(dev.data_ptr(), dev.shape[1], 16, res.data_ptr(), st.cuda_stream)
                    w.power_map_batch_dev_join(st.cuda_stream)
                    out = res.cpu().numpy()
                return self.pending.numpy().copy(), out
            if k == 3:
                return w.miso(th, ph, np.ascontiguousarray(other[:, :W]))
            return None

    one = _worker(0, "plain", None)
    one.stream_open(6)
    one_others = Others(one)
    together_maps, together_other = [], []
    for k in range(len(cuts) - 1):
        together_other.append(one_others.step(k))
        together_maps.append(session_step(one, k))    # k == 1: while the submitted batch is in flight
    alone_s, alone_o = _worker(0, "plain", None), _worker(0, "plain", None)
    alone_s.stream_open(6)
    apart_maps = [session_step(alone_s, k) for k in range(len(cuts) - 1)]
    apart_others = Others(alone_o)
    apart_other = [apart_others.step(k) for k in range(len(cuts) - 1)]
    assert sum(len(m) for _, m in apart_maps) >= 8
    for (f0, m0), (f1, m1) in zip(together_maps, apart_maps):
        assert f0 == f1 and np.array_equal(m0, m1)
    for x, y in zip(together_other, apart_other):
        if isinstance(x, tuple):
            assert all(np.array_equal(a, b) for a, b in zip(x, y))
        else:
            assert (x is None and y is None) or np.array_equal(x, y)
    for w in (one, alone_s, alone_o):
        w.close()


# ---- nothing leaks ---------------------------------------------------------------------------------------------------
TOLERANCE = 64 << 20      # as in test_handle_lifetime: far below what a cycle allocates, not derived from a measurement


def _free():
    import torch
    torch.cuda.synchronize(0)
    return torch.cuda.mem_get_info(0)[0]


def _cycle_drift(cycle):
    after = []
    for _ in range(3):
        before = _free()
        used = cycle()
        assert before - used > 1 << 30, "the cycle must allocate over 1 GiB"
        after.append(_free())
    return [after[0] - a for a in after[1:]]


@pytest.mark.gpu
def test_sessions_return_their_memory():
    """Three open / push / map / close cycles on one handle, and three handles destroyed with a session open, each give
    their device memory back (a cfg3 session of 1024 frames holds about 1.6 GB)."""
    import bflk
    c = cases.CONFIGS["cfg3"]
    stream = _stream(512, 3 * N + H + 1, seed=19)
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])

    def open_push_map(h):
        h.stream_open(1024)
        h.stream_push(stream)
        assert len(h.stream_power_maps(8)[1]) == 3
        h.stream_window(1)
        return _free()

    def close_cycle():
        used = open_push_map(w)
        w.stream_close()
        return used

    def destroy_cycle():
        h = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
        used = open_push_map(h)
        h.close()
        return used

    for cycle in (close_cycle, destroy_cycle):
        drift = _cycle_drift(cycle)
        print(f"{cycle.__name__}: free memory lost after cycles 2, 3 relative to cycle 1: {drift} bytes")
        assert all(d <= TOLERANCE for d in drift), drift
    w.close()
