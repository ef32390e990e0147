"""Power maps past the CUDA grid limits and at the edges of history and stream length, against a float64 restatement of
the map (power_ref).

Large batches: 65 571 frames (2 x 32 768 + 35) in one call cross the 32 768-pair slabs of the packing, tiled and
lane-broadcast kernels, the 65 535-frame slabs of the generic kernel, and the 65 535 blocks of grid.y that the finalize
kernels (frames longer than one block) and the multi-GPU assembly cover with grid-stride loops.  An 8-element line array keeps such a stream near 1 GB.  Every large call must give
the bits of the same frames mapped in calls of at most 16 384 frames.

Edges: histories other than 256 (odd ones flip the parity of the tiled kernel's staging origin), frames shorter than one
block and up to four blocks long, streams exactly as long as the last frame needs (its last tap is the stream's last
sample), and caller tables whose offsets span exactly [0, H] with fractions 0 and just below 1.  The automatic kernel
must meet the bar everywhere; a kernel chosen explicitly either meets it or refuses the call with BFLK_ERR_STATE."""
import numpy as np
import pytest

import cases

POWER_RTOL = 1e-4
ERR_STATE = -2

B_BIG = 2 * 32768 + 35        # > 32 768 block pairs and > 65 535 frames in one call
SLICE = 16384                 # frames per call of the reference concatenation
LINE = np.array([[0.02 * (k - 3.5), 0.0, 0.0] for k in range(8)], np.float32)   # 8 microphones, 2 cm apart
H_BIG = 256


def power_ref(stream, off, frac, index, N, frames):
    """float64 power maps [len(frames)][D] of frames `frames` (frame b starts at sample b * N) of stream [C][T] float32,
    for tables off / frac [D][C], channels `index` (None: all) in order:
    out[i] = sum_c f x[o + i] + (1 - f) x[o + i + 1] for i < N; MA_i = 0.5 out[i] - 0.25 (out[i - 1] + out[i + 1]) for
    i in [1, N - 2]; power = sum MA^2 / (N * usable).  A read past the end of the stream raises IndexError."""
    stream = np.asarray(stream)
    idx = np.arange(stream.shape[0]) if index is None else np.asarray(index, np.int64)
    taps = off[:, idx].astype(np.int64)[:, :, None] + np.arange(N)                # [D][usable][N]
    f = frac[:, idx].astype(np.float64)[:, :, None]
    rows = idx[None, :, None]
    maps = []
    for b in frames:
        x0 = stream[rows, b * N + taps].astype(np.float64)
        x1 = stream[rows, b * N + taps + 1].astype(np.float64)
        out = (f * x0 + (1.0 - f) * x1).sum(axis=1)
        ma = 0.5 * out[:, 1:-1] - 0.25 * (out[:, :-2] + out[:, 2:])
        maps.append((ma * ma).sum(axis=1) / (N * len(idx)))
    return np.array(maps)


def rel_err(a, b):
    return float(np.max(np.abs(np.asarray(a, np.float64) - b) / np.abs(b)))


def assert_meets_bar(p, ref, what):
    assert rel_err(p, ref) <= POWER_RTOL, (what, rel_err(p, ref))
    assert int(np.argmax(p)) == int(np.argmax(ref)), what


def ragged_mask(C):
    return np.array([i for i in range(C) if i % 7 != 3], np.int32)


# ---- the reference itself (no GPU) ---------------------------------------------------------------------------------------
def test_power_ref_matches_oracle(oracle, golden):
    from bflk import synth
    g = golden["snapshot"]
    xyz = oracle.create_antenna()
    off, fr = oracle.mimo_lut(xyz, 16, 16, 180.0)
    ref = power_ref(g["window"], off, fr, None, 256, [0])[0]
    assert rel_err(oracle.mimo_update(g["window"], off, fr), ref) <= 1e-5
    assert rel_err(g["power"], ref) <= 1e-5
    ref_m = power_ref(g["window"], off, fr, g["mask"], 256, [0])[0]
    assert rel_err(oracle.mimo_update(g["window"], off, fr, index=g["mask"]), ref_m) <= 1e-5
    mask = ragged_mask(64)
    for N in (100, 258, 512):
        for H in (64, 255):
            B, W = 3, H + N + 1
            stream = synth.make_stream(xyz, (B - 1) * N + W)          # tight: the last frame reads the last sample
            off, fr = oracle.mimo_lut(xyz, 12, 10, 150.0, H)
            ref = power_ref(stream, off, fr, mask, N, range(B))
            for b in range(B):
                po = oracle.mimo_update(np.ascontiguousarray(stream[:, b * N:b * N + W]), off, fr, index=mask, n=N)
                assert rel_err(po, ref[b]) <= 1e-5, (N, H, b)
    with pytest.raises(IndexError):
        power_ref(stream[:, :-1], off, fr, mask, N, [B - 1])           # one sample short


# ---- large batches (GPU) ---------------------------------------------------------------------------------------------------
def line_array(N, kernel=0):
    import bflk
    w = bflk.Beamformer(n_channels=8, frame_len=N, history=H_BIG, window_len=H_BIG + N + 1)
    w.set_geometry(LINE)
    w.set_grid_fov(6, 6, 120.0)
    w.set_kernel(kernel)
    return w


def even_samples(B, N, H=H_BIG):
    """The least even stream length that holds B frames: the tiled kernels read float rows of even length only."""
    T = (B - 1) * N + H + N + 1
    return T + (T & 1)


def synth_stream(xyz, T, N):
    """[C][T] float32 on the device: a 40-frame synthetic scene repeated, times a per-sample gain ramp (no two frames
    alike)."""
    import torch
    from bflk import synth
    base = torch.from_numpy(synth.make_stream(np.asarray(xyz, np.float64), 40 * N)).cuda()
    x = base.repeat(1, T // (40 * N) + 1)[:, :T].contiguous()
    x *= torch.linspace(0.5, 1.5, T, dtype=torch.float32, device="cuda")[None, :]
    return x


def dev_maps(w, x, B, submit=False):
    """bflk_power_map_batch_dev (or _dev_submit + _dev_join) of B frames of the device stream x [C][T] -> host [B][D]."""
    import torch
    out = torch.empty((B, w.n_directions()[2]), dtype=torch.float32, device=x.device)
    torch.cuda.synchronize()
    if submit:
        w.power_map_batch_dev_submit(x.data_ptr(), x.shape[1], B, out.data_ptr())
        w.power_map_batch_dev_join()
    else:
        w.power_map_batch_dev(x.data_ptr(), x.shape[1], B, out.data_ptr())
    torch.cuda.synchronize()
    return out.cpu().numpy()


def sliced_maps(w, x, B, N):
    """The same frames in calls of at most SLICE frames, each on its own tight copy of the samples it needs."""
    parts = []
    for b0 in range(0, B, SLICE):
        nb = min(SLICE, B - b0)
        xs = x[:, b0 * N:b0 * N + even_samples(nb, N)].contiguous()
        parts.append(dev_maps(w, xs, nb))
        del xs
    return np.concatenate(parts)


def edge_frames(N, B):
    """Frame 0, the last frame, the frames around 65 535 / 65 536 and the frames of the block pairs on both sides of every
    32 768-pair slab edge."""
    nblk = 1 if N <= 256 else (N - 2 + 253) // 254
    n_pairs = (B * nblk + 1) // 2
    f = {0, B - 1, 65534, 65535, 65536}
    for P in range(32768, n_pairs, 32768):
        f |= {(2 * P - 2) // nblk, (2 * P - 1) // nblk, (2 * P) // nblk, (2 * P + 1) // nblk}
    return sorted(b for b in f if b < B)


def check_frames(w, x, maps, N, frames, what):
    off, fr = w.tables()
    for b in frames:
        win = x[:, b * N:b * N + H_BIG + N + 1].cpu().numpy()
        assert_meets_bar(maps[b], power_ref(win, off, fr, None, N, [0])[0], (what, b))


def release(*objs):
    import torch
    for o in objs:
        if hasattr(o, "close"):
            o.close()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("N,kernels", [(256, (0, 1, 2, 3, 4)), (258, (0, 2, 3, 4)), (512, (0, 2, 3, 4))])
def test_large_device_batch_equals_sliced_calls(N, kernels):
    """N = 256: crosses the pair slabs of kernels 2-4 and the frame slab of the generic kernel.  N = 258 / 512 (2 and 3
    blocks a frame): more than 65 535 frames reach the finalize kernels."""
    B = B_BIG
    x = synth_stream(LINE, even_samples(B, N), N)
    frames = edge_frames(N, B)
    for kernel in kernels:
        w = line_array(N, kernel)
        big = dev_maps(w, x, B)
        assert w.kernel_info()[0] == (kernel or 4)
        assert big.shape == (B, 36) and np.all(np.isfinite(big)) and big.min() > 0
        assert np.array_equal(big, sliced_maps(w, x, B, N)), kernel
        check_frames(w, x, big, N, frames, kernel)
        release(w)
    del x
    release()


@pytest.mark.gpu
def test_large_device_batch_submit_join():
    N, B = 512, B_BIG
    x = synth_stream(LINE, even_samples(B, N), N)
    w = line_array(N)
    want = dev_maps(w, x, B)
    got = dev_maps(w, x, B, submit=True)
    assert w.kernel_info()[0] == 4
    assert np.array_equal(got, want)
    del x
    release(w)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [1, 3, 4])
def test_large_wire_batch_and_ingest(oracle, kernel):
    """2.2 M wire rows: more than 65 535 x 32, the sample tiles the ingest kernel converts (kernels 1 and 3 convert the wire
    first; kernel 4 packs it directly).  Same bits as the float batch on the oracle's conversion."""
    import torch
    from bflk import synth
    N = 256
    B = 8590
    T = even_samples(B, N)
    assert T > 65535 * 32
    x = synth_stream(LINE, T, N)
    wire = synth.to_wire_i32(x.cpu().numpy())                    # [T][8]
    exposure = oracle.ingest(wire)                               # [8][T]
    w = line_array(N, kernel)
    if kernel == 1:
        assert np.array_equal(w.ingest_i32(wire), exposure)
    wd = torch.from_numpy(wire).cuda()
    out = torch.empty((B, 36), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    w.power_map_batch_i32_dev(wd.data_ptr(), T, B, out.data_ptr())
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert w.kernel_info()[0] == kernel
    xe = torch.from_numpy(exposure).cuda()
    assert np.array_equal(got, dev_maps(w, xe, B))
    check_frames(w, xe, got, N, [0, 4095, B - 1], kernel)
    del x, wd, xe, out
    release(w)


@pytest.mark.gpu
def test_session_backlog_of_large_batch():
    """A session opened for 65 571 frames of 512 samples, filled in pieces, mapped in one call: the bits of the batch."""
    N, B = 512, B_BIG
    T = even_samples(B, N)
    x = synth_stream(LINE, T, N)
    w = line_array(N)
    want = dev_maps(w, x, B)
    w.stream_open(B)
    piece = 1 << 22
    for t0 in range(0, T, piece):
        w.stream_push(x[:, t0:t0 + piece].cpu().numpy())
    assert w.stream_status() == (T, 0, B, 0)
    first, maps = w.stream_power_maps(B)
    assert first == 0 and np.array_equal(maps, want)
    assert w.kernel_info()[0] == 4
    w.stream_close()
    del x
    release(w)


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs in one box")
def test_group_large_device_batch_equals_single_gpu():
    """Frame-sharded over two GPUs (one direction group), 65 571 frames: the assembly covers more than 65 535 frames."""
    import torch
    import bflk
    from bflk import synth
    N, B = 256, B_BIG
    org = cases.origins(1, 1)
    x = synth_stream(synth.tile_geometry(org), even_samples(B, N), N)
    single = bflk.MIMOWorker(org, 6, 6, 120.0)
    want = dev_maps(single, x, B)
    release(single)
    g = bflk.Group(org, 6, 6, 120.0, devices=[0, 1], dir_groups=1)
    ins = [x] + [x.to("cuda:1")]
    outs = [torch.zeros((B, 36), dtype=torch.float32, device=f"cuda:{i}") for i in range(2)]
    torch.cuda.synchronize(0)
    torch.cuda.synchronize(1)
    g.power_map_batch_dev([t.data_ptr() for t in ins], x.shape[1], B, [t.data_ptr() for t in outs])
    for o in outs:
        assert np.array_equal(o.cpu().numpy(), want)
    del x, ins, outs
    release(g)


# ---- history and stream-length edges (GPU) -----------------------------------------------------------------------------------
EDGES = [
    # H, N, W = H + N + 1, ragged channel mask + direction range
    (255, 256, 512, False),       # tight, even: the tiled kernels read the stream's last sample
    (256, 256, 513, True),        # tight, odd: stream rows of odd length
    (64, 258, 323, False),        # short history; two heavily overlapping blocks
    (301, 510, 812, True),        # odd history: the parity of the tiled kernel's staging origin flips
    (128, 1000, 1129, False),     # four blocks
    (200, 100, 301, True),        # shorter than one block: the generic kernel only
]


def all_entry_points(w, stream, B):
    """The maps of B frames through a pageable host batch, a page-locked host batch, a device batch and single frames."""
    import torch
    D = w.n_directions()[2]
    T = stream.shape[1]
    N, W = w.cfg.frame_len, w.cfg.window_len
    out = {"pageable": lambda: w.power_map_batch(stream, B)}

    def pinned():
        ps = torch.from_numpy(stream).pin_memory()
        o = np.zeros((B, D), np.float32)
        w.power_map_batch_ptr(ps.data_ptr(), T, B, o.ctypes.data)
        return o

    def device():
        return dev_maps(w, torch.from_numpy(stream).cuda(), B)

    def single():
        return np.stack([w.power_map(np.ascontiguousarray(stream[:, b * N:b * N + W])) for b in range(B)])
    out.update(pinned=pinned, device=device, single=single)
    return out


def expected_kernel(kernel, N, T):
    """The kernel that serves the call, or None where an explicit choice must be refused with BFLK_ERR_STATE: the tiled
    kernels need frames of whole even blocks and float rows of even length, the lane-broadcast kernel frames of >= 256."""
    tiled = N >= 256 and N % 2 == 0 and T % 2 == 0
    if kernel == 0:
        return 4 if tiled else 3 if N >= 256 else 1
    if kernel in (2, 4) and not tiled:
        return None
    if kernel == 3 and N < 256:
        return None
    return kernel


def run_edge_case(w, stream, B, kernel, index, first, count, what):
    import bflk
    import torch
    N = w.cfg.frame_len
    T = stream.shape[1]
    off, fr = w.tables()
    off, fr = off[first:first + count], fr[first:first + count]
    want_kernel = expected_kernel(kernel, N, T)
    got = {}
    for name, call in all_entry_points(w, stream, B).items():
        if want_kernel is None:
            with pytest.raises(bflk.BflkError) as e:
                call()
            assert e.value.code == ERR_STATE, (what, name, str(e.value))
            continue
        got[name] = call()
        assert w.kernel_info()[0] == want_kernel, (what, name)
    torch.cuda.synchronize()
    if want_kernel is None:
        return None
    ref = power_ref(stream, off, fr, index, N, range(B))
    for name, p in got.items():
        assert p.shape == (B, count)
        assert np.array_equal(p, got["pageable"]), (what, name)
    for b in range(B):
        assert_meets_bar(got["pageable"][b], ref[b], (what, b))
    return got["pageable"]


@pytest.mark.gpu
@pytest.mark.parametrize("slack", [0, 1])
@pytest.mark.parametrize("H,N,W,ragged", EDGES)
def test_history_and_stream_length_edges(H, N, W, ragged, slack):
    """slack = 0: the stream, and every single frame's window, is exactly as long as the last frame needs; 1: one sample
    more, which flips the parity of the rows (the tiled kernels take rows of even length only)."""
    import bflk
    from bflk import synth
    org = cases.origins(1, 1)
    B = 5
    assert W == H + N + 1
    T = (B - 1) * N + W + slack
    stream = synth.make_stream(synth.tile_geometry(org), T)
    index, first, count = None, 0, 120
    for kernel in range(5):
        w = bflk.MIMOWorker(org, 12, 10, 150.0, frame_len=N, history=H, window_len=W + slack)
        w.set_kernel(kernel)
        if ragged:
            index, first, count = ragged_mask(64), 13, 71
            w.set_channel_mask(index)
            w.set_direction_range(first, count)
        run_edge_case(w, stream, B, kernel, index, first, count, (H, N, W, T, kernel))
        w.close()


def edge_lut(rows, cols, C, H, rng):
    """Offsets of a rows x cols grid whose per-channel delays change linearly across the grid, spanning exactly [0, H],
    neighbouring directions at most 3 samples apart; fractions uniform with 0 and the float just below 1 included."""
    a = 2 * np.pi * np.arange(C) / C
    u, v = np.cos(a), np.sin(a)
    s = 1.0 / (np.abs(u) + np.abs(v))
    u, v = u * s, v * s                                         # |u| + |v| = 1; channel 0: u = 1, v = 0
    y = np.linspace(-1.0, 1.0, rows)[:, None, None]
    x = np.linspace(-1.0, 1.0, cols)[None, :, None]
    off = np.rint(H / 2 + H / 2 * (u * y + v * x)).astype(np.int32).reshape(rows * cols, C)
    fr = rng.random((rows * cols, C), dtype=np.float32)
    fr[::7] = 0.0
    fr[3::7] = np.nextafter(np.float32(1.0), np.float32(0.0))
    fr[:, 5] = 0.0
    fr[:, 6] = np.nextafter(np.float32(1.0), np.float32(0.0))
    return off, fr


@pytest.mark.gpu
@pytest.mark.parametrize("T_extra", [0, 1])
def test_caller_tables_spanning_the_whole_history(T_extra):
    """A caller LUT with H = 64 whose offsets reach both 0 and H and whose fractions include 0 and nextafter(1, 0),
    declared as a grid: the tiled kernels serve it.  T_extra = 0: the exact minimum stream (odd rows: the tiled kernels
    refuse float rows of odd length, the automatic choice falls back); 1: one sample more (even rows)."""
    import bflk
    from bflk import synth
    H, N, rows, cols, C, B = 64, 256, 24, 24, 64, 5
    off, fr = edge_lut(rows, cols, C, H, np.random.default_rng(5))
    assert off.min() == 0 and off.max() == H
    grid = off.reshape(rows, cols, C).astype(np.int64)
    assert np.abs(np.diff(grid, axis=0)).max() <= 3 and np.abs(np.diff(grid, axis=1)).max() <= 3
    assert (fr == 0.0).any() and (fr == np.nextafter(np.float32(1.0), np.float32(0.0))).any()
    W = H + N + 1 + T_extra
    T = (B - 1) * N + W
    xyz = synth.tile_geometry(cases.origins(1, 1))
    stream = synth.make_stream(xyz, T)
    for kernel in range(5):
        w = bflk.Beamformer(n_channels=C, frame_len=N, history=H, window_len=W)
        w.set_geometry(xyz.astype(np.float32))
        w.set_grid_tables(off, fr)
        w.set_grid_shape(rows, cols)
        w.set_kernel(kernel)
        got_off, got_fr = w.tables()
        assert np.array_equal(got_off, off) and np.array_equal(got_fr.view(np.uint32), fr.view(np.uint32))
        run_edge_case(w, stream, B, kernel, None, 0, rows * cols, ("lut", T, kernel))
        w.close()
