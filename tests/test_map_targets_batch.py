"""Targets of every map of a device batch or a session backlog in one launch (bflk_targets_batch_dev, bflk_session_targets).

Every map's records must be those oracle.map_targets defines (same directions in the same order, power and probability
bit for bit), with theta / phi of bflk_get_grid, row / col = divmod(direction, cols) and reserved 0, and the records
bflk_targets gives for the same map on the host.  The session call must take and consume frames exactly as
bflk_stream_power_maps does."""
import ctypes as C

import numpy as np
import pytest

import cases

BFLK_ERR_INVALID, BFLK_ERR_STATE = -1, -2
N, H, W = 256, 256, 1024
PARAMS = [(8, 0.05), (1, 0.5), (32, 0.001), (256, 0.0)]


# ---- no GPU ----------------------------------------------------------------------------------------------------------
def test_null_handle_is_invalid():
    import bflk
    L = bflk.load_library()
    buf = np.zeros(4096, np.float32)
    i64, i32 = C.c_int64(), C.c_int32()
    assert L.bflk_targets_batch_dev(None, buf.ctypes.data, 1, 8, 0.5, buf.ctypes.data, buf.ctypes.data, None) == BFLK_ERR_INVALID
    assert L.bflk_session_targets(None, 1, 8, 0.5, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, C.byref(i64),
                                  C.byref(i32)) == BFLK_ERR_INVALID


def test_target_dtype_decodes_records():
    import bflk
    recs = (bflk.Target * 6)()
    for i, t in enumerate(recs):
        t.theta, t.phi, t.power, t.probability, t.direction, t.row, t.col = 0.25 * i, -0.5 * i, 1.5 * i, 3.0, i, i // 3, i % 3
    got = bflk.decode_targets(bytes(recs), [2, 1])
    assert [len(m) for m in got] == [2, 1]
    assert got[1][0] == dict(theta=0.75, phi=-1.5, power=4.5, probability=3.0, direction=3, row=1, col=0)


# ---- helpers -----------------------------------------------------------------------------------------------------------
def records(w, maps, max_targets, min_rel, stream=0, presync=True):
    """bflk_targets_batch_dev on the rows of maps (a [B][D] float32 CUDA tensor): (TARGET_DTYPE records [B][max_targets],
    counts [B]); slots past a map's count are returned as the call left them.  presync: wait for the whole device first
    (the handle's stream, stream 0, does not wait for torch's); off, the call relies on the stream order alone"""
    import torch
    import bflk
    B = maps.shape[0]
    raw = torch.full((B, max_targets * bflk.TARGET_DTYPE.itemsize), 0xA5, dtype=torch.uint8, device=maps.device)
    n = torch.full((B,), -7, dtype=torch.int32, device=maps.device)
    if presync:
        torch.cuda.synchronize(maps.device)
    w.targets_batch_dev(maps.data_ptr(), B, raw.data_ptr(), n.data_ptr(), max_targets, min_rel, stream)
    torch.cuda.synchronize(maps.device)
    return np.frombuffer(raw.cpu().numpy().tobytes(), bflk.TARGET_DTYPE).reshape(B, max_targets), n.cpu().numpy()


def host_records(w, power, max_targets, min_rel):
    """bflk_targets on a host map: TARGET_DTYPE records [n]"""
    import bflk
    out = (bflk.Target * max_targets)()
    n = C.c_int32()
    src = np.ascontiguousarray(power, np.float32)
    w._check(w._L.bflk_targets(w._h, src.ctypes.data, max_targets, float(min_rel), out, C.byref(n)))
    return np.frombuffer(bytes(out), bflk.TARGET_DTYPE)[:n.value]


def assert_oracle(oracle, rec, n, power, rows, cols, theta, phi, max_targets, min_rel, what=""):
    """records rec[:n] of one map are the oracle's targets of `power`, with the grid's angles"""
    idx, pw, pr = oracle.map_targets(power, rows, cols, max_targets, min_rel)
    assert n == len(idx), (what, n, len(idx))
    r = rec[:n]
    assert np.array_equal(r["direction"], idx), what
    assert np.array_equal(r["power"].view(np.uint32), pw.view(np.uint32)), what
    assert np.array_equal(r["probability"].view(np.uint32), pr.view(np.uint32)), what
    assert np.array_equal(r["theta"].view(np.uint64), theta[idx].view(np.uint64)), what
    assert np.array_equal(r["phi"].view(np.uint64), phi[idx].view(np.uint64)), what
    assert np.array_equal(r["row"], idx // cols) and np.array_equal(r["col"], idx % cols), what
    assert not r["reserved"].any(), what


def device_maps(name, B, seed=0):
    """(worker, [B][D] CUDA tensor of maps) of B distinct frames of a cfg's geometry and grid"""
    import torch
    import bflk
    from bflk import synth
    c = cases.CONFIGS[name]
    w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
    T = (B - 1) * N + W
    s = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), T, seed=seed)
    s *= np.linspace(0.5, 1.5, T, dtype=np.float32)[None, :]          # no two frames alike
    x = torch.from_numpy(np.ascontiguousarray(s)).cuda()
    p = torch.zeros((B, c["rows"] * c["cols"]), dtype=torch.float32, device="cuda")
    w.power_map_batch_dev(x.data_ptr(), T, B, p.data_ptr())
    torch.cuda.synchronize()
    return w, p


def edge_maps(rows, cols, B, seed):
    """B maps of a rows x cols grid cycling through the edge cases: all zero, constant, plateaus with ties, NaN entries,
    negative values, peaks on the border, sparse spikes, random"""
    rng = np.random.default_rng(seed)
    D = rows * cols
    maps = np.empty((B, D), np.float32)
    for b in range(B):
        kind = b % 8
        if kind == 0:
            m = np.zeros(D, np.float32)
        elif kind == 1:
            m = np.full(D, rng.choice([1.0, 3e-7, np.inf]), np.float32)
        elif kind == 2:
            m = rng.integers(0, 3, D).astype(np.float32) * np.float32(rng.choice([0.5, 1.0]))
        elif kind == 3:
            m = rng.random(D, dtype=np.float32)
            m[rng.random(D) < 0.2] = np.nan
        elif kind == 4:
            m = rng.standard_normal(D).astype(np.float32)
        elif kind == 5:
            m = rng.random(D, dtype=np.float32) * 0.1
            g = m.reshape(rows, cols)
            g[0, :] += rng.random(cols, dtype=np.float32)
            g[:, -1] += rng.random(rows, dtype=np.float32)
        elif kind == 6:
            m = np.zeros(D, np.float32)
            m[rng.integers(0, D, 3)] = rng.random(3, dtype=np.float32) + 0.5
        else:
            m = rng.random(D, dtype=np.float32)
        maps[b] = m
    return maps


# ---- per-map parity ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("cfg1", 5), ("cfg2", 6), ("cfg3", 9)])
def test_batch_equals_oracle_and_bflk_targets(oracle, name, B):
    c = cases.CONFIGS[name]
    rows, cols = c["rows"], c["cols"]
    w, p = device_maps(name, B, seed=3)
    theta, phi = w.grid()
    maps = p.cpu().numpy()
    assert len({m.tobytes() for m in maps}) == B
    for max_targets, min_rel in PARAMS:
        rec, n = records(w, p, max_targets, min_rel)
        assert n.max() > 0
        for b in range(B):
            what = (name, max_targets, min_rel, b)
            assert_oracle(oracle, rec[b], n[b], maps[b], rows, cols, theta, phi, max_targets, min_rel, what)
            assert rec[b][:n[b]].tobytes() == host_records(w, maps[b], max_targets, min_rel).tobytes(), what
    w.close()


@pytest.mark.gpu
def test_edge_maps_past_the_grid_limit(oracle):
    """> 65 535 maps of a small grid in one call, every edge case many times over"""
    import torch
    import bflk
    rows, cols = 6, 7
    B = 65535 + 77
    w = bflk.MIMOWorker(cases.origins(1, 1), rows, cols, 180.0)
    theta, phi = w.grid()
    maps = edge_maps(rows, cols, B, seed=11)
    for max_targets, min_rel in [(8, 0.05), (3, 0.0)]:
        rec, n = records(w, torch.from_numpy(maps).cuda(), max_targets, min_rel)
        for b in range(B):
            assert_oracle(oracle, rec[b], n[b], maps[b], rows, cols, theta, phi, max_targets, min_rel, (b, b % 8))
    for b in range(8):
        assert rec[b][:n[b]].tobytes() == host_records(w, maps[b], 3, 0.0).tobytes(), b
    w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,max_targets", [(256, 256, 256), (512, 768, 24), (1400, 1400, 24)])
def test_large_grids(oracle, rows, cols, max_targets):
    """a cfg5-sized grid with every slot used; a grid whose candidate bitmask (48 KB) needs more than the default dynamic
    shared memory beside the kernel's static arrays; and a grid too large for any bitmask in shared memory (the candidates
    are evaluated again for every pick).  A few maps together, and the first alone through bflk_targets"""
    import torch
    import bflk
    w = bflk.MIMOWorker(cases.origins(1, 1), rows, cols, 60.0)
    theta, phi = w.grid()
    maps = edge_maps(rows, cols, 8, seed=rows)[[7, 5, 3, 4]]
    for min_rel in (0.0, 0.05):
        rec, n = records(w, torch.from_numpy(maps).cuda(), max_targets, min_rel)
        for b in range(len(maps)):
            assert_oracle(oracle, rec[b], n[b], maps[b], rows, cols, theta, phi, max_targets, min_rel, (min_rel, b))
        assert rec[0][:n[0]].tobytes() == host_records(w, maps[0], max_targets, min_rel).tobytes()
    assert n.max() == max_targets
    w.close()


# ---- direction ranges and groups ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_direction_range_is_not_consulted():
    name = "cfg3"
    c = cases.CONFIGS[name]
    w, p = device_maps(name, 4, seed=8)
    import bflk
    part = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
    part.set_direction_range(100, 300)
    for max_targets, min_rel in PARAMS:
        a, na = records(w, p, max_targets, min_rel)
        b, nb = records(part, p, max_targets, min_rel)
        assert np.array_equal(na, nb)
        for i in range(len(na)):
            assert a[i][:na[i]].tobytes() == b[i][:nb[i]].tobytes()
    w.close()
    part.close()


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs in one box")
def test_group_ranks_give_identical_records():
    import torch
    import bflk
    from bflk import synth
    from test_handle_lifetime import _group_handle
    c = cases.CONFIGS["cfg3"]
    B = 6
    T = (B - 1) * N + W
    stream = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), T)
    g = bflk.Group(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"], devices=[0, 1])
    ins = [torch.from_numpy(stream).to(f"cuda:{i}") for i in range(2)]
    outs = [torch.zeros((B, c["rows"] * c["cols"]), dtype=torch.float32, device=f"cuda:{i}") for i in range(2)]
    g.power_map_batch_dev([t.data_ptr() for t in ins], T, B, [t.data_ptr() for t in outs])
    got = []
    for i in range(2):
        with torch.cuda.device(i):
            got.append(records(_group_handle(g, i), outs[i], 16, 0.01))
    assert got[0][1].max() > 0 and np.array_equal(got[0][1], got[1][1])
    for b in range(B):
        assert got[0][0][b][:got[0][1][b]].tobytes() == got[1][0][b][:got[1][1][b]].tobytes()
    g.close()


# ---- stream ordering -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_side_stream_after_submit_and_join():
    import torch
    name = "cfg3"
    c = cases.CONFIGS[name]
    B = 64                                                 # the batch still runs when the side stream's call is enqueued
    w, p_sync = device_maps(name, B, seed=4)
    want, want_n = records(w, p_sync, 16, 0.01)
    from bflk import synth
    T = (B - 1) * N + W
    s = synth.make_stream(synth.tile_geometry(cases.origins(c["nx"], c["ny"])), T, seed=4)
    s *= np.linspace(0.5, 1.5, T, dtype=np.float32)[None, :]
    x = torch.from_numpy(np.ascontiguousarray(s)).cuda()
    p = torch.zeros_like(p_sync)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    w.power_map_batch_dev_submit(x.data_ptr(), T, B, p.data_ptr())
    w.power_map_batch_dev_join(side.cuda_stream)
    # no device-wide wait in between: only the join orders the side stream after the batch (torch's side stream also waits
    # for the legacy default stream, where records() fills its output buffers)
    got, got_n = records(w, p, 16, 0.01, side.cuda_stream, presync=False)
    assert np.array_equal(got_n, want_n) and got.tobytes() == want.tobytes()
    w.close()


@pytest.mark.gpu
def test_device_call_leaves_the_device_map():
    import torch
    import bflk
    from test_handle_lifetime import _assert_device_map_is, _window
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    p = w.power_map(_window())
    other = torch.rand((3, 256), device="cuda")
    side = torch.cuda.Stream()
    records(w, other, 8, 0.1, side.cuda_stream)
    records(w, other, 8, 0.1)
    _assert_device_map_is(w, p)
    w.close()


# ---- sessions ------------------------------------------------------------------------------------------------------------
def _session_stream(n_samples, seed):
    from bflk import synth
    s = synth.make_stream(synth.tile_geometry(cases.origins(1, 1)), n_samples, seed=seed)
    s *= np.linspace(0.5, 1.5, n_samples, dtype=np.float32)[None, :]
    return np.ascontiguousarray(s)


@pytest.mark.gpu
@pytest.mark.parametrize("max_targets,min_rel", [(8, 0.05), (256, 0.0)])
def test_session_targets_equal_maps_call_and_oracle(oracle, max_targets, min_rel):
    """Twin sessions, one taking maps and one taking maps with Targets, pushed the same samples and called with the same
    max_frames, including an overrun that skips frames and calls with nothing ready"""
    import bflk
    rows = cols = 24
    ws = [bflk.MIMOWorker(cases.origins(1, 1), rows, cols, 180.0) for _ in range(2)]
    theta, phi = ws[1].grid()
    T = 40 * N + W
    stream = _session_stream(T, seed=13)
    rng = np.random.default_rng(2)
    for w in ws:
        w.stream_open(6)
    taken = []

    def take(k):
        st = [w.stream_status() for w in ws]
        assert st[0] == st[1]
        f0, m0 = ws[0].stream_power_maps(k)
        f1, m1, tg = ws[1].stream_targets(k, max_targets, min_rel)
        assert f0 == f1 and np.array_equal(m0, m1) and len(tg) == len(m1)
        assert ws[0].stream_status() == ws[1].stream_status()
        for b in range(len(m1)):
            rec = np.array([(d["theta"], d["phi"], d["power"], d["probability"], d["direction"], d["row"], d["col"], 0)
                            for d in tg[b]], bflk.TARGET_DTYPE)
            assert_oracle(oracle, rec, len(rec), m1[b], rows, cols, theta, phi, max_targets, min_rel, (f1, b))
        taken.append(len(m1))

    t = 0
    while t < T:
        n = int(min(T - t, rng.integers(1, 3 * N)))
        for w in ws:
            w.stream_push(stream[:, t:t + n])
        t += n
        if not 16 * N < t < 26 * N:                       # in between, the ring of 6 frames overruns: frames are skipped
            take(int(rng.integers(1, 9)))
    while ws[1].stream_status()[2] > 0:
        take(8)
    assert sum(k > 1 for k in taken) > 2 and 0 in taken and ws[1].stream_status()[3] > 0
    before = ws[1].stream_status()
    f, m, tg = ws[1].stream_targets(4, max_targets, min_rel)                 # nothing ready: nothing changes
    assert (f, len(m), tg) == (before[1], 0, []) and ws[1].stream_status() == before
    for w in ws:
        w.close()


@pytest.mark.gpu
def test_session_targets_leave_a_single_frame_map():
    import bflk
    from test_stream_session import _heatmap, _targets
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    stream = _session_stream(8 * N + W, seed=9)
    w.stream_open(8)
    w.stream_push(stream[:, :N + H + 1])
    f, m, tg = w.stream_targets(4, 16, 0.05)
    assert (f, len(m)) == (0, 1)
    assert _targets(w) == _targets(w, m[0]) and _heatmap(w) == _heatmap(w, m[0])
    assert [(d["direction"], d["power"], d["probability"]) for d in tg[0]] == _targets(w, m[0])
    w.stream_push(stream[:, N + H + 1:4 * N + H + 1])
    f, m, tg = w.stream_targets(4, 16, 0.05)
    assert (f, len(m)) == (1, 3)
    with pytest.raises(bflk.BflkError) as e:
        _targets(w)
    assert e.value.code == BFLK_ERR_STATE
    w.close()


# ---- refusals ------------------------------------------------------------------------------------------------------------
def _code(fn, *args):
    import bflk
    with pytest.raises(bflk.BflkError) as e:
        fn(*args)
    return e.value.code


@pytest.mark.gpu
def test_refusals():
    import torch
    import bflk
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    p = torch.rand((2, 256), device="cuda")
    raw = torch.zeros((2, 257 * 40), dtype=torch.uint8, device="cuda")
    n = torch.zeros(2, dtype=torch.int32, device="cuda")
    dev = w.targets_batch_dev
    assert _code(dev, 0, 2, raw.data_ptr(), n.data_ptr(), 8, 0.1) == BFLK_ERR_INVALID
    assert _code(dev, p.data_ptr(), 2, 0, n.data_ptr(), 8, 0.1) == BFLK_ERR_INVALID
    assert _code(dev, p.data_ptr(), 2, raw.data_ptr(), 0, 8, 0.1) == BFLK_ERR_INVALID
    assert _code(dev, p.data_ptr(), 0, raw.data_ptr(), n.data_ptr(), 8, 0.1) == BFLK_ERR_INVALID
    for mt in (0, 257):
        assert _code(dev, p.data_ptr(), 2, raw.data_ptr(), n.data_ptr(), mt, 0.1) == BFLK_ERR_INVALID
    stream = _session_stream(4 * N + W, seed=1)
    w.stream_open(8)
    w.stream_push(stream)
    status = w.stream_status()
    assert status[2] > 0
    for mt in (0, 257):
        assert _code(w.stream_targets, 2, mt, 0.1) == BFLK_ERR_INVALID
    out, recs, cnt, i64, i32 = np.zeros((2, 256), np.float32), (bflk.Target * 16)(), np.zeros(2, np.int32), C.c_int64(), C.c_int32()
    L, h = w._L, w._h
    assert L.bflk_session_targets(h, 2, 8, 0.1, out.ctypes.data, None, cnt.ctypes.data, C.byref(i64), C.byref(i32)) == BFLK_ERR_INVALID
    assert L.bflk_session_targets(h, 2, 8, 0.1, out.ctypes.data, recs, None, C.byref(i64), C.byref(i32)) == BFLK_ERR_INVALID
    assert L.bflk_session_targets(h, 2, 8, 0.1, None, recs, cnt.ctypes.data, C.byref(i64), C.byref(i32)) == BFLK_ERR_INVALID
    w.set_direction_range(0, 200)                                              # a partial range: the session call refuses
    assert _code(w.stream_targets, 2, 8, 0.1) == BFLK_ERR_STATE
    assert w.stream_status() == status
    w.set_direction_range(0, 256)
    f, m, tg = w.stream_targets(2, 8, 0.1)
    assert f == status[1] and len(m) == 2
    # caller tables, without and with a shape: no angles, so no Targets
    off, fr = w.tables()
    for shape in (False, True):
        w.set_grid_tables(off, fr)
        if shape:
            w.set_grid_shape(16, 16)
        status = w.stream_status()
        assert _code(dev, p.data_ptr(), 2, raw.data_ptr(), n.data_ptr(), 8, 0.1) == BFLK_ERR_STATE
        assert _code(w.targets, p[0].cpu().numpy()) == BFLK_ERR_STATE
        assert _code(w.stream_targets, 2, 8, 0.1) == BFLK_ERR_STATE
        assert w.stream_status() == status
    w.set_grid_fov(16, 16, 180.0)
    dev(p.data_ptr(), 2, raw.data_ptr(), n.data_ptr(), 8, 0.1)
    torch.cuda.synchronize()
    w.close()
