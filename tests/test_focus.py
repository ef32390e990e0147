"""Near-field steering (bflk_set_focus): tables focused at a point r metres away instead of at a plane wave.

CPU: the focused delays of the CPU restatement (focus_oracle.py) against an independent float64 r - |r u - p|, against
the far field at a large distance, and against the arrival delays of synth.point_source_stream.
GPU: focused grid and steering tables bit for bit against the oracle; the far field untouched by the call; refusals that
change nothing; power maps, beams, sessions and Targets on a focused grid; focused MISO, FIR MISO and monopulse; the gain
of focusing on a point source at 5 m; a group of handles.

Bars as in test_dynamic_steering.py: tables, audio and kernel-2 beams bit for bit; powers within 1e-4 relative."""
import math

import numpy as np
import pytest

import cases
import focus_oracle as F
from test_dynamic_steering import SPEEDS, geometry, handle, hp_power, rel_err, same_bits, window_for

POWER_RTOL = 1e-4
BFLK_ERR_INVALID, BFLK_ERR_RANGE = -1, -5
TILED = {"cfg1": (1, 1), "cfg2": (4, 1), "cfg3": (4, 2)}


def tiled_xyz(oracle, name):
    return oracle.create_tiled_antenna(cases.origins(*TILED[name]))


def radius(xyz):
    """Largest |p| as the library computes it: float coordinates promoted to double."""
    p = np.asarray(xyz, np.float64)
    return float(np.max(np.sqrt((p[:, 0] * p[:, 0] + p[:, 1] * p[:, 1]) + p[:, 2] * p[:, 2])))


def exact_focus_delays(xyz, theta, phi, r, k):
    """r - |r u - p| in float64 from the float trig the library uses, times k, min-subtracted."""
    az, ay = np.float32(phi), -np.float32(theta)
    cz, sz = np.float32(math.cos(float(az))), np.float32(math.sin(float(az)))
    cy, sy = np.float32(math.cos(float(ay))), np.float32(math.sin(float(ay)))
    u = np.array([-float(sy) * float(cz), float(sy) * float(sz), float(cy)])
    d = (r - np.linalg.norm(r * u[None, :] - np.asarray(xyz, np.float64), axis=1)) * k
    return d - d.min()


def all_geometries(oracle):
    out = [(name, tiled_xyz(oracle, name), cases.origins(*TILED[name])) for name in TILED]
    for g, C in (("cube", 64), ("vertical", 64), ("tiles3d", 128)):
        xyz, origins = geometry(g, C, 0.3)
        out.append((g, xyz, origins))
    return out


# ---- the oracle (CPU) ------------------------------------------------------------------------------------------------
def test_focus_delays_match_float64(oracle):
    rng = np.random.default_rng(1)
    th, ph = np.r_[0.0, np.pi / 2, rng.random(6) * np.pi / 2], np.r_[0.0, 2.0, rng.random(6) * 2 * np.pi]
    for name, xyz, _ in all_geometries(oracle):
        for sr, c in SPEEDS:
            k = oracle.delay_scale(sr, c)
            for r in (radius(xyz) * 1.0001, 0.5, 3.0, 5.0, 20.0, 1e6):
                if r <= radius(xyz):
                    continue
                for t, p in zip(th, ph):
                    got = F.focus_delays(xyz, t, p, r, scale=k)
                    assert np.max(np.abs(got - exact_focus_delays(xyz, t, p, r, k))) <= 1e-4, (name, sr, c, r, t, p)


def test_focus_tends_to_the_far_field(oracle):
    rng = np.random.default_rng(2)
    for name, xyz, _ in all_geometries(oracle):
        for sr, c in SPEEDS:
            k = oracle.delay_scale(sr, c)
            for t, p in zip(rng.random(5) * np.pi / 2, rng.random(5) * 2 * np.pi):
                far = oracle.steering_vector_spherical(xyz, t, p, scale=k)
                assert np.max(np.abs(F.focus_delays(xyz, t, p, 1e7, scale=k) - far)) <= 1e-3, (name, sr, c)
    # the grid LUT is the per-direction tables
    xyz = tiled_xyz(oracle, "cfg3")
    off, fr = F.mimo_lut_focus(oracle, xyz, 5, 7, 150.0, 4.0, history=200)
    th, ph = oracle.mimo_grid(5, 7, 150.0)
    eo, ef = F.steer_tables_focus(xyz, th, ph, 4.0, history=200)
    assert np.array_equal(off, eo) and same_bits(fr, ef)


def test_focus_delays_are_the_point_source_arrival_delays(oracle):
    from bflk import synth
    for name in TILED:
        xyz = tiled_xyz(oracle, name)
        for sr, c in SPEEDS[:2]:
            for t, p, r in ((0.35, 0.52, 5.0), (1.1, 4.0, 1.0), (0.0, 0.0, 3.0)):
                tau = synth.point_source_delays(xyz, t, p, r, sr, c)
                assert np.max(np.abs(F.focus_delays(xyz, t, p, r, oracle.delay_scale(sr, c)) - tau)) <= 1e-4
    # the stream carries those delays: one noise-free tone is sin(2 pi f (t + tau) / fs)
    xyz = tiled_xyz(oracle, "cfg2")
    s = synth.point_source_stream(xyz, 300, [(0.4, 1.0, 2.0, 1000.0, 1.0)], sigma=0, dtype=np.float64)
    tau = synth.point_source_delays(xyz, 0.4, 1.0, 2.0)
    t = np.arange(300)
    assert np.allclose(s, np.sin(2 * np.pi * 1000.0 * (t[None, :] + tau[:, None]) / synth.SAMPLE_RATE), atol=1e-12)


# ---- tables (GPU) ------------------------------------------------------------------------------------------------------
def _tables_or_range(call, exp_off, exp_fr):
    """The oracle's bits when its largest delay fits the history, BFLK_ERR_RANGE when it does not."""
    import bflk
    if exp_off.min() < 0:
        with pytest.raises(bflk.BflkError) as e:
            call()
        assert e.value.code == BFLK_ERR_RANGE
        return False
    off, fr = call()
    assert np.array_equal(off, exp_off) and same_bits(fr, exp_fr)
    return True


@pytest.mark.gpu
@pytest.mark.parametrize("speed", SPEEDS)
def test_focused_tables_vs_oracle(oracle, speed):
    """set_focus then set_grid_fov, set_grid_fov then set_focus, and steer_tables: the oracle's focused tables bit for bit,
    from just outside the array to 1e6 m, on cfg1-3 and the 3-D geometries."""
    sr, c = speed
    k = oracle.delay_scale(sr, c)
    th, ph = np.r_[0.0, np.pi / 2, np.random.default_rng(5).random(14) * np.pi / 2], np.r_[0.0, 1.0, np.random.default_rng(6).random(14) * 7]
    import bflk
    checked = 0
    for name, xyz, origins in all_geometries(oracle):
        H = 256
        w = handle(xyz, origins, N=64, H=H, sample_rate=sr, speed=c)
        have_grid = False
        for r in (radius(xyz) * 1.001, 0.7, 2.0, 5.0, 1e6):
            if r <= radius(xyz):
                continue
            go, gf = F.mimo_lut_focus(oracle, xyz, 7, 9, 150.0, r, history=H, scale=k)
            if have_grid and go.min() < 0:            # the rebuild of the grid does not fit: refused
                with pytest.raises(bflk.BflkError) as e:
                    w.set_focus(r)
                assert e.value.code == BFLK_ERR_RANGE
                continue
            w.set_focus(r)
            if have_grid:                              # rebuilt at once
                off, fr = w.tables()
                assert np.array_equal(off, go) and same_bits(fr, gf), (name, r)

            def grid():
                w.set_grid_fov(7, 9, 150.0)
                return w.tables()
            have_grid = _tables_or_range(grid, go, gf)
            checked += have_grid
            eo, ef = F.steer_tables_focus(xyz, th, ph, r, history=H, scale=k)
            _tables_or_range(lambda: w.steer_tables(th, ph), eo, ef)
        w.close()
    assert checked >= 20


@pytest.mark.gpu
def test_focus_after_the_grid_equals_focus_before(oracle):
    c = cases.CONFIGS["cfg3"]
    import bflk
    a = bflk.MIMOWorker(cases.origins(4, 2), c["rows"], c["cols"], c["fov"])
    a.set_direction_range(100, 500)
    a.set_focus(3.0)
    assert a.n_directions() == (1024, 100, 500)          # the range survives the rebuild
    b = bflk.Beamformer(n_channels=512)
    b.set_tiled_geometry(cases.origins(4, 2))
    b.set_focus(3.0)
    b.set_grid_fov(c["rows"], c["cols"], c["fov"])
    eo, ef = F.mimo_lut_focus(oracle, tiled_xyz(oracle, "cfg3"), c["rows"], c["cols"], c["fov"], 3.0)
    for w in (a, b):
        off, fr = w.tables()
        assert np.array_equal(off, eo) and same_bits(fr, ef)
        th, ph = w.grid()
        assert np.array_equal((th, ph), oracle.mimo_grid(c["rows"], c["cols"], c["fov"]))   # angles unchanged
    a.close()
    b.close()


# ---- the far field is untouched ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_focus_zero_is_the_far_field(oracle):
    import bflk
    c = cases.CONFIGS["cfg3"]
    from bflk import synth
    stream = synth.make_stream(tiled_xyz(oracle, "cfg3"), 3 * c["N"] + c["W"])
    window = stream[:, :c["W"]]
    th, ph = np.deg2rad([20.0, 45.0, 70.0]), np.deg2rad([30.0, 200.0, 300.0])
    outs = []
    for calls in ([], [0.0], [5.0, 0.0], [1e6, 2.0, 0.0]):
        w = bflk.MIMOWorker(cases.origins(4, 2), c["rows"], c["cols"], c["fov"])
        for r in calls:
            w.set_focus(r)
        outs.append((w.tables(), w.steer_tables(th, ph), w.power_map_batch(stream, 4), w.miso(th, ph, window)))
        w.close()
    for o in outs[1:]:
        (off, fr), (so, sf), maps, (audio, power) = o
        (off0, fr0), (so0, sf0), maps0, (audio0, power0) = outs[0]
        assert np.array_equal(off, off0) and same_bits(fr, fr0) and np.array_equal(so, so0) and same_bits(sf, sf0)
        assert same_bits(maps, maps0) and same_bits(audio, audio0) and same_bits(power, power0)


# ---- refusals ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_change_nothing(oracle):
    import bflk
    c = cases.CONFIGS["cfg3"]
    xyz = tiled_xyz(oracle, "cfg3")
    # boresight and near it: no far-field delay, a few samples' focusing delay at 6 m and 20 samples next to the array
    H = 10
    w = bflk.MIMOWorker(cases.origins(4, 2), 1, 1, 90.0, history=H, window_len=300)
    th, ph = np.array([0.0, 0.01]), np.array([0.0, 2.1])
    w.set_focus(6.0)
    before = w.tables()
    assert np.array_equal(before[0], F.mimo_lut_focus(oracle, xyz, 1, 1, 90.0, 6.0, history=H)[0]) and before[0].min() < H
    steer_before = w.steer_tables(th, ph)
    eo, ef = F.steer_tables_focus(xyz, th, ph, 6.0, history=H)
    assert np.array_equal(steer_before[0], eo) and same_bits(steer_before[1], ef)
    R = radius(xyz)
    near = R * 1.01
    assert F.mimo_lut_focus(oracle, xyz, 1, 1, 90.0, near, history=H)[0].min() < 0
    for r, code in ((-1.0, BFLK_ERR_INVALID), (float("nan"), BFLK_ERR_INVALID), (float("inf"), BFLK_ERR_INVALID),
                    (-float("inf"), BFLK_ERR_INVALID), (R, BFLK_ERR_INVALID), (R * 0.5, BFLK_ERR_INVALID),
                    (near, BFLK_ERR_RANGE)):
        with pytest.raises(bflk.BflkError) as e:
            w.set_focus(r)
        assert e.value.code == code, r
        off, fr = w.tables()
        assert np.array_equal(off, before[0]) and same_bits(fr, before[1]), r
        so, sf = w.steer_tables(th, ph)                  # still focused at 6 m
        assert np.array_equal(so, steer_before[0]) and same_bits(sf, steer_before[1]), r
    # a geometry whose elements reach past the focus: every table build refuses it
    far_out = np.asarray(xyz).copy()
    far_out[0] = [7.0, 0.0, 0.0]
    w.set_geometry(far_out)
    window = window_for(512, 300, 1)
    for call in (lambda: w.set_grid_fov(1, 1, 90.0), lambda: w.steer_tables(th, ph), lambda: w.miso(th, ph, window),
                 lambda: w.monopulse(th, ph, window, 0.05, 1.4)):
        with pytest.raises(bflk.BflkError) as e:
            call()
        assert e.value.code == BFLK_ERR_INVALID
    import torch
    win_dev = torch.from_numpy(window).cuda()
    audio = torch.zeros((2, 256), device="cuda")
    with pytest.raises(bflk.BflkError) as e:
        w.miso_dev(th, ph, win_dev.data_ptr(), audio.data_ptr(), 0)
    assert e.value.code == BFLK_ERR_INVALID
    w.set_geometry(xyz)                      # back inside the focus: the focus of 6 m still holds
    w.set_grid_fov(1, 1, 90.0)
    off, fr = w.tables()
    assert np.array_equal(off, before[0]) and same_bits(fr, before[1])
    w.close()


# ---- power maps, beams, sessions and Targets on a focused grid -----------------------------------------------------
def _cpu_power(oracle, window, off, fr, n):
    import os
    if oracle.ref() is not None:
        return oracle.ref_mimo_update(window, off, fr, n=n, n_threads=os.cpu_count() or 1)
    return oracle.mimo_update(window, off, fr, n=n)


@pytest.mark.gpu
@pytest.mark.parametrize("name,r", [("cfg1", 1.0), ("cfg2", 3.0), ("cfg3", 5.0), ("cfg3", 2.0)])
def test_focused_power_maps_every_kernel(oracle, name, r):
    import bflk
    import torch
    from bflk import synth
    c = cases.CONFIGS[name]
    xyz = tiled_xyz(oracle, name)
    th, ph = oracle.mimo_grid(c["rows"], c["cols"], c["fov"])
    src = synth.nearest_direction(th, ph, np.deg2rad(20.0), np.deg2rad(30.0))
    stream = synth.point_source_stream(xyz, c["N"] + c["W"], [(th[src], ph[src], r, 9000.0, 1e-2)])
    window = np.ascontiguousarray(stream[:, :c["W"]])
    w = bflk.MIMOWorker(cases.origins(*TILED[name]), c["rows"], c["cols"], c["fov"])
    w.set_focus(r)
    off, fr = w.tables()
    eo, ef = F.mimo_lut_focus(oracle, xyz, c["rows"], c["cols"], c["fov"], r)
    assert np.array_equal(off, eo) and same_bits(fr, ef)
    ref = _cpu_power(oracle, window, off, fr, c["N"])
    for kernel in (1, 2, 3, 4):
        w.set_kernel(kernel)
        p = w.update(window)
        assert w.kernel_info()[0] == kernel
        assert rel_err(p, ref) <= POWER_RTOL and int(np.argmax(p)) == int(np.argmax(ref)), kernel
    w.set_kernel(0)
    w.set_channel_split(True)
    p = w.update(window)
    assert rel_err(p, ref) <= POWER_RTOL and int(np.argmax(p)) == int(np.argmax(ref))
    w.set_channel_split(False)
    # kernel 2 beams: the oracle's delayed sums bit for bit
    w.set_kernel(2)
    x = torch.from_numpy(stream).cuda()
    beams = torch.full((2, off.shape[0], c["N"]), float("nan"), device="cuda")
    power = torch.full((2, off.shape[0]), float("nan"), device="cuda")
    w.beams_batch_dev(x.data_ptr(), x.shape[1], 2, beams.data_ptr(), power.data_ptr())
    torch.cuda.synchronize()
    for b in range(2):
        exp = oracle.mimo_das(np.ascontiguousarray(stream[:, b * c["N"]:]), off, fr, None, c["N"])
        assert same_bits(beams[b].cpu().numpy(), exp), b
    w.close()


@pytest.mark.gpu
def test_focused_session_maps_beams_and_targets_equal_the_batch(oracle):
    import bflk
    import torch
    from bflk import synth
    c = cases.CONFIGS["cfg3"]
    N, H, B = c["N"], c["H"], 6
    xyz = tiled_xyz(oracle, "cfg3")
    th, ph = oracle.mimo_grid(c["rows"], c["cols"], c["fov"])
    src = synth.nearest_direction(th, ph, np.deg2rad(20.0), np.deg2rad(30.0))
    T = (B - 1) * N + H + N + 2
    stream = synth.point_source_stream(xyz, T, [(th[src], ph[src], 4.0, 9000.0, 1e-2), (0.0, 0.0, 8.0, 3000.0, 5e-3)])
    w = bflk.MIMOWorker(cases.origins(4, 2), c["rows"], c["cols"], c["fov"])
    w.set_focus(4.0)
    maps = w.power_map_batch(stream, B)
    x = torch.from_numpy(stream).cuda()
    beams = torch.empty((B, c["rows"] * c["cols"], N), device="cuda")
    power = torch.empty((B, c["rows"] * c["cols"]), device="cuda")
    w.beams_batch_dev(x.data_ptr(), T, B, beams.data_ptr(), power.data_ptr())
    torch.cuda.synchronize()
    beams = beams.cpu().numpy()
    assert same_bits(power.cpu().numpy(), maps)
    w.stream_open(16)
    w.stream_push(stream)
    f0, p0 = w.stream_power_maps(2)
    f1, b1, p1 = w.stream_beams(2)
    f2, p2, tg = w.stream_targets(2, max_targets=4, min_rel_power=0.2)
    assert (f0, f1, f2) == (0, 2, 4)
    assert same_bits(p0, maps[0:2]) and same_bits(p1, maps[2:4]) and same_bits(b1, beams[2:4]) and same_bits(p2, maps[4:6])
    for i, b in enumerate((4, 5)):
        assert tg[i] == w.targets(maps[b], max_targets=4, min_rel_power=0.2)
    assert tg[0][0]["direction"] == src                      # the focused source is the strongest peak
    w.close()


# ---- MISO, FIR MISO and monopulse ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("geom,speed,H,N,r", [("tiles3d", 0, 256, 256, 0.6), ("cube", 2, 100, 188, 3.0),
                                              ("vertical", 1, 255, 65, 1e5)])
def test_focused_miso_vs_oracle(oracle, geom, speed, H, N, r):
    import torch
    sr, c = SPEEDS[speed]
    k = oracle.delay_scale(sr, c)
    C = 128
    xyz, origins = geometry(geom, C, 0.25)
    W = H + N + 1
    w = handle(xyz, origins, N=N, H=H, W=W, sample_rate=sr, speed=c)
    mask = np.random.default_rng(N).permutation(C)[:97].astype(np.int32)
    w.set_channel_mask(mask)
    window = window_for(C, W, N + H)
    rng = np.random.default_rng(H)
    T = 140                                       # more than the directions passed inline
    th, ph = rng.random(T) * 1.4, rng.random(T) * 2 * np.pi
    w.set_focus(r)
    eo, ef = F.steer_tables_focus(xyz, th, ph, r, history=H, scale=k)
    assert eo.min() >= 0
    audio, power = w.miso(th, ph, window)
    for t in range(T):
        assert same_bits(audio[t], oracle.particle_das(window, eo[t], ef[t], index=mask, n=N)), t
        ref = oracle.particle_beam(window, eo[t], ef[t], index=mask, n=N)
        assert abs(power[t] - ref) <= POWER_RTOL * ref, t
    # bflk_miso_dev: the same bits
    win_dev = torch.from_numpy(window).cuda()
    a_dev = torch.full((T, N), float("nan"), device="cuda")
    p_dev = torch.full((T,), float("nan"), device="cuda")
    w.miso_dev(th, ph, win_dev.data_ptr(), a_dev.data_ptr(), p_dev.data_ptr())
    torch.cuda.synchronize()
    assert same_bits(a_dev.cpu().numpy(), audio) and same_bits(p_dev.cpu().numpy(), power)
    # monopulse: quadrant directions of the far-field code path, their beams on focused tables
    limit, spread = np.deg2rad(80.0), np.deg2rad(4.0)
    P = 9
    got = w.monopulse(th[:P], ph[:P], window, spread, limit)
    for p in range(P):
        theta_p, nth, nph = oracle.quadrant(th[p], ph[p], spread, limit)
        assert got[0][p] == theta_p and np.array_equal(got[1][p], nth) and np.array_equal(got[2][p], nph)
        qo, qf = F.steer_tables_focus(xyz, nth, nph, r, history=H, scale=k)
        q = [oracle.particle_beam(window, qo[j], qf[j], index=mask, n=N) for j in range(4)]
        assert rel_err(got[3][p], q) <= POWER_RTOL, p
    w.close()


@pytest.mark.gpu
def test_focused_fir_miso_vs_oracle(oracle, golden):
    coeffs = golden["fir"]["coeffs"]
    sr, c = SPEEDS[0]
    H, N, C = 64, 256, 128
    k = oracle.delay_scale(sr, c)
    xyz, _ = geometry("cube", C, 0.15)
    W = H + N + coeffs.shape[1] - 1
    w = handle(xyz, N=N, H=H, W=W, sample_rate=sr, speed=c)
    w.set_fir(coeffs)
    w.set_focus(0.8)
    window = window_for(C, W, 3)
    th, ph = np.random.default_rng(4).random(12) * 1.4, np.random.default_rng(5).random(12) * 6.3
    audio, power = w.miso(th, ph, window)
    eo, ef = F.steer_tables_focus(xyz, th, ph, 0.8, history=H, scale=k)
    for t in range(len(th)):
        exp = oracle.particle_das_fir(window, eo[t], ef[t], coeffs, n=N)
        assert same_bits(audio[t], exp), t
        assert abs(power[t] - hp_power(exp, N)) <= POWER_RTOL * hp_power(exp, N), t
    w.close()


# ---- physics ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_focusing_recovers_a_point_source_at_5m(oracle):
    """cfg3 (2 x 4 tiles, 0.64 m), a 9 kHz point source 5 m away on the grid node nearest theta 20, phi 30 deg: the focused
    map peaks at the source's cell, and the far-field map loses more than 15 % of the power there."""
    import bflk
    from bflk import synth
    c = cases.CONFIGS["cfg3"]
    xyz = tiled_xyz(oracle, "cfg3")
    th, ph = oracle.mimo_grid(c["rows"], c["cols"], c["fov"])
    src = synth.nearest_direction(th, ph, np.deg2rad(20.0), np.deg2rad(30.0))
    window = synth.point_source_stream(xyz, c["W"], [(th[src], ph[src], 5.0, 9000.0, 1e-2)])
    w = bflk.MIMOWorker(cases.origins(4, 2), c["rows"], c["cols"], c["fov"])
    far = w.update(window)
    w.set_focus(5.0)
    near = w.update(window)
    assert int(np.argmax(near)) == src
    assert far[src] / near[src] < 0.85, far[src] / near[src]
    w.close()


# ---- group ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_group_set_focus_equals_a_focused_handle(oracle):
    import torch
    import bflk
    from bflk import synth
    c = cases.CONFIGS["cfg3"]
    B = 5
    stream = synth.make_stream(tiled_xyz(oracle, "cfg3"), (B - 1) * c["N"] + c["W"])
    single = bflk.MIMOWorker(cases.origins(4, 2), c["rows"], c["cols"], c["fov"])
    single.set_focus(2.5)
    ref = single.power_map_batch(stream, B)
    n = min(torch.cuda.device_count(), 2)
    g = bflk.Group(cases.origins(4, 2), c["rows"], c["cols"], c["fov"], devices=list(range(n)))
    g.set_focus(2.5)
    assert np.array_equal(g.power_map_batch(stream, B), ref)
    with pytest.raises(bflk.BflkError) as e:
        g.set_focus(-3.0)
    assert e.value.code == BFLK_ERR_INVALID
    assert np.array_equal(g.power_map_batch(stream, B), ref)
    g.close()
    single.close()
