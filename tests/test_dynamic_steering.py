"""Dynamic steering against the CPU oracle across its configuration space: bflk_steer_tables and the grid tables of
bflk_set_grid_fov, the fused MISO kernel behind bflk_miso / bflk_miso_dev (it builds its steering table inside the kernel),
the FIR form of MISO, bflk_monopulse, and the order of MISO calls made on several streams.

Geometries are 3-D (random points in a cube, a vertical line, tiles at different heights), speeds of sound and sample rates
differ from the reference's constants, frame lengths straddle the kernel's 62-output slices, histories run from 0 to 1000,
masks are unsorted, and target counts straddle the switch between directions passed inline and staged ones.

Bars: steering tables (offsets and fraction bits), MISO audio and monopulse quadrant directions bit-exact; MISO power and
monopulse q within 1e-4 relative."""
import numpy as np
import pytest

import cases

POWER_RTOL = 1e-4
BFLK_ERR_INVALID, BFLK_ERR_RANGE = -1, -5
MISO_INLINE = 128           # directions that travel in the MISO kernel's parameter space (kMisoInline)
SPEEDS = [(48828.0, 343.0), (16000.0, 1480.0), (96000.0, 343.0), (48828.0, 1480.0)]   # (sample rate, propagation speed)


# ---- geometry and inputs --------------------------------------------------------------------------------------------
def cube(C, side, seed=1):
    """C points drawn uniformly from a cube of the given side, centred on the origin."""
    rng = np.random.default_rng(seed)
    return ((rng.random((C, 3)) - 0.5) * side).astype(np.float32)


def vertical_line(C, pitch):
    xyz = np.zeros((C, 3), np.float32)
    xyz[:, 2] = (np.arange(C) - (C - 1) / 2) * pitch
    return xyz


TILE_ORIGINS = np.array([[-0.08, -0.08, 0.0], [0.08, -0.08, 0.05], [-0.08, 0.08, -0.03], [0.08, 0.08, 0.11]], np.float32)


def geometry(name, C, extent):
    """(xyz, tile origins or None): the named 3-D geometry with its largest span about `extent` metres."""
    if name == "cube":
        return cube(C, extent / np.sqrt(3.0)), None
    if name == "vertical":
        return vertical_line(C, extent / (C - 1)), None
    assert name == "tiles3d" and C % 64 == 0
    from oracle import oracle as O
    origins = TILE_ORIGINS[:C // 64] * np.float32(extent / 0.35)
    return O.create_tiled_antenna(origins), origins


def fit_extent(H, sample_rate, speed, limit=0.3):
    """An array span whose largest delay stays within 90 % of a history of H samples."""
    return min(limit, 0.9 * H * speed / sample_rate) if H > 0 else limit


def window_for(C, W, seed):
    return np.random.default_rng(seed).standard_normal((C, W)).astype(np.float32)


def directions(T, seed, theta_max=np.pi / 2):
    rng = np.random.default_rng(seed)
    return rng.random(T) * theta_max, rng.random(T) * 2 * np.pi


def edge_directions():
    """theta 0 and pi / 2 with phi at 0, just below 2 pi, negative and above 2 pi."""
    th, ph = np.meshgrid([0.0, np.pi / 2], [0.0, np.nextafter(2 * np.pi, 0.0), -0.7, 2 * np.pi + 0.9])
    return th.ravel(), ph.ravel()


def hp_power(audio, N):
    """Particle::beam in double: the 3-tap high-pass of the delayed sum, mean square over N."""
    a = audio.astype(np.float64)
    ma = 0.5 * a[1:-1] - 0.25 * (a[2:] + a[:-2])
    return float(np.sum(ma * ma) / N)


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a, np.float32).view(np.uint32), np.ascontiguousarray(b, np.float32).view(np.uint32))


def handle(xyz, origins=None, N=256, H=256, W=None, sample_rate=48828.0, speed=340.0):
    import bflk
    w = bflk.Beamformer(n_channels=xyz.shape[0], frame_len=N, history=H, window_len=H + N + 1 if W is None else W,
                        sample_rate=sample_rate, propagation_speed=speed)
    if origins is not None:
        w.set_tiled_geometry(origins)
    else:
        w.set_geometry(xyz)
    assert np.array_equal(w.geometry(), xyz)
    return w


# ---- the oracle (CPU) ------------------------------------------------------------------------------------------------
def test_default_scale_reproduces_the_golden_tables(oracle, golden):
    """The delay scale threaded through the oracle keeps the bits of the reference's constants."""
    import hashlib
    g = golden["tables"]
    k = oracle.delay_scale()
    assert k == oracle.delay_scale(oracle.SAMPLE_RATE, oracle.PROPAGATION_SPEED) == float(np.float32(48828.0 / 340.0))
    for name in ("cfg1", "cfg3"):
        c = cases.CONFIGS[name]
        xyz = oracle.create_tiled_antenna(cases.origins(c["nx"], c["ny"]))
        off, fr = oracle.mimo_lut(xyz, c["rows"], c["cols"], c["fov"], c["H"], scale=k)
        assert hashlib.sha256(off.tobytes()).digest() == g[f"{name}_off_sha"].tobytes()
        assert hashlib.sha256(fr.tobytes()).digest() == g[f"{name}_frac_sha"].tobytes()
    th, ph = cases.cfg4_targets()
    xyz = oracle.create_tiled_antenna(cases.origins(4, 2))
    for scale in (None, k):
        off, fr = oracle.steer_tables(xyz, th, ph, history=256, scale=scale)
        assert np.array_equal(off, g["cfg4_off"]) and same_bits(fr, g["cfg4_frac"])
    # another scale changes the delays in proportion
    d1 = oracle.steering_vector_spherical(xyz, 0.5, 1.0, scale=k)
    d2 = oracle.steering_vector_spherical(xyz, 0.5, 1.0, scale=oracle.delay_scale(16000.0, 1480.0))
    assert np.allclose(d2, d1 * (16000.0 / 1480.0) / k, rtol=1e-5, atol=1e-4)


def test_unit_scale_boresight_delays_are_heights(oracle):
    """sample_rate == propagation_speed and integer heights: every boresight delay is exactly z - min z."""
    rng = np.random.default_rng(3)
    xyz = np.c_[rng.random((40, 2)) - 0.5, rng.integers(-7, 30, 40)].astype(np.float32)
    for phi in (0.0, 1.3, -0.4, 2 * np.pi + 0.2):
        d = oracle.steering_vector_spherical(xyz, 0.0, phi, scale=oracle.delay_scale(343.0, 343.0))
        assert np.array_equal(d, xyz[:, 2] - xyz[:, 2].min())
        off, fr = oracle.split_delays(d, 50)
        assert np.array_equal(off, 50 - (xyz[:, 2] - xyz[:, 2].min()).astype(np.int32)) and not fr.any()


def test_fir_delayed_sum_oracle(oracle, golden):
    """particle_das_fir: a one-tap table sums the shifted samples in mask order; the golden table through it agrees with
    the FIR power map of the same direction."""
    rng = np.random.default_rng(5)
    C, N, W = 12, 40, 80
    window = window_for(C, W, 6)
    off = rng.integers(0, 30, C).astype(np.int32)
    fr = rng.random(C).astype(np.float32)
    mask = rng.permutation(C)[:9].astype(np.int32)
    one_tap = np.zeros((5, 8), np.float32)
    one_tap[:, 3] = 1.0
    exp = np.zeros(N, np.float32)
    for c in mask:
        exp = (exp + window[c, off[c] + 3:off[c] + 3 + N]).astype(np.float32)
    assert same_bits(oracle.particle_das_fir(window, off, fr, one_tap, index=mask, n=N), exp)
    coeffs = golden["fir"]["coeffs"]
    audio = oracle.particle_das_fir(window, off, fr, coeffs, index=mask, n=N)
    p = oracle.mimo_update_fir(window, off[None], fr[None], coeffs, index=mask, n=N)[0]
    assert abs(hp_power(audio, N) / len(mask) - p) <= POWER_RTOL * p


# ---- steering tables ----------------------------------------------------------------------------------------------
def _expect_tables(got_fn, exp_off, exp_fr, H):
    """Bits of the oracle's tables when their largest delay fits the history, BFLK_ERR_RANGE when it does not."""
    import bflk
    if exp_off.min() < 0:                        # offset = H - delay: a delay beyond the history
        with pytest.raises(bflk.BflkError) as e:
            got_fn()
        assert e.value.code == BFLK_ERR_RANGE
        return False
    off, fr = got_fn()
    assert np.array_equal(off, exp_off) and same_bits(fr, exp_fr)
    return True


@pytest.mark.gpu
@pytest.mark.parametrize("geom", ["cube", "vertical", "tiles3d"])
@pytest.mark.parametrize("speed", SPEEDS)
def test_tables_vs_oracle(oracle, geom, speed):
    """bflk_steer_tables and the set_grid_fov tables, bit for bit, at every history; out of range: BFLK_ERR_RANGE."""
    sr, c = speed
    k = oracle.delay_scale(sr, c)
    C = 128 if geom == "tiles3d" else 64
    xyz, origins = geometry(geom, C, 0.3)
    th, ph = edge_directions()
    rth, rph = directions(24, 11)
    th, ph = np.r_[th, rth], np.r_[ph, rph]
    checked = 0
    for H in (16, 100, 255, 257, 1000):
        w = handle(xyz, origins, N=64, H=H, sample_rate=sr, speed=c)
        eo, ef = oracle.steer_tables(xyz, th, ph, history=H, scale=k)
        if not _expect_tables(lambda: w.steer_tables(th, ph), eo, ef, H):
            # the directions that fit still come out exact one by one
            fit = [t for t in range(len(th)) if eo[t].min() >= 0]
            if fit:
                assert _expect_tables(lambda: w.steer_tables(th[fit], ph[fit]), eo[fit], ef[fit], H)
        go, gf = oracle.mimo_lut(xyz, 7, 9, 150.0, H, scale=k)

        def grid():
            w.set_grid_fov(7, 9, 150.0)
            return w.tables()
        checked += _expect_tables(grid, go, gf, H)
        w.close()
    assert checked >= 3          # most histories hold the whole grid: the comparison is not vacuous


# ---- MISO audio and power -------------------------------------------------------------------------------------------
# (N, H, C, usable, T, geometry, speed index, window slack)
MISO_CASES = [
    (3, 17, 64, 64, 5, "cube", 0, 0),
    (4, 1, 64, 33, 7, "cube", 1, 0),
    (63, 64, 96, 63, 128, "vertical", 2, 0),
    (64, 255, 256, 31, 129, "tiles3d", 3, 0),
    (65, 17, 128, 65, 9, "cube", 0, 0),
    (66, 64, 64, 2, 3, "cube", 2, 0),
    (127, 1000, 512, 511, 16, "cube", 2, 0),
    (128, 64, 64, 1, 4, "vertical", 1, 0),
    (188, 255, 256, 32, 128, "tiles3d", 0, 0),
    (250, 17, 64, 64, 1, "cube", 3, 0),
    (256, 1000, 128, 128, 1000, "cube", 0, 0),
    (300, 64, 64, 64, 33, "vertical", 2, 37),
    (1000, 255, 128, 128, 8, "tiles3d", 1, 0),
    (4096, 17, 64, 64, 3, "cube", 0, 0),
]


def _check_miso(w, oracle, xyz, window, th, ph, H, N, k, mask=None, check_every=1):
    """bflk_miso against Particle::das / Particle::beam of the oracle; audio-only and power-only calls give the same bits."""
    audio, power = w.miso(th, ph, window)
    a2, none = w.miso(th, ph, window, want_power=False)
    none2, p2 = w.miso(th, ph, window, want_audio=False)
    assert none is None and none2 is None
    assert same_bits(a2, audio) and same_bits(p2, power)
    off, fr = oracle.steer_tables(xyz, th, ph, history=H, scale=k)
    for t in range(0, len(th), check_every):
        exp = oracle.particle_das(window, off[t], fr[t], index=mask, n=N)
        assert same_bits(audio[t], exp), t
        ref = oracle.particle_beam(window, off[t], fr[t], index=mask, n=N)
        assert abs(power[t] - ref) <= POWER_RTOL * ref, (t, power[t], ref)
    return audio, power


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,C,usable,T,geom,speed,slack", MISO_CASES)
def test_miso_vs_oracle(oracle, N, H, C, usable, T, geom, speed, slack):
    sr, c = SPEEDS[speed]
    k = oracle.delay_scale(sr, c)
    xyz, origins = geometry(geom, C, fit_extent(H, sr, c))
    W = H + N + 1 + slack
    w = handle(xyz, origins, N=N, H=H, W=W, sample_rate=sr, speed=c)
    mask = None
    if usable < C:   # unsorted: channels are summed in mask order
        mask = np.random.default_rng(N + C).permutation(C)[:usable].astype(np.int32)
        w.set_channel_mask(mask)
    window = window_for(C, W, N + H)
    th, ph = directions(T, N * 7 + H)
    _check_miso(w, oracle, xyz, window, th, ph, H, N, k, mask, check_every=1 if T <= 200 else 7)
    w.close()


@pytest.mark.gpu
def test_miso_4096_channels(oracle):
    """4096 channels: the MISO kernel's per-channel tables need 64 KB of shared memory, more than the default 48 KB."""
    sr, c = SPEEDS[0]
    H, N, C = 64, 256, 4096
    k = oracle.delay_scale(sr, c)
    xyz, _ = geometry("cube", C, fit_extent(H, sr, c))
    w = handle(xyz, N=N, H=H, sample_rate=sr, speed=c)
    window = window_for(C, H + N + 1, 41)
    th, ph = directions(4, 42)
    _check_miso(w, oracle, xyz, window, th, ph, H, N, k)
    off, fr = w.steer_tables(th, ph)
    eo, ef = oracle.steer_tables(xyz, th, ph, history=H, scale=k)
    assert np.array_equal(off, eo) and same_bits(fr, ef)
    w.close()


@pytest.mark.gpu
def test_miso_inline_staged_inline(oracle):
    """128 -> 129 -> 128 targets on one handle: directions in the kernel's parameters, then staged, then inline again."""
    sr, c = SPEEDS[2]
    H, N = 100, 188
    k = oracle.delay_scale(sr, c)
    xyz, origins = geometry("tiles3d", 128, fit_extent(H, sr, c))
    w = handle(xyz, origins, N=N, H=H, sample_rate=sr, speed=c)
    window = window_for(128, H + N + 1, 8)
    th, ph = directions(MISO_INLINE + 1, 9)
    a0, p0 = _check_miso(w, oracle, xyz, window, th[:MISO_INLINE], ph[:MISO_INLINE], H, N, k)
    a1, p1 = _check_miso(w, oracle, xyz, window, th, ph, H, N, k)
    assert same_bits(a1[:MISO_INLINE], a0) and same_bits(p1[:MISO_INLINE], p0)
    a2, p2 = w.miso(th[:MISO_INLINE], ph[:MISO_INLINE], window)
    assert same_bits(a2, a0) and same_bits(p2, p0)
    w.close()


@pytest.mark.gpu
def test_miso_without_history(oracle):
    """H = 0: boresight on a level array has no delay; a tilt below one sample still fits; one whose largest delay reaches a
    sample is out of range."""
    import bflk
    sr, c = SPEEDS[0]
    k = oracle.delay_scale(sr, c)
    N, C = 256, 64
    xyz = cube(C, 0.2)
    xyz[:, 2] = 0.0
    w = handle(xyz, N=N, H=0, sample_rate=sr, speed=c)
    window = window_for(C, N + 1, 12)
    span = float(np.ptp(xyz[:, 0]) + np.ptp(xyz[:, 1]))
    small = 0.5 / (k * span)                         # largest delay below half a sample
    _check_miso(w, oracle, xyz, window, np.array([0.0, small, small]), np.array([0.0, 0.3, 4.0]), 0, N, k)
    big = np.arcsin(min(1.0, 4.0 / (k * float(np.ptp(xyz[:, 0])))))   # about 4 samples along x
    assert oracle.steering_vector_spherical(xyz, big, 0.0, scale=k).max() >= 1.0
    with pytest.raises(bflk.BflkError) as e:
        w.miso([big], [0.0], window)
    assert e.value.code == BFLK_ERR_RANGE
    w.close()


# ---- the range boundary ------------------------------------------------------------------------------------------
def _heights_array(C, top, seed):
    """Microphones at integer heights 0..top (the far one at `top`, channel C - 1), small random x / y."""
    rng = np.random.default_rng(seed)
    z = np.r_[0, rng.integers(0, top, C - 2), top]
    return np.c_[rng.random((C, 2)) * 0.05, z].astype(np.float32)


@pytest.mark.gpu
def test_range_boundary(oracle):
    """Scale exactly 1 (sample_rate == propagation_speed) and integer heights: boresight delays are the heights.  A largest
    delay of H fits (offset 0); H + 1 does not: bflk_miso, bflk_steer_tables and set_grid_fov refuse it, bflk_miso_dev clamps
    it.  The range flag of a failed or clamped call does not leak into the next call."""
    import bflk
    import torch
    H, N, C = 40, 128, 64
    W = H + N + 1
    fits, over = _heights_array(C, H, 1), _heights_array(C, H + 1, 1)
    w = handle(fits, N=N, H=H, W=W, sample_rate=343.0, speed=343.0)
    window = window_for(C, W, 2)
    bore = (np.zeros(1), np.zeros(1))
    off, fr = w.steer_tables(*bore)
    assert off[0, C - 1] == 0 and np.array_equal(off[0], H - fits[:, 2].astype(np.int32)) and not fr.any()
    _check_miso(w, oracle, fits, window, *bore, H, N, 1.0)
    w.set_grid_fov(1, 1, 90.0)                                     # a 1 x 1 grid is boresight
    assert np.array_equal(w.tables()[0], off)

    w.set_geometry(over)
    for call in (lambda: w.miso(*bore, window), lambda: w.steer_tables(*bore), lambda: w.set_grid_fov(1, 1, 90.0)):
        with pytest.raises(bflk.BflkError) as e:
            call()
        assert e.value.code == BFLK_ERR_RANGE
    # bflk_miso_dev cannot report it: the offset is clamped to 0
    eo, ef = oracle.steer_tables(over, *bore, history=H, scale=1.0)
    assert eo[0, C - 1] == -1
    clamped = np.maximum(eo, 0)
    win_dev = torch.from_numpy(window).cuda()
    audio = torch.zeros((1, N), dtype=torch.float32, device="cuda")
    power = torch.zeros(1, dtype=torch.float32, device="cuda")
    w.miso_dev(*bore, win_dev.data_ptr(), audio.data_ptr(), power.data_ptr())
    torch.cuda.synchronize()
    assert same_bits(audio.cpu().numpy()[0], oracle.particle_das(window, clamped[0], ef[0], n=N))

    # the next valid call succeeds, after the clamped call and after a refused one
    w.set_geometry(fits)
    a1, _ = w.miso(*bore, window)
    w.set_geometry(over)
    with pytest.raises(bflk.BflkError):
        w.miso(*bore, window)
    w.set_geometry(fits)
    a2, _ = w.miso(*bore, window)
    assert same_bits(a1, a2)

    # the far microphone outside the mask: MISO checks the channels it sums, the table calls check every channel
    w.set_geometry(over)
    mask = np.arange(C - 2, -1, -1, dtype=np.int32)
    w.set_channel_mask(mask)
    am, pm = w.miso(*bore, window)
    assert same_bits(am[0], oracle.particle_das(window, eo[0], ef[0], index=mask, n=N))
    with pytest.raises(bflk.BflkError) as e:
        w.steer_tables(*bore)
    assert e.value.code == BFLK_ERR_RANGE
    w.close()


# ---- device calls ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("T", [16, 200])
def test_miso_dev_equals_miso(T):
    """bflk_miso_dev on an explicit window and on a borrowed resident one, on the handle's stream and on a caller's stream,
    gives the bits of bflk_miso."""
    import torch
    from oracle import oracle as O
    sr, c = SPEEDS[1]
    H, N, C = 255, 300, 192
    xyz, origins = geometry("tiles3d", C, fit_extent(H, sr, c))
    w = handle(xyz, origins, N=N, H=H, sample_rate=sr, speed=c)
    mask = np.random.default_rng(4).permutation(C)[:150].astype(np.int32)
    w.set_channel_mask(mask)
    window = window_for(C, H + N + 1, 13)
    th, ph = directions(T, 14)
    a_ref, p_ref = w.miso(th, ph, window)
    off, fr = O.steer_tables(xyz, th, ph, history=H, scale=O.delay_scale(sr, c))
    assert same_bits(a_ref[0], O.particle_das(window, off[0], fr[0], index=mask, n=N))
    win_dev = torch.from_numpy(window).cuda()
    st = torch.cuda.Stream()
    for resident in (False, True):
        w.set_window_dev(win_dev.data_ptr() if resident else None)
        for stream in (0, st.cuda_stream):
            audio = torch.full((T, N), np.nan, dtype=torch.float32, device="cuda")
            power = torch.full((T,), np.nan, dtype=torch.float32, device="cuda")
            w.miso_dev(th, ph, None if resident else win_dev.data_ptr(), audio.data_ptr(), power.data_ptr(), stream)
            torch.cuda.synchronize()
            assert same_bits(audio.cpu().numpy(), a_ref) and same_bits(power.cpu().numpy(), p_ref), (resident, stream)
    a_res, p_res = w.miso(th, ph)                               # bflk_miso on the borrowed window
    assert same_bits(a_res, a_ref) and same_bits(p_res, p_ref)
    w.set_window_dev(None)
    w.close()


# ---- FIR MISO -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("N", [63, 256, 300])
def test_fir_miso_vs_oracle(oracle, golden, N):
    """bflk_set_fir with the reference's 101 x 8 table: audio bit-exact against the FIR delayed sum, power within 1e-4; a
    window too short for the taps is refused."""
    import bflk
    coeffs = golden["fir"]["coeffs"]
    taps = coeffs.shape[1]
    sr, c = SPEEDS[0]
    H, C = 64, 128
    k = oracle.delay_scale(sr, c)
    xyz, _ = geometry("cube", C, fit_extent(H, sr, c))
    W = H + N + taps - 1
    w = handle(xyz, N=N, H=H, W=W, sample_rate=sr, speed=c)
    mask = np.random.default_rng(N).permutation(C)[:100].astype(np.int32)
    w.set_channel_mask(mask)
    w.set_fir(coeffs)
    window = window_for(C, W, N)
    th, ph = directions(12, N + 1)
    audio, power = w.miso(th, ph, window)
    off, fr = oracle.steer_tables(xyz, th, ph, history=H, scale=k)
    for t in range(len(th)):
        exp = oracle.particle_das_fir(window, off[t], fr[t], coeffs, index=mask, n=N)
        assert same_bits(audio[t], exp), t
        assert abs(power[t] - hp_power(exp, N)) <= POWER_RTOL * hp_power(exp, N)
    w.close()
    short = handle(xyz, N=N, H=H, W=W - 1, sample_rate=sr, speed=c)
    short.set_fir(coeffs)
    with pytest.raises(bflk.BflkError) as e:
        short.miso(th, ph, window[:, :W - 1])
    assert e.value.code == BFLK_ERR_INVALID
    short.close()


# ---- monopulse ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("geom,speed,H,N", [("tiles3d", 2, 100, 256), ("cube", 1, 17, 188), ("vertical", 3, 255, 65)])
@pytest.mark.parametrize("P", [1, 32, 33])
def test_monopulse_vs_oracle(oracle, geom, speed, H, N, P):
    """Quadrant directions bit-exact and q within 1e-4 on 3-D arrays at other speeds and histories, with a mask; phi near 0
    and 2 pi, theta at 0, at the limit and on the pull-in branch; reference 0 and > 0."""
    sr, c = SPEEDS[speed]
    k = oracle.delay_scale(sr, c)
    C = 128
    xyz, origins = geometry(geom, C, fit_extent(H, sr, c))
    w = handle(xyz, origins, N=N, H=H, sample_rate=sr, speed=c)
    mask = np.random.default_rng(P).permutation(C)[:77].astype(np.int32)
    w.set_channel_mask(mask)
    window = window_for(C, H + N + 1, P + H)
    limit, spread = np.deg2rad(80.0), np.deg2rad(4.0)
    rng = np.random.default_rng(P + 100)
    theta = np.r_[0.0, limit, np.pi / 2 - 0.01, limit - 1e-3, rng.random(max(0, P - 4)) * limit][:P]
    phi = np.r_[1e-9, np.nextafter(2 * np.pi, 0.0), 2 * np.pi - 1e-3, 0.0, rng.random(max(0, P - 4)) * 2 * np.pi][:P]
    for reference in (0.0, 3e-4):
        got = w.monopulse(theta, phi, window, spread, limit, reference=reference)
        exp = oracle.monopulse(xyz, theta, phi, window, spread, limit, reference=reference, index=mask, history=H, scale=k,
                               n=N)
        assert np.array_equal(got[0], exp[0])
        assert np.array_equal(got[1], exp[1]) and np.array_equal(got[2], exp[2])
        assert rel_err(got[3], exp[3]) <= POWER_RTOL
        div = reference if reference > 0 else 1.0
        scale = np.abs(exp[3]).sum(axis=1) / div
        assert np.all(np.abs(got[4][:, :2] - exp[4][:, :2]) <= 4 * POWER_RTOL * scale[:, None])
        assert np.all(np.abs(got[4][:, 2] - exp[4][:, 2]) <= POWER_RTOL * exp[4][:, 2])
        assert np.all(np.abs(got[5] - exp[5]) <= 8 * POWER_RTOL)
    if P > 2:
        assert got[0][2] < theta[2]                                 # the pull-in branch was taken
    w.close()


# ---- calls on several streams ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_miso_calls_on_two_streams_are_ordered():
    """MISO calls with power outputs share the handle's partial sums: bflk_miso_dev on stream A and then on stream B must
    not overlap, and a bflk_miso on the resident window right after a bflk_miso_dev on A sees what A did before it.  Both
    streams are held behind one event so that, unordered, their kernels would run at the same time; long frames make each
    kernel several waves of CTAs, so the two grids' slices of a target would interleave."""
    import torch
    sr, c = SPEEDS[0]
    H, N, C, T = 64, 4096, 128, 128
    xyz, origins = geometry("tiles3d", C, fit_extent(H, sr, c))
    w = handle(xyz, origins, N=N, H=H, sample_rate=sr, speed=c)
    wins = [torch.from_numpy(window_for(C, H + N + 1, s)).cuda() for s in (31, 32)]
    dirs = [directions(T, s) for s in (33, 34)]
    solo = [w.miso(*dirs[i], wins[i].cpu().numpy()) for i in range(2)]
    gate, sa, sb = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    outs = [[torch.empty((T, N), device="cuda"), torch.empty(T, device="cuda")] for _ in range(8)]

    def run(i, j, stream):
        w.miso_dev(*dirs[i], wins[i].data_ptr(), outs[j][0].data_ptr(), outs[j][1].data_ptr(), stream.cuda_stream)

    for s in (sa, sb):       # warm up: buffers sized, nothing left to reserve or synchronise between the gated calls
        run(0, 0, s)
    torch.cuda.synchronize()
    with torch.cuda.stream(gate):
        torch.cuda._sleep(20_000_000)
    ev = torch.cuda.Event()
    ev.record(gate)
    sa.wait_event(ev)
    sb.wait_event(ev)
    for j in range(0, 8, 2):
        run(0, j, sa)
        run(1, j + 1, sb)
    torch.cuda.synchronize()
    for j in range(8):
        a, p = solo[j % 2]
        assert same_bits(outs[j][0].cpu().numpy(), a) and same_bits(outs[j][1].cpu().numpy(), p), j

    # bflk_miso on the resident window right after a bflk_miso_dev on A: A fills the window before its call
    resident = torch.zeros_like(wins[1])
    w.set_window_dev(resident.data_ptr())
    with torch.cuda.stream(gate):
        torch.cuda._sleep(20_000_000)
    ev = torch.cuda.Event()
    ev.record(gate)
    sa.wait_event(ev)
    with torch.cuda.stream(sa):
        resident.copy_(wins[1])
    run(0, 0, sa)
    a, p = w.miso(*dirs[1])
    torch.cuda.synchronize()
    assert same_bits(a, solo[1][0]) and same_bits(p, solo[1][1])
    assert same_bits(outs[0][0].cpu().numpy(), solo[0][0]) and same_bits(outs[0][1].cpu().numpy(), solo[0][1])
    w.set_window_dev(None)
    w.close()
