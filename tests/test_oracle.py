"""CPU tests of the oracle: against the committed golden vectors and against the compiled,
unmodified reference kernel (oracle/_ref, built from /root/reference/src/dsp/delay.cpp + streams.hpp)."""
import hashlib

import numpy as np
import pytest

import cases


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def test_create_antenna_matches_reference_formula(oracle, golden):
    xyz = oracle.create_antenna()
    assert np.array_equal(xyz, golden["tables"]["antenna_xyz"])
    # src/geometry/antenna.cpp:68-76: element 0 at (-0.07, -0.07), pitch 0.02, row-major i = r*8 + c
    assert np.allclose(xyz[0], [-0.07, -0.07, 0.0], atol=1e-7)
    assert np.allclose(xyz[9] - xyz[0], [0.02, 0.02, 0.0], atol=1e-7)


@pytest.mark.parametrize("name", list(cases.CONFIGS))
def test_tables_match_golden(oracle, golden, name):
    c = cases.CONFIGS[name]
    g = golden["tables"]
    xyz = oracle.create_tiled_antenna(cases.origins(c["nx"], c["ny"]))
    off, fr = oracle.mimo_lut(xyz, c["rows"], c["cols"], c["fov"], c["H"])
    assert np.array_equal(sha(off), g[f"{name}_off_sha"])
    assert np.array_equal(sha(fr), g[f"{name}_frac_sha"])
    rows = g[f"{name}_rows"]
    assert np.array_equal(off[rows], g[f"{name}_off_rows"])
    assert np.array_equal(fr[rows].view(np.uint32), g[f"{name}_frac_rows"].view(np.uint32))
    # contract of the split (mimo.cpp:46-54): 0 <= fraction < 1, offset = H - int(delay) in [0, H]
    assert fr.min() >= 0.0 and fr.max() < 1.0
    assert off.max() <= c["H"] and off.min() == c["H"] - int(g[f"{name}_max_delay"]) >= 0
    # the closest element of every direction has zero delay (antenna.cpp:94)
    assert np.all((off == c["H"]).any(axis=1))


def test_odd_grid_degenerate_centre(oracle, golden):
    xyz = oracle.create_antenna()
    off, fr = oracle.mimo_lut(xyz, 9, 9, 120.0)
    assert np.array_equal(off, golden["tables"]["odd9_off"])
    assert np.array_equal(fr, golden["tables"]["odd9_frac"])
    th, ph = oracle.mimo_grid(9, 9, 120.0)
    # centre cell: x, y cancel to ~1e-17 (or exactly 0 -> defined as boresight), never NaN
    assert np.all(np.isfinite(th)) and np.all(np.isfinite(ph)) and th[40] < 1e-12
    assert np.all(off[40] == 256) and np.all(fr[40] < 1e-6)
    th3, ph3 = oracle.mimo_grid(1, 1, 90.0)          # exact 0/0 case
    assert th3[0] == 0.0 and ph3[0] == 0.0


def test_delay_kernel_semantics(oracle):
    # src/dsp/delay.cpp:16-26 probe from SURVEY.md 8c: ramp input, fraction 0.25
    sig = np.arange(512, dtype=np.float32)
    out = np.zeros(256, np.float32)
    oracle.delay(out, sig[253:].copy(), 0.25)
    assert out[0] == np.float32(253.75) and out[255] == np.float32(508.75)
    oracle.delay(out, sig[253:].copy(), 0.25)           # accumulates
    assert out[0] == np.float32(507.5)


def test_delay_bit_exact_vs_compiled_reference(oracle, golden):
    # the stored output of the compiled reference: its delayed sums of the golden snapshot (64 delay() calls per direction,
    # channel order, from zero), which make_golden.py asserted equal to the reference's before it saved them
    g = golden["snapshot"]
    window = np.ascontiguousarray(g["window"])
    off, fr = oracle.mimo_lut(oracle.create_antenna(), 16, 16, 180.0)
    for k, d in enumerate(g["das_sel"]):
        out = np.zeros(256, np.float32)
        for ch in range(window.shape[0]):
            oracle.delay(out, window[ch, off[d, ch]:off[d, ch] + 257].copy(), fr[d, ch])
        assert np.array_equal(out.view(np.uint32), g["das"][k].view(np.uint32))
    R = oracle.ref()
    if R is None:          # the live comparison needs the reference build (oracle/_ref), which is not in the repository
        return
    assert R.ref_n_samples() == 256
    rng = np.random.default_rng(1)
    for _ in range(50):
        sig = (rng.standard_normal(257) * 10.0 ** rng.integers(-6, 3)).astype(np.float32)
        acc = rng.standard_normal(256).astype(np.float32)
        f = np.float32(rng.random())
        a, b = acc.copy(), acc.copy()
        oracle.delay(a, sig, f)
        R.ref_delay(b, sig, f)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_window_semantics_vs_reference_streams(oracle):
    """a8: after forward(), position -> oldest block; get_signal(i, off) = ring[position/4 + off].  Without the reference
    build (oracle/_ref) the ring's output is the one the assertions below pin, and the oracle is checked on it."""
    R = oracle.ref()
    frames = np.arange(6 * 256, dtype=np.float32)
    window = np.zeros(1024, np.float32)
    probe = np.zeros(257, np.float32)
    if R is not None:
        assert R.ref_streams_window(frames, 6, window, 253, probe) == 1024
    else:
        window[:] = frames[512:1536]
        probe[:] = window[253:253 + 257]
    # six frames written: the ring holds frames 2..5, oldest first
    assert np.array_equal(window, frames[512:1536])
    assert window[0] == 512 and window[768] == 1280
    assert np.array_equal(probe, window[253:253 + 257])
    out = np.zeros(256, np.float32)
    oracle.delay(out, probe, 0.25)
    assert out[0] == np.float32(765.75)


def test_snapshot_matches_golden_and_reference(oracle, golden):
    g = golden["snapshot"]
    window = g["window"]
    xyz = oracle.create_antenna()
    off, fr = oracle.mimo_lut(xyz, 16, 16, 180.0)
    power = oracle.mimo_update(window, off, fr)
    das = oracle.mimo_das(window, off, fr)
    assert np.array_equal(power, g["power"])
    assert np.array_equal(das[g["das_sel"]], g["das"])
    # compiled reference delay(): delayed sums bit-identical, power within fast-math reassociation
    assert np.max(np.abs(g["ref_power"] - power) / power) < 1e-5
    assert int(np.argmax(power)) == int(np.argmax(g["ref_power"]))
    if oracle.ref() is not None:
        rp, rd = oracle.ref_mimo_update(window, off, fr, want_das=True)
        assert np.array_equal(rd, das)
        assert np.array_equal(rp, g["ref_power"])
        rp4 = oracle.ref_mimo_update(window, off, fr, n_threads=4)
        assert np.array_equal(rp4, rp)
    assert np.array_equal(oracle.mimo_update(window, off, fr, index=g["mask"]), g["power_masked"])
    # the reference's own synthetic tone (9 kHz from boresight, pipeline.cpp:115) wins after the high-pass
    assert int(np.argmax(power)) in (119, 120, 135, 136)


def test_particle_matches_golden(oracle, golden):
    g = golden["snapshot"]
    xyz = oracle.create_antenna()
    soff, sfr = oracle.steer_tables(xyz, g["miso_theta"], g["miso_phi"])
    assert np.array_equal(soff, g["miso_off"]) and np.array_equal(sfr, g["miso_frac"])
    for t in range(4):
        assert np.array_equal(oracle.particle_das(g["window"], soff[t], sfr[t]), g["miso_audio"][t])
        assert oracle.particle_beam(g["window"], soff[t], sfr[t]) == g["miso_beam"][t]
    # beam() normalises by N only, update() by N*count (particle.cpp:79 vs mimo.cpp:137)
    off, fr = oracle.mimo_lut(xyz, 16, 16, 180.0)
    p_mimo = oracle.mimo_update(g["window"], off[5:6], fr[5:6])[0]
    p_beam = oracle.particle_beam(g["window"], off[5], fr[5])
    assert np.isclose(p_beam / 64.0, p_mimo, rtol=1e-6)


def test_cfg4_tables_golden(oracle, golden):
    th, ph = cases.cfg4_targets()
    xyz = oracle.create_tiled_antenna(cases.origins(4, 2))
    off, fr = oracle.steer_tables(xyz, th, ph)
    assert np.array_equal(off, golden["tables"]["cfg4_off"])
    assert np.array_equal(fr, golden["tables"]["cfg4_frac"])


def test_heatmap_calibrate_ingest_golden(oracle, golden):
    g = golden["snapshot"]
    heat, arg, mx = oracle.populate_heatmap(g["power"])
    assert np.array_equal(heat, g["heat"]) and arg == int(g["heat_argmax"]) and mx == float(g["heat_max"])
    assert heat.max() == 255 and heat[arg] == 255
    cal = g["window"].copy()
    cal[5] *= 0.0
    cal[9] *= 3.0
    cal[33] *= 0.5
    idx, corr, med, mean = oracle.calibrate(cal)
    assert np.array_equal(idx, g["cal_index"]) and np.array_equal(corr, g["cal_corr"])
    assert med == float(g["cal_median"]) and mean == float(g["cal_mean"])
    assert 5 not in idx          # dead microphone gated out (aw_processing_unit.cpp:166)
    exposure = oracle.ingest(g["wire"])
    assert np.array_equal(exposure, g["exposure"])
    # un-flip + /2^23 restores the quantised signal
    q = np.rint(g["window"][:, :64].astype(np.float64) * 8388608.0) / 8388608.0
    assert np.array_equal(exposure, q.astype(np.float32))


def test_empty_and_ragged_masks(oracle, golden):
    g = golden["snapshot"]
    xyz = oracle.create_antenna()
    off, fr = oracle.mimo_lut(xyz, 4, 4, 90.0)
    one = oracle.mimo_update(g["window"], off, fr, index=np.array([7], np.int32))
    assert np.all(np.isfinite(one)) and one.max() > 0
    rev = oracle.mimo_update(g["window"], off, fr, index=np.arange(63, -1, -1, dtype=np.int32))
    fwd = oracle.mimo_update(g["window"], off, fr)
    assert np.allclose(rev, fwd, rtol=1e-3)     # same physics, different rounding order


def test_quadrant_directions_geometry(oracle):
    """Spherical::quadrant (geometry.cpp:181-217): four directions at angular distance `spread` from the particle, 90
    degrees apart around it; theta pulled in by spread / 2 only when theta + spread passes pi / 2; phi wrapped."""
    def unit(t, p):
        return np.array([np.sin(t) * np.cos(p), np.sin(t) * np.sin(p), np.cos(t)])
    spread = np.deg2rad(5.0)
    for theta, phi in [(0.3, 1.0), (1.2, 4.0), (0.0, 0.0), (np.pi / 2 - 0.02, 2.0)]:
        t2, nt, nph = oracle.quadrant(theta, phi, spread, np.pi / 2)
        pulled = theta + spread > np.pi / 2
        assert t2 == (theta - spread / 2 if pulled else theta)
        assert np.all((nph >= 0) & (nph < 2 * np.pi)) and np.all((nt >= 0) & (nt <= np.pi / 2))
        v = np.stack([unit(a, b) for a, b in zip(nt, nph)])
        # points * (Ry Rz) rotates the pole to a direction at polar angle (theta - spread if pulled) -- all four neighbours
        # sit `spread` away from it, and opposite ones (0,2) / (1,3) are 2 * spread apart
        centre = v.sum(axis=0) / np.linalg.norm(v.sum(axis=0))
        assert np.allclose(np.arccos(np.clip(v @ centre, -1, 1)), spread, atol=1e-9)
        assert np.isclose(np.arccos(np.clip(v[0] @ v[2], -1, 1)), 2 * spread, atol=1e-9)
        assert np.isclose(np.arccos(np.clip(v[1] @ v[3], -1, 1)), 2 * spread, atol=1e-9)
        assert np.isclose(np.arccos(centre[2]), theta - spread if pulled else theta, atol=1e-9)


# ---- f4: the FIR variant of delay() pinned against the reference file compiled without AVX2 --------------------------
def test_fir_delay_bit_exact_vs_golden_and_compiled_reference(oracle, golden):
    """delay.cpp compiles its `#elif USE_FILTER` branch (delay.cpp:28-40) exactly when __AVX2__ is undefined; oracle/_ref/
    libref_fir.so is that build of the unmodified file.  The known-answer vectors it produced are committed
    (tests/golden/fir.npz, with the reference's 101 x 8 table of src/dsp/filter.h as that object holds it)."""
    g = golden["fir"]
    co = np.ascontiguousarray(g["coeffs"])
    assert co.shape == (101, 8) and np.allclose(co.sum(axis=1), 1.0, atol=2e-6) and co[0, 3] > 0.9999
    L = oracle.lib()
    for k in range(g["kat_signal"].shape[0]):
        out = np.zeros(256, np.float32)
        L.orc_delay_fir(out, np.ascontiguousarray(g["kat_signal"][k]), float(g["kat_fraction"][k]), 256, co, 101, 8)
        assert np.array_equal(out.view(np.uint32), g["kat_out"][k].view(np.uint32))
    R = oracle.ref_fir()
    if R is None:          # the live comparison needs the reference build (oracle/_ref), which is not in the repository
        return
    assert np.array_equal(oracle.ref_filter_table(), co)
    rng = np.random.default_rng(2)
    for _ in range(50):
        sig = (rng.standard_normal(264) * 10.0 ** rng.integers(-6, 3)).astype(np.float32)
        acc = rng.standard_normal(256).astype(np.float32)
        f = np.float32(rng.random())
        a, b = acc.copy(), acc.copy()
        L.orc_delay_fir(a, sig, float(f), 256, co, 101, 8)
        R.ref_delay(b, sig, f)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_fir_power_map_matches_golden_and_compiled_reference(oracle, golden):
    g, snap = golden["fir"], golden["snapshot"]
    xyz = oracle.create_antenna()
    off, fr = oracle.mimo_lut(xyz, 16, 16, 180.0)
    p = oracle.mimo_update_fir(snap["window"], off, fr, g["coeffs"])
    assert np.array_equal(p, g["power"])
    assert np.max(np.abs(p - g["ref_power"]) / g["ref_power"]) < 1e-5      # same delayed sums, fast-math power sum
    assert int(np.argmax(p)) == int(np.argmax(g["ref_power"]))
    if oracle.ref_fir() is not None:
        assert np.array_equal(oracle.ref_mimo_update_fir(snap["window"], off, fr), g["ref_power"])


# ---- exposure of the one unpinned row: Eigen's evaluation order in steer() / compute_delays() -------------------------
def _tables_variant(xyz, theta, phi, variant, history=256):
    """Steering tables of antenna.cpp:89-107 under a different plausible evaluation of the Eigen expressions (numpy float32,
    every operation rounded where written; a float32 FMA is emulated in float64, exact up to double rounding)."""
    f32, f64 = np.float32, np.float64
    az, ay = f32(phi), -f32(theta)
    cz, sz = f32(np.cos(f64(az))), f32(np.sin(f64(az)))
    cy, sy = f32(np.cos(f64(ay))), f32(np.sin(f64(ay)))
    x, y, z = (xyz[:, k].astype(f32) for k in range(3))

    def fma(a, b, c):
        return (a.astype(f64) * b.astype(f64) + c.astype(f64)).astype(f32) if np.ndim(a) or np.ndim(b) or np.ndim(c) else f32(f64(a) * f64(b) + f64(c))

    def dot(r, v, order, fused):
        acc = np.zeros_like(v[0])
        for i, k in enumerate(order):
            rk = np.full_like(v[0], r[k])
            if fused:
                acc = fma(rk, v[k], acc)
            else:
                prod = (rk * v[k]).astype(f32)
                acc = prod if i == 0 else (acc + prod).astype(f32)
        return acc

    order = (2, 1, 0) if variant == "k_reversed" else (0, 1, 2)
    fused = variant not in ("no_fma", "no_fma_double_k")
    zero, one = f32(0), f32(1)
    p = (x, y, z)
    q = (dot((cz, -sz, zero), p, order, fused), dot((sz, cz, zero), p, order, fused), dot((zero, zero, one), p, order, fused))
    zz = dot((-sy, zero, cy), q, order, fused)
    if variant in ("double_k", "no_fma_double_k"):
        d = (zz.astype(f64) * (48828.0 / 340.0)).astype(f32)       # the double constant NOT narrowed first
    else:
        d = (zz * f32(48828.0 / 340.0)).astype(f32)
    d = (d - d.min()).astype(f32)
    ip = np.trunc(d.astype(f64))
    return (history - ip).astype(np.int32), (d.astype(f64) - ip).astype(f32), d


def test_exposure_of_unpinned_eigen_order(oracle):
    """Eigen is absent, so the rounding order of steer()'s 3x3 . 3xC product and of `row * (fs / c)` cannot be observed;
    the oracle fixes one (fma chain k = 0,1,2; float x float constant).  This test measures what the other plausible
    evaluations would change on cfg3 (the headline grid): how many (offset, fraction) entries differ, by how much the
    delays move, and that an entry whose offset flips does so ACROSS an integer boundary (delay continuous) -- i.e. the
    exposure of the "tables bit-exact" claim is a handful of ulps on a small share of entries, never a different beam."""
    c = cases.CONFIGS["cfg3"]
    xyz = oracle.create_tiled_antenna(cases.origins(c["nx"], c["ny"]))
    th, ph = oracle.mimo_grid(c["rows"], c["cols"], c["fov"])
    off0, fr0 = oracle.mimo_lut(xyz, c["rows"], c["cols"], c["fov"], c["H"])
    sel = np.arange(0, len(th), 7)                               # 147 directions x 512 channels
    report = {}
    for variant in ("oracle_order", "no_fma", "k_reversed", "double_k", "no_fma_double_k"):
        n_off = n_fr = n = 0
        worst = 0.0
        for d in sel:
            off, fr, dly = _tables_variant(xyz, th[d], ph[d], variant, c["H"])
            ref_delay = (c["H"] - off0[d]).astype(np.float64) + fr0[d].astype(np.float64)
            diff = np.abs(dly.astype(np.float64) - ref_delay)
            worst = max(worst, float(diff.max()))
            n_off += int(np.count_nonzero(off != off0[d]))
            n_fr += int(np.count_nonzero(fr.view(np.uint32) != fr0[d].view(np.uint32)))
            n += off.size
        report[variant] = (n_off / n, n_fr / n, worst)
    # the numpy model of the oracle's own order reproduces the oracle exactly (the model is sound)
    assert report["oracle_order"] == (0.0, 0.0, 0.0)
    for variant, (share_off, share_fr, worst) in report.items():
        print(f"eigen-order exposure, {variant}: {100 * share_off:.3f} % offsets, {100 * share_fr:.2f} % fractions differ, "
              f"largest delay change {worst:.2e} samples")
        # a delay is at most ~100 samples: one float ulp there is 7.6e-6; every alternative stays within a few ulps
        assert worst <= 4e-5
        assert share_off <= 2e-3                                 # offset flips only where a delay sits on an integer


# ---- f3: heat-map resize pinned against OpenCV, map peaks as Targets ---------------------------------------------------
def _resize_cases(g):
    k = 0
    while f"case{k}_src" in g:
        yield g[f"case{k}_src"], int(g[f"case{k}_shape"][0]), int(g[f"case{k}_shape"][1]), g[f"case{k}_sha"], g.get(f"case{k}_out")
        k += 1


def test_resize_matches_opencv_golden(oracle, golden):
    """cv::resize(..., INTER_LINEAR) on CV_8UC1 (aw_processing_unit.cpp:252): OpenCV is absent from /root/reference, the
    golden outputs come from the real cv2.resize (tests/golden/make_golden.py); the fixed-point restatement is bit-exact."""
    g = golden["resize"]
    big = oracle.resize_linear_u8(g["heat16"], 1024, 1024)
    assert np.array_equal(sha(big), g["heat16_to_1024_sha"]) and np.array_equal(big[::97], g["heat16_to_1024_rows"])
    for src, oh, ow, want_sha, want in _resize_cases(g):
        out = oracle.resize_linear_u8(src, oh, ow)
        assert np.array_equal(sha(out), want_sha)
        if want is not None:
            assert np.array_equal(out, want)
    try:
        import cv2
    except ImportError:
        return
    rng = np.random.default_rng(3)
    for _ in range(10):
        ih, iw, oh, ow = (int(v) for v in rng.integers(1, 70, 4))
        src = rng.integers(0, 256, (ih, iw), dtype=np.uint8)
        assert np.array_equal(oracle.resize_linear_u8(src, oh, ow), cv2.resize(src, (ow, oh), interpolation=cv2.INTER_LINEAR))


def test_map_targets_definition(oracle, golden):
    """Peaks of the map as Targets (new behaviour, see oracle.c): local maxima above a share of the peak, strongest first,
    probability = 1 / gradientError from the four grid neighbours."""
    g = golden["snapshot"]
    idx, pw, pr = oracle.map_targets(g["power"], 16, 16, max_targets=8, min_rel=0.05)
    assert idx[0] == int(np.argmax(g["power"])) and pw[0] == g["power"].max()
    assert np.all(np.diff(pw) <= 0) and len(set(idx.tolist())) == len(idx)
    m = g["power"].reshape(16, 16)
    for i in idx:
        r, c = divmod(int(i), 16)
        assert m[r, c] == m[max(r - 1, 0):r + 2, max(c - 1, 0):c + 2].max() and m[r, c] >= 0.05 * m.max()
    r, c = divmod(int(idx[0]), 16)
    err = (abs(float(m[r, c + 1]) - float(m[r, c - 1])) + abs(float(m[r + 1, c]) - float(m[r - 1, c]))) / (float(m[r, c - 1]) + float(m[r, c + 1]) + float(m[r - 1, c]) + float(m[r + 1, c]))
    assert np.isclose(pr[0], 1.0 / err, rtol=1e-6)
    # a plateau yields ONE target (the lowest index), a flat neighbourhood an (almost) infinite probability
    flat = np.zeros((6, 6), np.float32)
    flat[2:4, 2:4] = 1.0
    i2, p2, q2 = oracle.map_targets(flat, 6, 6, 4, 0.5)
    assert i2.tolist() == [14] and p2[0] == 1.0
    two = np.full((8, 8), 0.1, np.float32)
    two[1, 1], two[6, 5] = 3.0, 2.0
    i3, p3, _ = oracle.map_targets(two, 8, 8, 4, 0.5)
    assert i3.tolist() == [9, 53] and p3.tolist() == [3.0, 2.0]
    assert oracle.map_targets(two, 8, 8, 4, 0.9)[0].tolist() == [9]          # threshold relative to the peak
    assert oracle.map_targets(two, 8, 8, 1, 0.1)[0].tolist() == [9]          # k limits the list
