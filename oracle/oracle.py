"""ctypes binding of the CPU oracle (oracle/liboracle.so, oracle/_ref/libref.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product never imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
N_SAMPLES = 256
WINDOW = 1024
ELEMENTS = 64
SAMPLE_RATE = 48828.0         # src/geometry/antenna.h:17
PROPAGATION_SPEED = 340.0     # src/geometry/antenna.h:16

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")


def build():
    """(Re)build liboracle.so and, when /root/reference is present, _ref/libref.so."""
    subprocess.run(["make", "-C", _HERE, "all"], check=True, stdout=subprocess.DEVNULL)


def _load(path):
    if not os.path.exists(path):
        build()
    return C.CDLL(path)


_lib = None
_ref = None
_ref_fir = None


def lib():
    global _lib
    if _lib is None:
        L = _load(os.path.join(_HERE, "liboracle.so"))
        L.orc_create_antenna.argtypes = [_f32p, C.c_int, C.c_int, C.c_float]
        L.orc_create_tiled_antenna.argtypes = [_f32p, C.c_int, _f32p]
        L.orc_steering_vector_spherical.argtypes = [_f32p, C.c_int, C.c_double, C.c_double, _f32p]
        L.orc_steering_vector_spherical_k.argtypes = [_f32p, C.c_int, C.c_double, C.c_double, C.c_float, _f32p]
        L.orc_split_delays.argtypes = [_f32p, C.c_int, C.c_int, _i32p, _f32p]
        L.orc_mimo_grid.argtypes = [C.c_int, C.c_int, C.c_double, _f64p, _f64p]
        L.orc_mimo_lut.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, _i32p, _f32p]
        L.orc_mimo_lut_k.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_float, _i32p, _f32p]
        L.orc_delay.argtypes = [_f32p, _f32p, C.c_float, C.c_int]
        L.orc_mimo_update.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, C.c_int, _f32p]
        L.orc_mimo_das.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, C.c_int, _f32p]
        L.orc_particle_beam.argtypes = [_f32p, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, _f32p]
        L.orc_particle_beam.restype = C.c_double
        L.orc_mimo_update_fir.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, C.c_int, _f32p,
                                          C.c_int, C.c_int, _f32p]
        L.orc_mimo_update_fir.restype = None
        L.orc_delay_fir.argtypes = [_f32p, _f32p, C.c_float, C.c_int, _f32p, C.c_int, C.c_int]
        L.orc_delay_fir.restype = None
        L.orc_particle_das_fir.argtypes = [_f32p, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, _f32p, C.c_int, C.c_int,
                                           _f32p]
        L.orc_particle_das_fir.restype = None
        L.orc_quadrant.argtypes = [_f64p, C.c_double, C.c_double, C.c_double, _f64p, _f64p]
        L.orc_quadrant.restype = None
        L.orc_monopulse_gradient.argtypes = [_f64p, C.c_double, _f64p, _f64p]
        L.orc_monopulse_gradient.restype = None
        L.orc_particle_das.argtypes = [_f32p, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, _f32p]
        L.orc_populate_heatmap.argtypes = [_f32p, C.c_int, _u8p, C.POINTER(C.c_float)]
        L.orc_populate_heatmap.restype = C.c_int
        L.orc_calibrate.argtypes = [_f32p, C.c_int, C.c_float, _i32p, _f32p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.orc_calibrate.restype = C.c_int
        L.orc_ingest.argtypes = [_i32p, C.c_int, C.c_int, _f32p]
        L.orc_resize_linear_u8.argtypes = [_u8p, C.c_int, C.c_int, _u8p, C.c_int, C.c_int]
        L.orc_resize_linear_u8.restype = None
        L.orc_map_targets.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, C.c_float, _i32p, _f32p, _f32p]
        L.orc_map_targets.restype = C.c_int
        _lib = L
    return _lib


def ref():
    """The compiled UNMODIFIED reference kernel (None if oracle/_ref/libref.so is unavailable)."""
    global _ref
    if _ref is None:
        path = os.path.join(_HERE, "_ref", "libref.so")
        if not os.path.exists(path):
            if os.path.exists("/root/reference/src/dsp/delay.cpp"):
                build()
            if not os.path.exists(path):
                return None
        R = C.CDLL(path)
        R.ref_n_samples.restype = C.c_int
        R.ref_delay.argtypes = [_f32p, _f32p, C.c_float]
        R.ref_streams_window.argtypes = [_f32p, C.c_int, _f32p, C.c_int, _f32p]
        R.ref_streams_window.restype = C.c_int
        R.ref_mimo_update.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_int]
        _ref = R
    return _ref


def ref_fir():
    """The reference's delay.cpp compiled WITHOUT AVX2: its FIR variant of delay() (None if oracle/_ref/libref_fir.so is unavailable)."""
    global _ref_fir
    if _ref_fir is None:
        path = os.path.join(_HERE, "_ref", "libref_fir.so")
        if not os.path.exists(path):
            if os.path.exists("/root/reference/src/dsp/delay.cpp"):
                build()
            if not os.path.exists(path):
                return None
        R = C.CDLL(path)
        R.ref_delay.argtypes = [_f32p, _f32p, C.c_float]
        R.ref_filter_coeffs.restype = C.POINTER(C.c_float)
        R.ref_mimo_update.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, _i32p, C.c_int, _i32p, _f32p, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_int]
        assert R.ref_is_fir() == 1
        _ref_fir = R
    return _ref_fir


def ref_filter_table():
    """filter_coeffs[101][8] of src/dsp/filter.h as the compiled reference object holds it."""
    return np.ctypeslib.as_array(ref_fir().ref_filter_coeffs(), shape=(101, 8)).copy()


def ref_mimo_update_fir(window, offsets, fractions, index=None, n=N_SAMPLES, n_threads=1):
    """MIMOWorker::update loop around the compiled reference FIR delay() (W must cover offset + n + 7)."""
    R = ref_fir()
    window = np.ascontiguousarray(window, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    D = offsets.shape[0]
    power = np.zeros(D, np.float32)
    R.ref_mimo_update(window, Cn, W, n, index, len(index), np.ascontiguousarray(offsets, np.int32),
                      np.ascontiguousarray(fractions, np.float32), D, power.ctypes.data, None, n_threads)
    return power


# ---- geometry / tables ------------------------------------------------------------------------
def create_antenna(columns=8, rows=8, distance=0.02):
    xyz = np.zeros((rows * columns, 3), np.float32)
    lib().orc_create_antenna(xyz, columns, rows, distance)
    return xyz


def create_tiled_antenna(origins):
    origins = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
    xyz = np.zeros((origins.shape[0] * ELEMENTS, 3), np.float32)
    lib().orc_create_tiled_antenna(xyz, origins.shape[0], origins)
    return xyz


def delay_scale(sample_rate=SAMPLE_RATE, propagation_speed=PROPAGATION_SPEED):
    """Samples per metre of path difference, float(sample_rate / propagation_speed) as compute_delays() scales
    (antenna.cpp:90-92) and the library derives it from its config."""
    return float(np.float32(float(sample_rate) / float(propagation_speed)))


def steering_vector_spherical(xyz, theta, phi, scale=None):
    """Delays [C] in samples, min-subtracted; scale (delay_scale()) defaults to the reference's constants."""
    d = np.zeros(xyz.shape[0], np.float32)
    xyz = np.ascontiguousarray(xyz, np.float32)
    if scale is None:
        lib().orc_steering_vector_spherical(xyz, xyz.shape[0], float(theta), float(phi), d)
    else:
        lib().orc_steering_vector_spherical_k(xyz, xyz.shape[0], float(theta), float(phi), float(scale), d)
    return d


def split_delays(delays, history=N_SAMPLES):
    delays = np.ascontiguousarray(delays, np.float32)
    off = np.zeros(delays.shape[0], np.int32)
    fr = np.zeros(delays.shape[0], np.float32)
    lib().orc_split_delays(delays, delays.shape[0], history, off, fr)
    return off, fr


def mimo_grid(rows, cols, fov_deg):
    th = np.zeros(rows * cols, np.float64)
    ph = np.zeros(rows * cols, np.float64)
    lib().orc_mimo_grid(rows, cols, float(fov_deg), th, ph)
    return th, ph


def mimo_lut(xyz, rows, cols, fov_deg, history=N_SAMPLES, scale=None):
    Cn = xyz.shape[0]
    off = np.zeros((rows * cols, Cn), np.int32)
    fr = np.zeros((rows * cols, Cn), np.float32)
    xyz = np.ascontiguousarray(xyz, np.float32)
    if scale is None:
        lib().orc_mimo_lut(xyz, Cn, rows, cols, float(fov_deg), history, off, fr)
    else:
        lib().orc_mimo_lut_k(xyz, Cn, rows, cols, float(fov_deg), history, float(scale), off, fr)
    return off, fr


def steer_tables(xyz, thetas, phis, history=N_SAMPLES, scale=None):
    """Particle::steer for a list of directions -> offsets/fractions [T][C]."""
    T = len(thetas)
    off = np.zeros((T, xyz.shape[0]), np.int32)
    fr = np.zeros((T, xyz.shape[0]), np.float32)
    for t in range(T):
        off[t], fr[t] = split_delays(steering_vector_spherical(xyz, thetas[t], phis[t], scale), history)
    return off, fr


# ---- beamforming --------------------------------------------------------------------------------
def delay(out, signal, fraction, n=N_SAMPLES):
    lib().orc_delay(out, signal, fraction, n)


def _idx(index, Cn):
    return np.arange(Cn, dtype=np.int32) if index is None else np.ascontiguousarray(index, np.int32)


def mimo_update(window, offsets, fractions, index=None, n=N_SAMPLES):
    window = np.ascontiguousarray(window, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    D = offsets.shape[0]
    power = np.zeros(D, np.float32)
    lib().orc_mimo_update(window, Cn, W, n, index, len(index), np.ascontiguousarray(offsets, np.int32),
                          np.ascontiguousarray(fractions, np.float32), D, power)
    return power


def mimo_das(window, offsets, fractions, index=None, n=N_SAMPLES):
    window = np.ascontiguousarray(window, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    D = offsets.shape[0]
    out = np.zeros((D, n), np.float32)
    lib().orc_mimo_das(window, Cn, W, n, index, len(index), np.ascontiguousarray(offsets, np.int32),
                       np.ascontiguousarray(fractions, np.float32), D, out)
    return out


def particle_beam(window, offsets, fractions, index=None, n=N_SAMPLES):
    window = np.ascontiguousarray(window, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    scratch = np.zeros(n, np.float32)
    return lib().orc_particle_beam(window, W, n, index, len(index), np.ascontiguousarray(offsets, np.int32),
                                   np.ascontiguousarray(fractions, np.float32), scratch)


def particle_das(window, offsets, fractions, index=None, n=N_SAMPLES):
    window = np.ascontiguousarray(window, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    out = np.zeros(n, np.float32)
    lib().orc_particle_das(window, W, n, index, len(index), np.ascontiguousarray(offsets, np.int32),
                           np.ascontiguousarray(fractions, np.float32), out)
    return out


def populate_heatmap(power):
    power = np.ascontiguousarray(power, np.float32)
    heat = np.zeros(power.shape[0], np.uint8)
    mx = C.c_float()
    arg = lib().orc_populate_heatmap(power, power.shape[0], heat, C.byref(mx))
    return heat, arg, mx.value


def calibrate(signals, reference_power_level=1e-5):
    signals = np.ascontiguousarray(signals, np.float32)
    assert signals.shape[0] == ELEMENTS
    index = np.zeros(ELEMENTS, np.int32)
    corr = np.zeros(ELEMENTS, np.float32)
    med, mean = C.c_float(), C.c_float()
    n = lib().orc_calibrate(signals, signals.shape[1], reference_power_level, index, corr, C.byref(med), C.byref(mean))
    return index[:n].copy(), corr[:n].copy(), med.value, mean.value


def ingest(frames):
    frames = np.ascontiguousarray(frames, np.int32)
    n, ns = frames.shape
    out = np.zeros((ns, n), np.float32)
    lib().orc_ingest(frames, n, ns, out)
    return out


# ---- compiled reference (oracle/_ref) ---------------------------------------------------------------
def ref_mimo_update(window, offsets, fractions, index=None, n=N_SAMPLES, n_threads=1, want_das=False):
    R = ref()
    window = np.ascontiguousarray(window, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    D = offsets.shape[0]
    power = np.zeros(D, np.float32)
    das = np.zeros((D, n), np.float32) if want_das else None
    R.ref_mimo_update(window, Cn, W, n, index, len(index), np.ascontiguousarray(offsets, np.int32),
                      np.ascontiguousarray(fractions, np.float32), D, power.ctypes.data,
                      das.ctypes.data if want_das else None, n_threads)
    return (power, das) if want_das else power


def quadrant(theta, phi, spread, theta_limit):
    """Spherical::quadrant + normalizeSpherical (geometry.cpp:181-217, particle.h:24-27): (theta', near_theta[4], near_phi[4])."""
    t = np.array([theta], np.float64)
    nt, nph = np.zeros(4), np.zeros(4)
    lib().orc_quadrant(t, float(phi), float(spread), float(theta_limit), nt, nph)
    return float(t[0]), nt, nph


def monopulse(xyz, theta, phi, window, spread, theta_limit, reference=0.0, index=None, history=N_SAMPLES, scale=None,
              n=N_SAMPLES):
    """GradientParticle::findNearby + step() up to the gradient (gradient_ascend.cpp:18-81) for each particle, with the
    oracle's steer / beam: (theta', near_theta, near_phi, q, gradient, error)."""
    theta = np.asarray(theta, np.float64).ravel().copy()
    phi = np.asarray(phi, np.float64).ravel()
    P = theta.shape[0]
    nth, nph, q = np.zeros((P, 4)), np.zeros((P, 4)), np.zeros((P, 4))
    grad, err = np.zeros((P, 3)), np.zeros(P)
    for p in range(P):
        theta[p], nth[p], nph[p] = quadrant(theta[p], phi[p], spread, theta_limit)
        off, fr = steer_tables(xyz, nth[p], nph[p], history, scale)
        for k in range(4):
            q[p, k] = particle_beam(window, off[k], fr[k], index=index, n=n)
        e = np.zeros(1)
        lib().orc_monopulse_gradient(np.ascontiguousarray(q[p]), float(reference), grad[p], e)
        err[p] = e[0]
    return theta, nth, nph, q, grad, err


def particle_das_fir(window, offsets, fractions, coeffs, index=None, n=N_SAMPLES):
    """Particle::das around the FIR variant of delay() (delay.cpp:28-40) for one direction: out [n]; coeffs [n_phases][taps]."""
    window = np.ascontiguousarray(window, np.float32)
    coeffs = np.ascontiguousarray(coeffs, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    offsets = np.ascontiguousarray(offsets, np.int32)
    assert int(offsets[index].max()) + n + coeffs.shape[1] - 1 <= W, "the window is too short for the FIR taps"
    out = np.zeros(n, np.float32)
    lib().orc_particle_das_fir(window, W, n, index, len(index), offsets, np.ascontiguousarray(fractions, np.float32), coeffs,
                               coeffs.shape[0], coeffs.shape[1], out)
    return out


def mimo_update_fir(window, offsets, fractions, coeffs, index=None, n=N_SAMPLES):
    """MIMOWorker::update around the FIR variant of delay() (delay.cpp:28-40); coeffs [n_phases][taps]."""
    window = np.ascontiguousarray(window, np.float32)
    coeffs = np.ascontiguousarray(coeffs, np.float32)
    Cn, W = window.shape
    index = _idx(index, Cn)
    D = offsets.shape[0]
    power = np.zeros(D, np.float32)
    lib().orc_mimo_update_fir(window, Cn, W, n, index, len(index), np.ascontiguousarray(offsets, np.int32),
                              np.ascontiguousarray(fractions, np.float32), D, coeffs, coeffs.shape[0], coeffs.shape[1], power)
    return power


# ---- after the map: heat-map resize, peaks as Targets -----------------------------------------------------------
def resize_linear_u8(src, out_rows, out_cols):
    """cv::resize(..., INTER_LINEAR) on an 8-bit map (aw_processing_unit.cpp:252), fixed-point restatement."""
    src = np.ascontiguousarray(src, np.uint8)
    dst = np.zeros((out_rows, out_cols), np.uint8)
    lib().orc_resize_linear_u8(src, src.shape[0], src.shape[1], dst, out_rows, out_cols)
    return dst


def map_targets(power, rows, cols, max_targets=8, min_rel=0.5):
    """Peaks of a rows x cols power map: (index [n], power [n], probability [n])."""
    power = np.ascontiguousarray(power, np.float32).ravel()
    idx = np.zeros(max_targets, np.int32)
    pw = np.zeros(max_targets, np.float32)
    pr = np.zeros(max_targets, np.float32)
    n = lib().orc_map_targets(power, rows, cols, max_targets, min_rel, idx, pw, pr)
    return idx[:n].copy(), pw[:n].copy(), pr[:n].copy()
