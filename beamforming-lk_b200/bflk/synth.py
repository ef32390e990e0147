"""Synthetic microphone-array input (the repo's replacement for offline UDP replay, udp/README.md:56-67).

Seeded, reproducible plane-wave tones + white noise shaped like normalised 24-bit audio
(src/fpga/pipeline.cpp:290), SURVEY.md 8d: sources (theta, phi, f, A) = (20 deg, 30 deg, 3 kHz, 1e-2),
(45 deg, 200 deg, 6 kHz, 5e-3) and the reference's own synthetic 9 kHz / 1e-2 tone from boresight
(src/fpga/pipeline.cpp:115,129-132); noise sigma 1e-3, numpy Philox seed 0xB200.
"""
import numpy as np

from . import ELEMENTS, PROPAGATION_SPEED, SAMPLE_RATE

DEFAULT_SOURCES = (
    (np.deg2rad(20.0), np.deg2rad(30.0), 3000.0, 1e-2),
    (np.deg2rad(45.0), np.deg2rad(200.0), 6000.0, 5e-3),
    (0.0, 0.0, 9000.0, 1e-2),
)
SEED = 0xB200


def tile_geometry(origins, columns=8, rows=8, distance=0.02):
    """Element positions [C][3] of 8x8 tiles (float64 model of create_antenna; input synthesis only)."""
    origins = np.asarray(origins, np.float64).reshape(-1, 3)
    c = np.arange(columns) * distance - rows * distance / 2 + distance / 2
    r = np.arange(rows) * distance - columns * distance / 2 + distance / 2
    tile = np.stack([np.tile(c, rows), np.repeat(r, columns), np.zeros(rows * columns)], axis=1)
    return (origins[:, None, :] + tile[None, :, :]).reshape(-1, 3)


def arrival_delays(xyz, theta, phi, sample_rate=SAMPLE_RATE, speed=PROPAGATION_SPEED):
    """Per-element delay in samples of a plane wave from (theta, phi), min-subtracted (float64)."""
    xr = np.cos(phi) * xyz[:, 0] - np.sin(phi) * xyz[:, 1]
    z = np.sin(theta) * xr + np.cos(theta) * xyz[:, 2]
    d = z * (sample_rate / speed)
    return d - d.min()


def make_stream(xyz, n_samples, sources=DEFAULT_SOURCES, sigma=1e-3, seed=SEED, t0=0, dtype=np.float32):
    """stream[C][n_samples]: sum_j A_j sin(2 pi f_j (t + tau_jc) / fs) + sigma * n_c(t)."""
    xyz = np.asarray(xyz, np.float64)
    C = xyz.shape[0]
    t = np.arange(t0, t0 + n_samples, dtype=np.float64)
    out = np.zeros((C, n_samples), np.float64)
    for theta, phi, f, A in sources:
        tau = arrival_delays(xyz, theta, phi)
        out += A * np.sin(2.0 * np.pi * f * (t[None, :] + tau[:, None]) / SAMPLE_RATE)
    if sigma > 0:
        rng = np.random.Generator(np.random.Philox(seed))
        out += sigma * rng.standard_normal((C, n_samples))
    return out.astype(dtype)


def point_source_delays(xyz, theta, phi, r, sample_rate=SAMPLE_RATE, speed=PROPAGATION_SPEED):
    """Per-element delay in samples of a point source r metres from the origin in direction (theta, phi),
    (r - |s - p|) * fs / c with s = r u, min-subtracted (float64): the near-field counterpart of arrival_delays, whose
    plane-wave delay is u.p * fs / c with the same u = (sin theta cos phi, -sin theta sin phi, cos theta)."""
    xyz = np.asarray(xyz, np.float64)
    s = r * np.array([np.sin(theta) * np.cos(phi), -np.sin(theta) * np.sin(phi), np.cos(theta)])
    d = (r - np.linalg.norm(s[None, :] - xyz, axis=1)) * (sample_rate / speed)
    return d - d.min()


def point_source_stream(xyz, n_samples, sources, sigma=1e-3, seed=SEED, t0=0, sample_rate=SAMPLE_RATE,
                        speed=PROPAGATION_SPEED, dtype=np.float32):
    """stream[C][n_samples] of point sources (theta, phi, r, f, A) r metres away: sum_j A_j sin(2 pi f_j (t + tau_jc) / fs)
    + sigma * n_c(t), tau_jc = point_source_delays (the same amplitude at every element)."""
    xyz = np.asarray(xyz, np.float64)
    C = xyz.shape[0]
    t = np.arange(t0, t0 + n_samples, dtype=np.float64)
    out = np.zeros((C, n_samples), np.float64)
    for theta, phi, r, f, A in sources:
        tau = point_source_delays(xyz, theta, phi, r, sample_rate, speed)
        out += A * np.sin(2.0 * np.pi * f * (t[None, :] + tau[:, None]) / sample_rate)
    if sigma > 0:
        rng = np.random.Generator(np.random.Philox(seed))
        out += sigma * rng.standard_normal((C, n_samples))
    return out.astype(dtype)


def to_wire_i32(stream):
    """float stream[C][n] -> wire frames[n][C] int32 (round(x * 2^23)) with the serpentine column flip
    the FPGA applies (inverse of src/fpga/pipeline.cpp:273-287)."""
    C, n = stream.shape
    q = np.rint(stream.astype(np.float64) * 8388608.0).astype(np.int32)
    sensor = np.arange(C)
    grp = sensor // 8
    src = np.where(grp % 2 == 1, sensor, 8 * (1 + grp) - 1 - sensor % 8)
    wire = np.zeros((n, C), np.int32)
    wire[:, src] = q.T
    return wire


def nearest_direction(theta_grid, phi_grid, theta, phi):
    """Index of the grid direction closest (great-circle) to (theta, phi)."""
    g = np.stack([np.sin(theta_grid) * np.cos(phi_grid), np.sin(theta_grid) * np.sin(phi_grid), np.cos(theta_grid)], 1)
    v = np.array([np.sin(theta) * np.cos(phi), np.sin(theta) * np.sin(phi), np.cos(theta)])
    return int(np.argmax(g @ v))
