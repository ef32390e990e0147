"""CPU restatement of near-field steering (bflk_set_focus), the twin of steer.cuh: focus_z.  TEST INFRASTRUCTURE ONLY.

For direction (theta, phi) the far-field path takes the floats cz, sz = cos / sin of float(phi) and cy, sy = cos / sin of
-float(theta), each evaluated in double and rounded to float (rotateZ / rotateY, as oracle.c and the library's make_trig).
The focused delay of element p (float coordinates promoted to double) at distance r is then, in double,

    u  = (-sy cz, sy sz, cy)                       each entry a product of two floats: exact
    z  = (2 r (u.p) - p.p) / (r + |r u - p|)       dot products as (a0 b0 + a1 b1) + a2 b2

every operation rounded where it is written (numpy's float64 ufuncs round each operation and never fuse two; sqrt and
division are correctly rounded), and float(z) takes the far-field float path: times the delay scale k (float x float),
minus the minimum, offset = history - trunc, fraction = the rest (exact for a float).  The bits equal the device tables'."""
import math

import numpy as np

SAMPLE_RATE = 48828.0
PROPAGATION_SPEED = 340.0


def _scale(scale):
    return np.float32(SAMPLE_RATE / PROPAGATION_SPEED) if scale is None else np.float32(scale)


def _u(thetas, phis):
    """[T][3] float64 projection directions from the float trig of each direction."""
    u = np.empty((len(thetas), 3), np.float64)
    for t, (theta, phi) in enumerate(zip(thetas, phis)):
        az, ay = float(np.float32(phi)), -float(np.float32(theta))
        cz, sz = float(np.float32(math.cos(az))), float(np.float32(math.sin(az)))
        cy, sy = float(np.float32(math.cos(ay))), float(np.float32(math.sin(ay)))
        u[t] = (-sy * cz, sy * sz, cy)
    return u


def focus_delays_many(xyz, thetas, phis, r, scale=None):
    """Delays [T][C] in samples (float32), min-subtracted per direction, of point sources r metres away."""
    p = np.asarray(xyz, np.float32).astype(np.float64)
    u = _u(np.atleast_1d(thetas), np.atleast_1d(phis))[:, None, :]              # [T][1][3]
    p0, p1, p2 = p[None, :, 0], p[None, :, 1], p[None, :, 2]                   # [1][C]
    u0, u1, u2 = u[..., 0], u[..., 1], u[..., 2]                               # [T][1]
    up = (u0 * p0 + u1 * p1) + u2 * p2
    pp = (p0 * p0 + p1 * p1) + p2 * p2
    q0, q1, q2 = r * u0 - p0, r * u1 - p1, r * u2 - p2
    n = np.sqrt((q0 * q0 + q1 * q1) + q2 * q2)
    z = (((2.0 * r) * up - pp) / (r + n)).astype(np.float32)
    d = z * _scale(scale)
    return d - d.min(axis=1, keepdims=True)


def focus_delays(xyz, theta, phi, r, scale=None):
    """Delays [C] of one direction."""
    return focus_delays_many(xyz, [theta], [phi], r, scale)[0]


def split(delays, history):
    """offset = history - (int)ip, fraction = (float)modf((double)delay, &ip), as oracle.split_delays."""
    ip = np.trunc(delays)
    return (history - ip.astype(np.int32)).astype(np.int32), (delays - ip).astype(np.float32)


def steer_tables_focus(xyz, thetas, phis, r, history=256, scale=None):
    """Focused Particle::steer tables: offsets / fractions [T][C]."""
    return split(focus_delays_many(xyz, thetas, phis, r, scale), history)


def mimo_lut_focus(oracle, xyz, rows, cols, fov_deg, r, history=256, scale=None):
    """The focused LUT of a rows x cols grid (oracle.mimo_grid's directions): offsets / fractions [D][C]."""
    th, ph = oracle.mimo_grid(rows, cols, fov_deg)
    return steer_tables_focus(xyz, th, ph, r, history, scale)
