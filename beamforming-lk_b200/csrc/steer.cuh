// steer.cuh -- the device side of steering_vector_spherical, shared by the table kernel (tables.cu) and the fused MISO
// kernel (das_miso.cu) so both produce the same bits.  Every rounding is pinned (__f*_rn): see tables.cu.
#pragma once
#include "bflk_internal.h"

namespace bflk {

// z'' of steer() (src/geometry/antenna.cpp:99-107) for one element
__device__ __forceinline__ float steer_z(const DirTrig t, float px, float py, float pz) {
    // rotateZ(float(phi)) * p, k = 0,1,2 from a zero accumulator (documented evaluation order)
    float xr = __fmaf_rn(0.0f, pz, __fmaf_rn(-t.sz, py, __fmaf_rn(t.cz, px, 0.0f)));
    float yr = __fmaf_rn(0.0f, pz, __fmaf_rn(t.cz, py, __fmaf_rn(t.sz, px, 0.0f)));
    float zr = __fmaf_rn(1.0f, pz, __fmaf_rn(0.0f, py, __fmaf_rn(0.0f, px, 0.0f)));
    // row Z of rotateY(-float(theta)): (-sin, 0, cos)
    return __fmaf_rn(t.cy, zr, __fmaf_rn(0.0f, yr, __fmaf_rn(-t.sy, xr, 0.0f)));
}


// z'' of a point source at distance r (bflk_set_focus) on the direction steer_z projects on: r - |r u - p|, with
// u = (-sy cz, sy sz, cy) exact in double (each entry a product of two floats), written without the cancellation as
// (2 r u.p - p.p) / (r + |r u - p|).  Every double operation is rounded where it is written (tests/focus_oracle.py);
// as r grows the value tends to u.p, the far-field z''.
__device__ __forceinline__ float focus_z(const DirTrig t, float px, float py, float pz, double r) {
    const double u0 = __dmul_rn(-(double)t.sy, (double)t.cz), u1 = __dmul_rn((double)t.sy, (double)t.sz), u2 = t.cy;
    const double p0 = px, p1 = py, p2 = pz;
    const double up = __dadd_rn(__dadd_rn(__dmul_rn(u0, p0), __dmul_rn(u1, p1)), __dmul_rn(u2, p2));
    const double pp = __dadd_rn(__dadd_rn(__dmul_rn(p0, p0), __dmul_rn(p1, p1)), __dmul_rn(p2, p2));
    const double q0 = __dsub_rn(__dmul_rn(r, u0), p0), q1 = __dsub_rn(__dmul_rn(r, u1), p1), q2 = __dsub_rn(__dmul_rn(r, u2), p2);
    const double n = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(q0, q0), __dmul_rn(q1, q1)), __dmul_rn(q2, q2)));
    return __double2float_rn(__ddiv_rn(__dsub_rn(__dmul_rn(__dmul_rn(2.0, r), up), pp), __dadd_rn(r, n)));
}

// compute_delays() scale (antenna.cpp:90-92): row(Z) * float(SAMPLE_RATE / PROPAGATION_SPEED); FOCUS: of focus_z
template <bool FOCUS = false>
__device__ __forceinline__ float steer_delay(const DirTrig t, const float *__restrict__ xyz, int c, float k_scale, double r = 0.0) {
    const float px = xyz[3 * c + 0], py = xyz[3 * c + 1], pz = xyz[3 * c + 2];
    return __fmul_rn(FOCUS ? focus_z(t, px, py, pz, r) : steer_z(t, px, py, pz), k_scale);
}

}  // namespace bflk
