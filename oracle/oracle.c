/* oracle.c -- see oracle.h.  TEST INFRASTRUCTURE ONLY, never linked into the product.
 * Build with -O2 -ffp-contract=off -fno-fast-math so every float operation below rounds exactly
 * where it is written; explicit fmaf() marks the reference's fused operations. */
#include "oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ---- a1 ----------------------------------------------------------------------------------- */
void orc_create_antenna(float *xyz, int columns, int rows, float distance) {
    /* src/geometry/antenna.cpp:60-76.  Note the reference mixes rows/columns in the centring
     * terms (x uses rows, y uses columns); kept as written. */
    float half = distance / 2;
    int i = 0;
    for (int r = 0; r < rows; r++) {
        for (int c = 0; c < columns; c++) {
            xyz[3 * i + 0] = (float)c * distance - (float)rows * half + half;
            xyz[3 * i + 1] = (float)r * distance - (float)columns * half + half;
            xyz[3 * i + 2] = 0.f;
            i++;
        }
    }
}

void orc_create_tiled_antenna(float *xyz, int n_tiles, const float *origins) {
    float tile[3 * ORC_ELEMENTS];
    orc_create_antenna(tile, ORC_COLUMNS, ORC_ROWS, ORC_DISTANCE);
    for (int a = 0; a < n_tiles; a++)
        for (int e = 0; e < ORC_ELEMENTS; e++)
            for (int k = 0; k < 3; k++)
                xyz[3 * (a * ORC_ELEMENTS + e) + k] = tile[3 * e + k] + origins[3 * a + k];
}

/* ---- a2-a5 -------------------------------------------------------------------------------- */
void orc_steering_vector_spherical(const float *xyz, int C, double theta, double phi, float *delays) {
    orc_steering_vector_spherical_k(xyz, C, theta, phi, (float)(ORC_SAMPLE_RATE / ORC_PROPAGATION_SPEED), delays);
}

void orc_steering_vector_spherical_k(const float *xyz, int C, double theta, double phi, float k, float *delays) {
    /* steer(): rotateY(-float(theta)) * (rotateZ(float(phi)) * points), antenna.cpp:99-107.
     * Matrix entries: float(cos/sin((double)angle)), geometry.cpp:219-233.
     * Product evaluation order (Eigen 3.4 GEMM path, FMA-contracted, k = 0,1,2 from a zero
     * accumulator) is FIXED here as acc = fma(R[i][k], p[k], acc). */
    const float az = (float)phi;
    const float ay = -(float)theta;
    const float cz = (float)cos((double)az), sz = (float)sin((double)az);
    const float cy = (float)cos((double)ay), sy = (float)sin((double)ay);
    const float Rz[3][3] = {{cz, -sz, 0.0f}, {sz, cz, 0.0f}, {0.0f, 0.0f, 1.0f}};
    const float Ry[3][3] = {{cy, 0.0f, sy}, {0.0f, 1.0f, 0.0f}, {-sy, 0.0f, cy}};
    /* compute_delays(): row(Z) * k as float x float, k = float(SAMPLE_RATE / PROPAGATION_SPEED), then subtract the
     * minimum, antenna.cpp:89-97. */
    float mn = INFINITY;
    for (int c = 0; c < C; c++) {
        const float *p = &xyz[3 * c];
        float q[3];
        for (int i = 0; i < 3; i++) {
            float acc = 0.0f;
            for (int j = 0; j < 3; j++) acc = fmaf(Rz[i][j], p[j], acc);
            q[i] = acc;
        }
        float acc = 0.0f;
        for (int j = 0; j < 3; j++) acc = fmaf(Ry[2][j], q[j], acc);
        float d = acc * k;
        delays[c] = d;
        if (d < mn) mn = d;
    }
    for (int c = 0; c < C; c++) delays[c] = delays[c] - mn;
}

void orc_split_delays(const float *delays, int C, int history, int32_t *offsets, float *fractions) {
    for (int c = 0; c < C; c++) {
        double ip;
        float fraction = (float)modf((double)delays[c], &ip);
        offsets[c] = history - (int)ip;
        fractions[c] = fraction;
    }
}

/* ---- a6 ----------------------------------------------------------------------------------- */
void orc_mimo_grid(int rows, int cols, double fov_deg, double *theta, double *phi) {
    /* src/dsp/mimo.cpp:20-43; TO_RADIANS(a) = a * M_PI / 180.0 (geometry.h). */
    double fovRadian = fov_deg * (M_PI / 180.0);
    double separationRows = sin(fovRadian / 2.0) / ((double)rows / 2.0);
    double separationColumns = sin(fovRadian / 2.0) / ((double)cols / 2.0);
    int k = 0;
    for (int r = 0; r < rows; r++) {
        for (int c = 0; c < cols; c++) {
            double y = (double)r * separationRows - (double)rows * separationRows / 2.0 + separationRows / 2.0;
            double x = (double)c * separationColumns - (double)cols * separationColumns / 2.0 + separationColumns / 2.0;
            double norm = sqrt(pow(x, 2) + pow(y, 2));
            if (norm == 0.0) { theta[k] = 0.0; phi[k] = 0.0; k++; continue; }
            x /= norm;
            y /= norm;
            if (norm > 1.0) norm = 1.0;
            theta[k] = asin(norm);
            phi[k] = atan2(y, x);
            k++;
        }
    }
}

void orc_mimo_lut(const float *xyz, int C, int rows, int cols, double fov_deg, int history,
                  int32_t *offsets, float *fractions) {
    orc_mimo_lut_k(xyz, C, rows, cols, fov_deg, history, (float)(ORC_SAMPLE_RATE / ORC_PROPAGATION_SPEED), offsets, fractions);
}

void orc_mimo_lut_k(const float *xyz, int C, int rows, int cols, double fov_deg, int history, float k,
                    int32_t *offsets, float *fractions) {
    int D = rows * cols;
    double *theta = (double *)malloc(sizeof(double) * D), *phi = (double *)malloc(sizeof(double) * D);
    float *del = (float *)malloc(sizeof(float) * C);
    orc_mimo_grid(rows, cols, fov_deg, theta, phi);
    for (int d = 0; d < D; d++) {
        orc_steering_vector_spherical_k(xyz, C, theta[d], phi[d], k, del);
        orc_split_delays(del, C, history, &offsets[(size_t)d * C], &fractions[(size_t)d * C]);
    }
    free(theta); free(phi); free(del);
}

/* ---- a9 ----------------------------------------------------------------------------------- */
void orc_delay(float *out, const float *signal, float fraction, int n) {
    for (int i = 0; i < n; i++)
        out[i] = out[i] + fmaf(fraction, signal[i] - signal[i + 1], signal[i + 1]);
}

/* ---- a10 ---------------------------------------------------------------------------------- */
static float hp_power(const float *out, int n) {
    /* src/dsp/mimo.cpp:131-135 / particle.cpp:68-72; powf(MA, 2) == MA * MA; summed in index order. */
    float power = 0.0f;
    for (int i = 1; i < n - 1; i++) {
        float MA = out[i] * 0.5f - 0.25f * (out[i + 1] + out[i - 1]);
        power += MA * MA;
    }
    return power;
}

static void das_one(const float *window, int W, int n, const int *index, int usable,
                    const int32_t *offsets, const float *fractions, float *out) {
    memset(out, 0, sizeof(float) * n);
    for (int s = 0; s < usable; s++) {
        int i = index[s];
        orc_delay(out, &window[(size_t)i * W + offsets[i]], fractions[i], n);
    }
}

void orc_mimo_das(const float *window, int C, int W, int n, const int *index, int usable,
                  const int32_t *offsets, const float *fractions, int D, float *out) {
    for (int m = 0; m < D; m++)
        das_one(window, W, n, index, usable, &offsets[(size_t)m * C], &fractions[(size_t)m * C], &out[(size_t)m * n]);
}

void orc_mimo_update(const float *window, int C, int W, int n, const int *index, int usable,
                     const int32_t *offsets, const float *fractions, int D, float *power) {
    float *out = (float *)malloc(sizeof(float) * n);
    for (int m = 0; m < D; m++) {
        das_one(window, W, n, index, usable, &offsets[(size_t)m * C], &fractions[(size_t)m * C], out);
        float p = hp_power(out, n);
        p /= (float)(n * usable);   /* mimo.cpp:137, count == usable */
        power[m] = p;
    }
    free(out);
}

/* ---- a11 / a12 ---------------------------------------------------------------------------- */
double orc_particle_beam(const float *window, int W, int n, const int *index, int usable,
                         const int32_t *offsets, const float *fractions, float *out_scratch) {
    das_one(window, W, n, index, usable, offsets, fractions, out_scratch);
    float p = hp_power(out_scratch, n);
    p /= (float)n;                  /* particle.cpp:79 */
    return (double)p;
}

void orc_particle_das(const float *window, int W, int n, const int *index, int usable,
                      const int32_t *offsets, const float *fractions, float *out) {
    das_one(window, W, n, index, usable, offsets, fractions, out);
}

/* ---- a13 ---------------------------------------------------------------------------------- */
int orc_populate_heatmap(const float *power, int D, uint8_t *heat, float *max_out) {
    float maxV = 0.0f;
    int arg = 0;
    for (int i = 0; i < D; i++)
        if (power[i] > maxV) { maxV = power[i]; arg = i; }
    for (int i = 0; i < D; i++) {
        double db = pow((double)(power[i] / maxV), 1);   /* mimo.cpp:86: float division, widened */
        db *= 255.0;
        if (db < 0.0) db = 0.0;
        if (db > 255.0) db = 255.0;
        heat[i] = (uint8_t)db;
    }
    if (max_out) *max_out = maxV;
    return arg;
}

/* ---- a15 ---------------------------------------------------------------------------------- */
static int cmp_float(const void *a, const void *b) {
    float x = *(const float *)a, y = *(const float *)b;
    return (x > y) - (x < y);
}

int orc_calibrate(const float *signals, int W, float reference_power_level, int *index,
                  float *correction, float *median_out, float *mean_out) {
    /* src/aw_processing_unit/aw_processing_unit.cpp:126-200 */
    float power[ORC_ELEMENTS], medians[ORC_ELEMENTS];
    float mean = 0.0f;
    for (int s = 0; s < ORC_ELEMENTS; s++) {
        float pv = 0.0f;
        for (int i = 0; i < W; i++) pv += signals[(size_t)s * W + i] * signals[(size_t)s * W + i];
        pv /= (float)W;
        mean += pv;
        power[s] = pv;
    }
    memcpy(medians, power, sizeof(power));
    qsort(medians, ORC_ELEMENTS, sizeof(float), cmp_float);
    float median = (float)((medians[ORC_ELEMENTS / 2] + medians[ORC_ELEMENTS / 2 + 1]) / 2.0);
    int count = 0;
    for (int s = 0; s < ORC_ELEMENTS; s++) {
        float diff = fabsf(power[s] - median);
        if (diff > 1e-4) {
        } else if (power[s] < median * 1e-3) {
        } else {
            index[count] = s;
            count++;
            mean += power[s];
        }
    }
    mean /= (float)count;
    for (int s = 0; s < count; s++) correction[s] = reference_power_level / power[index[s]];
    if (median_out) *median_out = median;
    if (mean_out) *mean_out = mean;
    return count;
}

/* ---- f1 ----------------------------------------------------------------------------------- */
void orc_ingest(const int32_t *frames, int n, int n_sensors, float *exposure) {
    /* src/fpga/pipeline.cpp:260-297 */
    for (int i = 0; i < n; i++) {
        int inverted = 0;
        for (unsigned sensor_index = 0; sensor_index < (unsigned)n_sensors; sensor_index++) {
            unsigned index;
            if (sensor_index % ORC_COLUMNS == 0) inverted = !inverted;
            if (inverted) index = ORC_COLUMNS * (1 + sensor_index / ORC_COLUMNS) - 1 - sensor_index % ORC_COLUMNS;
            else index = sensor_index;
            exposure[(size_t)sensor_index * n + i] = (float)frames[(size_t)i * n_sensors + index] / 8388608.0f;
        }
    }
}

/* ---- f2: monopulse directions and gradient (next row of SURVEY 8f) ------------------------- */
/* Spherical::quadrant (src/geometry/geometry.cpp:181-217) with rotateTo (:120-142), toCartesian (:91-98) and
 * normalizeSpherical (src/dsp/particle.h:24-27; wrapAngle src/geometry/geometry.cpp:11-20).  All double.  The 3x3
 * and 4x3 products go through Eigen in the reference (absent here): the order is fixed as ((a0 b0 + a1 b1) + a2 b2),
 * no contraction.  *theta is pulled in by spread / 2 when theta + spread passes pi / 2, like the reference's
 * non-const member does to directionCurrent. */
static double dot3(const double *a, const double *b, int sb) { return (a[0] * b[0] + a[1] * b[sb]) + a[2] * b[2 * sb]; }

void orc_quadrant(double *theta, double phi, double spread, double theta_limit, double *near_theta, double *near_phi) {
    static const double deg[4] = {45.0, 315.0, 225.0, 135.0};
    double search[4][3];
    for (int i = 0; i < 4; i++) {
        const double a = deg[i] * (M_PI / 180.0);                 /* TO_RADIANS, geometry.h:18 */
        search[i][0] = 1.0 * sin(spread) * cos(a);                  /* radius * sin(theta) * cos(phi) */
        search[i][1] = 1.0 * sin(spread) * sin(a);
        search[i][2] = 1.0 * cos(spread);
    }
    double rt = *theta;
    if (rt + spread > M_PI / 2.0) {                                /* geometry.cpp:198-201 */
        rt -= spread;
        *theta -= spread / 2.0;
    }
    const double Rz[9] = {cos(phi), -sin(phi), 0.0, sin(phi), cos(phi), 0.0, 0.0, 0.0, 1.0};
    const double Ry[9] = {cos(rt), 0.0, sin(rt), 0.0, 1.0, 0.0, -sin(rt), 0.0, cos(rt)};
    double R[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) R[3 * i + j] = dot3(Ry + 3 * i, Rz + j, 3);   /* rotation = Ry * Rz */
    for (int i = 0; i < 4; i++) {
        double k[3];
        for (int j = 0; j < 3; j++) k[j] = dot3(search[i], R + j, 3);              /* rotated = points * rotation */
        double nt = acos(k[2]);
        double np = atan2(k[1], k[0]) - M_PI;
        np = fmod(np, 2.0 * M_PI);                                  /* wrapAngle */
        if (np < 0.0) np = 2.0 * M_PI + np;
        nt = nt < 0.0 ? 0.0 : (nt > theta_limit ? theta_limit : nt);   /* clip */
        near_theta[i] = nt;
        near_phi[i] = np;
    }
}

/* GradientParticle::step, quadrant form (src/dsp/gradient_ascend.cpp:50-78): q[4] -> {theta, phi, radius}, error */
void orc_monopulse_gradient(const double *q, double reference, double *gradient, double *error) {
    const double sum = q[0] + q[1] + q[2] + q[3];
    const double phi = (q[0] + q[3]) - (q[1] + q[2]);
    const double theta = (q[2] + q[3]) - (q[0] + q[1]);
    *error = (fabs(phi) + fabs(theta)) / sum;
    gradient[0] = reference > 0.0 ? theta / reference : theta;     /* RELATIVE 1 / 0 */
    gradient[1] = reference > 0.0 ? phi / reference : phi;
    gradient[2] = sum / 4;
}

/* ---- f4: FIR fractional-delay variant of delay() (src/dsp/delay.cpp:28-40, USE_FILTER build) ---------------- */
/* coeffs[n_phases][taps] is filter.h's table in the reference (101 x 8).  The reference compiles this branch only when
 * __AVX2__ is not defined (delay.cpp:8,28), i.e. on a host without AVX2 / FMA: oracle/_ref/libref_fir.so is that build
 * (same file, -mno-avx2 -mno-fma) and shows what it does -- the taps accumulate in order, each product rounded and then
 * added (no contraction).  tests/test_oracle.py pins this function to it bit for bit. */
void orc_delay_fir(float *out, const float *signal, float fraction, int n, const float *coeffs, int n_phases, int taps) {
    float get_filter = fraction * (float)(n_phases - 1) + 0.5f;     /* fraction * 100.0f + 0.5f */
    int delay_int = (int)get_filter;
    if (delay_int > n_phases - 1) delay_int = n_phases - 1;
    for (int k = 0; k < n; k++)
        for (int i = 0; i < taps; i++) out[k] = out[k] + coeffs[(size_t)delay_int * taps + i] * signal[k + i];
}

/* Particle::das with the FIR delay(): the delayed sum of one direction, channels in mask order */
void orc_particle_das_fir(const float *window, int W, int n, const int *index, int usable, const int32_t *offsets,
                          const float *fractions, const float *coeffs, int n_phases, int taps, float *out) {
    memset(out, 0, sizeof(float) * n);
    for (int s = 0; s < usable; s++) {
        int i = index[s];
        orc_delay_fir(out, &window[(size_t)i * W + offsets[i]], fractions[i], n, coeffs, n_phases, taps);
    }
}

void orc_mimo_update_fir(const float *window, int C, int W, int n, const int *index, int usable,
                         const int32_t *offsets, const float *fractions, int D, const float *coeffs, int n_phases,
                         int taps, float *power) {
    float *out = (float *)malloc(sizeof(float) * n);
    for (int m = 0; m < D; m++) {
        memset(out, 0, sizeof(float) * n);
        for (int s = 0; s < usable; s++) {
            int i = index[s];
            orc_delay_fir(out, &window[(size_t)i * W + offsets[(size_t)m * C + i]], fractions[(size_t)m * C + i], n, coeffs, n_phases, taps);
        }
        float p = hp_power(out, n);
        p /= (float)(n * usable);
        power[m] = p;
    }
    free(out);
}

/* ---- f3: the steps after the map: bilinear resize of the heat-map and peak -> Target ------------------------------ */
/* cv::resize(compact, normal, normal.size(), 0, 0, cv::INTER_LINEAR) on CV_8UC1 (src/aw_processing_unit/
 * aw_processing_unit.cpp:252).  OpenCV is a third-party dependency absent from /root/reference (libopencv-dev 4.5.4 in
 * the reference's Dockerfile); its 8-bit INTER_LINEAR path is fixed point: coefficients cvRound(c * 2048) as short,
 * horizontal pass in int, vertical pass ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16), then (v + 2) >> 2.
 * Horizontal coordinates clamp the fraction to 0 at the borders, vertical ones keep it and clip the row index.
 * Pinned: tests/golden/resize.npz holds cv2.resize outputs (opencv-python 4.13, generated by make_golden.py). */
static void resize_coeffs(int isz, int osz, int clamp, int *ofs, short *a0, short *a1) {
    const double inv = (double)osz / (double)isz, scale = 1.0 / inv;
    for (int d = 0; d < osz; d++) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int sx = (int)floorf(f);
        f -= (float)sx;
        if (clamp) {
            if (sx < 0) { f = 0.f; sx = 0; }
            if (sx >= isz - 1) { f = 0.f; sx = isz - 1; }
        }
        ofs[d] = sx;
        a0[d] = (short)lrintf((1.f - f) * 2048.f);
        a1[d] = (short)lrintf(f * 2048.f);
    }
}

void orc_resize_linear_u8(const uint8_t *src, int ih, int iw, uint8_t *dst, int oh, int ow) {
    int *xo = (int *)malloc(sizeof(int) * ow), *yo = (int *)malloc(sizeof(int) * oh);
    short *xa0 = (short *)malloc(2 * ow), *xa1 = (short *)malloc(2 * ow), *ya0 = (short *)malloc(2 * oh), *ya1 = (short *)malloc(2 * oh);
    resize_coeffs(iw, ow, 1, xo, xa0, xa1);
    resize_coeffs(ih, oh, 0, yo, ya0, ya1);
    for (int y = 0; y < oh; y++) {
        int y0 = yo[y] < 0 ? 0 : (yo[y] > ih - 1 ? ih - 1 : yo[y]);
        int y1 = yo[y] + 1 < 0 ? 0 : (yo[y] + 1 > ih - 1 ? ih - 1 : yo[y] + 1);
        for (int x = 0; x < ow; x++) {
            int x0 = xo[x], x1 = x0 + 1 > iw - 1 ? iw - 1 : x0 + 1;
            int S0 = src[y0 * iw + x0] * xa0[x] + src[y0 * iw + x1] * xa1[x];
            int S1 = src[y1 * iw + x0] * xa0[x] + src[y1 * iw + x1] * xa1[x];
            int v = ((ya0[y] * (S0 >> 4)) >> 16) + ((ya1[y] * (S1 >> 4)) >> 16);
            v = (v + 2) >> 2;
            dst[y * ow + x] = (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
        }
    }
    free(xo); free(yo); free(xa0); free(xa1); free(ya0); free(ya1);
}

/* Peaks of the MIMO map as Targets (a14: src/dsp/worker.h:32-61; the gradient worker is the reference's only producer,
 * src/dsp/gradient_ascend.cpp:399-408).  NEW behaviour, defined here and mirrored by the library: a grid direction is a
 * target when it is the maximum of its 3x3 neighbourhood (ties: lowest index) and carries at least min_rel of the map's
 * maximum; targets come in order of decreasing power (ties: index).  power = the map value (the tracker reports the mean
 * beam power around its direction); probability = 1 / gradientError like the tracker's, with gradientError formed from
 * the four grid neighbours instead of the four quadrant beams (gradient_ascend.cpp:62-76): (|right - left| + |down - up|)
 * / (left + right + up + down), a missing neighbour at the border replaced by the direction itself. */
int orc_map_targets(const float *power, int rows, int cols, int max_targets, float min_rel, int *index, float *pw, float *prob) {
    const int D = rows * cols;
    float maxV = 0.0f;
    for (int i = 0; i < D; i++) if (power[i] > maxV) maxV = power[i];
    const float thr = min_rel * maxV;
    unsigned char *taken = (unsigned char *)calloc(D, 1);
    int n = 0;
    while (n < max_targets) {
        int best = -1;
        for (int i = 0; i < D; i++) {
            if (taken[i]) continue;
            const float p = power[i];
            if (!(p >= thr) || !(p > 0.0f)) continue;
            const int r = i / cols, c = i % cols;
            int is_max = 1;
            for (int dr = -1; dr <= 1 && is_max; dr++)
                for (int dc = -1; dc <= 1; dc++) {
                    const int rr = r + dr, cc = c + dc;
                    if ((dr == 0 && dc == 0) || rr < 0 || rr >= rows || cc < 0 || cc >= cols) continue;
                    const int j = rr * cols + cc;
                    if (power[j] > p || (power[j] == p && j < i)) { is_max = 0; break; }
                }
            if (!is_max) continue;
            if (best < 0 || p > power[best]) best = i;      /* index order breaks ties towards the lower index */
        }
        if (best < 0) break;
        taken[best] = 1;
        const int r = best / cols, c = best % cols;
        const float p = power[best];
        const double ql = c > 0 ? power[best - 1] : p, qr = c < cols - 1 ? power[best + 1] : p;
        const double qu = r > 0 ? power[best - cols] : p, qd = r < rows - 1 ? power[best + cols] : p;
        const double err = (fabs(qr - ql) + fabs(qd - qu)) / (((ql + qr) + qu) + qd);
        double pr = 1.0 / err;
        if (!(pr < 3.4028234663852886e38)) pr = 3.4028234663852886e38;
        index[n] = best;
        pw[n] = p;
        prob[n] = (float)pr;
        n++;
    }
    free(taken);
    return n;
}
