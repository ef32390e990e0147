/* oracle.h -- CPU restatement of the reference's delay-and-sum hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it.
 * The product (beamforming-lk_b200/csrc) never links, imports or executes this code.
 *
 * Parity status: "parity unpinned" by the reference's own tests (they hold no golden vector or
 * known-answer test for this path, SURVEY.md 8c).  The restatement is instead pinned against the
 * reference's own compiled kernel: oracle/_ref builds /root/reference/src/dsp/delay.cpp and
 * src/fpga/streams.hpp verbatim (see Makefile) and tests/test_oracle_ref.py checks bit-equality of
 * orc_delay / window semantics against it.  Geometry goes through Eigen in the reference, which is
 * not available here; its evaluation order is fixed below and documented in DESIGN.md.
 *
 * All citations are relative to /root/reference.
 */
#ifndef BFLK_ORACLE_H
#define BFLK_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* reference constants */
#define ORC_SAMPLE_RATE 48828.0       /* src/geometry/antenna.h:17 */
#define ORC_PROPAGATION_SPEED 340.0   /* src/geometry/antenna.h:16 */
#define ORC_COLUMNS 8                 /* src/geometry/antenna.h:18 */
#define ORC_ROWS 8                    /* src/geometry/antenna.h:19 */
#define ORC_ELEMENTS 64               /* src/geometry/antenna.h:20 */
#define ORC_DISTANCE 0.02f            /* src/geometry/antenna.h:21 */
#define ORC_N_SAMPLES 256             /* src/fpga/streams.hpp:28 */
#define ORC_WINDOW 1024               /* src/fpga/streams.hpp:30-32 (PAGE_SIZE / sizeof(float)) */

/* a1: create_antenna, src/geometry/antenna.cpp:60-87. xyz is 3 x (rows*columns), column = element,
 * stored column-major like Eigen::MatrixXf(3, n): xyz[3*i + {0,1,2}]. */
void orc_create_antenna(float *xyz, int columns, int rows, float distance);

/* Multi-array generalisation (SURVEY.md 7 hard part 5): n_tiles copies of the 8x8 tile, tile a
 * translated by origins[3*a..], channel c = a*64 + e. */
void orc_create_tiled_antenna(float *xyz, int n_tiles, const float *origins);

/* a2-a5: steering_vector_spherical, src/geometry/antenna.cpp:89-107,126-134 and
 * src/geometry/geometry.cpp:219-233.  delays[C] in samples, min-subtracted. */
void orc_steering_vector_spherical(const float *xyz, int C, double theta, double phi, float *delays);
/* the same with the delay scale k (samples per metre, float(sample_rate / propagation_speed)) given; the entry point
 * above passes float(ORC_SAMPLE_RATE / ORC_PROPAGATION_SPEED) */
void orc_steering_vector_spherical_k(const float *xyz, int C, double theta, double phi, float k, float *delays);

/* a6/a7 split: fraction = (float)modf((double)del, &ip); offset = history - (int)ip
 * (src/dsp/mimo.cpp:46-54, src/dsp/particle.cpp:37-49; history == N_SAMPLES == 256 there). */
void orc_split_delays(const float *delays, int C, int history, int32_t *offsets, float *fractions);

/* a6: direction grid of MIMOWorker::computeDelayLUT, src/dsp/mimo.cpp:20-43.  theta/phi [rows*cols].
 * Degenerate centre cell (norm == 0, odd grids) is defined as theta = 0, phi = 0 (deviation: the
 * reference divides by zero there). */
void orc_mimo_grid(int rows, int cols, double fov_deg, double *theta, double *phi);

/* a6: full LUT, offsets/fractions [D][C] row-major, D = rows*cols, k = r*cols + c. */
void orc_mimo_lut(const float *xyz, int C, int rows, int cols, double fov_deg, int history,
                  int32_t *offsets, float *fractions);
void orc_mimo_lut_k(const float *xyz, int C, int rows, int cols, double fov_deg, int history, float k,
                    int32_t *offsets, float *fractions);

/* a9: delay(), src/dsp/delay.cpp:16-26 (AVX2 variant) == scalar twin :44-48 with the FMA pinned:
 * out[i] = out[i] + fma(fraction, signal[i] - signal[i+1], signal[i+1]), i in [0, n). */
void orc_delay(float *out, const float *signal, float fraction, int n);

/* a10: MIMOWorker::update, src/dsp/mimo.cpp:97-151.  window[C][W] physical-channel-major (the
 * snapshot signals[l] = ring of antenna.index[l], mimo.cpp:100-103); index[usable] = Antenna::index;
 * offsets/fractions [D][C] indexed by physical element; power[D].  n = frame length (256). */
void orc_mimo_update(const float *window, int C, int W, int n, const int *index, int usable,
                     const int32_t *offsets, const float *fractions, int D, float *power);
/* same, but also returns the delayed sum out[D][n] (for bit-exactness checks of the accumulate) */
void orc_mimo_das(const float *window, int C, int W, int n, const int *index, int usable,
                  const int32_t *offsets, const float *fractions, int D, float *out);

/* a11: Particle::beam, src/dsp/particle.cpp:51-82 (USE_BANDPASS 1): power / n only. */
double orc_particle_beam(const float *window, int W, int n, const int *index, int usable,
                         const int32_t *offsets, const float *fractions, float *out_scratch);
/* a12: Particle::das, src/dsp/particle.cpp:88-103. out[n]. */
void orc_particle_das(const float *window, int W, int n, const int *index, int usable,
                      const int32_t *offsets, const float *fractions, float *out);

/* a13: MIMOWorker::populateHeatmap, src/dsp/mimo.cpp:61-95 (USE_DB 0).  heat[D] uchar; returns argmax. */
int orc_populate_heatmap(const float *power, int D, uint8_t *heat, float *max_out);

/* a15: AWProcessingUnit::calibrate mask for one 64-element array, aw_processing_unit.cpp:134-200.
 * signals[64][W]; returns usable, fills index[], correction[] (reference_power_level / power). */
int orc_calibrate(const float *signals, int W, float reference_power_level, int *index,
                  float *correction, float *median_out, float *mean_out);

/* f1: receive_exposure conversion, src/fpga/pipeline.cpp:260-297: wire sample-major int32
 * frames[n][n_sensors] -> float exposure[n_sensors][n] with serpentine column un-flip and /2^23. */
void orc_ingest(const int32_t *frames, int n, int n_sensors, float *exposure);

/* f2: Spherical::quadrant + normalizeSpherical; GradientParticle::step (quadrant form) */
void orc_quadrant(double *theta, double phi, double spread, double theta_limit, double *near_theta, double *near_phi);
void orc_monopulse_gradient(const double *q, double reference, double *gradient, double *error);

/* f4: FIR variant of delay() (delay.cpp:28-40) and the power map built on it */
void orc_delay_fir(float *out, const float *signal, float fraction, int n, const float *coeffs, int n_phases, int taps);
void orc_mimo_update_fir(const float *window, int C, int W, int n, const int *index, int usable,
                         const int32_t *offsets, const float *fractions, int D, const float *coeffs, int n_phases,
                         int taps, float *power);
/* Particle::das around the FIR delay(): out[n] of one direction (window rows W apart, offset + n + taps - 1 <= W) */
void orc_particle_das_fir(const float *window, int W, int n, const int *index, int usable, const int32_t *offsets,
                          const float *fractions, const float *coeffs, int n_phases, int taps, float *out);

#ifdef __cplusplus
}
#endif
/* f3: cv::resize INTER_LINEAR on 8-bit maps (aw_processing_unit.cpp:252) and map peaks as Targets (worker.h:32-61) */
void orc_resize_linear_u8(const uint8_t *src, int ih, int iw, uint8_t *dst, int oh, int ow);
int orc_map_targets(const float *power, int rows, int cols, int max_targets, float min_rel, int *index, float *pw, float *prob);

#endif
