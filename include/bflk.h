/* bflk.h -- C ABI of the B200-native delay-and-sum path of beamforming-lk.
 *
 * This is the whole drop-in boundary: plain C types, caller-owned buffers, no exceptions, no torch
 * types.  Every entry point returns 0 on success or a negative bflk_status; the message of the last
 * failure on a handle is available from bflk_last_error().  A handle is "thread-compatible": use it
 * from one compute thread at a time (the reference calls Worker::update() under Worker::lock,
 * src/dsp/worker.h:219-222).  There is NO CPU fallback: without a usable CUDA device bflk_create fails.
 *
 * Reference interfaces replaced (paths relative to the reference repository):
 *   bflk_create / bflk_destroy      MIMOWorker / MISOWorker construction + destruction
 *                                   (src/dsp/mimo.cpp:7-13, src/dsp/miso.cpp:5-13, worker.h:111-114)
 *   bflk_set_geometry               Antenna::points as built by create_antenna (src/geometry/antenna.cpp:60-87)
 *   bflk_set_tiled_geometry         create_antenna + place_antenna for n arrays (antenna.cpp:56-87)
 *   bflk_set_channel_mask           Antenna::index / Antenna::usable written by
 *                                   AWProcessingUnit::calibrate (aw_processing_unit.cpp:190-200)
 *   bflk_set_grid_fov               MIMOWorker::computeDelayLUT (src/dsp/mimo.cpp:20-59)
 *   bflk_set_grid_tables            the same LUT supplied by the caller (offsetDelays / fractionalDelays, mimo.h:86-89)
 *   bflk_steer_tables               Particle::steer (src/dsp/particle.cpp:37-49)
 *   bflk_set_focus                  (no reference counterpart: the reference steers at plane waves only) the tables of
 *                                   all of the above focused at a point at a given distance
 *   bflk_power_map*                 MIMOWorker::update (src/dsp/mimo.cpp:97-151) -> powerdB
 *   bflk_beams_batch_dev, bflk_session_beams   the same, with the delayed sums out[] of every direction (mimo.cpp:121-130)
 *   bflk_power_map_batch*_submit / _wait / _join   the same in continuous operation (the reference's worker loop,
 *                                   src/dsp/worker.h:212-224, calls update() frame after frame): batches overlap their
 *                                   uploads, pre-passes and collectives with the kernels of their neighbours
 *   bflk_set_channel_split, bflk_launch_shape   latency shape of one live frame (MIMOWorker::update once per 5.24 ms)
 *   bflk_enable_timing / bflk_kernel_time_ms / bflk_launch_count   (no reference counterpart: measurement hooks)
 *   bflk_miso*                      Particle::steer + Particle::das + Particle::beam
 *                                   (src/dsp/particle.cpp:37-103) as used by MISOWorker::update (miso.cpp:39-46)
 *   bflk_heatmap                    MIMOWorker::populateHeatmap (src/dsp/mimo.cpp:61-95)
 *   bflk_resize_u8                  cv::resize(..., INTER_LINEAR) in AWProcessingUnit::draw (aw_processing_unit.cpp:245-259)
 *   bflk_targets                    Worker::tracking / getTargets (src/dsp/worker.h:32-61,136-142) for the MIMO map
 *   bflk_targets_batch_dev, bflk_session_targets   the same for every map of a device batch or a session backlog, in one launch
 *   bflk_calibrate                  AWProcessingUnit::calibrate mask (aw_processing_unit.cpp:126-200)
 *   bflk_ingest_i32, bflk_power_map_i32   Pipeline::receive_exposure conversion (src/fpga/pipeline.cpp:260-297)
 *   bflk_stream_*                   Streams (src/fpga/streams.hpp:152-182) + the worker loop (src/dsp/worker.h:212-224),
 *                                   kept on the device: push samples as they arrive, map every frame
 *   bflk_comm_*, bflk_shard_plan, bflk_power_map_batch_sharded*, bflk_group_*   (no reference counterpart: the reference
 *                                   is single-threaded per worker, src/dsp/worker.h:90; AWProcessingUnit::start,
 *                                   src/aw_processing_unit/aw_processing_unit.cpp:67-95, is where a group is created)
 */
#ifndef BFLK_H
#define BFLK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BFLK_VERSION 1

typedef enum bflk_status {
    BFLK_OK = 0,
    BFLK_ERR_INVALID = -1,   /* bad argument / inconsistent configuration */
    BFLK_ERR_STATE = -2,     /* call sequence: geometry / grid not set yet */
    BFLK_ERR_CUDA = -3,      /* CUDA runtime failure (message has the CUDA error string) */
    BFLK_ERR_NO_DEVICE = -4, /* no usable sm_100 device: there is no CPU fallback */
    BFLK_ERR_RANGE = -5      /* a delay does not fit the history / window the caller configured */
} bflk_status;

/* Runtime replacement for the reference's compile-time constants. Zero-initialise, then fill;
 * bflk_default_config() gives the reference's values. */
typedef struct bflk_config {
    int32_t n_channels;       /* C: physical microphones (n_arrays * 64; ELEMENTS, antenna.h:20) */
    int32_t frame_len;        /* N: samples per frame (N_SAMPLES 256, streams.hpp:28) */
    int32_t history;          /* H: offset = H - int(delay) (N_SAMPLES in mimo.cpp:50 / particle.cpp:44) */
    int32_t window_len;       /* W: floats per channel handed to single-frame calls (N_ITEMS_BUFFER 1024) */
    double sample_rate;       /* SAMPLE_RATE 48828.0, antenna.h:17 */
    double propagation_speed; /* PROPAGATION_SPEED 340.0, antenna.h:16 */
    int32_t device;           /* CUDA device ordinal */
    int32_t reserved;
} bflk_config;

typedef struct bflk_handle bflk_handle;

void bflk_default_config(bflk_config *cfg);
int bflk_version(void);

int bflk_create(const bflk_config *cfg, bflk_handle **out);
int bflk_destroy(bflk_handle *h);
/* Message of the last failure on h (h == NULL: last failure of bflk_create on this thread). */
const char *bflk_last_error(const bflk_handle *h);

/* ---- geometry, mask, steering tables ------------------------------------------------------------ */
/* xyz[C][3] in metres (row c = element c; same memory as the reference's column-major 3 x C matrix). */
int bflk_set_geometry(bflk_handle *h, const float *xyz, int32_t n_channels);
/* n_tiles 8x8 arrays at 2 cm pitch (create_antenna), tile a translated by origins[a][3]; C = 64*n_tiles. */
int bflk_set_tiled_geometry(bflk_handle *h, int32_t n_tiles, const float *origins);
int bflk_get_geometry(const bflk_handle *h, float *xyz);
/* index[usable]: physical channels summed, IN THIS ORDER (mimo.cpp:124-130). NULL = all channels. */
int bflk_set_channel_mask(bflk_handle *h, const int32_t *index, int32_t usable);

/* rows x cols direction grid over fov degrees; direction k = r*cols + c. Builds the LUT on the device. */
int bflk_set_grid_fov(bflk_handle *h, int32_t rows, int32_t cols, float fov_deg);
/* Caller-supplied LUT [D][C] (physical element index), offsets as in the reference (H - int(delay)). */
int bflk_set_grid_tables(bflk_handle *h, const int32_t *offsets, const float *fractions, int32_t n_directions);
/* Declares that a caller-supplied LUT is a row-major rows x cols grid of neighbouring directions (rows * cols = D): the
 * register-tiled kernels, which share sample windows inside 2x2 tiles of adjacent directions, then serve it like a
 * bflk_set_grid_fov grid; without it such tables run on the lane-broadcast kernel. */
int bflk_set_grid_shape(bflk_handle *h, int32_t rows, int32_t cols);
/* Multi-GPU sharding: this handle computes directions [first, first+count) of the grid only. */
int bflk_set_direction_range(bflk_handle *h, int32_t first, int32_t count);
int bflk_get_n_directions(const bflk_handle *h, int32_t *total, int32_t *first, int32_t *count);
int bflk_get_grid(const bflk_handle *h, double *theta, double *phi);            /* [D] each */
int bflk_get_tables(const bflk_handle *h, int32_t *offsets, float *fractions);  /* [D][C] */
/* Particle::steer for T directions: offsets / fractions [T][C], computed by the device table kernel. */
int bflk_steer_tables(bflk_handle *h, const double *theta, const double *phi, int32_t n_targets,
                      int32_t *offsets, float *fractions);
/* Near-field steering: every table the handle builds from angles steers at the point distance_m metres from the origin of
 * the geometry's frame in that direction, instead of at a plane wave from it.  For direction (theta, phi), with cz, sz,
 * cy, sy the floats of the far-field rotation (cos / sin of float(phi) and of -float(theta)), u = (-sy cz, sy sz, cy) in
 * double and element p promoted to double, the element's z'' becomes
 *     z = (2 r u.p - p.p) / (r + |r u - p|)    (= r - |r u - p|, without the cancellation),
 * every double operation rounded where it is written ((a0 b0 + a1 b1) + a2 b2 for dot products), then zf = float(z);
 * from zf on the float path is the far-field one (times the delay scale, minus the minimum, integer and fraction split).
 * As distance_m grows the tables tend to the far-field ones.  distance_m = 0 is the far field (the default): the tables
 * are then bit-identical to those of a handle that never called this.
 * The focus applies to: the bflk_set_grid_fov grid (rebuilt at once when one is set; later bflk_set_grid_fov calls use
 * the focus), bflk_steer_tables, bflk_miso and bflk_miso_dev (FIR form included) and bflk_monopulse.  Tables the caller
 * supplies (bflk_set_grid_tables) are not touched, and grid angles (bflk_get_grid, Target records) do not change.
 * BFLK_ERR_INVALID: distance_m negative, NaN or infinite, or not larger than the largest |p| of the geometry (the point
 * would lie inside the array); the table calls above check that again after a geometry change.  BFLK_ERR_RANGE: a
 * focused delay of the grid exceeds the history.  A refused call changes nothing: the previous focus and tables stay. */
int bflk_set_focus(bflk_handle *h, double distance_m);

/* ---- full-grid power map (MIMO) ------------------------------------------------------------------- */
/* window[C][W] channel-major snapshot exactly as read_stream() produces it (oldest sample first);
 * power_out[count] for this handle's direction range.  Host buffers; H2D + kernel + D2H, synchronous. */
int bflk_power_map(bflk_handle *h, const float *window, float *power_out);
/* Batched: stream[C][T] channel-major continuous samples; frame b uses window stream[c][b*N .. b*N+W'),
 * i.e. consecutive frames advance by N samples like Streams::forward().  T >= (B-1)*N + H + N + 1.
 * power_out[B][count].  Every batch call takes any B >= 1: batches beyond the 65 535 blocks of a CUDA grid dimension
 * run in slabs or grid-stride loops. */
int bflk_power_map_batch(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out);
/* Continuous operation: _submit returns as soon as the batch is enqueued (at most two batches in flight; a third submit
 * waits for the oldest), _wait blocks until the oldest batch in flight has delivered its maps into the power_out it was
 * submitted with.  The upload of batch i + 1 overlaps the kernels of batch i.  stream / power_out must stay valid and
 * untouched until the matching _wait; page-locked buffers (bflk_pin_host) are needed for the copies to overlap. */
int bflk_power_map_batch_submit(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out);
int bflk_power_map_batch_wait(bflk_handle *h);
/* One frame straight from the wire format: frames[W][C] int32, one row per time sample as the FPGA sends it
 * (src/fpga/receiver.h:24-30).  The conversion of Pipeline::receive_exposure (serpentine un-flip, / 2^23,
 * src/fpga/pipeline.cpp:260-297) runs on the device and feeds the power map without a host round trip. */
int bflk_power_map_i32(bflk_handle *h, const int32_t *frames, float *power_out);
/* A batch from the wire format: frames[T][C] int32 (T time samples, every sensor of the message in wire order), frame b
 * uses rows [b*N, b*N + H + N + 1).  One fused pass turns the wire samples into the kernel's staged layout (un-flip
 * folded into the column index, / 2^23, transpose, pair-interleave): no float copy of the stream exists, and the maps
 * are bit-identical to bflk_power_map_batch on the converted stream.  power_out[B][count].  At most 2^31 - 1 rows per
 * call (BFLK_ERR_INVALID beyond). */
int bflk_power_map_batch_i32(bflk_handle *h, const int32_t *frames, int64_t n_samples, int32_t n_frames, float *power_out);
int bflk_power_map_batch_i32_dev(bflk_handle *h, const int32_t *frames_dev, int64_t n_samples, int32_t n_frames,
                                 float *power_dev, void *cuda_stream);
/* Same with DEVICE pointers, asynchronous on cuda_stream (a cudaStream_t, NULL = the handle's stream). */
int bflk_power_map_batch_dev(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                             float *power_dev, void *cuda_stream);
/* The beams with the maps: beams_dev[B][count][N] = for frame b and direction first + k of the range, the delayed sum
 * out[i] (i < N) that its power squares (MIMOWorker::update, src/dsp/mimo.cpp:121-130, before the high-pass): the channels
 * in mask order over stream[c][b*N + offset + i], interpolated as the kernel in use interpolates.  Kernels 1, 2 and 3 give
 * the bits of the reference's delay(); kernel 4 (and the channel split) the two-FMA form's sums, within a few roundings
 * per channel of them; with bflk_set_fir the FIR sums.  power_dev[B][count] holds the bits bflk_power_map_batch_dev gives
 * on the same input.  stream_dev as there; beams_dev (8-byte aligned) and power_dev are required device buffers.
 * Asynchronous on cuda_stream; argument checks and error codes as bflk_power_map_batch_dev. */
int bflk_beams_batch_dev(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames, float *beams_dev,
                         float *power_dev, void *cuda_stream);
/* Continuous operation on DEVICE-resident streams: _dev_submit enqueues the batch on one of the handle's two compute streams
 * (alternating, each with its own scratch) once cuda_stream has reached the call, and returns; consecutive batches overlap --
 * the pack pre-pass of batch i + 1 runs under the kernel of batch i and its CTAs fill the SMs the last CTAs of batch i leave
 * idle.  power_dev of every batch submitted so far is complete for work enqueued on cuda_stream after
 * bflk_power_map_batch_dev_join(h, cuda_stream) (asynchronous: it enqueues a wait).  Batches in flight need their own
 * power_dev.  Same bits as bflk_power_map_batch_dev.  Grids the register-tiled kernels do not serve run in stream order. */
int bflk_power_map_batch_dev_submit(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                                    float *power_dev, void *cuda_stream);
int bflk_power_map_batch_dev_join(bflk_handle *h, void *cuda_stream);
/* Selects the kernel: 0 = automatic, 1 = generic per-direction kernel, 2 = register-tiled kernel with the reference's
 * exact operation triple (delayed sums bit-identical to delay(), src/dsp/delay.cpp:16-26), 3 = lane-broadcast kernel,
 * 4 = register-tiled kernel in two-FMA form (f*s[i] + (1-f)*s[i+1]: as accurate as the reference against exact
 * arithmetic, power maps within the 1e-4 bar, ~13 % faster than 2).  Automatic = 4 when the grid tiles, else 3, else 1.
 * 2 and 4 need an even frame_len >= 256 and float rows of even length (the row stride: T of a batch, W of a single frame;
 * wire rows have no such condition); 3 needs frame_len >= 256.  A call the chosen kernel cannot serve returns
 * BFLK_ERR_STATE; the automatic choice falls back instead. */
int bflk_set_kernel(bflk_handle *h, int32_t which);
/* Latency option for calls too small to fill the GPU (a live worker's single frame, MIMOWorker::update once per 5.24 ms,
 * src/dsp/mimo.cpp:97-151): on != 0 lets the two-FMA form (kernel 0 / 4) split the CHANNELS of a frame across a thread-block
 * cluster of 2 or 4 CTAs, whose partial delayed sums are added through distributed shared memory in a fixed order before
 * the power epilogue (cfg3 single frame: 16 CTAs become 128).  The result is deterministic and within the same 1e-4 bar, but
 * the channel sum is associated differently than in a large batch, so "a batch gives the same bits as its frames one by
 * one" holds only with the option off (the default).  Kernel 2 never splits (its sums stay bit-identical to delay()). */
int bflk_set_channel_split(bflk_handle *h, int32_t on);
/* The CTA shape a power-map call gets (pure arithmetic, no device needed): rows x cols directions (2x2 tiles), n_channels
 * usable channels, n_frames frames of frame_len samples on a GPU with n_sms SMs.  warps = warps per CTA, 0 = the throughput
 * shape (16-warp CTAs; every call that fills two waves of them); split = cluster size of the channel split (1 = none; 2 / 4
 * only with channel_split != 0).  The model behind it (waves x (fixed cost + channels x cycles per channel step for the warps
 * sharing a scheduler)) is fitted to B200 measurements: profiles/r2c_latency_shapes.txt. */
int bflk_launch_shape(int32_t rows, int32_t cols, int32_t n_channels, int32_t frame_len, int32_t n_frames, int32_t n_sms,
                      int32_t channel_split, int32_t *warps, int32_t *split);
/* Which kernel the last power-map call used (1 generic, 2 tiled exact, 3 lane-broadcast, 4 tiled two-FMA; 0 = none yet), the
 * largest offset spread inside a direction tile (or tile pair) for the current grid, and the window chunks of the tiled
 * variant in use. */
int bflk_get_kernel(const bflk_handle *h, int32_t *last_used, int32_t *tile_span, int32_t *window_chunks);
/* Number of kernel launches issued by this handle so far (bench.py's gpu_launches). */
int64_t bflk_launch_count(const bflk_handle *h);
/* Kernel timing for the roofline report: when enabled, every launch of the dominant delay-and-sum kernel
 * (and of the pack pre-pass) is bracketed by CUDA events on the stream it is launched on.
 * bflk_kernel_time_ms synchronises on those events, returns the accumulated milliseconds and launch
 * counts since the last call, and resets the accumulators. */
int bflk_enable_timing(bflk_handle *h, int32_t on);
/* FP32 throughput a packed-FMA saturation kernel reaches on this device right now (TFLOP/s, ~10 ms): the empirical
 * denominator reported next to the nominal FP32 roofline. */
int bflk_fp32_peak_tflops(bflk_handle *h, float *tflops);
int bflk_kernel_time_ms(bflk_handle *h, float *das_ms, int32_t *das_launches, float *pack_ms, int32_t *pack_launches);

/* ---- streaming session: samples in as they arrive, a power map for every frame ------------------------- */
/* The session keeps the history of every channel on the device (a mirrored ring, the twin of the reference's double-mapped
 * Streams, src/fpga/streams.hpp:152-182), so a live caller pushes only new samples and maps every frame -- where the
 * reference's worker loop drops the frames that arrive while it computes (src/dsp/worker.h:212-224).
 * Frame b is frame b of bflk_power_map_batch over everything pushed since bflk_stream_open: samples
 * [b*N, b*N + H + N + 1), plus n_taps - 2 with bflk_set_fir.  It is READY once that many samples have been pushed.
 *
 * bflk_stream_open (re)starts a session at sample 0, frame 0 with room for max_frames ready frames.  The session keeps raw
 * samples only: kernel, grid, mask, direction range and channel split are read by each maps call.  A bflk_set_fir that
 * lengthens a frame beyond what open sized the history for makes the maps calls fail with BFLK_ERR_STATE until the next
 * open.  bflk_stream_close (or bflk_destroy) frees the session.
 *
 * A push of n samples per channel (1 <= n <= the ring's capacity) returns once the caller's buffer may be reused; the
 * wire form needs n_channels % 8 == 0.  A push never blocks on or fails for a slow consumer: it overwrites the oldest
 * sample, and every frame whose first sample is gone is SKIPPED (next_frame moves past it, skipped counts it).
 *
 * bflk_stream_power_maps maps the oldest min(max_frames, ready) frames in ONE call -- a backlog as one batch, a single frame
 * in the latency shape -- into power_out[n][count] for the current direction range, reports the first frame and n, and
 * consumes them.  Nothing ready: *n_frames = 0, BFLK_OK, and nothing else changes.  Synchronous on the handle's stream;
 * after a call that returned one frame, bflk_targets / bflk_heatmap with a NULL map use it (as after bflk_power_map).
 * bflk_session_beams is bflk_stream_power_maps that also returns the frames' beams (bflk_beams_batch_dev):
 * beams_out[n][count][N] and power_out[n][count] on the host.  It takes and consumes frames exactly as the maps call does
 * (the two may be interleaved), and after a one-frame call bflk_targets / bflk_heatmap with a NULL map use that frame's map.
 * bflk_session_targets is bflk_stream_power_maps that also returns the Targets of every frame it maps (bflk_targets_batch_dev,
 * one launch for all of them): power_out[n][count], targets_out[n][max_targets] and n_targets[n] on the host; records past a
 * frame's count are not written.  It takes and consumes frames exactly as the other two (all three may be interleaved), and
 * after a one-frame call bflk_targets / bflk_heatmap with a NULL map use that frame's map.  It needs a bflk_set_grid_fov
 * grid and the whole grid on the handle (BFLK_ERR_STATE otherwise); a refused call consumes no frame.
 * bflk_stream_discard skips every ready frame but the newest `keep`.  bflk_stream_status: samples pushed per channel, the
 * next frame a maps call returns, frames ready, frames skipped so far.
 *
 * bflk_stream_window makes a pushed frame still held by the ring the resident window: bflk_miso, bflk_miso_dev and
 * bflk_monopulse with window == NULL then read it in place.  It is forgotten when the ring overwrites the frame, on close
 * and on a new open (MISO with NULL then fails with BFLK_ERR_INVALID).  A frame that is no longer held or not fully pushed:
 * BFLK_ERR_STATE.  Any session call without an open session: BFLK_ERR_STATE. */
int bflk_stream_open(bflk_handle *h, int32_t max_frames);
int bflk_stream_close(bflk_handle *h);
int bflk_stream_push(bflk_handle *h, const float *samples, int32_t n);      /* [C][n], channel-major */
int bflk_stream_push_i32(bflk_handle *h, const int32_t *rows, int32_t n);   /* [n][C], wire order */
int bflk_stream_power_maps(bflk_handle *h, int32_t max_frames, float *power_out, int64_t *first_frame, int32_t *n_frames);
int bflk_session_beams(bflk_handle *h, int32_t max_frames, float *beams_out, float *power_out, int64_t *first_frame,
                       int32_t *n_frames);
typedef struct bflk_target bflk_target;
int bflk_session_targets(bflk_handle *h, int32_t max_frames, int32_t max_targets, float min_rel_power, float *power_out,
                         bflk_target *targets_out, int32_t *n_targets, int64_t *first_frame, int32_t *n_frames);
int bflk_stream_discard(bflk_handle *h, int32_t keep);
int bflk_stream_status(const bflk_handle *h, int64_t *pushed, int64_t *next_frame, int32_t *ready, int64_t *skipped);
int bflk_stream_window(bflk_handle *h, int64_t frame);

/* ---- multi-GPU: the grid (x the frames of a batch) sharded across the GPUs of one box ---------------- */
/* Every direction's power is independent (src/dsp/mimo.cpp:121-151), so G ranks are arranged as G_d direction groups x
 * G_f frame groups (G = G_d * G_f): rank r computes direction slice r % G_d of the row-major grid for frame slice
 * r / G_d of a batch, and ONE NCCL all-gather per batch assembles the complete [B][D] maps on every rank.  Channels
 * are never sharded (that would reorder the channel sum).  dir_groups: G_d; 0 = automatic (2 when G is even, else 1);
 * dir_groups = G is the pure grid sharding, dir_groups = 1 the pure batch sharding.
 * NCCL is loaded at run time (libnccl.so.2); without it these calls fail and the single-GPU API is unaffected.
 *
 * (a) one process per GPU: rank 0 calls bflk_comm_unique_id, the caller broadcasts the 128 bytes, every rank calls
 *     bflk_comm_init_rank on its own handle (collective).  All ranks then set the same geometry / grid / mask and call
 *     the sharded entry points together. */
int bflk_comm_unique_id(uint8_t *id128);
int bflk_comm_init_rank(bflk_handle *h, const uint8_t *id128, int32_t n_ranks, int32_t rank, int32_t dir_groups);
int bflk_comm_info(const bflk_handle *h, int32_t *n_ranks, int32_t *rank, int32_t *dir_groups, int32_t *frame_groups,
                   int64_t *collectives);
/* The slice rank `rank` of `n_ranks` computes (pure arithmetic, needs no device). */
int bflk_shard_plan(int32_t n_directions, int32_t n_frames, int32_t n_ranks, int32_t dir_groups, int32_t rank,
                    int32_t *dir_first, int32_t *dir_count, int32_t *frame_first, int32_t *frame_count);
/* stream_dev[C][n_samples]: the SAME batch resident on every rank's device; power_all_dev[B][D] complete on every rank.
 * Asynchronous on cuda_stream (NULL = the handle's stream). */
int bflk_power_map_batch_sharded_dev(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                                     float *power_all_dev, void *cuda_stream);
/* Host buffers: every rank passes the same batch stream[C][n_samples] (pinned memory recommended) but reads only the
 * C / G_d channel rows of its own frame slice; the slice is replicated inside its frame group over NVLink, chunk by
 * chunk, overlapping the kernels.  power_out[B][D] (NULL on ranks that do not need the maps).  Synchronous. */
int bflk_power_map_batch_sharded(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out);
/* Continuous operation on DEVICE-resident streams (every rank alike): _dev_submit enqueues the rank's kernels on cuda_stream
 * and the all-gather + assembly on the communicator's own stream, in alternating buffer sets, so the kernels of batch i + 1
 * run under the collective of batch i (src/dsp/mimo.cpp:121-151: a rank's directions do not depend on the gather).
 * power_all_dev of every batch submitted so far is complete for work enqueued on cuda_stream after
 * bflk_power_map_batch_sharded_dev_join(h, cuda_stream) (asynchronous: it enqueues a wait, the host does not block). */
int bflk_power_map_batch_sharded_dev_submit(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                                            float *power_all_dev, void *cuda_stream);
int bflk_power_map_batch_sharded_dev_join(bflk_handle *h, void *cuda_stream);
/* Continuous operation (every rank alike): _submit enqueues a host batch and returns, _wait blocks until everything
 * submitted so far has delivered its maps; the uploads of batch i + 1 run under the kernels and collectives of batch i.
 * stream / power_out must stay valid until the _wait. */
int bflk_power_map_batch_sharded_submit(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out);
int bflk_power_map_batch_sharded_wait(bflk_handle *h);
/* (b) one process, several devices (single-process callers such as the reference's AWProcessingUnit): n_devices
 *     handles, one per device_ids[i], sharing one job; the setters apply to every member. */
typedef struct bflk_group bflk_group;
int bflk_group_create(const bflk_config *cfg, const int32_t *device_ids, int32_t n_devices, int32_t dir_groups, bflk_group **out);
int bflk_group_destroy(bflk_group *g);
int32_t bflk_group_size(const bflk_group *g);
bflk_handle *bflk_group_handle(bflk_group *g, int32_t i);
const char *bflk_group_last_error(const bflk_group *g);
int bflk_group_set_geometry(bflk_group *g, const float *xyz, int32_t n_channels);
int bflk_group_set_tiled_geometry(bflk_group *g, int32_t n_tiles, const float *origins);
int bflk_group_set_channel_mask(bflk_group *g, const int32_t *index, int32_t usable);
int bflk_group_set_grid_fov(bflk_group *g, int32_t rows, int32_t cols, float fov_deg);
int bflk_group_set_kernel(bflk_group *g, int32_t which);
int bflk_group_set_focus(bflk_group *g, double distance_m);
/* stream[C][n_samples] on the host -> power_out[B][D] on the host; all devices of the group work on it. */
int bflk_group_power_map_batch(bflk_group *g, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out);
/* stream_dev[i] / power_all_dev[i]: the batch and the [B][D] result on device i.  Asynchronous on each member's stream. */
int bflk_group_power_map_batch_dev(bflk_group *g, const float *const *stream_dev, int64_t n_samples, int32_t n_frames,
                                   float *const *power_all_dev);
int bflk_group_synchronize(bflk_group *g);

/* ---- dynamic steering (MISO) --------------------------------------------------------------------- */
/* Keep one frame's window[C][W] on the device across calls: the tracker evaluates many steps on the same frame
 * (src/dsp/gradient_ascend.cpp:301-409), and bflk_miso / bflk_monopulse with window == NULL use it instead of uploading
 * 4 * C * W bytes every time.  bflk_set_window copies a host buffer (NULL forgets it); bflk_set_window_dev borrows a
 * device buffer the caller keeps alive. */
int bflk_set_window(bflk_handle *h, const float *window);
int bflk_set_window_dev(bflk_handle *h, const float *window_dev);
/* For each target t: steer(theta[t], phi[t]); audio_out[t][N] = Particle::das; power_out[t] = Particle::beam.
 * Either output may be NULL. window[C][W] as in bflk_power_map, or NULL = the resident window.  One kernel launch:
 * the steering tables are built inside it (same bits as bflk_steer_tables); a delay beyond the history makes the
 * call return BFLK_ERR_RANGE.  Only the channels of the mask are checked: a microphone outside it may lie beyond the
 * history (its delay still counts for the minimum every delay is measured from), whereas bflk_steer_tables and
 * bflk_set_grid_fov check every channel. */
int bflk_miso(bflk_handle *h, const double *theta, const double *phi, int32_t n_targets, const float *window,
              float *audio_out, float *power_out);
/* Device pointers, asynchronous on cuda_stream (NULL = the handle's stream); window_dev == NULL = the resident window.
 * Being asynchronous it cannot return BFLK_ERR_RANGE: a delay beyond the history is clamped to it (validate the
 * directions once with bflk_steer_tables, or use bflk_miso).  With FIR interpolation set it builds its tables
 * synchronously and does return BFLK_ERR_RANGE.  It is ordered after the handle's earlier calls on other streams (and
 * bflk_miso after it), since all MISO calls share the handle's partial sums. */
int bflk_miso_dev(bflk_handle *h, const double *theta, const double *phi, int32_t n_targets,
                  const float *window_dev, float *audio_dev, float *power_dev, void *cuda_stream);

/* FIR fractional-delay interpolation instead of the 2-tap form: the reference's USE_FILTER build of delay()
 * (src/dsp/delay.cpp:28-40; coefficient table src/dsp/filter.h, 101 phases x 8 taps -- reference data, supplied by the
 * caller): phase = (int)(fraction * (n_phases - 1) + 0.5f), out[n] += coeffs[phase][i] * signal[n + i], i in order.
 * While set, power maps and MISO calls run through the generic kernel and a frame reads n_taps - 2 more samples;
 * coeffs = NULL restores the 2-tap form. */
int bflk_set_fir(bflk_handle *h, const float *coeffs, int32_t n_phases, int32_t n_taps);

/* Monopulse step of the gradient tracker (GradientParticle::findNearby + the beam part of GradientParticle::step,
 * quadrant form, src/dsp/gradient_ascend.cpp:18-81).  For each particle p: the four quadrant directions at angular
 * distance `spread` around (theta[p], phi[p]) (Spherical::quadrant, src/geometry/geometry.cpp:181-217 -- like the
 * reference it pulls theta[p] in by spread / 2 when theta + spread would pass pi / 2 and writes that back),
 * normalised to phi in [0, 2 pi), theta in [0, theta_limit] (normalizeSpherical, src/dsp/particle.h:24-27); their beam
 * powers q[p][4] (Particle::steer + Particle::beam) in ONE batched launch for all 4 * n_particles beams;
 * gradient[p][3] = {theta, phi, radius} = {((q3+q4)-(q1+q2)) / reference, ((q1+q4)-(q2+q3)) / reference, sum / 4}
 * (reference <= 0: not divided, the RELATIVE 0 build) and error[p] = (|phi| + |theta|) / sum of the undivided values.
 * The particle update itself (Particle::step, jump / tracking heuristics) stays with the caller.
 * near_theta / near_phi / q are [n_particles][4]; any output may be NULL. */
int bflk_monopulse(bflk_handle *h, double *theta, const double *phi, int32_t n_particles, double spread,
                   double theta_limit, double reference, const float *window, double *near_theta, double *near_phi,
                   double *q, double *gradient, double *error);

/* ---- neighbours of the path ------------------------------------------------------------------------ */
/* Page-lock a caller-owned host buffer (cudaHostRegister) so the H2D / D2H copies of the host-buffer entry points run at
 * full PCIe speed and asynchronously; the Worker adapter pins its snapshot buffer once. */
int bflk_pin_host(void *ptr, size_t bytes);
int bflk_unpin_host(void *ptr);
/* populateHeatmap: heat[count] = uchar(clip(255 * p / max)), argmax / max of the map.  power == NULL: the map the last
 * bflk_power_map call left on the device (n must equal its size). */
int bflk_heatmap(bflk_handle *h, const float *power, int32_t n, uint8_t *heat, int32_t *argmax, float *maxv);
/* cv::resize(compact, normal, normal.size(), 0, 0, cv::INTER_LINEAR) of the 8-bit heat-map (AWProcessingUnit::draw,
 * src/aw_processing_unit/aw_processing_unit.cpp:252): src[rows][cols] -> dst[out_rows][out_cols], bit-identical to
 * OpenCV's fixed-point 8-bit bilinear path. */
int bflk_resize_u8(bflk_handle *h, const uint8_t *src, int32_t rows, int32_t cols, int32_t out_rows, int32_t out_cols,
                   uint8_t *dst);
/* Peaks of the power map as Targets (struct Target, src/dsp/worker.h:32-61 -- what TargetHandler polls through
 * AWProcessingUnit::targets(), src/target_handler/target_handler.cpp:29-36).  The reference's MIMO worker never fills
 * Worker::tracking; this defines it: a grid direction is a target when it is the maximum of its 3x3 neighbourhood
 * (ties: lowest index) and carries at least min_rel_power of the map's maximum; strongest first.  power = the map
 * value; probability = 1 / gradientError as the gradient tracker reports it (src/dsp/gradient_ascend.cpp:62-76,406),
 * with the four grid neighbours in place of the four quadrant beams.  power == NULL: the map the last bflk_power_map
 * call left on the device (no upload).  Needs a bflk_set_grid_fov grid and the whole map on this handle: caller tables,
 * with or without bflk_set_grid_shape, or a direction range give BFLK_ERR_STATE.  max_targets: 1..256. */
struct bflk_target {         /* 40 bytes (typedef above) */
    double theta, phi;      /* Spherical direction of the grid cell (bflk_get_grid) */
    float power;
    float probability;
    int32_t direction;      /* r * cols + c */
    int32_t row, col;
    int32_t reserved;       /* 0 */
};
int bflk_targets(bflk_handle *h, const float *power, int32_t max_targets, float min_rel_power, bflk_target *out, int32_t *n_out);
/* The same for n_maps whole-grid maps on the DEVICE, one launch: power_dev[n_maps][D] (D = rows * cols; the handle's direction
 * range is not consulted, so a rank of a sharded job can pass its power_all_dev) -> targets_dev[n_maps][max_targets] (records
 * past a map's count are not written) and n_dev[n_maps], device buffers.  Each map's records are those bflk_targets gives for
 * it.  Asynchronous on cuda_stream (NULL = the handle's stream), ordered against the handle's earlier calls on other streams
 * as bflk_power_map_batch_dev is; the map bflk_targets / bflk_heatmap use with NULL is not touched.  Any n_maps >= 1;
 * max_targets 1..256.  Needs a bflk_set_grid_fov grid (BFLK_ERR_STATE otherwise). */
int bflk_targets_batch_dev(bflk_handle *h, const float *power_dev, int32_t n_maps, int32_t max_targets, float min_rel_power,
                           bflk_target *targets_dev, int32_t *n_dev, void *cuda_stream);
/* calibrate(): signals[64][W] of one array -> index[<=64], correction[<=64]; *usable = count. */
int bflk_calibrate(bflk_handle *h, const float *signals, int32_t window_len, float reference_power_level,
                   int32_t *index, float *correction, int32_t *usable, float *median, float *mean);
/* receive_exposure(): wire frames[n][n_sensors] int32 -> exposure[n_sensors][n] float (un-flip, / 2^23). */
int bflk_ingest_i32(bflk_handle *h, const int32_t *frames, int32_t n, int32_t n_sensors, float *exposure);

#ifdef __cplusplus
}
#endif
#endif /* BFLK_H */
