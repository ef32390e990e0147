// bflk_internal.h -- shared declarations of the B200-native DAS library (not part of the C ABI).
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <memory>
#include <string>
#include <vector>

#include "../../include/bflk.h"

namespace bflk {

// One steering direction as the device table kernel consumes it: the four rotation-matrix entries the
// reference evaluates in double and stores as float (src/geometry/geometry.cpp:219-233).
struct DirTrig {
    float cz, sz;  // cos / sin of float(phi)            (rotateZ)
    float cy, sy;  // cos / sin of -float(theta)         (rotateY)
};

// Packed per-(direction tile, usable channel) entry of the register-tiled kernel (das_tile.cu).
// base: even-aligned smallest offset of the tile's directions, delta[r] = offset[r] - base.
struct __align__(16) TileEntry {
    uint32_t win_off;   // byte offset of lane 0's window inside a packed row (padded layout); two 16-bit offsets
                        // (window A | window B << 16) in the two-window modes
    uint32_t deltas;    // 4 x 6 bit: delta of slot r in bits [6r, 6r+6); bits 24-25 (26-27): (first chunk) & 3 of window A (B)
    int32_t span;       // max delta of the tile for this channel
    int32_t reserved;
    float frac[4];      // fractional delays of the 4 directions
};

// Entry of the two-FMA ("fast", tolerance mode) variant: the four pad-class byte offsets of the window ready to add to the
// lane's row address (class m & 3 of window chunk m; no address arithmetic left in the kernel), and g = fl(1 - f).
struct __align__(16) TileEntryFast {
    uint32_t cls_off[4];  // byte offset of lane 0's window inside the STAGE (row offset (s % kTileCC) * row_bytes included) for chunk classes 0..3
    uint32_t deltas;      // 4 x 6 bit: delta of slot r in bits [6r, 6r+6)
    int32_t span;
    int32_t reserved[2];
    float frac[4];        // f
    float comp[4];        // g = 1 - f (rounded once, here)
};

// Two-window flavour of the same (modes 1 / 2): class offsets of window A (slots 0,1) and window B (slots 2,3); bit 28 of
// deltas = the whole tile fits window A for this channel (window B is not loaded).
struct __align__(16) TileEntryFastDual {
    uint32_t cls_a[4], cls_b[4];
    float frac[4], comp[4];
    uint32_t deltas;
    int32_t span;
    int32_t reserved[2];
};

// Tiling constants shared by the table builder (tables.cu) and the kernel (das_tile.cu).
constexpr int kTileCC = 8;      // channels per pipeline stage (a packed row holds two copies of the window data)
// Tile tables are stored per (tile group, stage) so that one bulk copy fetches a CTA's stage; a group is
// the `warps` direction tiles one CTA works on (one per compute warp):
// entry(tile t, channel slot s) = tiles[((t / warps) * n_stage + s / kTileCC) * warps * kTileCC
//                                       + (t % warps) * kTileCC + s % kTileCC],  n_stage = ceil(usable / kTileCC).
inline size_t tile_table_entries(int n_tiles, int usable, int warps) {
    const size_t groups = (n_tiles + warps - 1) / warps, stages = (usable + kTileCC - 1) / kTileCC;
    return groups * stages * warps * kTileCC;
}

// Tuning knobs (BFLK_* environment variables), read ONCE in bflk_create -- never on a call path.  0 / -1 = not set.
struct Tuning {
    int tile_nch = 0;        // BFLK_TILE_NCH: window chunks of the two-FMA variant (>= what the grid needs)
    int tile_warps = 0;      // BFLK_TILE_WARPS: 10, 11, 12 or 16 compute warps per CTA
    int tile_stages = 0;     // BFLK_TILE_STAGES: 3 or 4 stage buffers
    int tile_pairs = 0;      // BFLK_TILE_PAIRS: block pairs per CTA
    int tile_mode = -1;      // BFLK_TILE_MODE: 0 one window per 2x2 tile, 1 / 2 one window per direction pair
    int lat_warps = 0;       // BFLK_LAT_WARPS / BFLK_LAT_SPLIT: force the CTA shape / cluster size of small calls (measurements)
    int lat_split = 0;
    int no_ksplit = 0;       // BFLK_NO_KSPLIT=1: small calls never split the channels across a thread-block cluster
    int chunk_mib = 0;       // BFLK_CHUNK_MIB: host batches are uploaded in chunks of about this size
};

// Output blocks of a frame of frame_len samples: 256 samples each, 254 apart (das_common.cuh: the samples a block owns).
__host__ __device__ inline int blocks_per_frame(int frame_len) { return frame_len <= 256 ? 1 : (frame_len - 2 + 253) / 254; }

// Block pairs one CTA of the tiled kernel works on, one after the other: BFLK_TILE_PAIRS when set (tile_pairs > 0), else
// enough to hide a CTA's ramp-up and epilogue behind short channel lists (a CTA lives ~0.6 us per channel).
inline int block_pairs_per_cta(int tile_pairs, int usable) {
    return tile_pairs > 0 ? tile_pairs : std::max(1, std::min(8, 512 / std::max(1, usable)));
}

// Shape of the packed rows the tiled kernel stages (das_tile.cu).
struct TileGeometry {
    int stage_off = 0;   // first packed sample, relative to a block's first output sample (even)
    int nch = 0;         // 16-byte chunks per lane window the kernel variant loads (5 - 10; the exact form has no 9)
    int warps = 0;       // compute warps (= direction tiles) per CTA of the launch
    int tmpl_warps = 0;  // compiled variant (register budget / launch bound) the launch runs on; >= warps
    int fast = 0;        // 1: two-FMA form (TileEntryFast / TileEntryFastDual tables)
    int mode = 0;        // 0: one window per tile; 1 / 2: one window per direction pair (rows of a column / columns of a row)
    int row_chunks = 0;  // logical chunks per packed row
    int copy_bytes = 0;  // padded bytes of one copy of a packed row
    int row_bytes = 0;   // bytes per packed row: the even-aligned copy followed by the copy shifted by one sample pair
    int stages = 0;      // stage buffers that fit shared memory (4 or 3; 0 = the variant does not fit at all)
    int pairs_per_cta = 0;  // 0 = automatic
    int ksplit = 1;      // 2 / 4: a thread-block cluster of that size splits the channels of a block pair (small calls, two-FMA form)
};

// ---- lane-broadcast kernel (das_bcast.cu) -----------------------------------------------------------------
constexpr int kBcastCC = 8;  // channels per pipeline stage
struct BcastEntry {
    int32_t joff;  // byte offset of the lane's first row element (16 * (offset - smallest offset))
    float frac;    // fractional delay
};
struct BcastGeometry {
    int first_offset = 0;  // smallest offset in the LUT (history - max_delay)
    int first_sample = 0;  // block sample of row element 0
    int row_elems = 0;     // float4 elements per packed row
    int row_bytes = 0;
};

// n elements of T in device memory (cudaMalloc) or page-locked host memory (cudaMallocHost), freed by the destructor.
// Move-only.  reserve only grows: it frees the old block before it allocates the new one, and leaves n = 0 on failure.
enum class Mem { device, pinned };
template <typename T, Mem kind>
struct Buf {
    T *p = nullptr;
    size_t n = 0;
    Buf() = default;
    Buf(Buf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    Buf &operator=(Buf &&o) noexcept { std::swap(p, o.p); std::swap(n, o.n); return *this; }
    ~Buf() { reset(); }
    cudaError_t reserve(size_t count) {
        if (count <= n) return cudaSuccess;
        reset();
        cudaError_t e = kind == Mem::device ? cudaMalloc((void **)&p, count * sizeof(T)) : cudaMallocHost((void **)&p, count * sizeof(T));
        if (e == cudaSuccess) n = count;
        else p = nullptr;
        return e;
    }
  private:
    void reset() {
        if (p) kind == Mem::device ? cudaFree(p) : cudaFreeHost(p);
        p = nullptr;
        n = 0;
    }
};
template <typename T> using DevBuf = Buf<T, Mem::device>;
template <typename T> using PinBuf = Buf<T, Mem::pinned>;

// A non-blocking stream and an event, created by the constructor of the object that owns them and destroyed with it.
// A failed creation leaves a null handle and the error in cudaGetLastError(), which the owner's creator checks.  A stream
// is synchronised before it is destroyed.  An event that was never recorded is an empty set of work: waiting for it
// returns at once.
class Stream {
  public:
    Stream() { if (cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking) != cudaSuccess) s_ = nullptr; }
    Stream(const Stream &) = delete;
    Stream &operator=(const Stream &) = delete;
    ~Stream() {
        sync();
        if (s_) cudaStreamDestroy(s_);
    }
    void sync() const { if (s_) cudaStreamSynchronize(s_); }
    operator cudaStream_t() const { return s_; }
  private:
    cudaStream_t s_ = nullptr;
};

class Event {   // move-only
  public:
    Event() : Event(cudaEventDisableTiming) {}
    explicit Event(unsigned flags) { if (cudaEventCreateWithFlags(&e_, flags) != cudaSuccess) e_ = nullptr; }
    Event(Event &&o) noexcept : e_(o.e_) { o.e_ = nullptr; }
    Event &operator=(Event &&o) noexcept { std::swap(e_, o.e_); return *this; }
    ~Event() { if (e_) cudaEventDestroy(e_); }
    operator cudaEvent_t() const { return e_; }
  private:
    cudaEvent_t e_ = nullptr;
};

// Streaming session (bflk_stream_*): the last `cap` samples of every channel on the device, in a mirrored ring (the twin of
// the reference's double-mapped Streams, src/fpga/streams.hpp:152-182).  Sample t is stored at columns t % cap and
// t % cap + cap of its channel's row of 2 * cap floats, so any window of at most cap samples is contiguous: it starts at
// column start % cap, rows 2 * cap apart.  Nothing is ever moved, and cap is a multiple of N, so frame starts keep the
// alignment of the ring.  Created by bflk_stream_open with its buffers and events; bflk_stream_close deletes it.
struct Session {
    DevBuf<float> ring;          // [C][2 * cap]
    DevBuf<float> stage;         // one push: [C][n] float or [n][C] int32 (cap * C elements)
    Event copied;                // the push's upload has read the caller's buffer
    Event written;               // the push's samples are in the ring
    int64_t cap = 0;
    int64_t tail = 0;            // samples a frame needs beyond its own N, as the ring was sized for (frame_tail_samples)
    int64_t pushed = 0;          // samples per channel since bflk_stream_open
    int64_t next_frame = 0;      // oldest frame not yet mapped, discarded or skipped
    int64_t skipped = 0;         // frames passed over: overwritten before they were mapped, or discarded
    int64_t window_frame = -1;   // the frame that is the handle's resident window (bflk_stream_window), -1: none
};

}  // namespace bflk

struct bflk_comm;   // multi.cu: NCCL communicator state of a handle that is one rank of a multi-GPU job

// Created on its device by bflk_create, with all of its streams and events; bflk_destroy deletes it on that device.
struct bflk_handle {
    bflk_config cfg{};
    bflk::Tuning tuning;
    bflk_comm *comm = nullptr;
    bflk::Stream stream;
    int sm_count = 0;
    std::string error;
    int64_t launches = 0;
    int kernel_choice = 0;  // 0 auto, 1 generic, 2 tiled
    int kernel_last = 0;    // what the last power-map call ran
    bool allow_ksplit = false;  // bflk_set_channel_split: small two-FMA calls may split the channels across a thread-block cluster

    // geometry + mask (host copies are the source of truth; device copies feed the table kernels)
    bool have_geometry = false;
    std::vector<float> xyz;      // [C][3]
    std::vector<int32_t> index;  // [usable]
    bflk::DevBuf<float> d_xyz;
    bflk::DevBuf<int32_t> d_index;

    // steering grid
    bool have_grid = false;
    int32_t rows = 0, cols = 0;  // 0 x 0 when the tables were supplied by the caller
    int32_t n_dir = 0;           // D (whole grid)
    int32_t dir_first = 0, dir_count = 0;
    int32_t max_delay = 0;       // largest integer delay in the LUT
    std::vector<double> theta, phi;
    bflk::DevBuf<int32_t> d_off;  // [D][C]
    bflk::DevBuf<float> d_frac;   // [D][C]

    // register-tiled kernel tables (built lazily for the current grid / mask / range)
    bool tiles_valid = false;
    bool tiles_usable = false;   // false: grid shape / spreads do not fit the tiled kernel
    int tiles_fast = 0;          // the tables were built for the two-FMA variant
    int tiles_want_warps = 0;    // ... and for this CTA shape (0: throughput shape; 2..15: latency shape of small calls, latency_warps())
    int32_t n_tiles = 0;
    int32_t tile_smax = 0;       // compiled window slack the tables need
    bflk::DevBuf<char> d_tiles;             // tile_table_entries(n_tiles, usable) TileEntry / TileEntryFast, layout above
    bflk::DevBuf<int32_t> d_tile_dirs;      // [n_tiles][4] local direction index (or -1)
    bflk::TileGeometry tile_geom;

    // lane-broadcast kernel tables (built lazily for the current grid / mask / range)
    bool bcast_valid = false;
    int32_t bcast_tiles = 0;
    bflk::BcastGeometry bcast_geom;
    bflk::DevBuf<bflk::BcastEntry> d_bcast_table;  // [tile][stage][kBcastCC][32]
    bflk::DevBuf<int32_t> d_bcast_dirs;            // [tile][32] local direction index or -1
    bflk::DevBuf<int32_t> d_bcast_globals;         // [tile][32] grid direction index or -1

    // optional FIR interpolation (bflk_set_fir): coefficient table on the device
    bflk::DevBuf<float> d_fir;
    int32_t fir_phases = 0, fir_taps = 0;

    // window kept on the device across calls (bflk_set_window): MISO / monopulse iterations on one frame do not re-upload it
    const float *resident_window = nullptr;   // d_resident.p, a caller-owned device pointer (bflk_set_window_dev) or a session frame
    int64_t resident_stride = 0;              // its row stride: window_len, or 2 * cap of the session's ring
    std::unique_ptr<bflk::Session> session;   // bflk_stream_open .. bflk_stream_close
    bflk::DevBuf<int32_t> d_wire;
    bflk::DevBuf<uint8_t> d_bytes;            // heat-map / resize / peak-candidate scratch
    // bflk_power_map_batch_submit / _wait: two batches in flight, each with its own device buffers
    bflk::DevBuf<float> d_async_in[2], d_async_out[2];
    bflk::Event async_done[2];
    uint64_t async_seq = 0;
    int async_pending = 0;
    // maps of the synchronous host batches (bflk_power_map_batch, bflk_power_map_batch_i32); nothing else writes them
    bflk::DevBuf<float> d_maps;
    bool last_map_on_device = false;          // d_maps holds the [count] map of the last batch, which had one frame
    bflk::DevBuf<float> d_beams;              // delayed sums of a session's maps call that returns them (bflk_session_beams)
    bflk::DevBuf<float> d_post;               // host map of bflk_heatmap / bflk_targets, channel powers of bflk_calibrate
    bflk::DevBuf<float> d_resident;
    bflk::DevBuf<float> d_miso_out;           // [flag | audio | power]: one D2H copy per call
    bflk::DevBuf<float> d_miso_partial;
    bflk::DevBuf<unsigned> d_miso_counters;
    int32_t miso_epoch = 0;
    bflk::PinBuf<float> p_stage;              // pinned staging of single-frame inputs / small outputs
    bflk::Event caller_event;                 // orders work the library puts on a caller's stream against the handle's scratch
    cudaStream_t last_stream = nullptr;       // stream of the last asynchronous call

    // scratch
    bflk::DevBuf<float> d_window;
    bflk::DevBuf<bflk::DirTrig> d_trig;
    bflk::DevBuf<int32_t> d_soff;
    bflk::DevBuf<float> d_sfrac;
    bflk::DevBuf<int32_t> d_misc;
    bflk::PinBuf<float> p_out;
    bflk::PinBuf<bflk::DirTrig> p_trig;
    bflk::PinBuf<int32_t> p_misc;
    // host-buffer batches are cut into chunks: copies on copy_stream overlap compute on stream
    bflk::Stream copy_stream;
    std::vector<bflk::Event> chunk_events;    // grows with the chunk count of a batch
    // ... and the chunks' kernels alternate between two compute lanes (lanes_fork / lanes_join), each with its own scratch
    // set: a launch on its own ends with half a CTA lifetime of idle SMs on average (the CTAs of a launch all take equally
    // long and the SMs drift apart), which the next chunk's CTAs fill when they do not have to wait for it
    bflk::Stream lane[2];
    bflk::Event lane_done[2];
    struct {
        bflk::DevBuf<char> packed;     // pair-interleaved staging rows of the current batch
        bflk::DevBuf<float> partial;   // partial sums of frames longer than one block
    } scratch[2];                      // set 1 only for lane 1 (Launch::scratch)
    // device batches in continuous operation (power_map_dev_overlapped): they alternate between the two lanes too
    bflk::Event dev_in[2];                        // "the caller's stream has reached the submit" (inputs ready)
    uint64_t dev_seq = 0;
    bool caller_event_is_overlapped = false;      // the latest caller_event covers overlapped batches only (see power_map_dev_overlapped)

    // optional kernel timing (bflk_enable_timing): event pairs recorded on the launching stream
    bool timing = false;
    struct Timed {
        bflk::Event e0{cudaEventDefault}, e1{cudaEventDefault};
        int kind = 0;   // 0: delay-and-sum kernel, 1: pack pre-pass
    };
    std::vector<Timed> timed;

    ~bflk_handle();   // waits for the handle's and its communicator's streams before anything is freed

    int fail(int code, const char *fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        error = buf;
        return code;
    }
};

#define BFLK_CUDA(h, expr)                                                                              \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return (h)->fail(BFLK_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

namespace bflk {

// ---- tables.cu --------------------------------------------------------------------------------------
// delays -> (offset, fraction) for n_dir directions given their trig; also returns the largest integer
// delay through d_maxdelay (device int, atomically maxed).  off / frac are [n_dir][C].
cudaError_t launch_steer_tables(const DirTrig *d_trig, int n_dir, const float *d_xyz, int C, float k_scale,
                                int history, int32_t *d_off, float *d_frac, int32_t *d_maxdelay, cudaStream_t st);
cudaError_t launch_offset_range(const int32_t *d_off, size_t n, int32_t *d_maxoff, int32_t *d_minoff, cudaStream_t st);
// tile tables for directions [first, first+count) of a rows x cols grid, 2x2 direction tiles.
cudaError_t launch_build_tiles(const int32_t *d_off, const float *d_frac, int C, const int32_t *d_index, int usable,
                               int rows, int cols, int first, int count, int stage_off, int copy_bytes, int warps,
                               int mode, int pair_span, int fast, void *d_tiles, int32_t *d_tile_dirs, int n_tiles,
                               int32_t *d_maxspan, cudaStream_t st);

// ---- das_generic.cu ---------------------------------------------------------------------------------
struct GenericArgs {
    const float *stream;   // [C][T]
    int64_t row_stride;    // T
    int n_frames;          // B
    int frame_len;         // N
    int frame_stride;      // samples between consecutive frames' windows (N)
    const int32_t *off;    // [n_dir][C] (already offset to the first direction)
    const float *frac;
    int C;
    const int32_t *index;  // [usable]
    int usable;
    int n_dir;
    float *power;          // [B][n_dir] or nullptr
    float *audio;          // [B][n_dir][N] or nullptr
    float norm;            // power divisor: N*count (MIMO) or N (beam)
    const float *fir = nullptr;   // [fir_phases][fir_taps] coefficients: FIR interpolation instead of the 2-tap triple
    int fir_phases = 0, fir_taps = 0;
};
cudaError_t launch_das_generic(const GenericArgs &a, cudaStream_t st);

// ---- das_miso.cu ------------------------------------------------------------------------------------
constexpr int kMisoInline = 128;   // targets whose DirTrig travel in the kernel's parameter space (no H2D copy)
struct MisoArgs {
    const float *window;     // [C][row_stride]; frame b starts at window + b * frame_stride
    int64_t row_stride;
    int n_frames, frame_len, frame_stride;
    const DirTrig *trig;     // [n_targets] on the device (used when n_inline == 0)
    const float *xyz;        // [C][3]
    int C;
    const int32_t *index;    // [usable]
    int usable;
    float k_scale;           // float(sample_rate / propagation_speed)
    int history;
    int n_targets;
    float *audio;            // [B][T][N] or nullptr
    float *power;            // [B][T] or nullptr
    float *partial;          // [B][T][slices] scratch of the power reduction (power != nullptr)
    unsigned *counters;      // [B][T] zero-initialised, self-resetting arrival counters (power != nullptr)
    float norm;              // N (Particle::beam)
    int32_t *error_flag;     // set to `epoch` when a delay exceeds the history
    int32_t epoch;
    int32_t *off_out;        // optional [T][C] tables as built (nullptr: not stored)
    float *frac_out;
    int n_inline;            // n_targets when the directions are in trig_inline, else 0
    DirTrig trig_inline[kMisoInline];
};
cudaError_t launch_das_miso(const MisoArgs &a, cudaStream_t st);
int das_miso_slices(int frame_len);

// ---- staged kernels (das_tile.cu, das_bcast.cu): a pack pre-pass, the delay-and-sum kernel, finalize_kernel ------------
// The frames of a call and where their maps go, as both staged kernels take them.
struct FrameArgs {
    const float *stream = nullptr;   // [C][row_stride] channel-major rows; frame b starts at column b * frame_stride
    int64_t row_stride = 0;
    int64_t row_len = 0;             // valid samples per row from `stream` (chunked host batches pass row_len < row_stride)
    int n_frames = 0, frame_len = 0, frame_stride = 0;
    int usable = 0;
    int n_dir = 0;                   // directions in this handle's range (power row length)
    const int32_t *index = nullptr;  // [usable] channel mask (pack gathers rows in this order)
    void *packed = nullptr;          // packed_bytes() of scratch
    float *power = nullptr;          // [B][n_dir]
    float *partial = nullptr;        // [B * blocks_per_frame][n_dir] when frame_len > 256
    float *beams = nullptr;          // [B][n_dir][frame_len] delayed sums the power squares (8-byte aligned), or nullptr
    float norm = 0.f;
};
// bytes of the packed rows of a call: one row of row_bytes per (block pair, usable channel)
inline size_t packed_bytes(const FrameArgs &f, int row_bytes) {
    const int n_items = f.n_frames * blocks_per_frame(f.frame_len);
    return (size_t)((n_items + 1) / 2) * f.usable * row_bytes;
}
// frames longer than one block: power = the partial sums of each frame's blocks, added in block order, / norm (one launch)
cudaError_t launch_finalize(const FrameArgs &f, cudaStream_t st);
// hook(kind, begin): called right before (begin = true) and after each pack (kind 1) / main (kind 0) launch
typedef void (*TileLaunchHook)(void *ctx, int kind, bool begin, cudaStream_t st);

// ---- das_tile.cu ------------------------------------------------------------------------------------
struct TileArgs {
    FrameArgs f;
    const int32_t *wire = nullptr;   // when set: sample-major wire frames [row_len][wire_cols] instead of f.stream (pack_wire_kernel)
    int wire_cols = 0;
    const void *tiles = nullptr;     // tile_table_entries() entries (TileEntry, or TileEntryFast when geom.fast), grouped per (tile group, stage)
    const int32_t *tile_dirs = nullptr;   // [n_tiles][4]
    int n_tiles = 0;
    TileGeometry geom;
};
cudaError_t launch_das_tile(const TileArgs &a, int sm_count, cudaStream_t st, int *launches, TileLaunchHook hook = nullptr,
                            void *hook_ctx = nullptr);
int das_tile_max_span();
TileGeometry das_tile_geometry(int history, int max_delay, int max_span, int n_tiles = 0, int mode = 0, int fast = 0,
                               const Tuning *tuning = nullptr, int want_warps = 0);
// shared memory the variant needs with `stages` stage buffers
size_t das_tile_smem_bytes(const TileGeometry &g, int stages);
// can this geometry split the channels of a block pair across a cluster of `split` CTAs (compiled for some variants only)?
bool das_tile_ksplit_ok(const TileGeometry &g, int split);
size_t das_tile_entry_bytes(const TileGeometry &g);

// ---- das_bcast.cu -----------------------------------------------------------------------------------
struct BcastArgs {
    FrameArgs f;
    const BcastEntry *table = nullptr;
    const int32_t *tile_dirs = nullptr;   // [n_tiles][32] local direction index or -1
    int n_tiles = 0;
    BcastGeometry geom;
};
BcastGeometry das_bcast_geometry(int history, int max_delay);
bool das_bcast_fits(const BcastGeometry &g);
size_t das_bcast_table_entries(int n_tiles, int usable);
cudaError_t launch_bcast_table(const int32_t *d_off, const float *d_frac, int C, const int32_t *d_index, int usable,
                               const int32_t *d_tile_globals, int n_tiles, const BcastGeometry &g, BcastEntry *d_table,
                               cudaStream_t st);
cudaError_t launch_das_bcast(const BcastArgs &a, cudaStream_t st, int *launches, TileLaunchHook hook = nullptr,
                             void *hook_ctx = nullptr);

// ---- post.cu ----------------------------------------------------------------------------------------
cudaError_t launch_heatmap(const float *d_power, int n, uint8_t *d_heat, int32_t *d_argmax, float *d_max, cudaStream_t st);
cudaError_t launch_channel_power(const float *d_signals, int n_ch, int W, float *d_power, cudaStream_t st);
cudaError_t launch_ingest(const int32_t *d_frames, int64_t n, int n_sensors, float *d_exposure, cudaStream_t st);
// samples t0 .. t0 + n of every channel into a Session's ring: d_block [C][n] float, or d_wire [n][C] int32 when it is set
cudaError_t launch_history_push(const float *d_block, const int32_t *d_wire, int n, int C, int64_t t0, int cap, float *d_ring,
                                cudaStream_t st);
cudaError_t launch_ffma2_peak(float *d_out, int n_blocks, int iters, cudaStream_t st);
cudaError_t launch_resize_u8(const uint8_t *d_src, int ih, int iw, uint8_t *d_dst, int oh, int ow, const int32_t *d_tab, cudaStream_t st);
cudaError_t launch_map_targets(const float *d_power, int rows, int cols, int max_targets, float min_rel, uint8_t *d_cand,
                               int32_t *d_index, float *d_pw, float *d_prob, int32_t *d_n, cudaStream_t st);

// ---- bflk_api.cu internals used by multi.cu ---------------------------------------------------------------
// How power_map_dev runs.  A plain call orders itself against the handle's earlier calls through caller_event; a pipelined
// one runs on a lane between lanes_fork and lanes_join, which order the streams for it.
struct Launch {
    cudaStream_t st = nullptr;       // nullptr: the handle's stream
    int scratch = 0;                 // which of the handle's two scratch sets
    bool pipelined = false;          // on a lane: no caller_event wait or record; throughput CTA shape (tables built by lanes_fork)
    const int32_t *wire = nullptr;   // wire-format input [n_samples][C] instead of stream_dev
};
// stream_dev: first sample of frame 0; rows are row_stride floats apart and hold n_samples valid samples.  beams_dev: also
// the delayed sums the maps square, [n_frames][count][frame_len] (8-byte aligned), or nullptr
int power_map_dev(bflk_handle *h, const float *stream_dev, int64_t row_stride, int64_t n_samples, int32_t n_frames,
                  float *power_dev, const Launch &launch, float *beams_dev = nullptr);
// Continuous operation: the same as power_map_dev, but enqueued on one of the handle's two lanes (alternating, each with its
// own scratch) after `caller` has reached this point; *used = the stream the kernels are on.  Consecutive calls overlap: the
// pack pre-pass of batch i + 1 runs under the kernel of batch i and its CTAs fill the SMs the last CTAs of batch i leave
// idle.  caller_event afterwards covers everything enqueued so far.  Falls back to power_map_dev on `caller` (*used = caller)
// when the register-tiled kernels do not serve the grid.
int power_map_dev_overlapped(bflk_handle *h, const float *stream_dev, int64_t row_stride, int64_t n_samples, int32_t n_frames,
                             float *power_dev, cudaStream_t caller, cudaStream_t *used);
// Stream ordering of the handle's scratch and tables.  note_use records caller_event on st (the only place it is recorded):
// a later call on another stream waits for it.  overlapped: it covers overlapped device batches only.
int note_use(bflk_handle *h, cudaStream_t st, bool overlapped);
// lanes_fork: the two lanes wait for caller_event and for `after` (if given), once the tile tables are built; lanes_join:
// the handle's stream waits for them and caller_event is recorded there.  only = 0 / 1: just that lane (one overlapped
// device batch), which skips caller_event when it covers overlapped batches only (the lane's own are in its stream order).
int lanes_fork(bflk_handle *h, cudaEvent_t after, int only = -1);
int lanes_join(bflk_handle *h, int only = -1);
// -1 when the register-tiled kernels cannot serve a call (FIR, or kernel 1 / 3), else the `fast` flag for ensure_tiles
int tiled_form(const bflk_handle *h);
int ensure_tiles(bflk_handle *h, int fast, int want_warps = 0);
// CTA shape of a tiled call over n_tiles direction tiles and n_frames frames: warps = 0 (throughput shape) or 2..16
void latency_shape(long long n_tiles, int n_frames, int frame_len, int usable, int pairs_per_cta, int sms, bool may_split,
                   int *warps, int *split);
int64_t min_stream_samples(const bflk_handle *h, int n_frames);
// frames per chunk of a host batch of n_frames (whole CTA waves of the tiled kernel where it applies) and the samples a
// frame needs beyond its own N
int host_chunk_frames(bflk_handle *h, int n_frames, int *chunk_frames);
int64_t frame_tail_samples(const bflk_handle *h);
void comm_release(bflk_handle *h);   // multi.cu: deletes h->comm (bflk_comm is a complete type only there)

}  // namespace bflk
