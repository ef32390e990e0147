// tables.cu -- steering-delay tables on the device.
//
// Replaces steering_vector_spherical + the offset/fraction split of the reference
// (src/geometry/antenna.cpp:89-107,126-134; src/dsp/mimo.cpp:46-54; src/dsp/particle.cpp:37-49).
// Trigonometry is evaluated on the host in double exactly like rotateZ/rotateY
// (src/geometry/geometry.cpp:219-233) and arrives here as four floats per direction; the device does
// only correctly-rounded float mul / fma / sub with every rounding pinned (__f*_rn), so the tables are
// bit-identical to the host restatement in oracle/oracle.c.
#include "bflk_internal.h"
#include "steer.cuh"

namespace bflk {

// FOCUS: the delays of a point source at distance `focus` (focus_z) instead of a plane wave (steer_z)
template <bool FOCUS>
__global__ void __launch_bounds__(128) steer_tables_kernel(const DirTrig *__restrict__ trig, const float *__restrict__ xyz,
                                                           int C, float k_scale, int history, int32_t *__restrict__ off,
                                                           float *__restrict__ frac, int32_t *__restrict__ maxdelay,
                                                           double focus) {
    extern __shared__ float s_del[];
    __shared__ float s_red[4];
    const int d = blockIdx.x;
    const DirTrig t = trig[d];
    float mn = INFINITY;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float del = steer_delay<FOCUS>(t, xyz, c, k_scale, focus);  // compute_delays: row(Z) * float(SAMPLE_RATE / PROPAGATION_SPEED)
        s_del[c] = del;
        mn = fminf(mn, del);
    }
    for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = mn;
    __syncthreads();
    mn = fminf(fminf(s_red[0], s_red[1]), fminf(s_red[2], s_red[3]));
    int local_max = 0;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float del = __fsub_rn(s_del[c], mn);  // delays -= minCoeff
        float ip = truncf(del);               // modf((double)del, &ip): exact for a float argument
        float fr = __fsub_rn(del, ip);
        int di = (int)ip;
        off[(size_t)d * C + c] = history - di;
        frac[(size_t)d * C + c] = fr;
        local_max = max(local_max, di);
    }
    for (int o = 16; o > 0; o >>= 1) local_max = max(local_max, __shfl_xor_sync(0xffffffffu, local_max, o));
    if ((threadIdx.x & 31) == 0 && maxdelay) atomicMax(maxdelay, local_max);
}

cudaError_t launch_steer_tables(const DirTrig *d_trig, int n_dir, const float *d_xyz, int C, float k_scale, int history,
                                int32_t *d_off, float *d_frac, int32_t *d_maxdelay, double focus, cudaStream_t st) {
    if (n_dir <= 0) return cudaSuccess;
    auto kernel = focus > 0.0 ? steer_tables_kernel<true> : steer_tables_kernel<false>;
    kernel<<<n_dir, 128, C * sizeof(float), st>>>(d_trig, d_xyz, C, k_scale, history, d_off, d_frac, d_maxdelay, focus);
    return cudaGetLastError();
}

// maxoff / minoff: largest and smallest offset of a caller-supplied LUT (range validation).
__global__ void max_delay_kernel(const int32_t *__restrict__ off, size_t n, int32_t *maxoff, int32_t *minoff) {
    int mx = INT_MIN, mo = INT_MAX;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        int o = off[i];
        mx = max(mx, o);
        mo = min(mo, o);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        mo = min(mo, __shfl_xor_sync(0xffffffffu, mo, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(maxoff, mx);
        atomicMin(minoff, mo);
    }
}

cudaError_t launch_offset_range(const int32_t *d_off, size_t n, int32_t *d_maxoff, int32_t *d_minoff, cudaStream_t st) {
    int blocks = (int)((n + 255) / 256);
    if (blocks > 1184) blocks = 1184;
    if (blocks < 1) blocks = 1;
    max_delay_kernel<<<blocks, 256, 0, st>>>(d_off, n, d_maxoff, d_minoff);
    return cudaGetLastError();
}

// ---- tile tables ------------------------------------------------------------------------------------
// Tiles are 2x2 blocks of grid directions (r0..r0+1, c0..c0+1).  A handle's direction range
// [first, first+count) is a run of the row-major grid; tiles are enumerated over the rows the range
// touches and directions outside the range get tile_dirs = -1 (computed but not stored).
// mode 0: one window shared by the four directions of the tile.
// mode 1 / 2: two windows, each shared by a PAIR of directions (1: the two rows of a grid column, 2: the two columns
// of a grid row); directions are stored in "slot" order -- slots 0,1 use window A, slots 2,3 window B -- and
// tile_dirs follows the same order.  maxspan[mode] receives the largest delta of that mode.
__global__ void build_tiles_kernel(const int32_t *__restrict__ off, const float *__restrict__ frac, int C,
                                   const int32_t *__restrict__ index, int usable, int rows, int cols, int first,
                                   int count, int stage_off, int copy_bytes, int warps, int mode, int pair_span,
                                   int fast, void *__restrict__ tiles_raw,
                                   int32_t *__restrict__ tile_dirs, int n_tiles, int tile_cols, int row0,
                                   int32_t *__restrict__ maxspan) {
    const int t = blockIdx.x;
    if (t >= n_tiles) return;
    TileEntry *tiles = fast ? nullptr : static_cast<TileEntry *>(tiles_raw);
    TileEntryFast *tiles_fast = fast && mode == 0 ? static_cast<TileEntryFast *>(tiles_raw) : nullptr;
    TileEntryFastDual *tiles_fast2 = fast && mode != 0 ? static_cast<TileEntryFastDual *>(tiles_raw) : nullptr;
    const int tr = t / tile_cols, tc = t % tile_cols;
    int dirs[4];
#pragma unroll
    for (int slot = 0; slot < 4; slot++) {
        // grid position q = 2 * row + col of the direction in this slot
        const int q = mode == 1 ? ((slot & 1) << 1 | (slot >> 1)) : slot;
        int r = row0 + 2 * tr + (q >> 1), c = 2 * tc + (q & 1);
        dirs[slot] = (r < rows && c < cols) ? r * cols + c : -1;
    }
    // a direction that does not exist (odd grid edge) aliases the first existing direction of the tile
    int ref = dirs[0];
#pragma unroll
    for (int slot = 1; slot < 4; slot++)
        if (ref < 0) ref = dirs[slot];
    if (threadIdx.x < 4 && tile_dirs) {
        int g = dirs[threadIdx.x];
        tile_dirs[4 * t + threadIdx.x] = (g >= first && g < first + count) ? g - first : -1;
    }
    int span_max = 0;
    for (int s = threadIdx.x; s < usable; s += blockDim.x) {
        const int c = index[s];
        int o[4];
        TileEntry e;
#pragma unroll
        for (int slot = 0; slot < 4; slot++) {
            int g = dirs[slot] >= 0 ? dirs[slot] : ref;
            o[slot] = off[(size_t)g * C + c];
            e.frac[slot] = frac[(size_t)g * C + c];
        }
        unsigned packed = 0, need_last = 0;   // need_last: bit 29 / 30 = window A / B has a delta that reaches the last chunk
        int span = 0;
        if (mode == 0) {
            // window = smallest offset of the tile, exactly: an odd start reads the copy shifted by one sample pair
            const int base = min(min(o[0], o[1]), min(o[2], o[3]));
            const int odd = (base - stage_off) & 1;
            const int cb = (base - stage_off - odd) >> 1;                // first 16-byte chunk of lane 0's window
            e.win_off = (unsigned)(odd * copy_bytes) + 16u * (unsigned)(cb + (cb >> 2));  // one pad chunk after every four
            packed = (unsigned)(cb & 3) << 24;
#pragma unroll
            for (int slot = 0; slot < 4; slot++) {
                const int dlt = o[slot] - base;
                span = max(span, dlt);
                packed |= (unsigned)(dlt & 63) << (6 * slot);
            }
            if (span >= pair_span - 1) need_last = 1u << 29;
        } else {
            // one window per direction pair -- unless the whole tile fits a pair window for this channel: then slots 2,3
            // reuse window A (bit 28; the kernel skips the second load + differences)
            const int lo4 = min(min(o[0], o[1]), min(o[2], o[3])), hi4 = max(max(o[0], o[1]), max(o[2], o[3]));
            const bool same = hi4 - lo4 <= pair_span;
            e.win_off = 0;
#pragma unroll
            for (int w = 0; w < 2; w++) {
                const int base = same ? lo4 : min(o[2 * w], o[2 * w + 1]);
                const int odd = (base - stage_off) & 1;
                const int cb = (base - stage_off - odd) >> 1;
                e.win_off |= ((unsigned)(odd * copy_bytes) + 16u * (unsigned)(cb + (cb >> 2))) << (16 * w);
                packed |= (unsigned)(cb & 3) << (24 + 2 * w);
#pragma unroll
                for (int k = 0; k < 2; k++) {
                    const int dlt = o[2 * w + k] - base;
                    span = max(span, dlt);
                    packed |= (unsigned)(dlt & 63) << (6 * (2 * w + k));
                    // (a tile that fits window A: all four deltas are relative to it)
                    if (dlt >= pair_span - 1) need_last |= 1u << (same ? 29 : 29 + w);
                }
            }
            if (same) packed |= 1u << 28;
        }
        e.deltas = packed;
        e.span = span;
        e.reserved = 0;
        const int n_stage = (usable + kTileCC - 1) / kTileCC;
        const size_t slot = ((size_t)(t / warps) * n_stage + s / kTileCC) * (warps * kTileCC) + (t % warps) * kTileCC + s % kTileCC;
        if (tiles) tiles[slot] = e;
        if (tiles_fast) {  // mode 0 only
            TileEntryFast q;
            const unsigned r = (packed >> 24) & 3;
#pragma unroll
            for (int k = 0; k < 4; k++)
                q.cls_off[k] = (unsigned)(s % kTileCC) * 2u * (unsigned)copy_bytes + e.win_off + ((k > 0 && r >= (unsigned)(4 - k)) ? 16u : 0u);
            q.deltas = (packed & 0xffffffu) | need_last;
            q.span = span;
            q.reserved[0] = q.reserved[1] = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                q.frac[k] = e.frac[k];
                q.comp[k] = __fsub_rn(1.0f, e.frac[k]);
            }
            tiles_fast[slot] = q;
        }
        if (tiles_fast2) {  // modes 1 / 2
            TileEntryFastDual q;
#pragma unroll
            for (int w = 0; w < 2; w++) {
                const unsigned wo = (e.win_off >> (16 * w)) & 0xffffu, r = (packed >> (24 + 2 * w)) & 3;
#pragma unroll
                for (int k = 0; k < 4; k++)
                    (w ? q.cls_b : q.cls_a)[k] = (unsigned)(s % kTileCC) * 2u * (unsigned)copy_bytes + wo + ((k > 0 && r >= (unsigned)(4 - k)) ? 16u : 0u);
            }
            q.deltas = (packed & 0x10ffffffu) | need_last;
            q.span = span;
            q.reserved[0] = q.reserved[1] = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                q.frac[k] = e.frac[k];
                q.comp[k] = __fsub_rn(1.0f, e.frac[k]);
            }
            tiles_fast2[slot] = q;
        }
        span_max = max(span_max, span);
    }
    for (int o = 16; o > 0; o >>= 1) span_max = max(span_max, __shfl_xor_sync(0xffffffffu, span_max, o));
    if ((threadIdx.x & 31) == 0) atomicMax(maxspan + mode, span_max);
}

cudaError_t launch_build_tiles(const int32_t *d_off, const float *d_frac, int C, const int32_t *d_index, int usable,
                               int rows, int cols, int first, int count, int stage_off, int copy_bytes, int warps,
                               int mode, int pair_span, int fast, void *d_tiles, int32_t *d_tile_dirs, int n_tiles,
                               int32_t *d_maxspan, cudaStream_t st) {
    const int row0 = (first / cols) & ~1;
    const int tile_cols = (cols + 1) / 2;
    build_tiles_kernel<<<n_tiles, 128, 0, st>>>(d_off, d_frac, C, d_index, usable, rows, cols, first, count, stage_off,
                                                copy_bytes, warps, mode, pair_span, fast, d_tiles, d_tile_dirs, n_tiles, tile_cols, row0, d_maxspan);
    return cudaGetLastError();
}

}  // namespace bflk
