// das_tile.cu -- register-tiled delay-and-sum power map for sm_100a (the hot kernel).
//
// Replaces the loop nest of MIMOWorker::update (src/dsp/mimo.cpp:121-150) around delay()
// (src/dsp/delay.cpp:16-26).  Design (DESIGN.md "das_tile"):
//
//  * pack_kernel rewrites the channel-major stream once per batch into "pair-interleaved" rows:
//    element g of a row is float2{ blockA[g], blockB[g] } for two 256-sample output blocks A and B,
//    gathered in channel-mask order and laid out with one 16-byte pad every four 16-byte chunks.
//    With that layout (a) one FFMA2/FADD2 (fma.rn.f32x2 / add.rn.f32x2) advances the same output
//    sample of two blocks, for any delay parity, (b) a row is a contiguous byte range the main kernel
//    stages with cp.async.bulk (TMA bulk copy) + mbarrier, and (c) the 64-byte lane stride of the
//    per-thread windows becomes 80 bytes, which is bank-conflict-free for LDS.128.
//  * das_tile_kernel: one warp = one 2x2 tile of steering directions x two 256-sample blocks; lane l
//    owns output samples 8l..8l+7 of both blocks.  Per channel the warp loads ONE shared window of
//    sample pairs into registers (or one per direction pair on coarse grids) and serves the four
//    directions from registers through a warp-uniform dispatch on each direction's offset inside the
//    window.  Two accumulate forms (DESIGN.md 2, 4.1):
//      - exact triple (kernel 2): differences s[i]-s[i+1] formed once per window, then
//        acc = acc + fma(f, d, s[i+1]) per direction in mask order -- delayed sums bit-identical to
//        delay(); 2 + 1/4 FP32 lane-operations per (direction, channel, sample);
//      - two-FMA form (kernel 4, automatic; template parameter FAST): acc = fma(f, s[i], fma(g, s[i+1], acc)),
//        g = 1 - f from the table -- 16 FFMA2 per (direction, channel) and nothing else on the FP pipe,
//        the whole pipeline stage in one generated PTX block (das_tile_fast_asm.inc).
//  * epilogue: 3-tap high-pass + squares (mimo.cpp:131-135) with neighbour samples from lane +-1,
//    warp-shuffle reduction, one store per (block, direction); beams calls also store the delayed sums.
#include <algorithm>
#include <array>
#include <cstdlib>
#include <utility>

#include "bflk_internal.h"
#include "das_common.cuh"

namespace bflk {

namespace {

constexpr int kCC = kTileCC;         // channels per pipeline stage
constexpr int kMaxStages = 4;        // stage buffers (KernelArgs::stages: 4 when shared memory allows, else 3)
constexpr int kBlock = 256;          // output samples per block
constexpr int kK = 8;                // sample pairs per lane

// chunk (16 B = 2 sample pairs) c of a row lives at padded chunk c + (c >> 2)
__host__ __device__ __forceinline__ int padded_chunk(int c) { return c + (c >> 2); }

}  // namespace

// ---- packed tile entry as the kernel reads it -----------------------------------------------------------
// word0: byte offset of the warp's window inside a packed row (lane 0), word1: 4 x 6-bit deltas | r << 24,
// word2: span, word3: unused; then the four fractions.
static_assert(sizeof(TileEntry) == 32, "TileEntry is two 16-byte loads");

// ---- pack: stream[C][T] -> packed[pair][usable][row] of float2{A, B} -------------------------------------
struct PackArgs {
    const int32_t *wire;  // sample-major wire frames [row_len][wire_cols] (src/fpga/receiver.h:24-30) instead of `stream`
    int wire_cols;
    const float *stream;
    int64_t row_stride;   // T
    int64_t row_len;      // valid samples per row from the stream pointer (<= row_stride)
    int n_frames, frame_len, frame_stride;
    int blocks_per_frame;
    int n_items;          // n_frames * blocks_per_frame
    int pair0;            // first pair of this launch (grid.z is limited to 65535)
    const int32_t *index;
    int usable;
    int stage_off;        // first staged sample relative to a block start (even)
    int row_chunks;       // logical chunks per row
    int row_bytes;        // bytes per packed row = two padded copies (multiple of 16)
    int copy_bytes;       // bytes of one copy
    float4 *packed;
};

__global__ void __launch_bounds__(256) pack_kernel(PackArgs a) {
    const int pair = a.pair0 + blockIdx.z, s = blockIdx.y;
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= a.row_chunks) return;
    const int itemA = 2 * pair, itemB = min(2 * pair + 1, a.n_items - 1);
    const int64_t tA = item_first_sample(itemA, a.blocks_per_frame, a.frame_len, a.frame_stride) + a.stage_off + 2 * ch;
    const int64_t tB = item_first_sample(itemB, a.blocks_per_frame, a.frame_len, a.frame_stride) + a.stage_off + 2 * ch;
    const float *row = a.stream + (size_t)a.index[s] * a.row_stride;
    // samples 2ch, 2ch+1, 2ch+2 of both blocks (8-byte loads, zero beyond the end of the stream)
    auto load2 = [&](int64_t t) {
        float2 v = make_float2(0.f, 0.f);
        if (t + 1 < a.row_len) v = *reinterpret_cast<const float2 *>(row + t);
        else if (t < a.row_len) v.x = row[t];
        return v;
    };
    const float2 A = load2(tA), A2 = load2(tA + 2), B = load2(tB), B2 = load2(tB + 2);
    // copy 0 holds the pairs at even positions first (chunk ch = pairs 2ch, 2ch+1); copy 1 is shifted by one pair
    // (chunk ch = pairs 2ch+1, 2ch+2) so that a window starting at an odd pair is still a 16-byte aligned LDS.128
    char *dst = reinterpret_cast<char *>(a.packed) + ((size_t)pair * a.usable + s) * a.row_bytes + 16 * padded_chunk(ch);
    *reinterpret_cast<float4 *>(dst) = make_float4(A.x, B.x, A.y, B.y);
    *reinterpret_cast<float4 *>(dst + a.copy_bytes) = make_float4(A.y, B.y, A2.x, B2.x);
    // also fill the pad chunk that follows every fourth chunk: whole 32-byte sectors reach DRAM, no partial writes
    if ((ch & 3) == 3 && 16 * (padded_chunk(ch) + 2) <= a.copy_bytes) {
        *reinterpret_cast<float4 *>(dst + 16) = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4 *>(dst + a.copy_bytes + 16) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// ---- pack straight from the wire format (SURVEY 8f, f1) ---------------------------------------------------------
// The FPGA sends one message per time sample: int32 stream[n_sensors], daisy-chained arrays mirrored (receiver.h:24-30).
// Pipeline::receive_exposure turns that into per-channel float rows on the host (serpentine un-flip, / 2^23,
// src/fpga/pipeline.cpp:260-297) and MIMOWorker::update copies them again (mimo.cpp:100-103).  Here the conversion,
// the un-flip (folded into the column index), the transpose and the pair-interleave of pack_kernel are ONE pass: a CTA
// loads a [130 samples][32 channels] tile of both blocks of a pair with coalesced 128-byte rows, keeps it transposed in
// shared memory, and writes the same packed rows pack_kernel writes -- so the delay-and-sum kernel is unchanged and its
// result is bit-identical to the float path (int32 -> float and the power-of-two scale are exact for 24-bit samples).
constexpr int kWireCh = 32, kWireChunks = 64, kWireT = 2 * kWireChunks + 2, kWirePitch = kWireT + 1;

__global__ void __launch_bounds__(256) pack_wire_kernel(PackArgs a) {
    __shared__ float sm[2][kWireCh][kWirePitch];
    const int pair = a.pair0 + blockIdx.z, s0 = blockIdx.y * kWireCh, ch0 = blockIdx.x * kWireChunks;
    const int itemA = 2 * pair, itemB = min(2 * pair + 1, a.n_items - 1);
    const int64_t t0[2] = {item_first_sample(itemA, a.blocks_per_frame, a.frame_len, a.frame_stride) + a.stage_off + 2 * ch0,
                           item_first_sample(itemB, a.blocks_per_frame, a.frame_len, a.frame_stride) + a.stage_off + 2 * ch0};
    const int cl = threadIdx.x & 31, r = threadIdx.x >> 5;
    const int s = s0 + cl;
    int col = -1;
    if (s < a.usable) col = wire_column(a.index[s]);
#pragma unroll
    for (int h = 0; h < 2; h++)
        for (int t = r; t < kWireT; t += 8) {
            const int64_t ts = t0[h] + t;
            float v = 0.f;
            if (col >= 0 && ts < a.row_len) v = wire_to_float(a.wire[(size_t)ts * a.wire_cols + col]);
            sm[h][cl][t] = v;
        }
    __syncthreads();
    for (int o = threadIdx.x; o < kWireCh * kWireChunks; o += 256) {
        const int chl = o % kWireChunks, c2 = o / kWireChunks, ch = ch0 + chl;
        if (ch >= a.row_chunks || s0 + c2 >= a.usable) continue;
        const float *A = &sm[0][c2][2 * chl], *B = &sm[1][c2][2 * chl];
        char *dst = reinterpret_cast<char *>(a.packed) + ((size_t)pair * a.usable + s0 + c2) * a.row_bytes + 16 * padded_chunk(ch);
        *reinterpret_cast<float4 *>(dst) = make_float4(A[0], B[0], A[1], B[1]);
        *reinterpret_cast<float4 *>(dst + a.copy_bytes) = make_float4(A[1], B[1], A[2], B[2]);
        if ((ch & 3) == 3 && 16 * (padded_chunk(ch) + 2) <= a.copy_bytes) {
            *reinterpret_cast<float4 *>(dst + 16) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4 *>(dst + a.copy_bytes + 16) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

// ---- main kernel ---------------------------------------------------------------------------------------------
struct KernelArgs {
    const char *packed;          // [pair][usable][row_bytes]
    const char *tiles;           // TileEntry / TileEntryFast, grouped per (tile group, stage), see tile_table_entries()
    const int32_t *tile_dirs;    // [n_tiles][4]
    int n_tiles, usable, n_dir;
    int row_bytes;
    int n_items, blocks_per_frame, frame_len;
    int pair0, n_pairs;          // block pairs [pair0, pair0 + n_pairs) of this launch ...
    int pairs_per_cta;           // ... consecutive ones handled by one CTA (short channel lists: amortises the ramp-up)
    int stages;                  // stage buffers in shared memory (3 or 4)
    int launch_warps;            // warps per CTA of this launch (host side: <= the compiled variant's)
    float *out;                  // power [frames][n_dir] (blocks_per_frame == 1) or partial [items][n_dir]
    float norm;
    float *beams;                // delayed sums [frames][n_dir][frame_len] (BEAMS instantiations only; FrameArgs::beams)
};

#include "das_tile_asm.inc"
#include "das_tile_fast_asm.inc"

// DUAL: two NCH-chunk windows per channel, one per direction pair (tile tables built with mode 1 / 2), NCH 6 or 7
// FAST: two-FMA form acc += g s[i+1]; acc += f s[i] (TileEntryFast tables; power within 1e-4 of the reference instead of
//       bit-identical delayed sums) -- 16 FFMA2 per (direction, channel) and no other FP instruction.
// KSPLIT: the CTAs of a thread-block cluster (grid.z = cluster size 2 or 4) split the CHANNELS of a block pair between
//       them and add their partial delayed sums through distributed shared memory, in rank order, before the epilogue.
//       For calls too small to fill the SMs (a live worker's single frame: cfg3 is 16 CTAs): the serial channel loop gets
//       shorter by the cluster size.  The channel sum is re-associated (rank sums added at the end), so FAST only.
// BEAMS: the epilogue also stores the delayed sums (beams calls).  A template flag, not a run-time test: even a branch the
//       power-only calls never take changes how ptxas allocates registers around the channel loop (more moves inside it).
template <int NCH, int kWarps, bool DUAL = false, bool FAST = false, bool KSPLIT = false, bool BEAMS = false>
__global__ void __launch_bounds__(kWarps * 32, 1) das_tile_kernel(KernelArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int kEnt = FAST ? (DUAL ? (int)sizeof(TileEntryFastDual) : (int)sizeof(TileEntryFast)) : (int)sizeof(TileEntry);
    // layout: [stages] x { rows: kCC * row_bytes | tiles: kWarps * kCC * kEnt } then barriers
    const int stage_rows = kCC * a.row_bytes;
    const int stage_bytes = stage_rows + (int)(blockDim.x >> 5) * kCC * kEnt;
    const uint32_t smem = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const int kStages = a.stages;
    const uint32_t bars = smem + kStages * stage_bytes;  // full[kStages] mbarriers, then done[kStages] arrival counters
    unsigned *done_cnt = reinterpret_cast<unsigned *>(smem_raw + kStages * stage_bytes + 8 * kStages);

    // kWarps is the compiled register budget (launch bound); a launch may use fewer warps per CTA (single-frame calls:
    // more, smaller CTAs -- one warp per scheduler instead of four -- cut the latency of the serial channel loop)
    const int nwarps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_stage = (a.usable + kCC - 1) / kCC;
    // pipeline stages st_first, st_first + st_step, ... of every block pair are this CTA's: all of them, unless a cluster splits
    // the channels -- then round robin, so every rank sees the same mix of near and far microphones (the share of second
    // windows, i.e. the cost of a stage, depends on where on the array its channels sit)
    int st_first = 0, st_step = 1;
    unsigned crank = 0, csize = 1;
    if constexpr (KSPLIT) {
        asm("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
        asm("mov.u32 %0, %%cluster_nctarank;" : "=r"(csize));
        st_first = (int)crank;
        st_step = (int)csize;
    }
    const int tile0 = blockIdx.x * nwarps;
    const int my_tile = min(tile0 + warp, a.n_tiles - 1);
    const bool active = tile0 + warp < a.n_tiles;  // idle warps of the last tile group only keep the pipeline moving
    // this CTA works on block pairs [pair_lo, pair_hi) one after the other; the staging pipeline runs straight through
    // the pair boundaries, so the next pair's first stages load while this pair's epilogue runs
    const int pair_lo = a.pair0 + blockIdx.y * a.pairs_per_cta;
    const int pair_hi = min(pair_lo + a.pairs_per_cta, a.pair0 + a.n_pairs);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; s++) {
            mbar_init(bars + 8 * s, 1);
            done_cnt[s] = 0;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // producer: fills buffer buf with (block pair `pair`, channel chunk `st`).  There is no producer warp and no "empty"
    // barrier anybody waits on: the LAST warp to finish a stage (arrival counter in shared memory) refills the buffer it
    // just freed with the stage kStages ahead, so no warp ever waits for a slower one and the prefetch distance is the
    // whole ring.
    auto issue = [&](int pair, int st, int buf) {
        const int c0 = st * kCC, nc = min(kCC, a.usable - c0);
        const uint32_t dst = smem + buf * stage_bytes;
        const uint32_t full = bars + 8 * buf;
        const uint32_t tile_bytes = (uint32_t)(nwarps * kCC * kEnt);
        mbar_expect_tx(full, (uint32_t)(nc * a.row_bytes) + tile_bytes);
        bulk_g2s(dst, a.packed + ((size_t)pair * a.usable + c0) * a.row_bytes, (uint32_t)(nc * a.row_bytes), full);
        bulk_g2s(dst + stage_rows, a.tiles + ((size_t)blockIdx.x * n_stage + st) * (nwarps * kCC) * kEnt, tile_bytes, full);
    };
    // (pair, chunk) of the stage kStages ahead of the one being consumed, advanced once per stage by every warp
    int npair = pair_lo, nst = st_first;
    for (int g = 0; g < kStages; g++) {
        if (threadIdx.x == 0 && npair < pair_hi) issue(npair, nst, g);
        if ((nst += st_step) >= n_stage) { nst = st_first; npair++; }
    }

    const uint32_t lane_off = 80u * lane;  // 8 pairs = 4 chunks = 5 padded chunks per lane
    int buf = 0, ph = 0;                   // buffer and barrier parity of the stage being consumed
    for (int pair = pair_lo; pair < pair_hi; pair++) {
    u64 acc[4][kK];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
        for (int k = 0; k < kK; k++) acc[r][k] = 0ull;

    // one pipeline stage (kCC channels).  Whether the stage loop is left to the compiler's loop transformations changes how
    // ptxas allocates the 64 accumulator registers around the PTX block: measured on B200, the two-window variants are
    // 3 % faster with the loop kept as written (no in-loop register moves), the one-window variants 9 % slower.
    auto stage = [&](int st) {
            mbar_wait(bars + 8 * buf, ph);
            const uint32_t rows_s = smem + buf * stage_bytes;
            const uint32_t tiles_s = rows_s + stage_rows + warp * kCC * kEnt;
            const int nc = min(kCC, a.usable - st * kCC);
            if constexpr (FAST) {
                // the whole stage in one asm block: entry prefetch, window loads, four dispatched bodies, loop
                if (active) {
                    // (the entries' window offsets include the row's offset inside the stage)
                    if constexpr (DUAL) tile_stage_fast_dual<NCH>(acc, tiles_s, rows_s + lane_off, tiles_s + nc * kEnt);
                    else tile_stage_fast<NCH>(acc, tiles_s, rows_s + lane_off, tiles_s + nc * kEnt);
                }
            } else
            if (active) {
                uint32_t e0, e1;
                float f0, f1, f2, f3;
                uint32_t ent = tiles_s, row = rows_s + lane_off;
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(e0), "=r"(e1) : "r"(ent));
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(f0), "=f"(f1), "=f"(f2), "=f"(f3) : "r"(ent + 16));
#pragma unroll 1
                for (int c = 0; c < nc; c++) {
                    // window loads, differences, four accumulate bodies, prefetch of entry c + 1 into e0..f3 (the read past
                    // the last entry of a stage stays inside this CTA's shared memory and is never used)
                    ent += 32;
                    if constexpr (DUAL) tile_channel_step_dual<NCH>(acc, e0, e1, f0, f1, f2, f3, row, ent);
                    else tile_channel_step<NCH>(acc, e0, e1, f0, f1, f2, f3, row, ent);
                    row += a.row_bytes;
                }
            }
            __syncwarp();
            if (lane == 0) {
                // all of this warp's reads of the buffer have completed (their values were consumed above)
                if (atomicInc(&done_cnt[buf], nwarps - 1) == (unsigned)(nwarps - 1) && npair < pair_hi) issue(npair, nst, buf);
            }
            if ((nst += st_step) >= n_stage) { nst = st_first; npair++; }
            if (++buf == kStages) { buf = 0; ph ^= 1; }
    };
    if constexpr (DUAL && FAST) {
#pragma unroll 1
        for (int st = st_first; st < n_stage; st += st_step) stage(st);
    } else {
        for (int st = st_first; st < n_stage; st += st_step) stage(st);
    }

    if constexpr (KSPLIT) {
        // Tile t (= warp t of every rank) is finished by rank t % cluster size.  Every warp PUSHES its partial sums into the
        // finishing rank's shared memory (st.shared::cluster: nobody waits for a remote load), slot [source rank][t / cluster
        // size], 8 KB each, over the stage buffers -- which is why the first cluster barrier is there: every CTA must be done
        // with its rows first (no bulk copy is in flight: one block pair per CTA in this mode).  After the second barrier the
        // finishing warp adds the partials IN RANK ORDER from its own shared memory (its own included, read back the same
        // way: the result does not depend on which rank finishes the tile) and runs the epilogue; the others are done.
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        const int nfw = (nwarps + (int)csize - 1) / (int)csize;
        const unsigned dest = (unsigned)warp % csize;
        const int wl = warp / (int)csize;
        uint32_t remote;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem + (uint32_t)((((int)crank * nfw + wl) * 8192) + lane * 16)), "r"(dest));
#pragma unroll
        for (int j = 0; j < 16; j++)
            asm volatile("st.shared::cluster.v2.b64 [%0], {%1, %2};" ::"r"(remote + (uint32_t)(j * 512)), "l"(acc[j >> 2][2 * (j & 3)]),
                         "l"(acc[j >> 2][2 * (j & 3) + 1]) : "memory");
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        if (dest != crank) continue;
        for (int q = 0; q < (int)csize; q++) {
            const uint32_t src = smem + (uint32_t)(((q * nfw + wl) * 8192) + lane * 16);
#pragma unroll
            for (int j = 0; j < 16; j++) {
                u64 v0, v1;
                lds128(v0, v1, src + (uint32_t)(j * 512));
                acc[j >> 2][2 * (j & 3)] = q == 0 ? v0 : add2(acc[j >> 2][2 * (j & 3)], v0);
                acc[j >> 2][2 * (j & 3) + 1] = q == 0 ? v1 : add2(acc[j >> 2][2 * (j & 3) + 1], v1);
            }
        }
    }

    // ---- epilogue: MA = 0.5 out[j] - 0.25 (out[j+1] + out[j-1]); power = sum MA^2 (mimo.cpp:131-137) ----
    const int itemA = 2 * pair, itemB = 2 * pair + 1;
    int jlo[2], jhi[2];
#pragma unroll
    for (int h = 0; h < 2; h++) item_ma_range(min(h ? itemB : itemA, a.n_items - 1), a.blocks_per_frame, a.frame_len, jlo[h], jhi[h]);
#pragma unroll
    for (int r = 0; r < 4; r++) {
        u64 prev = __shfl_up_sync(0xffffffffu, acc[r][kK - 1], 1);
        u64 next = __shfl_down_sync(0xffffffffu, acc[r][0], 1);
        float pa = 0.f, pb = 0.f;
#pragma unroll
        for (int k = 0; k < kK; k++) {
            const u64 left = k == 0 ? prev : acc[r][k - 1];
            const u64 right = k == kK - 1 ? next : acc[r][k + 1];
            const int j = kK * lane + k;
            float ma = __fsub_rn(__fmul_rn(lo(acc[r][k]), 0.5f), __fmul_rn(0.25f, __fadd_rn(lo(right), lo(left))));
            float mb = __fsub_rn(__fmul_rn(hi(acc[r][k]), 0.5f), __fmul_rn(0.25f, __fadd_rn(hi(right), hi(left))));
            if (j >= jlo[0] && j <= jhi[0]) pa = __fmaf_rn(ma, ma, pa);
            if (j >= jlo[1] && j <= jhi[1]) pb = __fmaf_rn(mb, mb, pb);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            pa += __shfl_xor_sync(0xffffffffu, pa, o);
            pb += __shfl_xor_sync(0xffffffffu, pb, o);
        }
        if (lane == 0 && active) {
            const int dir = a.tile_dirs[4 * my_tile + r];
            if (dir >= 0) {
                if (a.blocks_per_frame == 1) {
                    a.out[(size_t)itemA * a.n_dir + dir] = __fdiv_rn(pa, a.norm);
                    if (itemB < a.n_items) a.out[(size_t)itemB * a.n_dir + dir] = __fdiv_rn(pb, a.norm);
                } else {
                    a.out[(size_t)itemA * a.n_dir + dir] = pa;
                    if (itemB < a.n_items) a.out[(size_t)itemB * a.n_dir + dir] = pb;
                }
            }
        }
        // beams calls: every block stores the frame samples it owns (item_beam_range); the bounds are even and rows start
        // at even samples, so a lane's samples go out in 8-byte pairs
        if (BEAMS && active) {
            const int dir = a.tile_dirs[4 * my_tile + r];
            if (dir >= 0) {
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int item = h ? itemB : itemA;
                    if (item >= a.n_items) continue;
                    int blo, bhi;
                    item_beam_range(item, a.blocks_per_frame, a.frame_len, blo, bhi);
                    const int b = item / a.blocks_per_frame, q = item - b * a.blocks_per_frame;
                    float *row = a.beams + ((size_t)b * a.n_dir + dir) * a.frame_len + block_first_sample(q, a.frame_len);
#pragma unroll
                    for (int k = 0; k < kK; k += 2) {
                        const int j = kK * lane + k;
                        const u64 v0 = acc[r][k], v1 = acc[r][k + 1];
                        if (j >= blo && j < bhi)
                            *reinterpret_cast<float2 *>(row + j) = h ? make_float2(hi(v0), hi(v1)) : make_float2(lo(v0), lo(v1));
                    }
                }
            }
        }
    }
    }  // block pairs of this CTA
}

// frames longer than one block (this kernel and das_bcast's): power[b][d] = (sum_q partial[b*nblk + q][d]) / norm, blocks
// in order; grid.y strides over the frames (it is limited to 65535)
__global__ void finalize_kernel(const float *__restrict__ partial, int n_frames, int nblk, int n_dir, float norm,
                                float *__restrict__ power) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n_dir) return;
    for (int b = blockIdx.y; b < n_frames; b += gridDim.y) {
        float p = 0.f;
        for (int q = 0; q < nblk; q++) p += partial[((size_t)b * nblk + q) * n_dir + d];
        power[(size_t)b * n_dir + d] = __fdiv_rn(p, norm);
    }
}

cudaError_t launch_finalize(const FrameArgs &f, cudaStream_t st) {
    dim3 fg((f.n_dir + 255) / 256, std::min(f.n_frames, 65535));
    finalize_kernel<<<fg, 256, 0, st>>>(f.partial, f.n_frames, blocks_per_frame(f.frame_len), f.n_dir, f.norm, f.power);
    return cudaGetLastError();
}

// ---- host side ---------------------------------------------------------------------------------------------------
int das_tile_max_span() { return 11; }

// Every compiled instantiation das_tile_kernel<nch, warps, dual, fast, ksplit>: the kernel is instantiated from this list
// (kTileLaunchers), and it alone answers which variants exist.  warps is the register budget (launch bound); a launch may
// run fewer warps per CTA on it.  The exact form has no 9-chunk window, and the channel split is two-FMA and 16 warps only.
struct TileVariant {
    int nch, warps;
    bool dual, fast, ksplit;
};
constexpr TileVariant kTileVariants[] = {
    // two-FMA form, channels split across a cluster
    {5, 16, false, true, true}, {6, 16, false, true, true}, {7, 16, false, true, true},
    {8, 16, false, true, true}, {9, 16, false, true, true}, {10, 16, false, true, true},
    {6, 16, true, true, true}, {7, 16, true, true, true},
    // two-FMA form
    {5, 10, false, true, false}, {5, 11, false, true, false}, {5, 12, false, true, false}, {5, 16, false, true, false},
    {6, 10, false, true, false}, {6, 11, false, true, false}, {6, 12, false, true, false}, {6, 16, false, true, false},
    {7, 10, false, true, false}, {7, 11, false, true, false}, {7, 12, false, true, false}, {7, 16, false, true, false},
    {8, 10, false, true, false}, {8, 11, false, true, false}, {8, 12, false, true, false}, {8, 16, false, true, false},
    {9, 10, false, true, false}, {9, 11, false, true, false}, {9, 12, false, true, false}, {9, 16, false, true, false},
    {10, 10, false, true, false}, {10, 11, false, true, false}, {10, 12, false, true, false}, {10, 16, false, true, false},
    {6, 10, true, true, false}, {6, 11, true, true, false}, {6, 12, true, true, false}, {6, 16, true, true, false},
    {7, 10, true, true, false}, {7, 11, true, true, false}, {7, 12, true, true, false}, {7, 16, true, true, false},
    // exact form
    {5, 10, false, false, false}, {5, 11, false, false, false}, {5, 12, false, false, false}, {5, 16, false, false, false},
    {6, 10, false, false, false}, {6, 11, false, false, false}, {6, 12, false, false, false}, {6, 16, false, false, false},
    {7, 10, false, false, false}, {7, 11, false, false, false}, {7, 12, false, false, false}, {7, 16, false, false, false},
    {8, 10, false, false, false}, {8, 11, false, false, false}, {8, 12, false, false, false}, {8, 16, false, false, false},
    {10, 10, false, false, false}, {10, 11, false, false, false}, {10, 12, false, false, false}, {10, 16, false, false, false},
    {6, 10, true, false, false}, {6, 11, true, false, false}, {6, 12, true, false, false}, {6, 16, true, false, false},
    {7, 10, true, false, false}, {7, 11, true, false, false}, {7, 12, true, false, false},
};
constexpr int kNumTileVariants = (int)(sizeof(kTileVariants) / sizeof(kTileVariants[0]));

// index of the variant in kTileVariants, -1 when it is not compiled
static int tile_variant(int nch, int warps, bool dual, bool fast, bool ksplit) {
    for (int i = 0; i < kNumTileVariants; i++) {
        const TileVariant &v = kTileVariants[i];
        if (v.nch == nch && v.warps == warps && v.dual == dual && v.fast == fast && v.ksplit == ksplit) return i;
    }
    return -1;
}

// experiment switch (read once): BFLK_NO_PACK_CARVEOUT=1 leaves the pack kernels' L1 / shared split to the driver
static bool getenv_once_no_carveout() {
    static const bool v = [] { const char *e = getenv("BFLK_NO_PACK_CARVEOUT"); return e && e[0] == '1'; }();
    return v;
}

size_t das_tile_entry_bytes(const TileGeometry &g);

size_t das_tile_smem_bytes(const TileGeometry &g, int stages) {
    // + 256: the fast variant's entry prefetch reads one entry past the last stage buffer's table (never used), and a window
    // whose last chunk no direction reads loads that chunk from [entry pointer + up to 192] instead (one broadcast wavefront)
    return (size_t)stages * (kCC * g.row_bytes + g.warps * kCC * das_tile_entry_bytes(g)) + stages * (8 + 4) + 256;
}

TileGeometry das_tile_geometry(int history, int max_delay, int max_span, int n_tiles, int mode, int fast, const Tuning *tuning, int want_warps) {
    TileGeometry g;
    g.mode = mode;
    g.fast = fast;
    g.stage_off = (history - max_delay) & ~1;
    // chunks per lane window: 9 + span sample pairs, two per chunk (two-window modes exist for spans up to 5)
    g.nch = max_span <= 1 && mode == 0 ? 5 : (max_span <= 3 ? 6 : (max_span <= 5 ? 7 : (max_span <= 7 ? 8 : 10)));
    if (fast) {
        g.nch = std::max(mode ? 6 : 5, (9 + max_span + 1) / 2);
        if (tuning && tuning->tile_nch > 0) g.nch = std::min(mode ? 7 : 10, std::max(g.nch, tuning->tile_nch));
    }
    // Warps (= direction tiles) per CTA, among the compiled variants of this window.  The kernel is issue-bound (an FFMA2 /
    // FADD2 holds a scheduler's issue port for two cycles), so more resident warps help only while registers allow: the
    // 6-chunk and the two-FMA variants fit 128 registers (16 warps, +5 % over 12); the exact 7- to 10-chunk variants need
    // ~150-165 (12 warps; at 16 they spill, so only BFLK_TILE_WARPS=16 runs them).  Smaller CTAs only when a small direction
    // shard (multi-GPU) would leave the last CTA mostly idle.
    const bool dual = mode != 0;
    const bool policy16 = fast || g.nch <= 6;
    const int n_cand = 4;
    const int cand[n_cand] = {16, 12, 11, 10};
    const double tlp[n_cand] = {policy16 ? 1.05 : 0.0, 1.0, 0.95, 0.88};
    const int forced = tuning && tile_variant(g.nch, tuning->tile_warps, dual, fast, false) >= 0 ? tuning->tile_warps : 0;
    // the largest logical chunk a lane can touch: (H - stage_off)/2 + 4*31 + nch - 1
    g.row_chunks = (history - g.stage_off) / 2 + 4 * 31 + g.nch;
    g.copy_bytes = 16 * (padded_chunk(g.row_chunks - 1) + 1);
    g.row_bytes = 2 * g.copy_bytes;  // even-aligned copy + copy shifted by one sample pair
    // pick the best-scoring CTA shape whose stage ring fits shared memory (long arrays: packed rows grow with the largest
    // delay); 4 stage buffers where they fit, else 3; stages == 0 tells the caller that no shape fits
    double best = 0.0;
    g.warps = 0;
    g.stages = 0;
    for (int i = 0; i < n_cand; i++) {
        if (forced ? cand[i] != forced : tlp[i] <= 0.0) continue;
        if (tile_variant(g.nch, cand[i], dual, fast, false) < 0) continue;
        TileGeometry t = g;
        t.warps = cand[i];
        int stages = tuning && tuning->tile_stages == 3 ? 3 : kMaxStages;
        if (das_tile_smem_bytes(t, stages) > 227 * 1024) stages = 3;
        if (das_tile_smem_bytes(t, stages) > 227 * 1024) continue;
        const int tiles = n_tiles > 0 ? n_tiles : 1 << 20;
        const int groups = (tiles + cand[i] - 1) / cand[i];
        const double score = (forced ? 1.0 : tlp[i]) * tiles / (double)(groups * cand[i]);
        if (score > best + 1e-9) { best = score; g.warps = cand[i]; g.stages = stages; }
    }
    g.tmpl_warps = g.warps;
    if (want_warps > 0 && want_warps <= 16 && g.stages >= 3) {
        // latency shape (single-frame calls): fewer warps per CTA than the throughput shape, run on the largest compiled
        // variant the policy allows (its register budget is an upper bound); the stage ring of a smaller CTA always fits if
        // the large one does
        const int tmpl = policy16 && tile_variant(g.nch, 16, dual, fast, false) >= 0 ? 16 : 12;
        TileGeometry t = g;
        t.warps = std::min(want_warps, tmpl);
        int stages = tuning && tuning->tile_stages == 3 ? 3 : kMaxStages;
        if (das_tile_smem_bytes(t, stages) > 227 * 1024) stages = 3;
        if (das_tile_smem_bytes(t, stages) <= 227 * 1024) {
            g.tmpl_warps = tmpl;
            g.warps = t.warps;
            g.stages = stages;
        }
    }
    if (g.warps == 0) g.warps = g.tmpl_warps = 12;   // nothing fits: stages stays 0
    g.pairs_per_cta = tuning && tuning->tile_pairs > 0 ? tuning->tile_pairs : 0;
    return g;
}

bool das_tile_ksplit_ok(const TileGeometry &g, int split) {
    // the exchange area (8 KB per (source rank, tile finished here)) reuses the stage buffers' rows
    return (split == 2 || split == 4) && tile_variant(g.nch, g.tmpl_warps, g.mode != 0, g.fast, true) >= 0 && g.stages >= 3 &&
           (size_t)split * ((g.warps + split - 1) / split) * 8192 <= (size_t)g.stages * kCC * g.row_bytes;
}

size_t das_tile_entry_bytes(const TileGeometry &g) {
    return g.fast ? (g.mode ? sizeof(TileEntryFastDual) : sizeof(TileEntryFast)) : sizeof(TileEntry);
}

template <int NCH, int WARPS, bool DUAL = false, bool FAST = false, bool KSPLIT = false, bool BEAMS = false>
static cudaError_t launch_main(const KernelArgs &k, dim3 grid, size_t smem, cudaStream_t st) {
    // the attribute is per device and only ever grows: set it when a larger request appears there, not per launch
    static size_t configured[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || smem > configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(das_tile_kernel<NCH, WARPS, DUAL, FAST, KSPLIT, BEAMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = smem;
    }
    const int warps = k.launch_warps > 0 && k.launch_warps <= WARPS ? k.launch_warps : WARPS;
    if constexpr (KSPLIT) {
        // grid.z CTAs = one thread-block cluster per (tile group, block pair): they split the channels
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = grid;
        cfg.blockDim = dim3(warps * 32);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr{};
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = 1;
        attr.val.clusterDim.y = 1;
        attr.val.clusterDim.z = grid.z;
        cfg.attrs = &attr;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, das_tile_kernel<NCH, WARPS, DUAL, FAST, KSPLIT, BEAMS>, k);
    }
    das_tile_kernel<NCH, WARPS, DUAL, FAST, KSPLIT, BEAMS><<<grid, warps * 32, smem, st>>>(k);
    return cudaGetLastError();
}

using TileLauncher = cudaError_t (*)(const KernelArgs &, dim3, size_t, cudaStream_t);
template <bool BEAMS, size_t... I>
static constexpr std::array<TileLauncher, sizeof...(I)> tile_launchers(std::index_sequence<I...>) {
    return {launch_main<kTileVariants[I].nch, kTileVariants[I].warps, kTileVariants[I].dual, kTileVariants[I].fast,
                        kTileVariants[I].ksplit, BEAMS>...};
}
// kTileLaunchers[beams][i] launches kTileVariants[i], the power-only or the beams instantiation
static constexpr std::array<TileLauncher, kNumTileVariants> kTileLaunchers[2] = {
    tile_launchers<false>(std::make_index_sequence<kNumTileVariants>()),
    tile_launchers<true>(std::make_index_sequence<kNumTileVariants>())};

cudaError_t launch_das_tile(const TileArgs &a, int sm_count, cudaStream_t st, int *launches, TileLaunchHook hook, void *hook_ctx) {
    (void)sm_count;
    const FrameArgs &f = a.f;
    const int nblk = blocks_per_frame(f.frame_len);
    const int n_items = f.n_frames * nblk;
    const int n_pairs = (n_items + 1) / 2;
    if (f.frame_len < kBlock || (!a.wire && (f.row_stride & 1)) || (f.frame_stride & 1) || (f.frame_len & 1)) return cudaErrorInvalidValue;
    // channel split across a cluster (latency shape of small calls): das_tile_ksplit_ok allows it where it is compiled
    const int ksplit = std::max(1, a.geom.ksplit);
    const int variant = tile_variant(a.geom.nch, a.geom.tmpl_warps, a.geom.mode != 0, a.geom.fast, ksplit > 1);
    const int stages = a.geom.stages;
    if (stages < 3 || variant < 0) return cudaErrorInvalidConfiguration;   // ensure_tiles never selects such a geometry
    const size_t smem = das_tile_smem_bytes(a.geom, stages);

    PackArgs p{};
    p.wire = a.wire;
    p.wire_cols = a.wire_cols;
    p.stream = f.stream;
    p.row_stride = f.row_stride;
    p.row_len = f.row_len;
    p.n_frames = f.n_frames;
    p.frame_len = f.frame_len;
    p.frame_stride = f.frame_stride;
    p.blocks_per_frame = nblk;
    p.n_items = n_items;
    p.index = f.index;
    p.usable = f.usable;
    p.stage_off = a.geom.stage_off;
    p.row_chunks = a.geom.row_chunks;
    p.row_bytes = a.geom.row_bytes;
    p.copy_bytes = a.geom.copy_bytes;
    p.packed = reinterpret_cast<float4 *>(f.packed);
    const int kWarps = a.geom.warps;

    KernelArgs k{};
    k.packed = reinterpret_cast<const char *>(f.packed);
    k.tiles = static_cast<const char *>(a.tiles);
    k.tile_dirs = a.tile_dirs;
    k.n_tiles = a.n_tiles;
    k.usable = f.usable;
    k.n_dir = f.n_dir;
    k.row_bytes = a.geom.row_bytes;
    k.n_items = n_items;
    k.blocks_per_frame = nblk;
    k.frame_len = f.frame_len;
    k.pairs_per_cta = ksplit > 1 ? 1 : block_pairs_per_cta(a.geom.pairs_per_cta, f.usable);
    k.out = nblk == 1 ? f.power : f.partial;
    k.beams = f.beams;
    k.norm = f.norm;
    k.stages = stages;
    k.launch_warps = kWarps;

    // the main kernel needs (nearly) all of an SM's shared memory: ask for the same L1 / shared split for the pack pre-pass
    // (it streams, an L1 hit rate does not matter to it), so the SMs do not have to be reconfigured between the two launches
    // of every call
    static bool carveout_set[64] = {false};
    {
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 64 && !carveout_set[dev] && !getenv_once_no_carveout()) {
            cudaFuncSetAttribute(pack_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            cudaFuncSetAttribute(pack_wire_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            carveout_set[dev] = true;
        }
    }
    // grid.y / grid.z are limited to 65535: process the pairs in slabs
    const int max_slab = 32768;
    for (int p0 = 0; p0 < n_pairs; p0 += max_slab) {
        const int np = min(max_slab, n_pairs - p0);
        PackArgs ps = p;
        KernelArgs ks = k;
        ps.pair0 = p0;
        ks.pair0 = p0;
        dim3 pg((a.geom.row_chunks + 255) / 256, f.usable, np);
        dim3 wg((a.geom.row_chunks + kWireChunks - 1) / kWireChunks, (f.usable + kWireCh - 1) / kWireCh, np);
        if (hook) hook(hook_ctx, 1, true, st);
        if (a.wire) pack_wire_kernel<<<wg, 256, 0, st>>>(ps);
        else pack_kernel<<<pg, 256, 0, st>>>(ps);
        if (hook) hook(hook_ctx, 1, false, st);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        ks.n_pairs = np;
        dim3 grid((a.n_tiles + kWarps - 1) / kWarps, (np + ks.pairs_per_cta - 1) / ks.pairs_per_cta, ksplit);
        if (hook) hook(hook_ctx, 0, true, st);
        e = kTileLaunchers[f.beams != nullptr][variant](ks, grid, smem, st);
        if (hook) hook(hook_ctx, 0, false, st);
        if (e != cudaSuccess) return e;
        *launches += 2;
    }
    if (nblk > 1) {
        cudaError_t e = launch_finalize(f, st);
        if (e != cudaSuccess) return e;
        *launches += 1;
    }
    return cudaSuccess;
}

}  // namespace bflk
