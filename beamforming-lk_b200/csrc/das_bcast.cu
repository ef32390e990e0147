// das_bcast.cu -- lane-per-direction delay-and-sum power map for sm_100a ("broadcast" kernel).
//
// Replaces the loop nest of MIMOWorker::update (src/dsp/mimo.cpp:121-150) around delay()
// (src/dsp/delay.cpp:16-26).  Design (DESIGN.md "das_bcast"):
//
//  * bcast_pack_kernel rewrites the channel-major stream once per batch into rows of
//    float4{ A[t], B[t], A[t-1]-A[t], B[t-1]-B[t] } for two 256-sample output blocks A and B (channel-mask
//    order).  The subtraction of delay() is thereby done ONCE per input sample instead of once per
//    (direction, sample): the inner loop is a single 16-byte shared-memory load feeding one FFMA2
//    (fma.rn.f32x2) and one FADD2 per two (direction, channel, sample) units -- 2 FP32 lane-operations
//    per unit, the reference's exact operation order, bit-identical delayed sums.
//  * bcast_kernel: one CTA = 32 adjacent steering directions x two 256-sample blocks; lane = direction,
//    warp w = output samples 16w..16w+15.  The 32 lanes of a warp read the same few neighbouring row
//    elements (their integer offsets differ by a few samples), so every LDS.128 is served by one or two
//    shared-memory wavefronts through the hardware's lane broadcast: the row is reused 32x from shared
//    memory and 16x across warps.  No data-dependent control flow, no alignment cases.
//  * rows and per-(channel, lane) {offset, fraction} tables are staged with cp.async.bulk (TMA bulk
//    copy) into a 3-stage mbarrier pipeline, 8 channels per stage.
//  * epilogue: 3-tap high-pass + squares (mimo.cpp:131-135); chunk-edge samples are exchanged through
//    shared memory, per-direction sums reduced across the 16 warps in fixed order; beams calls also store the
//    delayed sums.
#include "bflk_internal.h"
#include "das_common.cuh"

namespace bflk {

namespace {

constexpr int kWarps = 16;            // 16 warps x 16 sample pairs = one 256-sample block pair
constexpr int kThreads = kWarps * 32;
constexpr int kK = 16;                // sample pairs per lane
constexpr int kCC = kBcastCC;         // channels per pipeline stage
constexpr int kStages = 3;
constexpr int kBlock = 256;

struct PackArgs {
    const float *stream;
    int64_t row_stride, row_len;
    int frame_len, frame_stride, nblk, n_items, pair0;
    const int32_t *index;
    int usable;
    int first_sample;   // row element j <-> block sample first_sample + j
    int row_elems;      // float4 elements per row
    float4 *packed;     // [pair][usable][row_elems]
};

__global__ void __launch_bounds__(256) bcast_pack_kernel(PackArgs a) {
    const int pair = a.pair0 + blockIdx.z, s = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.row_elems) return;
    const int itemA = 2 * pair, itemB = min(2 * pair + 1, a.n_items - 1);
    const long long tA = item_first_sample(itemA, a.nblk, a.frame_len, a.frame_stride) + a.first_sample + j;
    const long long tB = item_first_sample(itemB, a.nblk, a.frame_len, a.frame_stride) + a.first_sample + j;
    const float *row = a.stream + (size_t)a.index[s] * a.row_stride;
    auto at = [&](long long t) { return (t >= 0 && t < a.row_len) ? __ldg(row + t) : 0.0f; };
    const float a1 = at(tA), a0 = at(tA - 1), b1 = at(tB), b0 = at(tB - 1);
    // current - next, rounded once exactly like _mm256_sub_ps(current_vec, next_vec) in delay.cpp:24
    a.packed[((size_t)pair * a.usable + s) * a.row_elems + j] = make_float4(a1, b1, __fsub_rn(a0, a1), __fsub_rn(b0, b1));
}

struct KernelArgs {
    const float4 *packed;       // [pair][usable][row_elems]
    const BcastEntry *table;    // [tile][n_stage][kCC][32]
    const int32_t *tile_dirs;   // [n_tiles][32] local direction index or -1
    int usable, n_dir, row_bytes;
    int n_items, nblk, frame_len, pair0;
    float *out;                 // power [frames][n_dir] (nblk == 1) or partial [items][n_dir]
    float norm;
    float *beams;               // delayed sums [frames][n_dir][frame_len] (BEAMS instantiation only; FrameArgs::beams)
};

// BEAMS: the epilogue also stores the delayed sums (beams calls); a template flag, so that the power-only kernel is compiled
// exactly as without it
template <bool BEAMS>
__global__ void __launch_bounds__(kThreads, 1) bcast_kernel(KernelArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int stage_rows = kCC * a.row_bytes;
    const int stage_bytes = stage_rows + kCC * 32 * (int)sizeof(BcastEntry);
    const uint32_t smem = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const uint32_t bars = smem + kStages * stage_bytes;  // full[kStages], empty[kStages]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x;
    const int pair = a.pair0 + blockIdx.y;
    const int n_stage = (a.usable + kCC - 1) / kCC;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; s++) {
            mbar_init(bars + 8 * s, 1);
            mbar_init(bars + 8 * (kStages + s), kWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const char *rows_g = reinterpret_cast<const char *>(a.packed) + (size_t)pair * a.usable * a.row_bytes;
    const BcastEntry *tbl_g = a.table + (size_t)tile * n_stage * (kCC * 32);
    auto issue = [&](int st) {
        const int buf = st % kStages;
        const int c0 = st * kCC, nc = min(kCC, a.usable - c0);
        const uint32_t dst = smem + buf * stage_bytes;
        const uint32_t full = bars + 8 * buf;
        constexpr uint32_t tbl_bytes = kCC * 32 * (uint32_t)sizeof(BcastEntry);
        mbar_expect_tx(full, (uint32_t)(nc * a.row_bytes) + tbl_bytes);
        bulk_g2s(dst, rows_g + (size_t)c0 * a.row_bytes, (uint32_t)(nc * a.row_bytes), full);
        bulk_g2s(dst + stage_rows, tbl_g + (size_t)st * (kCC * 32), tbl_bytes, full);
    };
    if (threadIdx.x == 0)
        for (int st = 0; st < min(kStages - 1, n_stage); st++) issue(st);

    u64 acc[kK];
#pragma unroll
    for (int k = 0; k < kK; k++) acc[k] = 0ull;

    const uint32_t lane_sample = 16u * (uint32_t)(kK * warp);  // byte offset of this warp's first sample pair
    for (int st = 0; st < n_stage; st++) {
        const int buf = st % kStages;
        if (threadIdx.x == 0 && st + kStages - 1 < n_stage) {
            if (st >= 1) mbar_wait(bars + 8 * (kStages + (st - 1) % kStages), ((st - 1) / kStages) & 1);
            issue(st + kStages - 1);
        }
        mbar_wait(bars + 8 * buf, (st / kStages) & 1);
        const uint32_t rows_s = smem + buf * stage_bytes;
        const uint32_t tbl_s = rows_s + stage_rows + 8 * lane;
        const int nc = min(kCC, a.usable - st * kCC);
        for (int c = 0; c < nc; c++) {
            uint32_t joff;
            float f;
            asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(joff), "=f"(f) : "r"(tbl_s + c * 256));
            const uint32_t addr = rows_s + c * a.row_bytes + joff + lane_sample;
            const u64 ff = dup2(f);
            u64 nx[kK], dd[kK];
#pragma unroll
            for (int k = 0; k < kK; k++) lds128(nx[k], dd[k], addr + 16 * k);
#pragma unroll
            for (int k = 0; k < kK; k++) acc[k] = add2(acc[k], fma2(ff, dd[k], nx[k]));  // out += fma(f, cur - next, next)
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + 8 * (kStages + buf));
    }

    // ---- epilogue ----------------------------------------------------------------------------------------
    __syncthreads();  // every warp is done with the stage buffers: reuse them
    u64 *edge = reinterpret_cast<u64 *>(smem_raw);                 // [kWarps][32][2]: first / last sample of each chunk
    float2 *part = reinterpret_cast<float2 *>(smem_raw + kWarps * 32 * 16);  // [kWarps][32]
    edge[(warp * 32 + lane) * 2 + 0] = acc[0];
    edge[(warp * 32 + lane) * 2 + 1] = acc[kK - 1];
    __syncthreads();
    const u64 prev = warp > 0 ? edge[((warp - 1) * 32 + lane) * 2 + 1] : 0ull;
    const u64 next = warp < kWarps - 1 ? edge[((warp + 1) * 32 + lane) * 2 + 0] : 0ull;
    const int itemA = 2 * pair, itemB = 2 * pair + 1;
    int jloA, jhiA, jloB, jhiB;
    item_ma_range(min(itemA, a.n_items - 1), a.nblk, a.frame_len, jloA, jhiA);
    item_ma_range(min(itemB, a.n_items - 1), a.nblk, a.frame_len, jloB, jhiB);
    float pa = 0.f, pb = 0.f;
#pragma unroll
    for (int k = 0; k < kK; k++) {
        const u64 left = k == 0 ? prev : acc[k - 1];
        const u64 right = k == kK - 1 ? next : acc[k + 1];
        const int j = kK * warp + k;
        // MA = 0.5 out[j] - 0.25 (out[j+1] + out[j-1]); power += MA^2   (mimo.cpp:133-134)
        const float ma = __fsub_rn(__fmul_rn(lo(acc[k]), 0.5f), __fmul_rn(0.25f, __fadd_rn(lo(right), lo(left))));
        const float mb = __fsub_rn(__fmul_rn(hi(acc[k]), 0.5f), __fmul_rn(0.25f, __fadd_rn(hi(right), hi(left))));
        if (j >= jloA && j <= jhiA) pa = __fmaf_rn(ma, ma, pa);
        if (j >= jloB && j <= jhiB) pb = __fmaf_rn(mb, mb, pb);
    }
    // beams calls: every block stores the frame samples it owns (item_beam_range), a lane its direction's 16 samples in
    // 8-byte pairs (even bounds, rows start at even samples)
    if constexpr (BEAMS) {
        const int dir = a.tile_dirs[tile * 32 + lane];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int item = h ? itemB : itemA;
            if (dir < 0 || item >= a.n_items) continue;
            int blo, bhi;
            item_beam_range(item, a.nblk, a.frame_len, blo, bhi);
            const int b = item / a.nblk, q = item - b * a.nblk;
            float *row = a.beams + ((size_t)b * a.n_dir + dir) * a.frame_len + block_first_sample(q, a.frame_len);
#pragma unroll
            for (int k = 0; k < kK; k += 2) {
                const int j = kK * warp + k;
                if (j >= blo && j < bhi)
                    *reinterpret_cast<float2 *>(row + j) = h ? make_float2(hi(acc[k]), hi(acc[k + 1])) : make_float2(lo(acc[k]), lo(acc[k + 1]));
            }
        }
    }
    part[warp * 32 + lane] = make_float2(pa, pb);
    __syncthreads();
    if (warp == 0) {
        float sa = 0.f, sb = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; w++) {
            const float2 p = part[w * 32 + lane];
            sa += p.x;
            sb += p.y;
        }
        const int dir = a.tile_dirs[tile * 32 + lane];
        if (dir >= 0) {
            if (a.nblk == 1) {
                sa = __fdiv_rn(sa, a.norm);
                sb = __fdiv_rn(sb, a.norm);
            }
            a.out[(size_t)itemA * a.n_dir + dir] = sa;
            if (itemB < a.n_items) a.out[(size_t)itemB * a.n_dir + dir] = sb;
        }
    }
}

// table[tile][stage][cc][lane] = { byte offset of the lane's first element inside a packed row, fraction }
__global__ void bcast_table_kernel(const int32_t *__restrict__ off, const float *__restrict__ frac, int C,
                                   const int32_t *__restrict__ index, int usable, const int32_t *__restrict__ tile_globals,
                                   int first_offset, BcastEntry *__restrict__ table) {
    const int tile = blockIdx.x, lane = threadIdx.x & 31;
    const int n_stage = (usable + kCC - 1) / kCC;
    int g = tile_globals[tile * 32 + lane];
    if (g < 0) g = tile_globals[tile * 32];  // padding lanes shadow the tile's first direction
    for (int s = threadIdx.x >> 5; s < n_stage * kCC; s += blockDim.x >> 5) {
        BcastEntry e;
        e.joff = 0;
        e.frac = 0.f;
        if (s < usable) {
            const int c = index[s];
            e.joff = 16 * (off[(size_t)g * C + c] - first_offset);
            e.frac = frac[(size_t)g * C + c];
        }
        table[((size_t)tile * n_stage * kCC + s) * 32 + lane] = e;
    }
}

}  // namespace

BcastGeometry das_bcast_geometry(int history, int max_delay) {
    BcastGeometry g;
    g.first_offset = history - max_delay;         // smallest offset in the LUT
    g.first_sample = g.first_offset + 1;          // row element 0 <-> "next" sample of output 0 at the smallest offset
    g.row_elems = max_delay + kBlock;             // offsets [first_offset, history] x outputs [0, 256)
    g.row_bytes = g.row_elems * 16;
    return g;
}

size_t das_bcast_table_entries(int n_tiles, int usable) {
    return (size_t)n_tiles * ((usable + kCC - 1) / kCC) * kCC * 32;
}

cudaError_t launch_bcast_table(const int32_t *d_off, const float *d_frac, int C, const int32_t *d_index, int usable,
                               const int32_t *d_tile_globals, int n_tiles, const BcastGeometry &g, BcastEntry *d_table,
                               cudaStream_t st) {
    bcast_table_kernel<<<n_tiles, 256, 0, st>>>(d_off, d_frac, C, d_index, usable, d_tile_globals, g.first_offset, d_table);
    return cudaGetLastError();
}

static size_t bcast_smem_bytes(const BcastGeometry &g) {
    return (size_t)kStages * (kCC * g.row_bytes + kCC * 32 * sizeof(BcastEntry)) + 2 * kStages * 8;
}

// packed rows grow with the largest delay: beyond ~330 samples of history the stage ring no longer fits shared memory
bool das_bcast_fits(const BcastGeometry &g) {
    const size_t smem = bcast_smem_bytes(g);
    return smem <= 227 * 1024 && smem >= (size_t)kWarps * 32 * 24;
}

cudaError_t launch_das_bcast(const BcastArgs &a, cudaStream_t st, int *launches, TileLaunchHook hook, void *hook_ctx) {
    const FrameArgs &f = a.f;
    const int nblk = blocks_per_frame(f.frame_len);
    const int n_items = f.n_frames * nblk;
    const int n_pairs = (n_items + 1) / 2;
    if (f.frame_len < kBlock) return cudaErrorInvalidValue;
    const size_t smem = bcast_smem_bytes(a.geom);
    if (!das_bcast_fits(a.geom)) return cudaErrorInvalidConfiguration;
    void (*const kernel)(KernelArgs) = f.beams ? bcast_kernel<true> : bcast_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;

    PackArgs p{};
    p.stream = f.stream;
    p.row_stride = f.row_stride;
    p.row_len = f.row_len;
    p.frame_len = f.frame_len;
    p.frame_stride = f.frame_stride;
    p.nblk = nblk;
    p.n_items = n_items;
    p.index = f.index;
    p.usable = f.usable;
    p.first_sample = a.geom.first_sample;
    p.row_elems = a.geom.row_elems;
    p.packed = reinterpret_cast<float4 *>(f.packed);

    KernelArgs k{};
    k.packed = p.packed;
    k.table = a.table;
    k.tile_dirs = a.tile_dirs;
    k.usable = f.usable;
    k.n_dir = f.n_dir;
    k.row_bytes = a.geom.row_bytes;
    k.n_items = n_items;
    k.nblk = nblk;
    k.frame_len = f.frame_len;
    k.out = nblk == 1 ? f.power : f.partial;
    k.beams = f.beams;
    k.norm = f.norm;

    const int max_slab = 32768;  // grid.y / grid.z limits
    for (int p0 = 0; p0 < n_pairs; p0 += max_slab) {
        const int np = min(max_slab, n_pairs - p0);
        p.pair0 = k.pair0 = p0;
        dim3 pg((a.geom.row_elems + 255) / 256, f.usable, np);
        if (hook) hook(hook_ctx, 1, true, st);
        bcast_pack_kernel<<<pg, 256, 0, st>>>(p);
        if (hook) hook(hook_ctx, 1, false, st);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        dim3 grid(a.n_tiles, np);
        if (hook) hook(hook_ctx, 0, true, st);
        kernel<<<grid, kThreads, smem, st>>>(k);
        if (hook) hook(hook_ctx, 0, false, st);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        *launches += 2;
    }
    if (nblk > 1) {
        if ((e = launch_finalize(f, st)) != cudaSuccess) return e;
        *launches += 1;
    }
    return cudaSuccess;
}

}  // namespace bflk
