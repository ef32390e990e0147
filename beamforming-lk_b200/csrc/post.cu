// post.cu -- the steps either side of the delay-and-sum path.
//   heat-map normalisation + peak  : MIMOWorker::populateHeatmap, src/dsp/mimo.cpp:61-95
//   per-microphone power           : AWProcessingUnit::calibrate, src/aw_processing_unit/aw_processing_unit.cpp:134-146
//   wire int32 -> float exposure   : Pipeline::receive_exposure, src/fpga/pipeline.cpp:260-297
//   streaming history              : the device twin of Streams' double-mapped ring, src/fpga/streams.hpp:152-182
#include "bflk_internal.h"
#include "das_common.cuh"

namespace bflk {

// ---- heat-map ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) heatmap_kernel(const float *__restrict__ power, int n, uint8_t *__restrict__ heat,
                                                      int32_t *__restrict__ argmax, float *__restrict__ maxv) {
    __shared__ float s_v[32];
    __shared__ int s_i[32];
    // maxV starts at 0.0 and is replaced on strict '>' (mimo.cpp:62-69): first occurrence of the maximum
    float best = 0.0f;
    int besti = 0x7fffffff;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float v = power[i];
        if (v > best) { best = v; besti = i; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, best, o);
        int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
    }
    if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = besti; }
    __syncthreads();
    if (threadIdx.x < 32) {
        best = threadIdx.x < (blockDim.x >> 5) ? s_v[threadIdx.x] : 0.0f;
        besti = threadIdx.x < (blockDim.x >> 5) ? s_i[threadIdx.x] : 0x7fffffff;
        for (int o = 16; o > 0; o >>= 1) {
            float ov = __shfl_xor_sync(0xffffffffu, best, o);
            int oi = __shfl_xor_sync(0xffffffffu, besti, o);
            if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
        }
        if (threadIdx.x == 0) { s_v[0] = best; s_i[0] = besti == 0x7fffffff ? 0 : besti; }
    }
    __syncthreads();
    const float mx = s_v[0];
    if (threadIdx.x == 0) { *argmax = s_i[0]; *maxv = mx; }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double db = (double)__fdiv_rn(power[i], mx);  // pow(powerdB[i] / maxV, 1), mimo.cpp:86
        db *= 255.0;
        db = db < 0.0 ? 0.0 : (db > 255.0 ? 255.0 : db);  // clip(); NaN (all-zero map) falls through to 0
        heat[i] = (uint8_t)db;
    }
}

cudaError_t launch_heatmap(const float *d_power, int n, uint8_t *d_heat, int32_t *d_argmax, float *d_max, cudaStream_t st) {
    heatmap_kernel<<<1, 1024, 0, st>>>(d_power, n, d_heat, d_argmax, d_max);
    return cudaGetLastError();
}

// ---- per-channel power (calibration) --------------------------------------------------------------------
// Sequential float accumulation per channel in sample order, as the reference loop does
// (aw_processing_unit.cpp:136-141), so the median gate sees the same bits as the CPU restatement.
__global__ void channel_power_kernel(const float *__restrict__ signals, int n_ch, int W, float *__restrict__ power) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_ch) return;
    const float *s = signals + (size_t)c * W;
    float pv = 0.0f;
    for (int i = 0; i < W; i++) {
        float x = s[i];
        pv = __fadd_rn(pv, __fmul_rn(x, x));
    }
    power[c] = __fdiv_rn(pv, (float)W);
}

cudaError_t launch_channel_power(const float *d_signals, int n_ch, int W, float *d_power, cudaStream_t st) {
    channel_power_kernel<<<(n_ch + 31) / 32, 32, 0, st>>>(d_signals, n_ch, W, d_power);
    return cudaGetLastError();
}

// ---- ingest -------------------------------------------------------------------------------------------
// frames[n][n_sensors] (one UDP message per time sample, src/fpga/receiver.h:24-30) ->
// exposure[n_sensors][n]: serpentine column un-flip + int32 / 2^23 (exact), 32x32 transpose tiles.  Sample tiles on grid.x
// (grid.y is limited to 65535 tiles, 2 M samples), sensor tiles on grid.y.
__global__ void __launch_bounds__(256) ingest_kernel(const int32_t *__restrict__ frames, int64_t n, int n_sensors,
                                                    float *__restrict__ exposure) {
    __shared__ float tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.x * 32;
    const int s0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int64_t i = i0 + r;
        const int sensor = s0 + tx;
        if (i < n && sensor < n_sensors) tile[r][tx] = wire_to_float(frames[(size_t)i * n_sensors + wire_column(sensor)]);
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int64_t i = i0 + tx;
        const int sensor = s0 + r;
        if (i < n && sensor < n_sensors) exposure[(size_t)sensor * n + i] = tile[tx][r];
    }
}

cudaError_t launch_ingest(const int32_t *d_frames, int64_t n, int n_sensors, float *d_exposure, cudaStream_t st) {
    dim3 grid((unsigned)((n + 31) / 32), (n_sensors + 31) / 32);
    ingest_kernel<<<grid, 256, 0, st>>>(d_frames, n, n_sensors, d_exposure);
    return cudaGetLastError();
}

// ---- streaming history (bflk_stream_push) ------------------------------------------------------------------------
// A block of n new samples per channel, samples t0 .. t0 + n of the session, into the mirrored ring: sample t goes to
// columns t % cap and t % cap + cap of its channel's row of 2 * cap floats.  Float blocks are channel-major [C][n] and are
// copied four samples per thread where ring and block stay 16-byte aligned; wire blocks [n][C] int32 go through the
// transposing 32 x 32 tile of ingest_kernel, with the same un-flip and scale, so the ring holds the floats ingest_kernel
// and pack_wire_kernel produce.
__global__ void __launch_bounds__(256) history_push_kernel(const float *__restrict__ block, const int32_t *__restrict__ wire,
                                                          int n, int C, int64_t t0, int cap, float *__restrict__ ring) {
    const int64_t pitch = 2 * (int64_t)cap;
    if (wire) {   // grid: (sample tiles, channel tiles)
        __shared__ float tile[32][33];
        const int i0 = blockIdx.x * 32, s0 = blockIdx.y * 32;
        const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
        for (int r = ty; r < 32; r += 8) {
            const int i = i0 + r, sensor = s0 + tx;
            if (i < n && sensor < C) tile[r][tx] = wire_to_float(wire[(size_t)i * C + wire_column(sensor)]);
        }
        __syncthreads();
        for (int r = ty; r < 32; r += 8) {
            const int sensor = s0 + r, i = i0 + tx;
            if (i < n && sensor < C) {
                float *row = ring + sensor * pitch + (t0 + i) % cap;
                row[0] = row[cap] = tile[tx][r];
            }
        }
        return;
    }
    // grid: (1024-sample pieces, channels)
    const float *src = block + (size_t)blockIdx.y * n;
    float *row = ring + blockIdx.y * pitch;
    const int i0 = blockIdx.x * 1024;
    if (((t0 | n | cap) & 3) == 0) {
        const int i = i0 + 4 * threadIdx.x;
        if (i < n) {
            const float4 v = *reinterpret_cast<const float4 *>(src + i);
            float4 *dst = reinterpret_cast<float4 *>(row + (t0 + i) % cap);
            dst[0] = v;
            dst[cap / 4] = v;
        }
    } else {
        for (int i = i0 + threadIdx.x; i < min(n, i0 + 1024); i += 256) row[(t0 + i) % cap] = row[(t0 + i) % cap + cap] = src[i];
    }
}

cudaError_t launch_history_push(const float *d_block, const int32_t *d_wire, int n, int C, int64_t t0, int cap, float *d_ring,
                                cudaStream_t st) {
    const dim3 grid = d_wire ? dim3((n + 31) / 32, (C + 31) / 32) : dim3((n + 1023) / 1024, C);
    history_push_kernel<<<grid, 256, 0, st>>>(d_block, d_wire, n, C, t0, cap, d_ring);
    return cudaGetLastError();
}

// ---- heat-map resize: cv::resize(compact, normal, normal.size(), 0, 0, cv::INTER_LINEAR) on CV_8UC1 -------------------
// (src/aw_processing_unit/aw_processing_unit.cpp:252).  OpenCV's 8-bit bilinear path is fixed point; the coefficient
// tables (offset, two shorts per output column / row) are built on the host exactly like cv::resize builds them and the
// kernel does the two integer passes per output pixel -- bit-identical to OpenCV (tests/golden/resize.npz, made with cv2).
__global__ void resize_u8_kernel(const uint8_t *__restrict__ src, int ih, int iw, uint8_t *__restrict__ dst, int oh, int ow,
                                 const int32_t *__restrict__ tab) {
    // tab: xo[ow] | xa[ow] (a0 | a1 << 16) | yo[oh] | ya[oh]
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= ow || y >= oh) return;
    const int x0 = tab[x], xa = tab[ow + x], yo = tab[2 * ow + y], ya = tab[2 * ow + oh + y];
    const int xa0 = (short)(xa & 0xffff), xa1 = (short)(xa >> 16), ya0 = (short)(ya & 0xffff), ya1 = (short)(ya >> 16);
    const int x1 = min(x0 + 1, iw - 1);
    const int y0 = min(max(yo, 0), ih - 1), y1 = min(max(yo + 1, 0), ih - 1);
    const int S0 = src[y0 * iw + x0] * xa0 + src[y0 * iw + x1] * xa1;
    const int S1 = src[y1 * iw + x0] * xa0 + src[y1 * iw + x1] * xa1;
    int v = ((ya0 * (S0 >> 4)) >> 16) + ((ya1 * (S1 >> 4)) >> 16);
    v = (v + 2) >> 2;
    dst[(size_t)y * ow + x] = (uint8_t)min(max(v, 0), 255);
}

cudaError_t launch_resize_u8(const uint8_t *d_src, int ih, int iw, uint8_t *d_dst, int oh, int ow, const int32_t *d_tab, cudaStream_t st) {
    dim3 grid((ow + 255) / 256, oh);
    resize_u8_kernel<<<grid, 256, 0, st>>>(d_src, ih, iw, d_dst, oh, ow, d_tab);
    return cudaGetLastError();
}

// ---- peaks of the map as Targets (src/dsp/worker.h:32-61) -----------------------------------------------------------
// One CTA.  Pass 1 marks the directions that are the maximum of their 3x3 neighbourhood (ties: lowest index) and carry at
// least min_rel of the map's maximum; pass 2 picks the max_targets strongest of them in order (power descending, index
// ascending) and forms the tracker-style probability 1 / gradientError from the four grid neighbours
// (src/dsp/gradient_ascend.cpp:62-76).  Same definition as oracle.c orc_map_targets.
__global__ void __launch_bounds__(1024) map_targets_kernel(const float *__restrict__ power, int rows, int cols, int max_targets,
                                                          float min_rel, uint8_t *__restrict__ cand, int32_t *__restrict__ out_index,
                                                          float *__restrict__ out_power, float *__restrict__ out_prob,
                                                          int32_t *__restrict__ out_n) {
    __shared__ float s_v[32];
    __shared__ int s_i[32];
    __shared__ float s_max;
    __shared__ int s_best;
    const int D = rows * cols;
    float mx = 0.0f;
    for (int i = threadIdx.x; i < D; i += blockDim.x) mx = fmaxf(mx, power[i]);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) s_v[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        float m = 0.0f;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) m = fmaxf(m, s_v[w]);
        s_max = m;
    }
    __syncthreads();
    const float thr = __fmul_rn(min_rel, s_max);
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
        const float p = power[i];
        bool is_max = p >= thr && p > 0.0f;
        if (is_max) {
            const int r = i / cols, c = i - r * cols;
            for (int dr = -1; dr <= 1 && is_max; dr++)
                for (int dc = -1; dc <= 1; dc++) {
                    const int rr = r + dr, cc = c + dc;
                    if ((dr == 0 && dc == 0) || rr < 0 || rr >= rows || cc < 0 || cc >= cols) continue;
                    const int j = rr * cols + cc;
                    const float q = power[j];
                    if (q > p || (q == p && j < i)) { is_max = false; break; }
                }
        }
        cand[i] = is_max ? 1 : 0;
    }
    __syncthreads();
    int n = 0;
    for (; n < max_targets; n++) {
        float best = -1.0f;
        int besti = 0x7fffffff;
        for (int i = threadIdx.x; i < D; i += blockDim.x)
            if (cand[i]) {
                const float p = power[i];
                if (p > best || (p == best && i < besti)) { best = p; besti = i; }
            }
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
            if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
        }
        if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = best; s_i[threadIdx.x >> 5] = besti; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); w++)
                if (s_v[w] > best || (s_v[w] == best && s_i[w] < besti)) { best = s_v[w]; besti = s_i[w]; }
            s_best = best >= 0.0f ? besti : -1;
            if (s_best >= 0) {
                const int i = s_best, r = i / cols, c = i - r * cols;
                const float p = power[i];
                const double ql = c > 0 ? power[i - 1] : p, qr = c < cols - 1 ? power[i + 1] : p;
                const double qu = r > 0 ? power[i - cols] : p, qd = r < rows - 1 ? power[i + cols] : p;
                const double err = (fabs(qr - ql) + fabs(qd - qu)) / (((ql + qr) + qu) + qd);
                double pr = 1.0 / err;
                if (!(pr < 3.4028234663852886e38)) pr = 3.4028234663852886e38;
                out_index[n] = i;
                out_power[n] = p;
                out_prob[n] = (float)pr;
                cand[i] = 0;
            }
        }
        __syncthreads();
        if (s_best < 0) break;
    }
    if (threadIdx.x == 0) *out_n = n;
}

cudaError_t launch_map_targets(const float *d_power, int rows, int cols, int max_targets, float min_rel, uint8_t *d_cand,
                               int32_t *d_index, float *d_pw, float *d_prob, int32_t *d_n, cudaStream_t st) {
    map_targets_kernel<<<1, 1024, 0, st>>>(d_power, rows, cols, max_targets, min_rel, d_cand, d_index, d_pw, d_prob, d_n);
    return cudaGetLastError();
}

// ---- FP32 saturation micro-benchmark (the empirical roofline denominator, SURVEY 8d) -------------------------------
// 16 independent packed-FMA chains per thread, 16 warps per SM, one CTA per SM: what the FP32 pipe delivers on this chip
// at the clock it runs at under load (tools/ubench measures the same: 127.6 of 128 lane-operations per clock per SM).
__global__ void __launch_bounds__(512) ffma2_peak_kernel(float *out, int iters, float seed) {
    unsigned long long p[16];
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const float v = seed + (float)(i + threadIdx.x);
        p[i] = ((unsigned long long)__float_as_uint(v) << 32) | __float_as_uint(v * 0.5f);
    }
    const float f = seed * 0.999f, g = seed * 1e-3f;
    const unsigned long long f2 = ((unsigned long long)__float_as_uint(f) << 32) | __float_as_uint(f);
    const unsigned long long g2 = ((unsigned long long)__float_as_uint(g) << 32) | __float_as_uint(g);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(p[i]) : "l"(f2), "l"(g2));
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; i++) s += __uint_as_float((unsigned)p[i]) + __uint_as_float((unsigned)(p[i] >> 32));
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

cudaError_t launch_ffma2_peak(float *d_out, int n_blocks, int iters, cudaStream_t st) {
    ffma2_peak_kernel<<<n_blocks, 512, 0, st>>>(d_out, iters, 1.0f);
    return cudaGetLastError();
}

}  // namespace bflk
