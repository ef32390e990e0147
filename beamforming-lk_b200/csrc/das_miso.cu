// das_miso.cu -- dynamic steering in ONE launch: T targets x B frames, tables computed in the kernel.
//
// Replaces, per target, Particle::steer + Particle::das + Particle::beam (src/dsp/particle.cpp:37-103) as MISOWorker::update
// uses them (src/dsp/miso.cpp:39-46) and the 4 x P beams of a monopulse step (src/dsp/gradient_ascend.cpp:30-81).  The
// reference recomputes a 64-entry steering table on the host for every steer(); here the direction arrives as the four
// rotation-matrix entries the reference evaluates in double (DirTrig, in the kernel's parameter space) and every CTA of a
// target builds its (offset, fraction) table in shared memory with the same pinned operations as the table kernel
// (steer.cuh) -- no table round trip through HBM, no host synchronisation between "steer" and "das": the largest-delay
// check of the host path is a flag the kernel raises.  Arithmetic per (target, channel, sample) is the reference's delay()
// triple in mask order (delay.cpp:24), so the audio block is bit-identical to Particle::das.
//
// The work is tiny (cfg4: 16 targets x 512 channels x 256 samples = 8.4 MFLOP) and LATENCY-bound: the adds of one output
// sample form a dependent chain over the channels.  What was measured on B200 (tools/miso_time.py, cfg4, per call):
//   one CTA per target, 256 threads, plain unrolled channel loop        95 us  (one L2 latency exposed per channel)
//   + two register sets of 16 channels (loads of the next batch first)   33 us  (L1 wavefront queue: 2 x 512 scalar loads x 8 warps)
//   + cp.async 4-byte staging, 4 stages                                  48 us  (LDGSTS issue rate)
//   + TMA bulk copies of the aligned row segments, 6 stages              93 us  (512 one-kilobyte copies issued by one thread)
// -> the frame is cut into slices of 62 high-pass outputs (64 samples with the neighbours the 3-tap filter needs): 5 CTAs
// of two warps per target spread the loads over five SMs, each thread keeps two register sets of 32 channels in flight,
// and the slices' partial powers are summed in slice order by the last CTA to finish (deterministic).
#include "bflk_internal.h"
#include "steer.cuh"

namespace bflk {

constexpr int kMisoThreads = 64;            // samples per CTA: 62 high-pass outputs + the neighbour on either side
constexpr int kMisoOut = kMisoThreads - 2;
constexpr int kBatch = 32;                  // channels per register set

// FOCUS: the tables of a point source at a.focus (focus_z); the far-field instantiation is the kernel as it was before
template <bool FOCUS>
__global__ void __launch_bounds__(kMisoThreads) miso_kernel(MisoArgs a) {
    extern __shared__ __align__(8) unsigned char s_raw[];
    __shared__ float s_red[kMisoThreads / 32];
    __shared__ float s_out[kMisoThreads];
    __shared__ int s_flag, s_last;
    long long *s_addr = reinterpret_cast<long long *>(s_raw);                          // [usable] element offset of the first tap
    float *s_frac = reinterpret_cast<float *>(s_raw + sizeof(long long) * a.usable);   // [usable]
    float *s_del = s_frac + a.usable;                                                  // [C] raw delays
    const int t = blockIdx.x, k = blockIdx.y, b = blockIdx.z, N = a.frame_len, n_slices = gridDim.y;
    const DirTrig trig = a.n_inline ? a.trig_inline[t] : a.trig[t];
    if (threadIdx.x == 0) s_flag = 0;

    // ---- Particle::steer: steering_vector_spherical + split (particle.cpp:37-49), all C elements for the minimum ----
    float mn = INFINITY;
    for (int c = threadIdx.x; c < a.C; c += kMisoThreads) {
        const float del = steer_delay<FOCUS>(trig, a.xyz, c, a.k_scale, a.focus);
        s_del[c] = del;
        mn = fminf(mn, del);
    }
    for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = mn;
    __syncthreads();
    mn = fminf(s_red[0], s_red[1]);
    for (int s = threadIdx.x; s < a.usable; s += kMisoThreads) {
        const int c = a.index[s];
        const float del = __fsub_rn(s_del[c], mn);   // delays -= minCoeff (antenna.cpp:94)
        const float ip = truncf(del);                // modf((double)del, &ip): exact for a float argument
        int di = (int)ip;
        if (di > a.history) {                        // the host path's BFLK_ERR_RANGE: raised here, reported after the call
            s_flag = 1;
            di = a.history;
        }
        s_addr[s] = (long long)c * a.row_stride + (a.history - di);
        s_frac[s] = __fsub_rn(del, ip);
        if (a.off_out && b == 0 && k == 0) {
            a.off_out[(size_t)t * a.C + c] = a.history - di;
            a.frac_out[(size_t)t * a.C + c] = s_frac[s];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_flag) atomicExch(a.error_flag, a.epoch);

    // ---- Particle::das (particle.cpp:88-103): out[i] += delay(channel s), s in mask order ----
    // slice k owns high-pass outputs [1 + 62 k, 1 + 62 k + 62) and therefore needs samples [62 k, 62 k + 64); the last slice
    // is shifted back so it ends at the frame's last sample (N >= 64; shorter frames run one clamped slice)
    const int i_lo = max(0, min(kMisoOut * k, N - kMisoThreads));
    const int i = min(i_lo + (int)threadIdx.x, N - 1);
    const float *sig0 = a.window + (size_t)b * a.frame_stride + i;
    const int last = a.usable - 1;
    float acc = 0.0f;
    {
        float curA[kBatch], nxtA[kBatch], curB[kBatch], nxtB[kBatch];
        auto load = [&](float (&cur)[kBatch], float (&nxt)[kBatch], int s0) {
#pragma unroll
            for (int u = 0; u < kBatch; u++) {
                const float *sig = sig0 + s_addr[min(s0 + u, last)];
                asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(cur[u]) : "l"(sig));
                asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(nxt[u]) : "l"(sig + 1));
            }
        };
        auto sum = [&](const float (&cur)[kBatch], const float (&nxt)[kBatch], int s0) {
#pragma unroll
            for (int u = 0; u < kBatch; u++)
                if (s0 + u <= last) acc = __fadd_rn(acc, __fmaf_rn(s_frac[s0 + u], __fsub_rn(cur[u], nxt[u]), nxt[u]));
        };
        load(curA, nxtA, 0);
        for (int s0 = 0; s0 < a.usable; s0 += 2 * kBatch) {
            load(curB, nxtB, s0 + kBatch);
            sum(curA, nxtA, s0);
            load(curA, nxtA, s0 + 2 * kBatch);
            sum(curB, nxtB, s0 + kBatch);
        }
    }
    // every sample is stored by exactly one slice: slice k stores [62 k, 62 k + 62), the last one everything up to N
    const int own_lo = kMisoOut * k, own_hi = k == n_slices - 1 ? N : kMisoOut * (k + 1);
    const int idx = i_lo + (int)threadIdx.x;
    if (a.audio && idx >= own_lo && idx < own_hi && idx < N) a.audio[((size_t)b * a.n_targets + t) * N + idx] = acc;
    if (!a.power) return;
    s_out[threadIdx.x] = acc;
    __syncthreads();
    // ---- Particle::beam (particle.cpp:68-79): 3-tap high-pass, mean square over N; this slice's outputs only ----
    const int hp_lo = 1 + kMisoOut * k, hp_hi = k == n_slices - 1 ? N - 1 : 1 + kMisoOut * (k + 1);
    float p = 0.0f;
    if (idx >= hp_lo && idx < hp_hi && threadIdx.x > 0 && threadIdx.x < kMisoThreads - 1) {
        const float ma = __fsub_rn(__fmul_rn(s_out[threadIdx.x], 0.5f),
                                   __fmul_rn(0.25f, __fadd_rn(s_out[threadIdx.x + 1], s_out[threadIdx.x - 1])));
        p = __fmul_rn(ma, ma);
    }
    for (int o = 16; o > 0; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = p;
    __syncthreads();
    if (threadIdx.x == 0) {
        float *part = a.partial + ((size_t)b * a.n_targets + t) * n_slices;
        part[k] = s_red[0] + s_red[1];
        __threadfence();
        s_last = atomicInc(a.counters + (size_t)b * a.n_targets + t, n_slices - 1) == (unsigned)(n_slices - 1);
        if (s_last) {
            __threadfence();
            float tot = 0.0f;
            for (int q = 0; q < n_slices; q++) tot += __ldcg(part + q);      // slice order: deterministic
            a.power[(size_t)b * a.n_targets + t] = __fdiv_rn(tot, a.norm);
        }
    }
}

int das_miso_slices(int frame_len) { return frame_len <= kMisoThreads ? 1 : (frame_len - 2 + kMisoOut - 1) / kMisoOut; }

cudaError_t launch_das_miso(const MisoArgs &a, cudaStream_t st) {
    if (a.n_targets <= 0 || a.n_frames <= 0) return cudaSuccess;
    const size_t smem = (size_t)a.usable * (sizeof(long long) + sizeof(float)) + (size_t)a.C * sizeof(float);
    if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
    auto kernel = a.focus > 0.0 ? miso_kernel<true> : miso_kernel<false>;
    if (smem > 48 * 1024) {   // beyond the default limit (thousands of channels): per device, so set per launch
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const int n_slices = das_miso_slices(a.frame_len);
    for (int b0 = 0; b0 < a.n_frames; b0 += 65535) {   // grid.z is limited to 65535
        MisoArgs s = a;
        s.n_frames = std::min(65535, a.n_frames - b0);
        s.window = a.window + (size_t)b0 * a.frame_stride;
        if (a.audio) s.audio = a.audio + (size_t)b0 * a.n_targets * a.frame_len;
        if (a.power) s.power = a.power + (size_t)b0 * a.n_targets;
        if (a.partial) s.partial = a.partial + (size_t)b0 * a.n_targets * n_slices;
        if (a.counters) s.counters = a.counters + (size_t)b0 * a.n_targets;
        dim3 grid(a.n_targets, n_slices, s.n_frames);
        kernel<<<grid, kMisoThreads, smem, st>>>(s);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace bflk
