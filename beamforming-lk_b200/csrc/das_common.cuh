// das_common.cuh -- PTX helpers shared by the delay-and-sum kernels: packed FP32 (FFMA2 / FADD2),
// mbarrier and TMA bulk-copy wrappers for sm_100a; the wire-format un-flip and scale of the ingest kernels.
#pragma once
#include <cuda/std/cstdint>

namespace bflk {
namespace {

typedef unsigned long long u64;

__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
    u64 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b) {
    u64 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 dup2(float f) {
    u64 d;
    asm("mov.b64 %0, {%1, %1};" : "=l"(d) : "f"(f));
    return d;
}
__device__ __forceinline__ float lo(u64 v) { return __uint_as_float((unsigned)v); }
__device__ __forceinline__ float hi(u64 v) { return __uint_as_float((unsigned)(v >> 32)); }

__device__ __forceinline__ void lds128(u64 &a, u64 &b, uint32_t addr) {
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}


// Wire format (one int32 row per time sample, src/fpga/receiver.h:24-30): the row column that holds a sensor -- every
// second group of 8 is mirrored (daisy-chained arrays, pipeline.cpp:273-287) -- and the sample as a float (/ 2^23, exact
// for 24-bit samples).  Every kernel that reads wire rows goes through these two, so they all hold the same floats.
__device__ __forceinline__ int wire_column(int sensor) {
    const int grp = sensor >> 3;
    return (grp & 1) ? sensor : 8 * (1 + grp) - 1 - (sensor & 7);
}
__device__ __forceinline__ float wire_to_float(int32_t v) { return __fdiv_rn((float)v, 8388608.0f); }

// output block q of a frame: first sample s_q = min(254 q, N - 256); it owns the high-pass outputs
// MA_i for i in [254 q + 1, min(254 q + 254, N - 2)]  (N = 256: one block, i in [1, 254], mimo.cpp:132); blocks_per_frame
// (bflk_internal.h) counts the blocks
__device__ __forceinline__ int block_first_sample(int q, int frame_len) { return min(254 * q, frame_len - 256); }
__device__ __forceinline__ long long item_first_sample(int item, int nblk, int frame_len, int frame_stride) {
    const int b = item / nblk, q = item - b * nblk;
    return (long long)b * frame_stride + block_first_sample(q, frame_len);
}
__device__ __forceinline__ void item_ma_range(int item, int nblk, int frame_len, int &jlo, int &jhi) {
    const int q = item % nblk;
    const int s = block_first_sample(q, frame_len);
    jlo = 254 * q + 1 - s;
    jhi = min(254 * q + 254, frame_len - 2) - s;
}
// the delayed sums (beams) block q of a frame stores, so that every frame sample is written exactly once: frame samples
// [254 q, 254 q + 254), the last block [254 q, N) -- as block samples [jlo, jhi), inside [0, 256), both bounds even
__device__ __forceinline__ void item_beam_range(int item, int nblk, int frame_len, int &jlo, int &jhi) {
    const int q = item % nblk;
    const int s = block_first_sample(q, frame_len);
    jlo = 254 * q - s;
    jhi = (q == nblk - 1 ? frame_len : 254 * q + 254) - s;
}

}  // namespace
}  // namespace bflk
