// decnet_b200/csrc/tma_utils.cuh -- TMA / mbarrier helpers (sm_100a) and host-side tensor-map
// encoding through the driver entry point (no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include "common.cuh"

namespace decnet {

// ------------------------------------------------------------------ host
// Encodes a tiled tensor map; returns 0 or a DECNET error code.  rank <= 5.
int encode_tensor_map(CUtensorMap *out, CUtensorMapDataType dtype, int rank, const void *gaddr,
                      const uint64_t *dims, const uint64_t *strides_bytes /* rank-1 */,
                      const uint32_t *box, CUtensorMapSwizzle swizzle,
                      CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B);

// ------------------------------------------------------------------ device
#ifdef __CUDACC__
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// non-blocking probe (try_wait may suspend the thread up to a hardware time limit before it answers)
__device__ __forceinline__ bool mbar_test_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// try_wait with a suspend-time hint (ns): the hardware parks the thread until the phase completes or the hint elapses, instead of
// answering "not yet" at once.  Every failed probe is a shared-memory access on the same L1 data pipe the tensor core fetches
// its operands through: in the 3xTF32 conv kernels (pipe 90 % busy) the 16 spinning epilogue warps made 4.5 M probes per launch,
// a third of the operand wavefronts (ncu source view, round 2).
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t *bar, uint32_t parity, uint32_t ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(ns) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait_hint(bar, parity, 20000u)) { }
}
// for waiters that are many (16 epilogue warps) or far ahead (producer)
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait_hint(bar, parity, 20000u)) { }
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *tm, int x, int y, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *tm, int x, int y, int z, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void *dst, const CUtensorMap *tm, int c0, int c1, int c2, int c3, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
          "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_5d(void *dst, const CUtensorMap *tm, int c0, int c1, int c2, int c3, int c4,
                                            uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4),
          "r"(smem_u32(bar)) : "memory");
}
#endif

// fp16 correction operands of the split = 2 conv modes: arithmetic for two neighbouring elements (a, b) -> packed halves, a in
// the low half:
//   lo16 = fp16(2^11 * (x - trunc_tf32(x)))   (the residual has <= 13 significant bits; fp16 keeps 11, like the TF32 lo part)
//   hi16 = fp16(x)                            (multiplies the 2^-11-sized lo part of the weights: its 2^-11 rounding is 2^-22 overall)
__device__ __forceinline__ uint32_t lo16x2(uint32_t a, uint32_t b) {
    const float fa = (__uint_as_float(a) - __uint_as_float(a & 0xFFFFE000u)) * 2048.f;
    const float fb = (__uint_as_float(b) - __uint_as_float(b & 0xFFFFE000u)) * 2048.f;
    return cvt_f16x2_sat(fb, fa);
}
__device__ __forceinline__ uint32_t hi16x2(uint32_t a, uint32_t b) { return cvt_f16x2_sat(__uint_as_float(b), __uint_as_float(a)); }


}  // namespace decnet
