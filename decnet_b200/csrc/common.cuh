// decnet_b200/csrc/common.cuh -- shared host/device helpers for libdecnet_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>
#include <utility>
#include "../../include/decnet_b200.h"

namespace decnet {

// thread-local error text behind decnet_last_error()
void set_error(const char *fmt, ...);
// records + returns DECNET_ERR_CUDA_BASE + err when err != cudaSuccess, else 0
int cuda_status(cudaError_t err, const char *what);
// checks cudaGetLastError() after a launch and bumps the per-thread launch counter
int after_launch(const char *kernel_name);
int sm_count_cached();

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline size_t round_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

#define DECNET_REQUIRE(cond, ...)                 \
    do {                                          \
        if (!(cond)) {                            \
            ::decnet::set_error(__VA_ARGS__);     \
            return DECNET_ERR_INVALID;            \
        }                                         \
    } while (0)

#define DECNET_CUDA(expr)                                         \
    do {                                                          \
        int _st = ::decnet::cuda_status((expr), #expr);           \
        if (_st) return _st;                                      \
    } while (0)

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__
// Programmatic dependent launch (the persistent tensor-core kernels follow one another dozens of times per step): a kernel
// launched with launch_pdl() may start while its predecessor in the stream is still running -- it sets up barriers, allocates
// TMEM, loads its weights -- and must call pdl_wait() before its first access to anything the predecessor wrote or still reads.
// pdl_wait() returns once the predecessor grid has completed and its memory operations are visible to this grid; every access
// that is ordered after the waiting thread's loads (through mbarriers) is ordered after it too.  pdl_trigger() lets the NEXT kernel
// be scheduled as soon as every CTA of this one has started.  Both are no-ops in a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// true unless DECNET_PDL=0 (read once)
bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void cp_async_16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_4(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_u32(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

__device__ __forceinline__ float group_max(float v, int G) {
    for (int o = G >> 1; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float group_sum(float v, int G) {
    for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// two fp32 -> packed fp16 halves (round to nearest, saturating to +-65504), lo_half in the low 16 bits
__device__ __forceinline__ uint32_t cvt_f16x2_sat(float hi_half, float lo_half) {
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi_half), "f"(lo_half));
    return d;
}

// "split16" storage of the activations the channels-last conv stacks chain on (conv2d_nhwc_tcgen05.cu, split = 3): the same
// 4 bytes per channel as fp32, and already the operand the conv's fp16 MMAs read.  Per 32-channel chunk of cl channels
// (cl = min(32, cp - c0), cp % 16 == 0) a pixel holds the halves
//     [fp16(2^11 * (x - h)) x cl | h x cl],   h = fp16(x),   both rounded to nearest and saturating (cvt.rn.satfinite),
// so x = h + 2^-11 * lo to ~2^-22 relative for |x| < 65504; beyond that both halves saturate and stay finite.  Zero encodes
// as zero bits: zero border pixels and zero padding channels are written exactly as in fp32.
// split16_store writes channels [c, c + N) of one pixel (pixel: its 4*cp bytes); N = 1, 4 or 16, c a multiple of N.
template <int N>
__device__ __forceinline__ void split16_store(void *pixel, int cp, int c, const float (&v)[N])
{
    static_assert(N == 1 || N == 4 || N == 16, "runs of 1, 4 or 16 channels");
    const int c0 = c & ~31, cl = min(32, cp - c0), k = c - c0;
    uint16_t *q = reinterpret_cast<uint16_t *>(pixel) + 2 * c0;
    if constexpr (N == 1) {
        const uint32_t h = cvt_f16x2_sat(0.f, v[0]);
        float hf;
        asm("{.reg .b16 t, u;\n\tmov.b32 {t, u}, %1;\n\tcvt.f32.f16 %0, t;}" : "=f"(hf) : "r"(h));
        q[k] = (uint16_t)cvt_f16x2_sat(0.f, (v[0] - hf) * 2048.f);
        q[cl + k] = (uint16_t)h;
    } else {
        uint32_t lo[N / 2], hi[N / 2];
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            hi[i] = cvt_f16x2_sat(v[2 * i + 1], v[2 * i]);
            float h0, h1;
            asm("{.reg .b16 t, u;\n\tmov.b32 {t, u}, %2;\n\tcvt.f32.f16 %0, t;\n\tcvt.f32.f16 %1, u;}" : "=f"(h0), "=f"(h1) : "r"(hi[i]));
            lo[i] = cvt_f16x2_sat((v[2 * i + 1] - h1) * 2048.f, (v[2 * i] - h0) * 2048.f);
        }
        if constexpr (N == 4) {
            *reinterpret_cast<uint2 *>(q + k) = make_uint2(lo[0], lo[1]);
            *reinterpret_cast<uint2 *>(q + cl + k) = make_uint2(hi[0], hi[1]);
        } else {
#pragma unroll
            for (int i = 0; i < N / 2; i += 4) {
                *reinterpret_cast<uint4 *>(q + k + 2 * i) = make_uint4(lo[i], lo[i + 1], lo[i + 2], lo[i + 3]);
                *reinterpret_cast<uint4 *>(q + cl + k + 2 * i) = make_uint4(hi[i], hi[i + 1], hi[i + 2], hi[i + 3]);
            }
        }
    }
}
#endif

}  // namespace decnet
