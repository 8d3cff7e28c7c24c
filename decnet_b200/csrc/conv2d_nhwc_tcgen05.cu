// decnet_b200/csrc/conv2d_nhwc_tcgen05.cu -- the GEMM-sized 3x3 Conv2d layers of DynamicUpsampling.weight_learning
// (modules/submodule.py:571-575: 9C+1 -> 81 -> 81 -> 81 channels at the coarse resolution of each level) as a TF32
// implicit GEMM on channels-last tensors that carry their own zero border.
//
// conv3d_tcgen05.cu's Conv2d mode loads one A tile per tap: nine TMA fills of the same pixels per channel chunk, and its
// main loop waits for operands (DESIGN.md section 3.4).  Here the activations live in a PADDED channels-last layout
// [B, h+2, w+2, C] (one zero pixel all around each image, written by the producing kernel), so that in the flattened
// pixel index p a tap (kh, kw) is the constant offset (kh-1)*(w+2) + (kw-1).  A tile is 128 consecutive padded pixels:
//   * per (row tap kh, 32-channel chunk) ONE TMA box of 130 pixels x 128 B lands in shared memory (SWIZZLE_128B);
//   * the three column taps read it at +0 / +1 / +2 pixel rows: the UMMA descriptor's start address simply moves by
//     128 B -- the MMA swizzles on absolute shared-memory address bits, so a start that is not 1 KB aligned is fine
//     (scripts/micro/umma_rowshift.cu);
//   * the weights of the three column taps arrive as one box {32 ch, NP, 3 taps}.
// One stage = 12 MMAs (3 taps x 4 K-steps of 8) behind one barrier round trip instead of 4, and 1.6x fewer bytes
// from L2 per tile.  Border pixels of the output are written as zeros, so the next layer needs no padding pass; image
// boundaries inside the flattened index are covered by the borders, the ends of the tensor by TMA's zero fill.
//
// split = 1 ("3xTF32", fp32-class results: the mode the parity gates run on): the activations arrive as plain fp32, four
// converter warps write lo = rna_tf32(x - trunc_tf32(x)) beside the raw tile (whose truncation by the MMA is the hi part), the weights arrive as hi and lo
// parts ([18][NP][cp]: taps 0-8 hi, 9-17 lo), and every column tap issues lo*hi + hi*lo + hi*hi into the same accumulator
// (36 MMAs per stage).  A stage is then 2 x 17 KB of A and 2 x 3 x NP x 128 B of B.
// The tensor core adds into its fp32 accumulator with truncation, a bias that grows with the length of the accumulation
// chain (measured: 5e-8 x K relative, i.e. 3e-4 at K = 9 x 649 -- irrelevant for TF32, not for an fp32-class result).  In
// split mode the hi*hi products therefore accumulate in chains of kGroup stages (24 MMAs) that alternate between two
// TMEM slots; the epilogue warps drain the finished slot into REGISTERS with round-to-nearest fp32 adds while the next
// chain runs (two-level accumulation).  The two small terms go to a third accumulator that lives for the whole tile
// (its values, and so its truncation steps, are 2^-11 of the big one's) and is added last; the registers are biased,
// activated and stored once per tile.  NP <= 128 (4 x NP TMEM columns).
//
// split = 2 (the default of the Python side): the two small terms as ONE kind::f16 MMA per column tap and K-step: the converters
// write [fp16(2^11 * lo(x)) x cl | fp16(x) x cl] (cl = channels of the chunk, 4 bytes per channel like the fp32 tile) beside the
// raw tile, taps 9-17 of the weights hold [fp16(hi(w) * 2^sw) x cl | fp16(lo(w) * 2^(11+sw)) x cl] per row, and the small-term
// accumulator is drained with the factor 2^-(11+sw) (bias[np]).  24 MMAs per stage instead of 36.  In the split modes the
// activation tile completes its own mbarrier, so the converters start while the (4x larger) weight part of the stage is still in
// flight (DESIGN.md section 3.4).
//
// split = 3 (split16 input, the default inside the DynamicUpsampling and wide Refinement stacks): the activations arrive already
// as the operand the fp16 MMAs read, stored by the producing kernel as [fp16(2^11 * (x - h)) x cl | h x cl], h = fp16(x)
// (common.cuh: split16_store; same 4 bytes per channel as fp32, so the same tensor map loads it).  The converters idle, the hi
// taps of the weights are gone ([9][NP][cp]: only the fp16 taps of split = 2), and per column tap the issuer runs
//   small terms: [lo | h] * [hi16(w) ; lo16(w)]   (split = 2's correction MMA, cl/8 K-steps)  -> small-term accumulator
//   big term:    h * hi16(w)                       (A at +2*cl bytes, the hi16 half of B, cl/16 K-steps) -> the chain slot,
// which sum to x*hi(w) + h*lo(w) -- the 3xTF32 budget (lo*lo dropped, 11 bits per part).  The chain is drained with 2^-sw
// (bias[np + 1]).  A stage is 17 KB + 3 x NP x 128 B instead of twice that, so the ring is twice as deep.
// round_out (the output's storage format): 0 fp32, 1 fp32 rounded to TF32 (for a following split = 0 layer), 2 split16 (for a
// following split = 3 layer; ldc == np).
//
// Warp roles as in conv3d_tcgen05.cu: 0 TMA producer, 1 MMA issuer, 2-5 epilogue, 6-9 converters (split modes 1 and 2 only);
// persistent CTAs, two TMEM slots.
#include "common.cuh"
#include "tma_utils.cuh"
#include <mutex>

namespace decnet {
namespace conv2dnhwc {

constexpr int kMaxStages = 6;
constexpr int kThreads = 320;
constexpr int kConvWarps = 4;
constexpr int kGroup = 4;                          // split mode: stages per hi*hi accumulation chain
constexpr int kTileM = 128;
constexpr int kARows = 130;                        // 128 pixels + one halo pixel on each side
constexpr int kABytes = 17 * 1024;                 // 130 rows x 128 B rounded up to the 1 KB swizzle period

struct Params {
    const float *bias;                             // [NP]
    float *out;                                    // padded channels-last [B, h+2, w+2, NP]
    int B, h, w;                                   // interior size
    int cp, np;
    int nchunks, last_ksteps;
    long long P;                                   // B * (h+2) * (w+2) padded pixels
    int relu, out_format, tmem_cols, num_tiles, stages;
    int split;                                     // 0 TF32, 1 3xTF32, 2 TF32 + fp16 corrections, 3 split16 input
    int taps;                                      // 3: 3x3 conv on the zero-bordered layout; 1: plain GEMM (1x1 conv) over P rows
    int border;                                    // 1: rows are pixels of [B, h+2, w+2] and border pixels are stored as zeros
    int ldc;                                       // output row stride in floats (>= np: writes a channel slice of a wider tensor)
    int dst_h, dst_w;                              // > 0 (GEMM mode, border = 0): row p = (b, y, x) of a flat [B, dst_h, dst_w]
                                                   // grid is stored at the interior pixel (b, y+1, x+1) of a zero-bordered one
    int na_slots;                                  // pair kernel: slots of the A ring (the B ring has two)
    long long *trace;                              // tuning only (decnet_conv2d_nhwc_debug_trace): clock64 timeline of CTA 0,
                                                   // [256 stages][8]: 0 slot free (TMA issued), 1 landed, 2 converted, 3 issuer saw it,
                                                   // 4 MMAs + commit issued; then [256 drains][2]: chain finished, drained
    int dbg;                                       // tuning only (variant 100 + mask): 1 converters idle, 2 no correction MMAs,
                                                   // 4 no hi*hi MMAs, 8 no weight TMA after the first ring fill, 16 no drains
};

__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// KSTEPS K-steps of 8 tf32 (32 bytes: +2 in the descriptor's 16-byte address field) of one column tap: one election
#define DN_NEXT(OFF)                                                               \
        "add.u64 a, %1, " #OFF ";\n\t"                                              \
        "add.u64 b, %2, " #OFF ";\n\t"                                              \
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], a, b, %3, t;\n\t"
#define DN_HEAD                                                                    \
        "{\n\t.reg .pred p, e, t;\n\t.reg .b64 a, b;\n\t"                            \
        "elect.sync _|e, 0xffffffff;\n\t"                                           \
        "setp.ne.b32 p, %4, 0;\n\t"                                                 \
        "setp.eq.b32 t, 0, 0;\n\t"                                                  \
        "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
template <int KSTEPS>
__device__ __forceinline__ void umma_tap(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate_first) {
    if constexpr (KSTEPS == 4)
        asm volatile(DN_HEAD DN_NEXT(2) DN_NEXT(4) DN_NEXT(6) "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
    else if constexpr (KSTEPS == 3)
        asm volatile(DN_HEAD DN_NEXT(2) DN_NEXT(4) "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
    else if constexpr (KSTEPS == 2)
        asm volatile(DN_HEAD DN_NEXT(2) "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
    else
        asm volatile(DN_HEAD "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
}
__device__ __forceinline__ void umma_taps3(int ksteps, uint32_t acc, uint64_t da, uint64_t db, uint32_t db_tap_step,
                                           uint32_t idesc, uint32_t first, int ntaps = 3) {
    // the column taps (3, or 1 in GEMM mode): A moves one pixel row (128 B = 8 sixteen-byte units), B one tap block
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
        if (kw >= ntaps) break;
        const uint64_t a = da + (uint64_t)(8 * kw), b = db + (uint64_t)(kw * db_tap_step);
        const uint32_t acc_first = (kw == 0) ? first : 1u;
        switch (ksteps) {
            case 4: umma_tap<4>(acc, a, b, idesc, acc_first); break;
            case 3: umma_tap<3>(acc, a, b, idesc, acc_first); break;
            case 2: umma_tap<2>(acc, a, b, idesc, acc_first); break;
            default: umma_tap<1>(acc, a, b, idesc, acc_first); break;
        }
    }
}
// The same column-tap block for kind::f16 operands (K-steps of 16 halves = the same 32 bytes): the correction terms of split = 2.
#define DH_NEXT(OFF)                                                               \
        "add.u64 a, %1, " #OFF ";\n\t"                                              \
        "add.u64 b, %2, " #OFF ";\n\t"                                              \
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], a, b, %3, t;\n\t"
#define DH_HEAD                                                                    \
        "{\n\t.reg .pred p, e, t;\n\t.reg .b64 a, b;\n\t"                            \
        "elect.sync _|e, 0xffffffff;\n\t"                                           \
        "setp.ne.b32 p, %4, 0;\n\t"                                                 \
        "setp.eq.b32 t, 0, 0;\n\t"                                                  \
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
template <int KSTEPS>
__device__ __forceinline__ void umma_tap_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate_first) {
    if constexpr (KSTEPS == 4)
        asm volatile(DH_HEAD DH_NEXT(2) DH_NEXT(4) DH_NEXT(6) "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
    else if constexpr (KSTEPS == 3)
        asm volatile(DH_HEAD DH_NEXT(2) DH_NEXT(4) "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
    else if constexpr (KSTEPS == 2)
        asm volatile(DH_HEAD DH_NEXT(2) "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
    else
        asm volatile(DH_HEAD "}" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate_first) : "memory");
}
__device__ __forceinline__ void umma_taps3_f16(int ksteps, uint32_t acc, uint64_t da, uint64_t db, uint32_t db_tap_step,
                                               uint32_t idesc, uint32_t first, int ntaps = 3) {
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
        if (kw >= ntaps) break;
        const uint64_t a = da + (uint64_t)(8 * kw), b = db + (uint64_t)(kw * db_tap_step);
        const uint32_t acc_first = (kw == 0) ? first : 1u;
        switch (ksteps) {
            case 4: umma_tap_f16<4>(acc, a, b, idesc, acc_first); break;
            case 3: umma_tap_f16<3>(acc, a, b, idesc, acc_first); break;
            case 2: umma_tap_f16<2>(acc, a, b, idesc, acc_first); break;
            default: umma_tap_f16<1>(acc, a, b, idesc, acc_first); break;
        }
    }
}
// split = 2 converter: the fp16 correction operand of one landed activation tile.  Row r of the second tile =
// [lo16 of the chunk's channels | fp16 of the same channels], 4 bytes per channel, K-major SWIZZLE_128B like the raw tile (16-byte
// unit j of row r sits at unit j ^ (r & 7)).  A thread converts 8 channels of one row: two 16-byte reads, two 16-byte writes; a
// quarter warp covers rows (q, q ^ 5) of an 8-row group, which keeps the four reads and the four writes of both rows on distinct
// bank groups.  cl8 = 8-channel groups in this chunk (4, or last_ksteps in the last chunk); cw = converter warp 0..kConvWarps-1.
__device__ __forceinline__ void convert_tile_f16(const unsigned char *raw, unsigned char *a2, int a_rows, int cl8, int cw, int lane)
{
    const int qw = lane >> 3, u = lane & 7, c8 = u & 3;
    const int rsub = u < 4 ? qw : (qw ^ 5);
    if (c8 >= cl8) return;
    // all reads of the thread first (the stores could alias them for the compiler, and a shared-memory round trip is long while
    // the MMAs of the other stage stream their operands): one latency, not five
    constexpr int kPass = (kARows + kConvWarps * 8 - 1) / (kConvWarps * 8);
    const int r0 = cw * 8 + rsub, x7 = r0 & 7;                        // r & 7 is the same in every pass
    const unsigned char *src = raw + r0 * 128;
    unsigned char *dst = a2 + r0 * 128;
    const int o0 = ((2 * c8) ^ x7) << 4, o1 = ((2 * c8 + 1) ^ x7) << 4;
    const int ol = (c8 ^ x7) << 4, oh = ((cl8 + c8) ^ x7) << 4;
    uint4 v0[kPass], v1[kPass];
#pragma unroll
    for (int k = 0; k < kPass; ++k)
        if (r0 + k * (kConvWarps * 8) < a_rows) {
            v0[k] = *reinterpret_cast<const uint4 *>(src + k * (kConvWarps * 8 * 128) + o0);
            v1[k] = *reinterpret_cast<const uint4 *>(src + k * (kConvWarps * 8 * 128) + o1);
        }
#pragma unroll
    for (int k = 0; k < kPass; ++k)
        if (r0 + k * (kConvWarps * 8) < a_rows) {
            uint4 l, h;
            l.x = lo16x2(v0[k].x, v0[k].y); l.y = lo16x2(v0[k].z, v0[k].w);
            l.z = lo16x2(v1[k].x, v1[k].y); l.w = lo16x2(v1[k].z, v1[k].w);
            h.x = hi16x2(v0[k].x, v0[k].y); h.y = hi16x2(v0[k].z, v0[k].w);
            h.z = hi16x2(v1[k].x, v1[k].y); h.w = hi16x2(v1[k].z, v1[k].w);
            *reinterpret_cast<uint4 *>(dst + k * (kConvWarps * 8 * 128) + ol) = l;
            *reinterpret_cast<uint4 *>(dst + k * (kConvWarps * 8 * 128) + oh) = h;
        }
}

__device__ __forceinline__ void umma_commit_elect(uint32_t bar_addr) {
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(bar_addr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__global__ void __launch_bounds__(kThreads, 1)
conv2d_nhwc_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Params p)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages];
    __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
    __shared__ __align__(8) uint64_t ready_bar[kMaxStages];   // split mode: hi/lo tiles written by the converters
    __shared__ __align__(8) uint64_t afull_bar[kMaxStages];   // split mode: the activation tile landed (the converters start
                                                              // while the 4x larger weight part of the stage is still in flight)
    __shared__ __align__(8) uint64_t tmem_full_bar[2];
    __shared__ __align__(8) uint64_t tmem_empty_bar[2];
    __shared__ __align__(8) uint64_t small_full_bar[2];       // split mode: the per-tile accumulator of the small terms
    __shared__ __align__(8) uint64_t small_empty_bar[2];
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned char *base = reinterpret_cast<unsigned char *>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int b_tap_bytes = p.np * 128;                       // one column tap of the weights: NP rows x 128 B
    const bool conv_mode = p.split == 1 || p.split == 2;      // the converters build a second A tile, two weight blocks
    const int nsplit = conv_mode ? 2 : 1;
    const int T = p.taps;                                     // taps per dimension: 3 (conv) or 1 (GEMM)
    const int a_rows = T == 3 ? kARows : kTileM;
    const int b_off = nsplit * kABytes;                       // stage: [A hi][A lo][B hi (T taps)][B lo (T taps)]
    const int stage_bytes = nsplit * (kABytes + T * b_tap_bytes);
    const int tx_bytes = a_rows * 128 + nsplit * T * b_tap_bytes;   // bytes TMA actually delivers per stage
    const int kStages = p.stages;
    const int acc_stride = p.split ? p.tmem_cols >> 2 : p.tmem_cols >> 1;   // split: 2 chain slots + 2 small-term slots
    const int pitch = p.w + 2;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB);
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); mbar_init(&ready_bar[s], kConvWarps); mbar_init(&afull_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], 4);
            mbar_init(&small_full_bar[a], 1); mbar_init(&small_empty_bar[a], 4);
        }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&tmem_base_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_trigger();                                            // see common.cuh: the next kernel may be scheduled from here on
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            pdl_wait();                                       // first access to the previous kernel's output: the activation tiles
            int s = 0; uint32_t ph = 0;
            int nfill = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
                const int p0 = tile * kTileM;
                for (int kh = 0; kh < T; ++kh)
                    for (int ck = 0; ck < p.nchunks; ++ck) {
                        mbar_wait(&empty_bar[s], ph ^ 1u);
                        unsigned char *sa = base + (size_t)s * stage_bytes;
                        const bool skip_b = (p.dbg & 8) && nfill >= kStages;
                        if (p.trace && blockIdx.x == 0 && nfill < 256) p.trace[nfill * 8 + 0] = clock64();
                        ++nfill;
                        // converter modes: the activation tile completes its own barrier, which is all the converters wait for
                        uint64_t *abar = conv_mode ? &afull_bar[s] : &full_bar[s];
                        if (conv_mode) {
                            mbar_arrive_expect_tx(abar, (uint32_t)(a_rows * 128));
                            if (skip_b) mbar_arrive(&full_bar[s]);
                            else mbar_arrive_expect_tx(&full_bar[s], (uint32_t)(tx_bytes - a_rows * 128));
                        } else {
                            mbar_arrive_expect_tx(&full_bar[s], (uint32_t)(skip_b ? a_rows * 128 : tx_bytes));
                        }
                        tma_load_2d(sa, &tmA, ck * 32, T == 3 ? p0 + (kh - 1) * pitch - 1 : p0, abar);
                        if (!skip_b) {
                        tma_load_3d(sa + b_off, &tmB, ck * 32, 0, kh * T, &full_bar[s]);
                        if (conv_mode) tma_load_3d(sa + b_off + T * b_tap_bytes, &tmB, ck * 32, 0, T * T + kh * T, &full_bar[s]);
                        }
                        if (++s == kStages) { s = 0; ph ^= 1u; }
                    }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // c_format F32, a/b TF32, both K-major, N = np, M = 128
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.np >> 3) << 17) | (8u << 24);
        const uint32_t idesc16 = (1u << 4) | ((uint32_t)(p.np >> 3) << 17) | (8u << 24);     // a/b format F16 (0)
        const uint32_t smem_base = smem_u32(base);
        const uint32_t empty_base = smem_u32(&empty_bar[0]);
        const uint32_t db_tap_step = (uint32_t)(b_tap_bytes >> 4);
        int s = 0; uint32_t ph = 0;
        bool ready = false;
        if (p.split) {
            // two-level accumulation: hi*hi in chains of kGroup stages alternating between TMEM slots 0/1 (drained by the
            // epilogue into registers), the small terms in slot 2 + (tile & 1) for the whole tile
            const uint32_t full_base = smem_u32(&tmem_full_bar[0]);
            const int nst = T * p.nchunks;
            uint32_t it = 0, j = 0;
            int nmma = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++j) {
                const uint32_t sj = j & 1u;
                mbar_wait(&small_empty_bar[sj], ((j >> 1) & 1u) ^ 1u);
                const uint32_t acc_s = tmem_base + (2u + sj) * (uint32_t)acc_stride;
                uint32_t acc_b = 0, slot = 0, first_s = 0u, first_b = 0u;
                int st = 0;
                for (int kh = 0; kh < T; ++kh)
                    for (int ck = 0; ck < p.nchunks; ++ck, ++st) {
                        const int gpos = st % kGroup;
                        if (gpos == 0) {
                            slot = it & 1u;
                            mbar_wait(&tmem_empty_bar[slot], ((it >> 1) & 1u) ^ 1u);
                            acc_b = tmem_base + slot * (uint32_t)acc_stride;
                            first_b = 0u;
                        }
                        if (!ready && conv_mode) mbar_wait(&ready_bar[s], ph);
                        mbar_wait(&full_bar[s], ph);                      // the weights of the stage (split = 3: the whole stage)
                        const bool tr = p.trace && blockIdx.x == 0 && lane == 0 && nmma < 256;
                        if (tr) p.trace[nmma * 8 + 3] = clock64();
                        tc_fence_after();
                        const uint32_t sa = smem_base + (uint32_t)(s * stage_bytes);
                        const uint64_t da = make_desc_sw128(sa), da_lo = make_desc_sw128(sa + (uint32_t)kABytes);
                        const uint64_t db = make_desc_sw128(sa + (uint32_t)b_off);
                        const uint64_t db_lo = make_desc_sw128(sa + (uint32_t)(b_off + T * b_tap_bytes));
                        int sn = s + 1; uint32_t phn = ph;
                        if (sn == kStages) { sn = 0; phn ^= 1u; }
                        ready = conv_mode && mbar_test_wait(&ready_bar[sn], phn);
                        const int ks = ck == p.nchunks - 1 ? p.last_ksteps : 4;
                        if (p.split == 3) {
                            // split16 tile [lo | h] (cl = 8 ks channels): small terms over all 2 cl halves, h * hi16(w) over the
                            // h half (ks 16-byte units in) and the hi16 half of B
                            if (!(p.dbg & 2)) umma_taps3_f16(ks, acc_s, da, db, db_tap_step, idesc16, first_s, T);
                            if (!(p.dbg & 4)) umma_taps3_f16(ks >> 1, acc_b, da + (uint64_t)ks, db, db_tap_step, idesc16, first_b, T);
                        } else if (p.dbg & 2) {
                        } else if (p.split == 2) {
                            // [lo16(x) | fp16(x)] * [hi16(w) ; lo16(w)]: both correction terms, K-concatenated fp16
                            umma_taps3_f16(ks, acc_s, da_lo, db_lo, db_tap_step, idesc16, first_s, T);
                        } else {
                            umma_taps3(ks, acc_s, da_lo, db, db_tap_step, idesc, first_s, T); // lo(x) * hi(w)
                            umma_taps3(ks, acc_s, da, db_lo, db_tap_step, idesc, 1u, T);      // hi(x) * lo(w)
                        }
                        if (!(p.dbg & 4) && p.split != 3)
                        umma_taps3(ks, acc_b, da, db, db_tap_step, idesc, first_b, T);        // hi(x) * hi(w)
                        first_s = 1u; first_b = 1u;
                        umma_commit_elect(empty_base + (uint32_t)(s * 8));
                        if (gpos == kGroup - 1 || st == nst - 1) { umma_commit_elect(full_base + slot * 8u); ++it; }
                        if (tr) p.trace[nmma * 8 + 4] = clock64();
                        ++nmma;
                        s = sn; ph = phn;
                    }
                umma_commit_elect(smem_u32(&small_full_bar[sj]));
            }
        } else {
            int j = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++j) {
                const int slot = j & 1;
                mbar_wait(&tmem_empty_bar[slot], ((uint32_t)(j >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t acc = tmem_base + (uint32_t)(slot * acc_stride);
                uint32_t first = 0u;                              // 0: overwrite the accumulator
                for (int kh = 0; kh < T; ++kh)
                    for (int ck = 0; ck < p.nchunks; ++ck) {
                        if (!ready) mbar_wait(&full_bar[s], ph);
                        tc_fence_after();
                        const uint32_t sa = smem_base + (uint32_t)(s * stage_bytes);
                        const uint64_t da = make_desc_sw128(sa);
                        const uint64_t db = make_desc_sw128(sa + (uint32_t)b_off);
                        int sn = s + 1; uint32_t phn = ph;
                        if (sn == kStages) { sn = 0; phn ^= 1u; }
                        ready = mbar_test_wait(&full_bar[sn], phn);
                        umma_taps3(ck == p.nchunks - 1 ? p.last_ksteps : 4, acc, da, db, db_tap_step, idesc, first, T);
                        umma_commit_elect(empty_base + (uint32_t)(s * 8));
                        first = 1u;
                        s = sn; ph = phn;
                    }
                umma_commit_elect(smem_u32(&tmem_full_bar[slot]));
            }
        }
    } else if (warp >= 6) {
        // ===================== converters (warps 6..9, split modes 1 and 2): hi in place, lo beside it =====================
        if (conv_mode) {
            const int ctid = threadIdx.x - 6 * 32;
            const int n16 = a_rows * 128 / 16;                    // 16-byte words TMA delivered for A
            int s = 0; uint32_t ph = 0;
            int nconv = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x)
                for (int it = 0; it < T * p.nchunks; ++it) {
                    mbar_wait(&afull_bar[s], ph);
                    const bool tr = p.trace && blockIdx.x == 0 && warp == 6 && lane == 0 && nconv < 256;
                    if (tr) p.trace[nconv * 8 + 1] = clock64();
                    uint4 *st = reinterpret_cast<uint4 *>(base + (size_t)s * stage_bytes);
                    uint4 *sl = reinterpret_cast<uint4 *>(base + (size_t)s * stage_bytes + kABytes);
                    if (p.dbg & 1) {
                    } else if (p.split == 2) {
                        convert_tile_f16(reinterpret_cast<const unsigned char *>(st), reinterpret_cast<unsigned char *>(sl), a_rows,
                                         (it % p.nchunks == p.nchunks - 1) ? p.last_ksteps : 4, warp - 6, lane);
                    } else
#pragma unroll 4
                    for (int i = ctid; i < n16; i += kConvWarps * 32) {
                        // hi = trunc_tf32(x): what the MMA reads from the raw tile (no store); lo = rna(x - hi) beside it
                        const uint4 v = st[i];
                        uint4 l;
                        l.x = (__float_as_uint(__uint_as_float(v.x) - __uint_as_float(v.x & 0xFFFFE000u)) + 0x1000u) & 0xFFFFE000u;
                        l.y = (__float_as_uint(__uint_as_float(v.y) - __uint_as_float(v.y & 0xFFFFE000u)) + 0x1000u) & 0xFFFFE000u;
                        l.z = (__float_as_uint(__uint_as_float(v.z) - __uint_as_float(v.z & 0xFFFFE000u)) + 0x1000u) & 0xFFFFE000u;
                        l.w = (__float_as_uint(__uint_as_float(v.w) - __uint_as_float(v.w & 0xFFFFE000u)) + 0x1000u) & 0xFFFFE000u;
                        sl[i] = l;
                    }
                    fence_proxy_async_smem();                     // generic-proxy writes -> visible to the MMA's async proxy
                    __syncwarp();
                    if (tr) p.trace[nconv * 8 + 2] = clock64();
                    ++nconv;
                    if (lane == 0) mbar_arrive(&ready_bar[s]);
                    if (++s == kStages) { s = 0; ph ^= 1u; }
                }
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const long long per_img = (long long)(p.h + 2) * pitch;
        // where row `pix` lands, and whether it carries a value (border pixels of the bordered layout are stored as zeros)
        auto place = [&](long long pix, bool inside, long long &dst, bool &interior) {
            dst = pix; interior = inside;
            if (p.border) {
                const long long rem = pix % per_img;
                const int yy = (int)(rem / pitch), xx = (int)(rem - (long long)yy * pitch);
                interior = inside && yy >= 1 && yy <= p.h && xx >= 1 && xx <= p.w;
            } else if (p.dst_h > 0 && inside) {
                const long long hw = (long long)p.dst_h * p.dst_w, b = pix / hw, rem = pix - b * hw;
                const int yy = (int)(rem / p.dst_w), xx = (int)(rem - (long long)yy * p.dst_w);
                dst = (b * (p.dst_h + 2) + yy + 1) * (p.dst_w + 2) + xx + 1;
            }
        };
        // bias / ReLU / storage format (out_format) / zero border, 16 channels from c0
        auto store16 = [&](const float (&v)[16], long long pix, bool interior, int c0) {
            const float4 *bp = reinterpret_cast<const float4 *>(p.bias + c0);
            float o[16];
#pragma unroll
            for (int i4 = 0; i4 < 4; ++i4) {
                const float4 bv = interior ? __ldg(bp + i4) : make_float4(0.f, 0.f, 0.f, 0.f);
                o[4 * i4] = v[4 * i4] + bv.x; o[4 * i4 + 1] = v[4 * i4 + 1] + bv.y;
                o[4 * i4 + 2] = v[4 * i4 + 2] + bv.z; o[4 * i4 + 3] = v[4 * i4 + 3] + bv.w;
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                if (p.relu) o[i] = fmaxf(o[i], 0.f);
                if (p.out_format == 1) o[i] = __uint_as_float((__float_as_uint(o[i]) + 0x1000u) & 0xFFFFE000u);
                if (!interior) o[i] = 0.f;
            }
            if (p.out_format == 2) {
                split16_store<16>(p.out + pix * p.ldc, p.np, c0, o);
            } else {
                float4 *op = reinterpret_cast<float4 *>(p.out + pix * p.ldc + c0);
#pragma unroll
                for (int i4 = 0; i4 < 4; ++i4) op[i4] = make_float4(o[4 * i4], o[4 * i4 + 1], o[4 * i4 + 2], o[4 * i4 + 3]);
            }
        };
        if (p.split) {
            // two-level accumulation: drain every finished hi*hi chain into registers with round-to-nearest adds, the small
            // terms' accumulator once at the end of the tile
            constexpr int kMaxChunks = 8;                             // NP <= 128
            float acc[kMaxChunks][16];
            const int ngroups = (T * p.nchunks + kGroup - 1) / kGroup;
            const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
            auto drain = [&](uint32_t trow, float scale) {
#pragma unroll
                for (int c = 0; c < kMaxChunks; ++c)
                    if (c * 16 < p.np) {
                        float v[16];
                        tmem_ld16(trow + (uint32_t)(c * 16), v);
#pragma unroll
                        for (int i = 0; i < 16; ++i) acc[c][i] = fmaf(v[i], scale, acc[c][i]);
                    }
                tc_fence_before();
                __syncwarp();
            };
            // split = 2, 3: the correction accumulator holds 2^(11+sw) x the value (see the weight packer); bias[np] = 2^-(11+sw);
            // split = 3: the chains hold 2^sw x the big term; bias[np + 1] = 2^-sw
            const float small_scale = p.split >= 2 ? __ldg(p.bias + p.np) : 1.f;
            const float big_scale = p.split == 3 ? __ldg(p.bias + p.np + 1) : 1.f;
            uint32_t it = 0, j = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++j) {
                const long long pix = (long long)tile * kTileM + r;
                const bool inside = pix < p.P;
                long long dst; bool interior;
                place(pix, inside, dst, interior);
#pragma unroll
                for (int c = 0; c < kMaxChunks; ++c)
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[c][i] = 0.f;
                for (int g = 0; g < ngroups; ++g, ++it) {
                    const uint32_t slot = it & 1u;
                    mbar_wait(&tmem_full_bar[slot], (it >> 1) & 1u);
                    const bool tr = p.trace && blockIdx.x == 0 && warp == 2 && lane == 0 && it < 256;
                    if (tr) p.trace[2048 + it * 2] = clock64();
                    tc_fence_after();
                    drain(lane_base + slot * (uint32_t)acc_stride, big_scale);
                    if (tr) p.trace[2048 + it * 2 + 1] = clock64();
                    if (lane == 0) mbar_arrive(&tmem_empty_bar[slot]);
                }
                const uint32_t sj = j & 1u;
                mbar_wait(&small_full_bar[sj], (j >> 1) & 1u);
                tc_fence_after();
                drain(lane_base + (2u + sj) * (uint32_t)acc_stride, small_scale);
                if (lane == 0) mbar_arrive(&small_empty_bar[sj]);
                if (inside) {
#pragma unroll
                    for (int c = 0; c < kMaxChunks; ++c)
                        if (c * 16 < p.np) store16(acc[c], dst, interior, c * 16);
                }
            }
        } else {
            int j = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++j) {
                const long long pix = (long long)tile * kTileM + r;
                const bool inside = pix < p.P;
                long long dst; bool interior;
                place(pix, inside, dst, interior);
                const int slot = j & 1;
                mbar_wait(&tmem_full_bar[slot], (uint32_t)(j >> 1) & 1u);
                tc_fence_after();
                const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(slot * acc_stride);
                for (int c0 = 0; c0 < p.np; c0 += 16) {
                    float v[16];
                    tmem_ld16(trow + (uint32_t)c0, v);
                    if (inside) store16(v, dst, interior, c0);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty_bar[slot]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}


// =============================================================================================================================
// Pair kernel (3xTF32 mode, NP <= 96): TWO 128-pixel tiles per CTA share every weight stage.
//
// OPT-IN EXPERIMENT (decnet_conv2d_nhwc_set_variant(2)), exact but SLOWER than the kernel above: 81 -> 81 at 180x324, B = 8:
// 497 us against 427 us.  It was built to test the hypothesis that the kernel above is bound by the L2 -> SM traffic of its weight
// tiles (72 KB of hi + lo weights per 17 KB activation tile, re-fetched for every 128-pixel tile: 3 GB per launch at 6.5 TB/s).
// Here the weights of a (row tap, channel chunk) stage are loaded ONCE for two consecutive tiles -- 106 KB instead of 178 KB per
// 72 MMAs -- and the time per tile-stage does not move (4180 cycles either way): the bound is SHARED-MEMORY bandwidth, not L2.
// Per stage the tensor core fetches 36 x 7 KB of operands, TMA writes 89 KB and the converters move 51 KB: 392 KB in 4180 cycles
// = 94 B/clk of the 128 B/clk crossbar (TF32 mode: 83 B/clk; this kernel: 85 B/clk).  Kept as the record of that measurement.
// Structure: a ring of two B slots (hi + lo taps) and a ring of A slots (hi + lo tile each).  TMEM holds four accumulators: per tile the current hi*hi
// chain (drained into registers every kGroup stages by that tile's four epilogue warps while the OTHER tile's MMAs run -- so one
// slot per tile is enough) and the small-term accumulator of the whole tile.
// Warps: 0 TMA producer, 1 MMA issuer, 2-5 epilogue of tile 0, 6-9 epilogue of tile 1, 10-13 converters (448 threads).
// =============================================================================================================================
constexpr int kPairThreads = 448;
constexpr int kPairChunks = 6;                     // NP <= 96: 96 accumulator registers per epilogue thread
constexpr int kMaxASlots = 4;

__global__ void __launch_bounds__(kPairThreads, 1)
conv2d_nhwc_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Params p)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t a_full[kMaxASlots], a_ready[kMaxASlots], a_empty[kMaxASlots];
    __shared__ __align__(8) uint64_t b_full[2], b_empty[2];
    __shared__ __align__(8) uint64_t big_full[2], big_empty[2], small_full[2], small_empty[2];
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned char *base = reinterpret_cast<unsigned char *>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int T = p.taps;
    const int a_rows = T == 3 ? kARows : kTileM;
    const int b_tap_bytes = p.np * 128;
    const int b_slot_bytes = 2 * T * b_tap_bytes;             // hi taps, then lo taps
    const int a_slot_bytes = 2 * kABytes;                     // hi tile, lo tile
    unsigned char *a_base = base + 2 * b_slot_bytes;
    const int NA = p.na_slots;
    const int acc_stride = p.tmem_cols >> 2;                  // big[0], big[1], small[0], small[1]
    const int pitch = p.w + 2;
    const int nst = T * p.nchunks;
    const int num_pairs = (p.num_tiles + 1) >> 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB);
        for (int s = 0; s < NA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_ready[s], kConvWarps); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1);
            mbar_init(&big_full[s], 1); mbar_init(&big_empty[s], 4);
            mbar_init(&small_full[s], 1); mbar_init(&small_empty[s], 4);
        }
        fence_mbar_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&tmem_base_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int sa = 0, sb = 0; uint32_t pha = 0, phb = 0;
            for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x)
                for (int kh = 0; kh < T; ++kh)
                    for (int ck = 0; ck < p.nchunks; ++ck) {
                        mbar_wait(&b_empty[sb], phb ^ 1u);
                        unsigned char *bs = base + (size_t)sb * b_slot_bytes;
                        mbar_arrive_expect_tx(&b_full[sb], (uint32_t)b_slot_bytes);
                        tma_load_3d(bs, &tmB, ck * 32, 0, kh * T, &b_full[sb]);
                        tma_load_3d(bs + T * b_tap_bytes, &tmB, ck * 32, 0, T * T + kh * T, &b_full[sb]);
                        if (++sb == 2) { sb = 0; phb ^= 1u; }
                        for (int m = 0; m < 2; ++m) {
                            const int p0 = (2 * pair + m) * kTileM;      // beyond P for the odd tail: TMA zero-fills
                            mbar_wait(&a_empty[sa], pha ^ 1u);
                            mbar_arrive_expect_tx(&a_full[sa], (uint32_t)(a_rows * 128));
                            tma_load_2d(a_base + (size_t)sa * a_slot_bytes, &tmA, ck * 32,
                                        T == 3 ? p0 + (kh - 1) * pitch - 1 : p0, &a_full[sa]);
                            if (++sa == NA) { sa = 0; pha ^= 1u; }
                        }
                    }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.np >> 3) << 17) | (8u << 24);
        const uint32_t idesc16 = (1u << 4) | ((uint32_t)(p.np >> 3) << 17) | (8u << 24);
        const uint32_t b_base_u = smem_u32(base), a_base_u = smem_u32(a_base);
        const uint32_t db_tap_step = (uint32_t)(b_tap_bytes >> 4);
        int sa = 0, sb = 0; uint32_t pha = 0, phb = 0;
        uint32_t chain[2] = {0u, 0u};
        uint32_t j = 0;
        for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x, ++j) {
            mbar_wait(&small_empty[0], (j & 1u) ^ 1u);
            mbar_wait(&small_empty[1], (j & 1u) ^ 1u);
            uint32_t first_s[2] = {0u, 0u}, first_b[2] = {0u, 0u};
            int st = 0;
            for (int kh = 0; kh < T; ++kh)
                for (int ck = 0; ck < p.nchunks; ++ck, ++st) {
                    const int gpos = st % kGroup;
                    const bool chain_end = gpos == kGroup - 1 || st == nst - 1;
                    mbar_wait(&b_full[sb], phb);
                    const uint32_t sbu = b_base_u + (uint32_t)(sb * b_slot_bytes);
                    const uint64_t db = make_desc_sw128(sbu), db_lo = make_desc_sw128(sbu + (uint32_t)(T * b_tap_bytes));
                    const int ks = ck == p.nchunks - 1 ? p.last_ksteps : 4;
#pragma unroll
                    for (int m = 0; m < 2; ++m) {
                        if (gpos == 0) {
                            mbar_wait(&big_empty[m], (chain[m] & 1u) ^ 1u);     // this tile's previous chain was drained
                            first_b[m] = 0u;
                        }
                        mbar_wait(&a_ready[sa], pha);
                        tc_fence_after();
                        const uint32_t sau = a_base_u + (uint32_t)(sa * a_slot_bytes);
                        const uint64_t da = make_desc_sw128(sau), da_lo = make_desc_sw128(sau + (uint32_t)kABytes);
                        const uint32_t acc_b = tmem_base + (uint32_t)(m * acc_stride);
                        const uint32_t acc_s = tmem_base + (uint32_t)((2 + m) * acc_stride);
                        if (p.split == 2) {
                            umma_taps3_f16(ks, acc_s, da_lo, db_lo, db_tap_step, idesc16, first_s[m], T);  // both corrections, fp16
                        } else {
                            umma_taps3(ks, acc_s, da_lo, db, db_tap_step, idesc, first_s[m], T); // lo(x) * hi(w)
                            umma_taps3(ks, acc_s, da, db_lo, db_tap_step, idesc, 1u, T);        // hi(x) * lo(w)
                        }
                        umma_taps3(ks, acc_b, da, db, db_tap_step, idesc, first_b[m], T);       // hi(x) * hi(w)
                        first_s[m] = 1u; first_b[m] = 1u;
                        umma_commit_elect(smem_u32(&a_empty[sa]));
                        if (chain_end) { umma_commit_elect(smem_u32(&big_full[m])); ++chain[m]; }
                        if (++sa == NA) { sa = 0; pha ^= 1u; }
                    }
                    umma_commit_elect(smem_u32(&b_empty[sb]));
                    if (++sb == 2) { sb = 0; phb ^= 1u; }
                }
            umma_commit_elect(smem_u32(&small_full[0]));
            umma_commit_elect(smem_u32(&small_full[1]));
        }
    } else if (warp >= 10) {
        // ===================== converters (warps 10..13): hi in place, lo beside it =====================
        const int ctid = threadIdx.x - 10 * 32;
        const int n16 = a_rows * 128 / 16;
        int sa = 0; uint32_t pha = 0;
        for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x)
            for (int it = 0; it < 2 * nst; ++it) {
                mbar_wait(&a_full[sa], pha);
                uint4 *sh = reinterpret_cast<uint4 *>(a_base + (size_t)sa * a_slot_bytes);
                uint4 *sl = reinterpret_cast<uint4 *>(a_base + (size_t)sa * a_slot_bytes + kABytes);
                if (p.split == 2) {
                    convert_tile_f16(reinterpret_cast<const unsigned char *>(sh), reinterpret_cast<unsigned char *>(sl), a_rows,
                                     ((it >> 1) % p.nchunks == p.nchunks - 1) ? p.last_ksteps : 4, warp - 10, lane);
                } else
#pragma unroll 4
                for (int i = ctid; i < n16; i += kConvWarps * 32) {
                    const uint4 v = sh[i];
                    uint4 h, l;
                    h.x = (v.x + 0x1000u) & 0xFFFFE000u; h.y = (v.y + 0x1000u) & 0xFFFFE000u;
                    h.z = (v.z + 0x1000u) & 0xFFFFE000u; h.w = (v.w + 0x1000u) & 0xFFFFE000u;
                    l.x = (__float_as_uint(__uint_as_float(v.x) - __uint_as_float(h.x)) + 0x1000u) & 0xFFFFE000u;
                    l.y = (__float_as_uint(__uint_as_float(v.y) - __uint_as_float(h.y)) + 0x1000u) & 0xFFFFE000u;
                    l.z = (__float_as_uint(__uint_as_float(v.z) - __uint_as_float(h.z)) + 0x1000u) & 0xFFFFE000u;
                    l.w = (__float_as_uint(__uint_as_float(v.w) - __uint_as_float(h.w)) + 0x1000u) & 0xFFFFE000u;
                    sh[i] = h;
                    sl[i] = l;
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_ready[sa]);
                if (++sa == NA) { sa = 0; pha ^= 1u; }
            }
    } else {
        // ===================== epilogue: warps 2-5 own tile 0 of the pair, warps 6-9 tile 1 =====================
        const int m = warp >= 6 ? 1 : 0;
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const long long per_img = (long long)(p.h + 2) * pitch;
        const int ngroups = (nst + kGroup - 1) / kGroup;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        float acc[kPairChunks][16];
        uint32_t chain = 0, j = 0;
        for (int pair = blockIdx.x; pair < num_pairs; pair += gridDim.x, ++j) {
            const long long pix = (long long)(2 * pair + m) * kTileM + r;
            const bool inside = pix < p.P;
            long long dst = pix; bool interior = inside;
            if (p.border) {
                const long long rem = pix % per_img;
                const int yy = (int)(rem / pitch), xx = (int)(rem - (long long)yy * pitch);
                interior = inside && yy >= 1 && yy <= p.h && xx >= 1 && xx <= p.w;
            } else if (p.dst_h > 0 && inside) {
                const long long hw = (long long)p.dst_h * p.dst_w, b = pix / hw, rem = pix - b * hw;
                const int yy = (int)(rem / p.dst_w), xx = (int)(rem - (long long)yy * p.dst_w);
                dst = (b * (p.dst_h + 2) + yy + 1) * (p.dst_w + 2) + xx + 1;
            }
#pragma unroll
            for (int c = 0; c < kPairChunks; ++c)
#pragma unroll
                for (int i = 0; i < 16; ++i) acc[c][i] = 0.f;
            auto drain = [&](uint32_t trow, float scale) {
#pragma unroll
                for (int c = 0; c < kPairChunks; ++c)
                    if (c * 16 < p.np) {
                        float v[16];
                        tmem_ld16(trow + (uint32_t)(c * 16), v);
#pragma unroll
                        for (int i = 0; i < 16; ++i) acc[c][i] = fmaf(v[i], scale, acc[c][i]);
                    }
                tc_fence_before();
                __syncwarp();
            };
            for (int g = 0; g < ngroups; ++g, ++chain) {
                mbar_wait(&big_full[m], chain & 1u);
                tc_fence_after();
                drain(lane_base + (uint32_t)(m * acc_stride), 1.f);
                if (lane == 0) mbar_arrive(&big_empty[m]);
            }
            mbar_wait(&small_full[m], j & 1u);
            tc_fence_after();
            drain(lane_base + (uint32_t)((2 + m) * acc_stride), p.split == 2 ? __ldg(p.bias + p.np) : 1.f);
            if (lane == 0) mbar_arrive(&small_empty[m]);
            if (inside) {
#pragma unroll
                for (int c = 0; c < kPairChunks; ++c)
                    if (c * 16 < p.np) {
                        const int c0 = c * 16;
                        const float4 *bp = reinterpret_cast<const float4 *>(p.bias + c0);
                        float4 *op = reinterpret_cast<float4 *>(p.out + dst * p.ldc + c0);
#pragma unroll
                        for (int i4 = 0; i4 < 4; ++i4) {
                            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (interior) {
                                const float4 bv = __ldg(bp + i4);
                                o = make_float4(acc[c][4 * i4] + bv.x, acc[c][4 * i4 + 1] + bv.y, acc[c][4 * i4 + 2] + bv.z,
                                                acc[c][4 * i4 + 3] + bv.w);
                                if (p.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                            }
                            op[i4] = o;
                        }
                    }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

}  // namespace conv2dnhwc
}  // namespace decnet

using namespace decnet;
using namespace decnet::conv2dnhwc;

static thread_local int g_halo_variant = 0;
static thread_local long long *g_halo_trace = nullptr;

extern "C" {

// Shared launcher.  taps = 3: 3x3 conv on the zero-bordered layout [B, h+2, w+2, cp] -> [B, h+2, w+2, ldc] (np channels
// written from out_pad); taps = 1: GEMM over P rows of cp channels (border = 1: the rows are the pixels of such a bordered
// tensor and border rows are stored as zeros; dst_h > 0: the P = B*dst_h*dst_w rows of a flat grid are stored at the interior
// pixels of a bordered [B, dst_h+2, dst_w+2, ldc] tensor).
static int launch_nhwc(const float *x, const float *w_packed, const float *bias, float *out, long long P, int B, int h, int w,
                       int cp, int np, int taps, int border, int relu, int round_out, int split, int ldc, int dst_h, int dst_w,
                       void *stream)
{
    DECNET_REQUIRE(x && w_packed && bias && out, "null pointer");
    DECNET_REQUIRE(P > 0, "non-positive size");
    DECNET_REQUIRE(cp % 8 == 0 && cp >= 8 && cp <= 8192, "cp=%d must be a multiple of 8", cp);
    DECNET_REQUIRE(np % 16 == 0 && np >= 16 && np <= 256, "np=%d must be a multiple of 16 in [16,256]", np);
    DECNET_REQUIRE(split >= 0 && split <= 3, "split must be 0 (TF32), 1 (3xTF32), 2 (TF32 + fp16 corrections) or 3 (split16 input)");
    DECNET_REQUIRE(!split || np <= 128, "split (3xTF32) mode accumulates in registers: np=%d must be <= 128", np);
    DECNET_REQUIRE(split != 3 || cp % 16 == 0, "split16 input needs cp %% 16 == 0, got cp=%d", cp);
    DECNET_REQUIRE(ldc >= np && ldc % 4 == 0, "ldc=%d must be a multiple of 4 and >= np=%d", ldc, np);
    DECNET_REQUIRE(round_out >= 0 && round_out <= 2, "round_out=%d must be 0 (fp32), 1 (TF32-rounded) or 2 (split16)", round_out);
    DECNET_REQUIRE(round_out != 2 || ldc == np, "split16 output needs ldc == np");
    DECNET_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15u) == 0 && (reinterpret_cast<uintptr_t>(w_packed) & 15u) == 0 &&
                   (reinterpret_cast<uintptr_t>(out) & 15u) == 0 && (reinterpret_cast<uintptr_t>(bias) & 15u) == 0,
                   "pointers must be 16-byte aligned");
    Params p{};
    p.bias = bias; p.out = out; p.B = B; p.h = h; p.w = w; p.cp = cp; p.np = np;
    p.taps = taps; p.border = border; p.ldc = ldc; p.dst_h = dst_h; p.dst_w = dst_w;
    p.dbg = g_halo_variant >= 100 ? g_halo_variant - 100 : 0;
    p.trace = g_halo_trace;
    p.nchunks = (cp + 31) / 32;
    p.last_ksteps = (cp - (p.nchunks - 1) * 32) / 8;
    p.P = P;
    DECNET_REQUIRE(p.P + 2ll * (w + 3) < (1ll << 31), "tensor too large for 32-bit TMA coordinates");
    p.relu = relu; p.out_format = round_out; p.split = split;
    const bool conv_mode = split == 1 || split == 2;
    p.tmem_cols = np <= 16 ? 32 : np <= 32 ? 64 : np <= 64 ? 128 : np <= 128 ? 256 : 512;
    if (p.split) p.tmem_cols *= 2;                                  // two chain slots + two small-term slots
    p.num_tiles = (int)((p.P + kTileM - 1) / kTileM);
    const size_t stage_bytes = ((size_t)kABytes + (size_t)taps * np * 128) * (conv_mode ? 2 : 1);
    p.stages = (int)((226 * 1024 - 1024) / stage_bytes);
    if (p.stages > kMaxStages) p.stages = kMaxStages;
    DECNET_REQUIRE(p.stages >= 2, "stage too large (np=%d)", np);
    const size_t smem = (size_t)p.stages * stage_bytes + 1024;
    CUtensorMap tmA, tmB;
    {
        const uint64_t dims[2] = {(uint64_t)cp, (uint64_t)p.P};
        const uint64_t strides[1] = {(uint64_t)cp * 4};
        const uint32_t box[2] = {32u, (uint32_t)(taps == 3 ? kARows : kTileM)};
        int rc = encode_tensor_map(&tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, x, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
        if (rc) return rc;
    }
    {
        const uint64_t dims[3] = {(uint64_t)cp, (uint64_t)np, (uint64_t)(taps * taps * (conv_mode ? 2 : 1))};
        const uint64_t strides[2] = {(uint64_t)cp * 4, (uint64_t)np * cp * 4};
        const uint32_t box[3] = {32u, (uint32_t)np, (uint32_t)taps};
        int rc = encode_tensor_map(&tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, w_packed, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
        if (rc) return rc;
    }
    {
        static std::mutex mu;
        static size_t set_for[64] = {0};
        int dev = 0;
        DECNET_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> lk(mu);
        if (dev < 0 || dev >= 64 || set_for[dev] < smem) {
            DECNET_CUDA(cudaFuncSetAttribute(conv2d_nhwc_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            if (dev >= 0 && dev < 64) set_for[dev] = smem;
        }
    }
    const int sms = sm_count_cached();
    // opt-in (variant 2): two tiles per CTA share each weight stage (pair kernel; exact, measured slower: see its header)
    if (conv_mode && np <= 16 * kPairChunks && p.num_tiles >= 2 * sms && g_halo_variant == 2 && !round_out) {
        const size_t b_slot = (size_t)2 * taps * np * 128, a_slot = (size_t)2 * kABytes;
        int na = (int)((226 * 1024 - 1024 - 2 * b_slot) / a_slot);
        if (na > kMaxASlots) na = kMaxASlots;
        if (na >= 2) {
            p.na_slots = na;
            p.tmem_cols = np <= 8 ? 32 : np <= 16 ? 64 : np <= 32 ? 128 : np <= 64 ? 256 : 512;       // 4 accumulators
            const size_t smem2 = 2 * b_slot + (size_t)na * a_slot + 1024;
            static std::mutex mu2;
            static size_t set_for2[64] = {0};
            int dev = 0;
            DECNET_CUDA(cudaGetDevice(&dev));
            {
                std::lock_guard<std::mutex> lk(mu2);
                if (dev < 0 || dev >= 64 || set_for2[dev] < smem2) {
                    DECNET_CUDA(cudaFuncSetAttribute(conv2d_nhwc_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
                    if (dev >= 0 && dev < 64) set_for2[dev] = smem2;
                }
            }
            const int pairs = (p.num_tiles + 1) / 2;
            conv2d_nhwc_pair_kernel<<<(unsigned)(pairs < sms ? pairs : sms), kPairThreads, smem2, static_cast<cudaStream_t>(stream)>>>(tmA, tmB, p);
            return after_launch("conv2d_nhwc_pair_kernel");
        }
    }
    const unsigned grid = (unsigned)(p.num_tiles < sms ? p.num_tiles : sms);
    DECNET_CUDA(launch_pdl(conv2d_nhwc_halo_kernel, dim3(grid), dim3(kThreads), smem, static_cast<cudaStream_t>(stream), tmA, tmB, p));
    return after_launch("conv2d_nhwc_halo_kernel");
}

// 0 / 1 = the one-tile-per-CTA kernel (default); 2 = pair kernel for 3xTF32 launches with >= 2 tiles per SM and np <= 96.  Per thread.
void decnet_conv2d_nhwc_set_variant(int variant) { g_halo_variant = variant; }
// tuning only: device buffer of 2560 int64 that CTA 0 of the following launches fills with its clock64 timeline, or null.  Per thread.
void decnet_conv2d_nhwc_debug_trace(void *buffer) { g_halo_trace = static_cast<long long *>(buffer); }

int decnet_conv2d_tc_nhwc_halo(const float *x_pad, const float *w_packed, const float *bias, float *out_pad,
                               int B, int h, int w, int cp, int np, int relu, int round_out, int split, void *stream)
{
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0, "non-positive size");
    return launch_nhwc(x_pad, w_packed, bias, out_pad, (long long)B * (h + 2) * (w + 2), B, h, w, cp, np, 3, 1, relu,
                       round_out, split, np, 0, 0, stream);
}

int decnet_conv2d_tc_nhwc_halo_ldc(const float *x_pad, const float *w_packed, const float *bias, float *out_pad,
                                   int B, int h, int w, int cp, int np, int ldc, int relu, int split, void *stream)
{
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0, "non-positive size");
    return launch_nhwc(x_pad, w_packed, bias, out_pad, (long long)B * (h + 2) * (w + 2), B, h, w, cp, np, 3, 1, relu, 0, split,
                       ldc, 0, 0, stream);
}

int decnet_gemm_tc_nhwc(const float *x, const float *w_packed, const float *bias, float *out, long long P, int cp, int np,
                        int ldc, int relu, int split, int border_B, int border_h, int border_w, int dst_h, int dst_w, void *stream)
{
    const int border = border_B > 0 ? 1 : 0;
    if (border)
        DECNET_REQUIRE(P == (long long)border_B * (border_h + 2) * (border_w + 2) && dst_h == 0,
                       "bordered rows: P=%lld must be B*(h+2)*(w+2)", P);
    if (dst_h > 0) DECNET_REQUIRE(dst_w > 0 && P % ((long long)dst_h * dst_w) == 0, "P=%lld is not a whole number of %dx%d grids", P, dst_h, dst_w);
    return launch_nhwc(x, w_packed, bias, out, P, border_B, border_h, border ? border_w : 0, cp, np, 1, border, relu, 0, split, ldc,
                       dst_h, dst_w, stream);
}

int decnet_conv2d_tf32_nhwc_halo(const float *x_pad, const float *w_packed, const float *bias, float *out_pad,
                                 int B, int h, int w, int cp, int np, int relu, int round_out_tf32, void *stream)
{
    return decnet_conv2d_tc_nhwc_halo(x_pad, w_packed, bias, out_pad, B, h, w, cp, np, relu, round_out_tf32, 0, stream);
}

}  // extern "C"
