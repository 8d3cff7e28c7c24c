// decnet_b200/csrc/codec.cu -- SURVEY.md section 8f rank 4: the data formats either side of the path, on the device.
//   image_prepare_u8 : uint8 RGB HWC image -> top/left zero pad to the network size (demo.py:75-81 `padding`), /255
//                      (the input of detailDetection, demo.py:158-162) and ToTensor + Normalize(mean, std)
//                      (demo.py:82-88 `transform`), NCHW fp32 -- one pass, a quarter of the upload bytes of fp32 images.
//   disp_to_u16      : the KITTI-style 16-bit disparity image demo.py:191-197 writes: clamp(pred * 256, 0, 65535)
//                      truncated to uint16, cropped to the last ori_h rows / ori_w columns (the PNG deflate stays on the host).
//   epe_3px          : modules/loss.py:427-437 `test_loss_func`: EPE and 3-px / 5 % error over 0 < gt < max_disp.
//   mirror_swap_u8   : the input of the reverse direction of StereoMatcher's left-right check: (mirror(right), mirror(left)).
//   lr_check         : the left-right consistency check itself, on the forward and mirrored reverse predictions.
//   lr_check_fill    : the check fused with background hole filling of the pixels it rejects (oracle/lr_fill.py): a row
//                      pass (check + nearest valid neighbours in the row) and a pass over the rows without a valid pixel.
//                      None of the last three has a counterpart in the reference.
#include "common.cuh"
#include <algorithm>
#include <cstdint>

namespace decnet {
namespace codec {

constexpr int kBlock = 256;

__global__ void __launch_bounds__(kBlock)
image_prepare_u8_kernel(const unsigned char *__restrict__ img, float *__restrict__ out01, float *__restrict__ norm,
                        float m0, float m1, float m2, float s0, float s1, float s2, int h, int w, int H, int W, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;      // over B*H*W padded pixels
    if (i >= n) return;
    const int x = (int)(i % W), y = (int)((i / W) % H);
    const long long b = i / ((long long)W * H);
    const int ry = H - h, rx = W - w;                                      // residual rows / columns come FIRST
    float v[3] = {0.f, 0.f, 0.f};
    if (y >= ry && x >= rx) {
        const unsigned char *p = img + ((b * h + (y - ry)) * (long long)w + (x - rx)) * 3;
        v[0] = __fdiv_rn((float)p[0], 255.f); v[1] = __fdiv_rn((float)p[1], 255.f); v[2] = __fdiv_rn((float)p[2], 255.f);
    }
    const long long plane = (long long)H * W, o = b * 3 * plane + (long long)y * W + x;
    if (out01) { out01[o] = v[0]; out01[o + plane] = v[1]; out01[o + 2 * plane] = v[2]; }
    if (norm) {
        norm[o] = __fdiv_rn(__fsub_rn(v[0], m0), s0);
        norm[o + plane] = __fdiv_rn(__fsub_rn(v[1], m1), s1);
        norm[o + 2 * plane] = __fdiv_rn(__fsub_rn(v[2], m2), s2);
    }
}

// demo.py:191-197 for one value: clamp(d * 256, 0, 65535) truncated; shared by disp_to_u16, lr_check and the fill kernels.
__device__ __forceinline__ unsigned short disp_u16(float d)
{
    float v = __fmul_rn(d, 256.f);
    v = v < 0.f ? 0.f : v;                                                 // also sends NaN comparisons' false branch through
    v = v > 65535.f ? 65535.f : v;
    return (unsigned short)(v == v ? v : 0.f);                             // truncation like numpy's astype('uint16')
}

__global__ void __launch_bounds__(kBlock)
disp_to_u16_kernel(const float *__restrict__ pred, unsigned short *__restrict__ out, int H, int W, int oh, int ow, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;      // over B*oh*ow cropped pixels
    if (i >= n) return;
    const int x = (int)(i % ow), y = (int)((i / ow) % oh);
    const long long b = i / ((long long)ow * oh);
    out[i] = disp_u16(pred[(b * H + (H - oh + y)) * (long long)W + (W - ow + x)]);
}

// Reverse order of 4 RGB pixels held in 3 little-endian words: pixel k is bytes 3k..3k+2 of (a, b, c).
__device__ __forceinline__ void reverse4(unsigned a, unsigned b, unsigned c, unsigned &o0, unsigned &o1, unsigned &o2)
{
    o0 = __byte_perm(c, b, 0x6321);                                        // p3 (c1 c2 c3), p2[0] (b2)
    o1 = __byte_perm(__byte_perm(b, c, 0x0043), a, 0x3710);                // p2[1..2] (b3 c0), p1[0..1] (a3 b0)
    o2 = __byte_perm(b, a, 0x6541);                                        // p1[2] (b1), p0 (a0 a1 a2)
}

// out_left = mirror(right), out_right = mirror(left) on uint8 RGB [B,h,w,3].  Each thread writes P output pixels of one row
// (view 0: out_left, view 1: out_right): P = 16 as three 16-byte accesses, P = 4 as three words, P = 1 byte by byte.
template <int P>
__global__ void __launch_bounds__(kBlock)
mirror_swap_u8_kernel(const unsigned char *__restrict__ left, const unsigned char *__restrict__ right,
                      unsigned char *__restrict__ out_left, unsigned char *__restrict__ out_right, int w, long long rows)
{
    const int nc = w / P;                                                  // chunks per row (w % P == 0)
    const long long per_view = rows * nc;
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (i >= 2 * per_view) return;
    const int view = (int)(i / per_view);
    const long long j = i - view * per_view, row = j / nc;
    const int c = (int)(j - row * nc);
    const unsigned char *src = (view ? left : right) + (row * w + (w - (c + 1) * P)) * 3;    // the mirrored chunk, read forward
    unsigned char *dst = (view ? out_right : out_left) + (row * w + c * P) * 3;
    if constexpr (P == 16) {
        const uint4 *s = reinterpret_cast<const uint4 *>(src);
        const uint4 v0 = __ldg(s), v1 = __ldg(s + 1), v2 = __ldg(s + 2);
        const unsigned in[12] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w};
        unsigned o[12];
#pragma unroll
        for (int g = 0; g < 4; ++g)                                        // output group g = reversed input group 3 - g
            reverse4(in[9 - 3 * g], in[10 - 3 * g], in[11 - 3 * g], o[3 * g], o[3 * g + 1], o[3 * g + 2]);
        uint4 *d = reinterpret_cast<uint4 *>(dst);
        d[0] = make_uint4(o[0], o[1], o[2], o[3]);
        d[1] = make_uint4(o[4], o[5], o[6], o[7]);
        d[2] = make_uint4(o[8], o[9], o[10], o[11]);
    } else if constexpr (P == 4) {
        const unsigned *s = reinterpret_cast<const unsigned *>(src);
        unsigned *d = reinterpret_cast<unsigned *>(dst);
        unsigned o0, o1, o2;
        reverse4(__ldg(s), __ldg(s + 1), __ldg(s + 2), o0, o1, o2);
        d[0] = o0; d[1] = o1; d[2] = o2;
    } else {
        dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
    }
}

// Whether one cropped pixel passes the left-right check (oracle/lr_check.py): x is its column in the crop, rev the padded row
// of the mirrored reverse prediction, whose value at crop column u sits at padded column W-1-u.
// dl = fwd[W - ow + x] is the forward value, loaded by the caller.  Shared by lr_check and lr_check_fill_rows.
__device__ __forceinline__ bool lr_valid(float dl, const float *rev, int W, int ow, int x, float tol)
{
    const float u = floorf(__fadd_rn(__fsub_rn((float)x, dl), 0.5f));      // NaN / inf dl fail every test below
    const bool inside = isfinite(dl) && u >= 0.f && u < (float)ow;
    const float dr = rev[W - 1 - (inside ? (int)u : 0)];                   // unconditional: a caller's loads can overlap
    return inside && fabsf(__fsub_rn(dl, dr)) <= tol;                      // NaN dr: false
}

// Left-right consistency check over the cropped pixels of the forward half of pred [2B,H,W]; the reverse half holds the
// mirrored run.
__global__ void __launch_bounds__(kBlock)
lr_check_kernel(const float *__restrict__ pred, int B, int H, int W, int oh, int ow, float tol, float *__restrict__ out_f32,
                unsigned short *__restrict__ out_u16, unsigned char *__restrict__ out_valid, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;      // over B*oh*ow cropped pixels
    if (i >= n) return;
    const int x = (int)(i % ow), y = (int)((i / ow) % oh);
    const long long b = i / ((long long)ow * oh);
    const float *fwd = pred + (b * H + (H - oh + y)) * (long long)W;
    const float *rev = pred + ((b + B) * H + (H - oh + y)) * (long long)W;
    const float dl = fwd[W - ow + x];
    const bool valid = lr_valid(dl, rev, W, ow, x, tol);
    if (out_f32) out_f32[i] = valid ? dl : 0.f;
    if (out_u16) out_u16[i] = valid ? disp_u16(dl) : (unsigned short)0;
    if (out_valid) out_valid[i] = valid ? 1 : 0;
}

// Background hole filling (oracle/lr_fill.py), row phase, fused with the check: one CTA per cropped row (b, y).  An invalid
// pixel takes the smaller value of its nearest valid neighbours L (left) and R (right) in the row -- R's only when strictly
// smaller, so ties keep L's bits -- or the one that exists; valid pixels keep dl.
// The row is processed in chunks of kFillChunk columns, thread t owning columns c0 + i*kBlock + t.  Per chunk the checked
// values are staged in shared memory and the validity as one warp ballot per 32 columns; L and R come from a block-wide max
// scan of valid column indices (carried from the previous chunks) and a min scan (carrying in the first valid column after
// the chunk).  A row of up to kFillChunk columns (every row up to Middlebury's 2916 px) is one chunk and one pass over the
// predictions.  For a wider row that first valid column after the chunk comes from a look-ahead that recomputes the check
// ahead of the chunk; it only moves forward, so the row is swept at most twice.  A neighbour outside the chunk is valid, so
// its value is its forward prediction, read back from pred.
// out_f32 always receives the row-phase values (0 on a row without a valid pixel: lr_fill_empty_rows_kernel reads them),
// out_u16 / out_valid when requested, row_flags[b*oh + y] whether the row has a valid pixel.
constexpr int kFillItems = 16;                                             // columns per thread per chunk
constexpr int kFillChunk = kBlock * kFillItems;                            // 4096 columns, 16 KB of staged values
constexpr int kFillWarps = kBlock / 32;

__global__ void __launch_bounds__(kBlock)
lr_check_fill_rows_kernel(const float *__restrict__ pred, int B, int H, int W, int oh, int ow, float tol,
                          float *__restrict__ out_f32, unsigned short *__restrict__ out_u16,
                          unsigned char *__restrict__ out_valid, unsigned char *__restrict__ row_flags)
{
    __shared__ float sv[kFillChunk];                                       // checked values of the chunk (dl where valid)
    __shared__ unsigned sbits[kFillItems * kFillWarps];                    // validity: ballot of entry e = i*kFillWarps + warp
    __shared__ int spre[kFillItems * kFillWarps];                          // last valid column before entry e (-1: none)
    __shared__ int ssuf[kFillItems * kFillWarps];                          // first valid column after entry e (ow: none)
    __shared__ int scarry, snext;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const long long row = blockIdx.x;                                      // b * oh + y
    const long long b = row / oh;
    const int y = (int)(row - b * oh);
    const float *fwd = pred + (b * H + (H - oh + y)) * (long long)W;
    const float *rev = pred + ((b + B) * H + (H - oh + y)) * (long long)W;
    const float *fwd_crop = fwd + (W - ow);
    const long long o = row * ow;
    int carry = -1;                                                        // last valid column left of the chunk
    int next = -1;                                                         // first valid column >= the chunk's end, once known

    for (int c0 = 0; c0 < ow; c0 += kFillChunk) {
        const int c1 = min(c0 + kFillChunk, ow);
        if (c1 == ow) {
            next = ow;
        } else if (next < c1) {                                            // look ahead (rows wider than one chunk only)
            if (t == 0) snext = ow;
            __syncthreads();
            for (int a = c1; a < ow; a += kFillChunk) {
                int m = ow;
#pragma unroll 1
                for (int i = 0; i < kFillItems; ++i) {                     // a thread's columns ascend: its first hit is its min
                    const int x = a + i * kBlock + t;
                    if (x < ow && lr_valid(fwd_crop[x], rev, W, ow, x, tol)) { m = x; break; }
                }
                m = __reduce_min_sync(0xffffffffu, m);
                if (lane == 0) atomicMin(&snext, m);
                __syncthreads();
                next = snext;
                __syncthreads();                                           // every thread has read snext before the next atomics
                if (next < ow) break;
            }
        }
        const int nseg = (c1 - c0 + kBlock - 1) / kBlock, nent = nseg * kFillWarps;
        unsigned vmask = 0;                                                // bit i: column c0 + i*kBlock + t is valid
        for (int i0 = 0; i0 < nseg; i0 += 4) {                             // 4 columns per thread, their loads in flight together
            float d[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) d[k] = fwd_crop[min(c0 + (i0 + k) * kBlock + t, ow - 1)];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int x = c0 + (i0 + k) * kBlock + t, xc = min(x, ow - 1);
                const bool v = (x < ow) & lr_valid(d[k], rev, W, ow, xc, tol);
                vmask |= (unsigned)v << (i0 + k);
                sv[(i0 + k) * kBlock + t] = v ? d[k] : 0.f;
            }
        }
#pragma unroll
        for (int i = 0; i < kFillItems; ++i) {
            if (i >= nseg) break;
            const unsigned bits = __ballot_sync(0xffffffffu, (vmask >> i) & 1u);
            if (lane == 0) sbits[i * kFillWarps + warp] = bits;
        }
        __syncthreads();
        if (warp < 2) {                                                    // warp 0: exclusive max scan, warp 1: min scan
            // lane l owns entries 4l..4l+3 (column order); entry e covers columns c0 + (e / kFillWarps)*kBlock + (e % kFillWarps)*32 + 0..31
            int agg[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int e = 4 * lane + k;
                const unsigned bits = e < nent ? sbits[e] : 0u;
                const int base = c0 + (e / kFillWarps) * kBlock + (e % kFillWarps) * 32;
                agg[k] = warp == 0 ? (bits ? base + 31 - __clz(bits) : -1) : (bits ? base + __ffs(bits) - 1 : ow);
            }
            if (warp == 0) {
                const int tot = max(max(agg[0], agg[1]), max(agg[2], agg[3]));
                int incl = tot;
                for (int s = 1; s < 32; s <<= 1) {
                    const int u = __shfl_up_sync(0xffffffffu, incl, s);
                    if (lane >= s) incl = max(incl, u);
                }
                int run = max(carry, __shfl_up_sync(0xffffffffu, incl, 1));
                if (lane == 0) run = carry;
#pragma unroll
                for (int k = 0; k < 4; ++k) { spre[4 * lane + k] = run; run = max(run, agg[k]); }
                if (lane == 31) scarry = run;
            } else {
                const int tot = min(min(agg[0], agg[1]), min(agg[2], agg[3]));
                int incl = tot;
                for (int s = 1; s < 32; s <<= 1) {
                    const int u = __shfl_down_sync(0xffffffffu, incl, s);
                    if (lane + s < 32) incl = min(incl, u);
                }
                int run = min(next, __shfl_down_sync(0xffffffffu, incl, 1));
                if (lane == 31) run = next;
#pragma unroll
                for (int k = 3; k >= 0; --k) { ssuf[4 * lane + k] = run; run = min(run, agg[k]); }
            }
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < kFillItems; ++i) {
            const int x = c0 + i * kBlock + t;
            if (i >= nseg || x >= ow) break;
            const int e = i * kFillWarps + warp, base = x - lane;
            const unsigned bits = sbits[e];
            const bool v = (bits >> lane) & 1u;
            float d = sv[x - c0];
            if (!v) {
                const unsigned lo = bits & ((1u << lane) - 1u), hi = bits & ~((2u << lane) - 1u);
                const int L = lo ? base + 31 - __clz(lo) : spre[e];
                const int R = hi ? base + __ffs(hi) - 1 : ssuf[e];
                const float dL = L < 0 ? 0.f : L >= c0 ? sv[L - c0] : fwd_crop[L];
                const float dR = R >= ow ? 0.f : R < c1 ? sv[R - c0] : fwd_crop[R];
                d = L < 0 ? dR : R >= ow ? dL : dR < dL ? dR : dL;         // neither: a row without a valid pixel, 0
            }
            out_f32[o + x] = d;
            if (out_u16) out_u16[o + x] = disp_u16(d);
            if (out_valid) out_valid[o + x] = v ? 1 : 0;
        }
        carry = scarry;
        __syncthreads();                                                   // sv, sbits and scarry are rewritten by the next chunk
    }
    if (t == 0) row_flags[row] = carry >= 0 ? 1 : 0;
}

// Background hole filling, column phase: a row without a valid pixel (row_flags 0) in an image that has a non-empty row takes,
// column by column, the smaller row-phase value of the nearest non-empty rows A (above) and C (below) -- C's only when
// strictly smaller -- or the one that exists.  One CTA per cropped row; non-empty rows, the common case, exit at once.  It
// reads the neighbours from the float rows the row phase wrote (the wrapper allocates them when only uint16 was asked for)
// and writes disp_u16 of the chosen value: reading the uint16 rows instead would also be exact, since disp_u16 is monotone,
// but would not give the float output.
__global__ void __launch_bounds__(kBlock)
lr_fill_empty_rows_kernel(int oh, int ow, float *__restrict__ out_f32, unsigned short *__restrict__ out_u16,
                          const unsigned char *__restrict__ row_flags)
{
    const long long row = blockIdx.x;
    if (row_flags[row]) return;
    __shared__ int sa, sc;
    const int t = threadIdx.x;
    const long long b = row / oh;
    const int y = (int)(row - b * oh);
    const unsigned char *flags = row_flags + b * oh;
    if (t == 0) { sa = -1; sc = oh; }
    __syncthreads();
    int a = -1, c = oh;
    for (int yy = t; yy < oh; yy += kBlock)
        if (flags[yy]) {
            if (yy < y) a = yy;                                            // ascending: the last hit above is the nearest
            else if (c == oh) c = yy;
        }
    a = __reduce_max_sync(0xffffffffu, a);
    c = __reduce_min_sync(0xffffffffu, c);
    if ((t & 31) == 0) { atomicMax(&sa, a); atomicMin(&sc, c); }
    __syncthreads();
    a = sa; c = sc;
    if (a < 0 && c == oh) return;                                          // no valid pixel in the image: it stays 0
    const float *ra = out_f32 + (b * oh + max(a, 0)) * (long long)ow, *rc = out_f32 + (b * oh + min(c, oh - 1)) * (long long)ow;
    const long long o = row * ow;
    for (int x = t; x < ow; x += kBlock) {
        const float da = a < 0 ? 0.f : ra[x], dc = c == oh ? 0.f : rc[x];
        const float d = a < 0 ? dc : c == oh ? da : dc < da ? dc : da;
        out_f32[o + x] = d;
        if (out_u16) out_u16[o + x] = disp_u16(d);
    }
}

__global__ void __launch_bounds__(kBlock)
epe_3px_kernel(const float *__restrict__ pred, const float *__restrict__ gt, float max_disp, double *__restrict__ sums, long long n)
{
    double e = 0.0, ok = 0.0, cnt = 0.0;
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < n; i += (long long)gridDim.x * kBlock) {
        const float g = gt[i];
        if (g < max_disp && g > 0.f) {
            const float err = fabsf(pred[i] - g);
            e += err; cnt += 1.0;
            ok += (err < 3.f || err < 0.05f * g) ? 1.0 : 0.0;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        e += __shfl_xor_sync(0xffffffffu, e, o); ok += __shfl_xor_sync(0xffffffffu, ok, o); cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sums[0], e); atomicAdd(&sums[1], ok); atomicAdd(&sums[2], cnt); }
}

}  // namespace codec
}  // namespace decnet

using namespace decnet;
using namespace decnet::codec;

extern "C" {

int decnet_image_prepare_u8(const unsigned char *img_hwc, float *out01, float *out_norm, const float *mean3_host,
                            const float *std3_host, int B, int h, int w, int H, int W, void *stream)
{
    DECNET_REQUIRE(img_hwc && (out01 || out_norm) && mean3_host && std3_host, "null pointer");
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0 && H >= h && W >= w, "padded size %dx%d must cover the image %dx%d", H, W, h, w);
    const long long n = (long long)B * H * W;
    image_prepare_u8_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
        img_hwc, out01, out_norm, mean3_host[0], mean3_host[1], mean3_host[2], std3_host[0], std3_host[1], std3_host[2], h, w, H, W, n);
    return after_launch("image_prepare_u8_kernel");
}

int decnet_disp_to_u16(const float *pred, unsigned short *out, int B, int H, int W, int ori_h, int ori_w, void *stream)
{
    DECNET_REQUIRE(pred && out, "null pointer");
    DECNET_REQUIRE(B > 0 && ori_h > 0 && ori_w > 0 && ori_h <= H && ori_w <= W, "crop %dx%d outside the %dx%d map", ori_h, ori_w, H, W);
    const long long n = (long long)B * ori_h * ori_w;
    disp_to_u16_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(pred, out, H, W, ori_h, ori_w, n);
    return after_launch("disp_to_u16_kernel");
}

int decnet_mirror_swap_u8(const unsigned char *left, const unsigned char *right, unsigned char *out_left,
                          unsigned char *out_right, int B, int h, int w, void *stream)
{
    DECNET_REQUIRE(left && right && out_left && out_right, "null pointer");
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0, "empty image batch %dx%dx%d", B, h, w);
    const long long rows = (long long)B * h;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    auto aligned = [&](unsigned a) {
        return ((reinterpret_cast<uintptr_t>(left) | reinterpret_cast<uintptr_t>(right) | reinterpret_cast<uintptr_t>(out_left) |
                 reinterpret_cast<uintptr_t>(out_right)) & (a - 1)) == 0;
    };
    auto grid = [&](int P) { return (unsigned)((2 * rows * (w / P) + kBlock - 1) / kBlock); };
    if (w % 16 == 0 && aligned(16))                                        // rows and chunks start at multiples of 48 bytes
        mirror_swap_u8_kernel<16><<<grid(16), kBlock, 0, st>>>(left, right, out_left, out_right, w, rows);
    else if (w % 4 == 0 && aligned(4))
        mirror_swap_u8_kernel<4><<<grid(4), kBlock, 0, st>>>(left, right, out_left, out_right, w, rows);
    else
        mirror_swap_u8_kernel<1><<<grid(1), kBlock, 0, st>>>(left, right, out_left, out_right, w, rows);
    return after_launch("mirror_swap_u8_kernel");
}

int decnet_lr_check(const float *pred, int B, int H, int W, int ori_h, int ori_w, float tol, float *out_f32,
                    unsigned short *out_u16, unsigned char *out_valid, void *stream)
{
    DECNET_REQUIRE(pred && (out_f32 || out_u16 || out_valid), "null prediction or no output requested");
    DECNET_REQUIRE(B > 0 && ori_h > 0 && ori_w > 0 && ori_h <= H && ori_w <= W, "crop %dx%d outside the %dx%d map", ori_h, ori_w, H, W);
    DECNET_REQUIRE(tol >= 0.f && tol <= 3.402823466e38f, "tolerance must be finite and >= 0");
    const long long n = (long long)B * ori_h * ori_w;
    lr_check_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
        pred, B, H, W, ori_h, ori_w, tol, out_f32, out_u16, out_valid, n);
    return after_launch("lr_check_kernel");
}

int decnet_lr_check_fill(const float *pred, int B, int H, int W, int ori_h, int ori_w, float tol, float *out_f32,
                         unsigned short *out_u16, unsigned char *out_valid, unsigned char *row_flags, void *stream)
{
    DECNET_REQUIRE(pred && out_f32 && row_flags, "null prediction, float rows or row flags");
    DECNET_REQUIRE(B > 0 && ori_h > 0 && ori_w > 0 && ori_h <= H && ori_w <= W, "crop %dx%d outside the %dx%d map", ori_h, ori_w, H, W);
    DECNET_REQUIRE(tol >= 0.f && tol <= 3.402823466e38f, "tolerance must be finite and >= 0");
    const long long rows = (long long)B * ori_h;
    DECNET_REQUIRE(rows <= 0x7fffffffLL, "%lld rows exceed the grid", rows);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    lr_check_fill_rows_kernel<<<(unsigned)rows, kBlock, 0, st>>>(pred, B, H, W, ori_h, ori_w, tol, out_f32, out_u16, out_valid,
                                                                 row_flags);
    if (int s = after_launch("lr_check_fill_rows_kernel")) return s;
    lr_fill_empty_rows_kernel<<<(unsigned)rows, kBlock, 0, st>>>(ori_h, ori_w, out_f32, out_u16, row_flags);
    return after_launch("lr_fill_empty_rows_kernel");
}

int decnet_epe_3px(const float *pred, const float *gt, float max_disp, double *sums3, long long n, void *stream)
{
    DECNET_REQUIRE(pred && gt && sums3 && n > 0, "null pointer or empty input");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DECNET_CUDA(cudaMemsetAsync(sums3, 0, 3 * sizeof(double), st));
    epe_3px_kernel<<<(unsigned)std::min<long long>((n + kBlock - 1) / kBlock, 148 * 8), kBlock, 0, st>>>(pred, gt, max_disp, sums3, n);
    return after_launch("epe_3px_kernel");
}

}  // extern "C"
