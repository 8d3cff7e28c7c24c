// decnet_b200/csrc/codec.cu -- SURVEY.md section 8f rank 4: the data formats either side of the path, on the device.
//   image_prepare_u8 : uint8 RGB HWC image -> top/left zero pad to the network size (demo.py:75-81 `padding`), /255
//                      (the input of detailDetection, demo.py:158-162) and ToTensor + Normalize(mean, std)
//                      (demo.py:82-88 `transform`), NCHW fp32 -- one pass, a quarter of the upload bytes of fp32 images.
//                      Its _shift form reads the image shifted by a column offset: the right view of a search range
//                      [min_disp, max_disp) that does not start at 0.
//   disp_add         : the minimum disparity added back to the prediction of that shifted search (fp32, rounded to nearest).
//   disp_to_u16      : the KITTI-style 16-bit disparity image demo.py:191-197 writes: clamp(pred * 256, 0, 65535)
//                      truncated to uint16, cropped to the last ori_h rows / ori_w columns (the PNG deflate stays on the host).
//   epe_3px          : modules/loss.py:427-437 `test_loss_func`: EPE and 3-px / 5 % error over 0 < gt < max_disp.
//   mirror_swap_u8   : the input of the reverse direction of StereoMatcher's left-right check: (mirror(right), mirror(left)).
//   lr_check         : the left-right consistency check itself, on the forward and mirrored reverse predictions.
//   lr_check_fill    : the check fused with background hole filling of the pixels it rejects (oracle/lr_fill.py): a row
//                      pass (check + nearest valid neighbours in the row) and a pass over the rows without a valid pixel.
//   lr_check_guided_fill : lr_check_fill, then edge-aware filling guided by the left image (oracle/lr_guided.py): three
//                      iterations of tridiagonal solves along every row and every column, and a compose pass.
//   lr_check_speckle : the check, then a speckle filter (oracle/lr_speckle.py: small connected regions invalidated) by a
//                      block-based union-find labeller, then either fill or none.
//                      None of the last five has a counterpart in the reference.
#include "common.cuh"
#include <algorithm>
#include <cstdint>

namespace decnet {
namespace codec {

constexpr int kBlock = 256;

// kShift: the image is read shifted right by col_shift columns (image column x - col_shift, black outside [0, w)), the
// right view of StereoMatcher's minimum disparity; |col_shift| <= w.  Without it col_shift is unused and the code is the
// unshifted kernel's.
template <bool kShift>
__global__ void __launch_bounds__(kBlock)
image_prepare_u8_kernel(const unsigned char *__restrict__ img, float *__restrict__ out01, float *__restrict__ norm,
                        float m0, float m1, float m2, float s0, float s1, float s2, int h, int w, int H, int W, long long n,
                        int col_shift)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;      // over B*H*W padded pixels
    if (i >= n) return;
    const int x = (int)(i % W), y = (int)((i / W) % H);
    const long long b = i / ((long long)W * H);
    const int ry = H - h, rx = W - w;                                      // residual rows / columns come FIRST
    const int sx = kShift ? x - rx - col_shift : x - rx;                   // source column in the image
    float v[3] = {0.f, 0.f, 0.f};
    if (y >= ry && x >= rx && (!kShift || (sx >= 0 && sx < w))) {
        const unsigned char *p = img + ((b * h + (y - ry)) * (long long)w + sx) * 3;
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

// pred[i] = pred[i] + offset in fp32, rounded to nearest (StereoMatcher's minimum disparity).  Threads 0..nvec-1 each take
// one float4 of the 16-byte aligned body p[head, head + 4*nvec); the rest take one float of the unaligned head and the tail.
__global__ void __launch_bounds__(kBlock)
disp_add_kernel(float *__restrict__ p, float offset, long long head, long long nvec, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (i < nvec) {
        float4 *q = reinterpret_cast<float4 *>(p + head) + i;
        float4 v = *q;
        v.x = __fadd_rn(v.x, offset); v.y = __fadd_rn(v.y, offset); v.z = __fadd_rn(v.z, offset); v.w = __fadd_rn(v.w, offset);
        *q = v;
        return;
    }
    const long long j = i - nvec, k = j < head ? j : j + 4 * nvec;        // scalar j: head element, then tail element
    if (k < n) p[k] = __fadd_rn(p[k], offset);
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
// valid_of(d, rev, W, ow, x, tol, o) says whether crop column x of the row (value d, row offset o = row * ow) is valid:
// CheckValid runs the check, SpeckleValid (below) reads the speckle filter's planes.
constexpr int kFillItems = 16;                                             // columns per thread per chunk
constexpr int kFillChunk = kBlock * kFillItems;                            // 4096 columns, 16 KB of staged values
constexpr int kFillWarps = kBlock / 32;

struct CheckValid {
    __device__ bool operator()(float d, const float *rev, int W, int ow, int x, float tol, long long) const
    {
        return lr_valid(d, rev, W, ow, x, tol);
    }
};

template <class Valid>
__global__ void __launch_bounds__(kBlock)
lr_check_fill_rows_kernel(const float *__restrict__ pred, int B, int H, int W, int oh, int ow, float tol,
                          float *__restrict__ out_f32, unsigned short *__restrict__ out_u16,
                          unsigned char *__restrict__ out_valid, unsigned char *__restrict__ row_flags, const Valid valid_of)
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
                    if (x < ow && valid_of(fwd_crop[x], rev, W, ow, x, tol, o)) { m = x; break; }
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
                const bool v = (x < ow) & valid_of(d[k], rev, W, ow, xc, tol, o);
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

// Speckle filter (oracle/lr_speckle.py) between the check and the fill: valid 4-neighbours whose values differ by at most
// max_diff (|a - b| in fp32) are joined, and every region of at most max_size pixels is invalidated.  A block-based
// union-find labeller over the cropped pixels, with int32 labels (a pixel index, -1 on an invalid pixel) in three passes:
//   speckle_tile_kernel   one CTA per kTile x kTile tile: the check, then the tile's unions in shared memory; writes the
//                         checked values val (dl where valid, else 0), each pixel's tile-local root as a global index, and
//                         zeroes the region sizes
//   speckle_merge_kernel  one thread per pair of 4-neighbours across a tile border: unions of the global trees
//   speckle_count_kernel  one CTA per tile: each pixel's label becomes its root, and the region sizes are counted, per CTA
//                         into one shared counter for the root most of the tile shares, so a region covering the image
//                         costs about one global atomic per tile rather than one per pixel
// Both unions are the lock-free atomic-min union of Playne & Hawick (IEEE TPDS 2018): a root is linked under the smaller
// one with atomicMin, and a link that lost a race is retried from the value it found.  Labels only ever point to smaller
// indices, so every chain ends.  Which pixel is a region's root depends on the race, the regions and sizes do not.
// Then valid' = valid && size[root] > max_size, applied by speckle_apply_kernel (no fill) or by
// lr_check_fill_rows_kernel<SpeckleValid> (the fills).
constexpr int kTile = 32;
constexpr int kTileRows = 8;                                               // a CTA is kTile x kTileRows threads, 4 rows each

__device__ __forceinline__ bool speckle_joined(float a, float b, float max_diff)
{
    return fabsf(__fsub_rn(a, b)) <= max_diff;                             // an overflow to inf does not join
}

template <class P>
__device__ __forceinline__ int uf_find(P lab, int x)
{
    for (int p = lab[x]; p != x; p = lab[x]) x = p;
    return x;
}

// Join the trees of a and b in lab (shared or global), concurrently with other threads' unions.
__device__ __forceinline__ void uf_union(int *lab, int a, int b)
{
    volatile int *v = lab;
    for (;;) {
        a = uf_find(v, a);
        b = uf_find(v, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(lab + b, a);                             // link the larger root under the smaller
        if (old == b) return;
        b = old;                                                           // b was linked meanwhile: continue from there
    }
}

// Tile t of the [B, oh, ow] crop -> its image b and its first row y0 and column x0.
__device__ __forceinline__ void speckle_tile(int oh, int ow, long long &b, int &y0, int &x0)
{
    const int tx = (ow + kTile - 1) / kTile, ty = (oh + kTile - 1) / kTile;
    const long long t = blockIdx.x;
    b = t / ((long long)tx * ty);
    const int r = (int)(t - b * tx * ty);
    y0 = r / tx * kTile;
    x0 = (r - r / tx * tx) * kTile;
}

__global__ void __launch_bounds__(kTile * kTileRows)
speckle_tile_kernel(const float *__restrict__ pred, int B, int H, int W, int oh, int ow, float tol, float max_diff,
                    float *__restrict__ val, int *__restrict__ label, int *__restrict__ size)
{
    __shared__ float sv[kTile * kTile];
    __shared__ int sl[kTile * kTile];                                      // tile-local parent, -1: invalid
    long long b;
    int y0, x0;
    speckle_tile(oh, ow, b, y0, x0);
    const int lx = threadIdx.x, x = x0 + lx;
#pragma unroll
    for (int k = 0; k < kTile / kTileRows; ++k) {
        const int ly = threadIdx.y + k * kTileRows, y = y0 + ly, i = ly * kTile + lx;
        bool v = false;
        float d = 0.f;
        if (x < ow && y < oh) {
            const float *fwd = pred + (b * H + (H - oh + y)) * (long long)W;
            const float *rev = pred + ((b + B) * H + (H - oh + y)) * (long long)W;
            const float dl = fwd[W - ow + x];
            v = lr_valid(dl, rev, W, ow, x, tol);
            d = v ? dl : 0.f;
        }
        sv[i] = d;
        sl[i] = v ? i : -1;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kTile / kTileRows; ++k) {                          // join each pixel to its left and upper neighbours
        const int ly = threadIdx.y + k * kTileRows, i = ly * kTile + lx;
        if (sl[i] < 0) continue;                                           // a valid pixel's parent stays >= 0
        if (lx > 0 && sl[i - 1] >= 0 && speckle_joined(sv[i], sv[i - 1], max_diff)) uf_union(sl, i - 1, i);
        if (ly > 0 && sl[i - kTile] >= 0 && speckle_joined(sv[i], sv[i - kTile], max_diff)) uf_union(sl, i - kTile, i);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kTile / kTileRows; ++k) {
        const int ly = threadIdx.y + k * kTileRows, y = y0 + ly, i = ly * kTile + lx;
        if (x >= ow || y >= oh) continue;
        const long long g = (b * oh + y) * ow + x;
        int root = -1;
        if (sl[i] >= 0) {
            const int r = uf_find(sl, i);
            root = (int)((b * oh + y0 + r / kTile) * ow + x0 + r % kTile);
        }
        val[g] = sv[i];
        label[g] = root;
        size[g] = 0;
    }
}

// Pair e of 4-neighbours across a tile border: the first nv pairs straddle the vertical borders (row, kTile*k - 1 | kTile*k),
// the rest the horizontal ones (kTile*k - 1 | kTile*k, x).
__global__ void __launch_bounds__(kBlock)
speckle_merge_kernel(const float *__restrict__ val, int *label, int oh, int ow, float max_diff, long long nv, long long n)
{
    const long long e = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (e >= n) return;
    const int tx = (ow + kTile - 1) / kTile, ty = (oh + kTile - 1) / kTile;
    long long c, a;
    if (e < nv) {
        const long long row = e / (tx - 1);
        c = row * ow + (long long)(e - row * (tx - 1) + 1) * kTile;
        a = c - 1;
    } else {
        const long long j = e - nv, q = j / ow, b = q / (ty - 1);
        c = (b * oh + (q - b * (ty - 1) + 1) * kTile) * ow + (j - q * ow);
        a = c - ow;
    }
    if (label[a] < 0 || label[c] < 0 || !speckle_joined(val[a], val[c], max_diff)) return;
    uf_union(label, (int)a, (int)c);
}

__global__ void __launch_bounds__(kTile * kTileRows)
speckle_count_kernel(int *label, int *__restrict__ size, int oh, int ow)
{
    __shared__ int sdom, scount;                                           // a root of the tile and its pixel count
    long long b;
    int y0, x0;
    speckle_tile(oh, ow, b, y0, x0);
    const int lx = threadIdx.x, x = x0 + lx;
    if (lx == 0 && threadIdx.y == 0) { sdom = -1; scount = 0; }
    __syncthreads();
    int roots[kTile / kTileRows];
#pragma unroll
    for (int k = 0; k < kTile / kTileRows; ++k) {
        const int y = y0 + threadIdx.y + k * kTileRows;
        roots[k] = -1;
        if (x >= ow || y >= oh) continue;
        const long long g = (b * oh + y) * ow + x;
        const int l = label[g];
        if (l < 0) continue;
        const int r = uf_find(label, l);                                   // the trees no longer change: concurrent
        if (r != l) label[g] = r;                                          // compressions only store ancestors
        roots[k] = r;
        if (sdom < 0) atomicCAS(&sdom, -1, r);
    }
    __syncthreads();
    const int dom = sdom;
#pragma unroll
    for (int k = 0; k < kTile / kTileRows; ++k) {
        const int r = roots[k];
        const unsigned peers = __match_any_sync(0xffffffffu, r);
        if (r < 0 || lx != __ffs(peers) - 1) continue;
        if (r == dom) atomicAdd(&scount, __popc(peers));
        else atomicAdd(size + r, __popc(peers));
    }
    __syncthreads();
    if (lx == 0 && threadIdx.y == 0 && scount) atomicAdd(size + dom, scount);
}

// lr_check_fill_rows_kernel's validity under the speckle filter; the kernel then reads its values from the plane val, passed
// as pred with H = oh, W = ow and no reverse half (B = 0).
struct SpeckleValid {
    const int *label, *size;
    int max_size;
    __device__ bool operator()(float, const float *, int, int, int x, float, long long o) const
    {
        const int r = label[o + x];
        return r >= 0 && size[r] > max_size;
    }
};

// The speckle filter without a fill: the requested outputs of valid' and its values.
__global__ void __launch_bounds__(kBlock)
speckle_apply_kernel(const float *__restrict__ val, const int *__restrict__ label, const int *__restrict__ size, int max_size,
                     float *__restrict__ out_f32, unsigned short *__restrict__ out_u16, unsigned char *__restrict__ out_valid,
                     long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const int r = label[i];
    const bool v = r >= 0 && size[r] > max_size;
    const float d = v ? val[i] : 0.f;
    if (out_f32) out_f32[i] = d;
    if (out_u16) out_u16[i] = disp_u16(d);
    if (out_valid) out_valid[i] = v ? 1 : 0;
}

// Edge-aware ("guided") hole filling (oracle/lr_guided.py): the fast global smoother's line solves over the background-
// filled output of the two kernels above.  Every operation is an explicitly rounded intrinsic in the oracle's order, so
// nothing is contracted into an FMA; subnormals are kept (the build has no -ftz), which the weight table and den need.
// Scratch (decnet_lr_guided_fill_scratch_floats): the weight table, then five planes of B*h*w floats: the row and column
// edge weights wh (pixel x to x+1, 0 in the last column) and wv (y to y+1, 0 in the last row), num, den and g (the solver's
// g_i, kept for the back substitution).
constexpr int kGuideTable = 766;                                           // k = sum_c |dI_c| in 0..765
constexpr int kGuideTableFloats = 768;                                     // the planes after it stay 16-byte aligned
constexpr int kGuideIters = 3;

// w(k) = float32(exp(-k / sigma)) in double: every entry of sigma = 2.6 but w(0) = 1 lies more than 6e5 double ulps from a
// float32 rounding boundary, so any double exp within a few ulps gives the oracle's table.
__global__ void guided_table_kernel(double sigma, float *__restrict__ table)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < kGuideTable) table[k] = (float)exp(-(double)k / sigma);
}

__device__ __forceinline__ int guide_l1(const unsigned char *p, const unsigned char *q)
{
    return abs((int)p[0] - (int)q[0]) + abs((int)p[1] - (int)q[1]) + abs((int)p[2] - (int)q[2]);
}

// Per cropped pixel: the edge weights to its right and lower neighbours, and the right-hand sides num = valid ? f : 0 and
// den = valid ? 1 : 0 (f is the check's value on valid pixels).
__global__ void __launch_bounds__(kBlock)
guided_prep_kernel(const unsigned char *__restrict__ guide, const float *__restrict__ f, const unsigned char *__restrict__ valid,
                   const float *__restrict__ table, int h, int w, long long n, float *__restrict__ wh, float *__restrict__ wv,
                   float *__restrict__ num, float *__restrict__ den)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;      // over B*h*w pixels
    if (i >= n) return;
    const int x = (int)(i % w), y = (int)((i / w) % h);
    const unsigned char *p = guide + i * 3;
    wh[i] = x < w - 1 ? table[guide_l1(p, p + 3)] : 0.f;
    wv[i] = y < h - 1 ? table[guide_l1(p, p + 3ll * w)] : 0.f;
    const bool v = valid[i];
    num[i] = v ? f[i] : 0.f;
    den[i] = v ? 1.f : 0.f;
}

// One forward-elimination step of oracle.lr_guided.solve_line for both right-hand sides: a = lam_t * w(k_i), the carried
// state is (a_(i-1), g_(i-1), y_(i-1) of num and den); in place: w -> g_i, fn -> y_i of num, fd -> y_i of den.
__device__ __forceinline__ void thomas_step(float lt, float &w, float &fn, float &fd, float &ap, float &gp, float &yn, float &yd)
{
    const float a = __fmul_rn(lt, w);
    const float m = __fsub_rn(__fadd_rn(__fadd_rn(1.f, ap), a), __fmul_rn(ap, gp));
    const float r = __frcp_rn(m);
    const float g = __fmul_rn(a, r);
    yn = __fmul_rn(__fadd_rn(fn, __fmul_rn(ap, yn)), r);
    yd = __fmul_rn(__fadd_rn(fd, __fmul_rn(ap, yd)), r);
    ap = a; gp = g;
    w = g; fn = yn; fd = yd;
}

// Back substitution x_i = y_i + g_i x_(i+1) (x_(n-1) = y_(n-1): last), in place on y.
__device__ __forceinline__ void thomas_back(bool last, float g, float &yn, float &yd, float &xn, float &xd)
{
    if (!last) {
        yn = __fadd_rn(yn, __fmul_rn(g, xn));
        yd = __fadd_rn(yd, __fmul_rn(g, xd));
    }
    xn = yn; xd = yd;
}

__device__ __forceinline__ void cp_async_wait_one() { asm volatile("cp.async.wait_group 1;\n" ::: "memory"); }

// Row solves of one iteration: one warp per 32 consecutive rows of the [B*h, w] planes, lane l solving row r0 + l.  The rows
// pass through shared memory in 32 x 32 tiles (a warp's loads and stores stay coalesced, the lanes' reads are conflict-free
// with the padded stride), double-buffered with cp.async: the next tile's loads are in flight while the current tile's
// dependent chain of steps runs.  Forward: (w, num, den) -> (g, y_num, y_den), then backward over the tiles in reverse:
// (g, y_num, y_den) -> x into num and den.
constexpr int kRowTile = 32;

__global__ void __launch_bounds__(32)
guided_rows_kernel(const float *__restrict__ wh, float *num, float *den, float *gbuf, float lt, long long rows, int n)
{
    __shared__ float s[2][3][kRowTile][kRowTile + 1];
    const int lane = threadIdx.x;
    const long long r0 = (long long)blockIdx.x * kRowTile;
    const int ntiles = (n + kRowTile - 1) / kRowTile;
    auto load = [&](int tile, int buf, const float *p0, const float *p1, const float *p2) {
        const int x = min(tile * kRowTile + lane, n - 1);
#pragma unroll 4
        for (int j = 0; j < kRowTile; ++j) {
            const long long o = min(r0 + j, rows - 1) * n + x;
            cp_async_4(&s[buf][0][j][lane], p0 + o);
            cp_async_4(&s[buf][1][j][lane], p1 + o);
            cp_async_4(&s[buf][2][j][lane], p2 + o);
        }
        cp_async_commit();
    };
    auto store = [&](int tile, int buf, float *p0, float *p1, float *p2) {
        const int x = tile * kRowTile + lane;
        __syncwarp();
        if (x < n)
            for (int j = 0; j < kRowTile && r0 + j < rows; ++j) {
                const long long o = (r0 + j) * n + x;
                if (p0) p0[o] = s[buf][0][j][lane];
                p1[o] = s[buf][1][j][lane];
                p2[o] = s[buf][2][j][lane];
            }
        __syncwarp();                                                      // the tile is read before a copy refills it
    };

    float ap = 0.f, gp = 0.f, yn = 0.f, yd = 0.f;
    load(0, 0, wh, num, den);
    for (int t = 0; t < ntiles; ++t) {
        const int buf = t & 1;
        if (t + 1 < ntiles) { load(t + 1, buf ^ 1, wh, num, den); cp_async_wait_one(); }
        else cp_async_wait_all();
        __syncwarp();
        const int cnt = min(kRowTile, n - t * kRowTile);
        float (*sw)[kRowTile + 1] = s[buf][0], (*sn)[kRowTile + 1] = s[buf][1], (*sd)[kRowTile + 1] = s[buf][2];
#pragma unroll 8
        for (int k = 0; k < cnt; ++k) thomas_step(lt, sw[lane][k], sn[lane][k], sd[lane][k], ap, gp, yn, yd);
        store(t, buf, gbuf, num, den);
    }
    float xn = 0.f, xd = 0.f;
    load(ntiles - 1, 0, gbuf, num, den);
    for (int t = ntiles - 1, i = 0; t >= 0; --t, ++i) {
        const int buf = i & 1;
        if (t > 0) { load(t - 1, buf ^ 1, gbuf, num, den); cp_async_wait_one(); }
        else cp_async_wait_all();
        __syncwarp();
        const int cnt = min(kRowTile, n - t * kRowTile);
        float (*sg)[kRowTile + 1] = s[buf][0], (*sn)[kRowTile + 1] = s[buf][1], (*sd)[kRowTile + 1] = s[buf][2];
#pragma unroll 8
        for (int k = cnt - 1; k >= 0; --k) thomas_back(t * kRowTile + k == n - 1, sg[lane][k], sn[lane][k], sd[lane][k], xn, xd);
        store(t, buf, nullptr, num, den);
    }
}

// Column solves of one iteration: one thread per column of the [B, h, w] planes (a warp's accesses are 32 consecutive
// columns of one row).  The next kColGroup rows' loads are issued before the current group's chain of steps.
constexpr int kColGroup = 8;
constexpr int kColBlock = 128;

__global__ void __launch_bounds__(kColBlock)
guided_cols_kernel(const float *__restrict__ wv, float *num, float *den, float *gbuf, float lt, int B, int h, int w)
{
    const long long col = (long long)blockIdx.x * kColBlock + threadIdx.x;
    if (col >= (long long)B * w) return;
    const long long b = col / w;
    const long long base = b * h * (long long)w + (col - b * w);
    auto at = [&](int y) { return base + (long long)min(max(y, 0), h - 1) * w; };
    float cw[kColGroup], cn[kColGroup], cd[kColGroup];
#pragma unroll
    for (int k = 0; k < kColGroup; ++k) { const long long o = at(k); cw[k] = wv[o]; cn[k] = num[o]; cd[k] = den[o]; }
    float ap = 0.f, gp = 0.f, yn = 0.f, yd = 0.f;
    for (int y0 = 0; y0 < h; y0 += kColGroup) {
        float nw[kColGroup], nn[kColGroup], nd[kColGroup];
#pragma unroll
        for (int k = 0; k < kColGroup; ++k) { const long long o = at(y0 + kColGroup + k); nw[k] = wv[o]; nn[k] = num[o]; nd[k] = den[o]; }
#pragma unroll
        for (int k = 0; k < kColGroup; ++k) {
            if (y0 + k >= h) break;
            thomas_step(lt, cw[k], cn[k], cd[k], ap, gp, yn, yd);
            const long long o = at(y0 + k);
            gbuf[o] = cw[k]; num[o] = cn[k]; den[o] = cd[k];
        }
#pragma unroll
        for (int k = 0; k < kColGroup; ++k) { cw[k] = nw[k]; cn[k] = nn[k]; cd[k] = nd[k]; }
    }
    // backward, groups of kColGroup rows from the bottom: group q covers rows top - k, k = 0..kColGroup-1
    int top = h - 1;
#pragma unroll
    for (int k = 0; k < kColGroup; ++k) { const long long o = at(top - k); cw[k] = gbuf[o]; cn[k] = num[o]; cd[k] = den[o]; }
    float xn = 0.f, xd = 0.f;
    for (; top >= 0; top -= kColGroup) {
        float nw[kColGroup], nn[kColGroup], nd[kColGroup];
#pragma unroll
        for (int k = 0; k < kColGroup; ++k) { const long long o = at(top - kColGroup - k); nw[k] = gbuf[o]; nn[k] = num[o]; nd[k] = den[o]; }
#pragma unroll
        for (int k = 0; k < kColGroup; ++k) {
            if (top - k < 0) break;
            thomas_back(top - k == h - 1, cw[k], cn[k], cd[k], xn, xd);
            const long long o = at(top - k);
            num[o] = cn[k]; den[o] = cd[k];
        }
#pragma unroll
        for (int k = 0; k < kColGroup; ++k) { cw[k] = nw[k]; cn[k] = nn[k]; cd[k] = nd[k]; }
    }
}

// Compose: an invalid pixel whose den is a normal float takes num / den, any other keeps the background value out_f32
// already holds (valid pixels keep their bits); out_u16 = disp_u16 of the result.
__global__ void __launch_bounds__(kBlock)
guided_compose_kernel(const float *__restrict__ num, const float *__restrict__ den, const unsigned char *__restrict__ valid,
                      float *__restrict__ out_f32, unsigned short *__restrict__ out_u16, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    float d = out_f32[i];
    if (!valid[i]) {
        const float c = den[i];
        if (c >= 1.17549435e-38f) { d = __fdiv_rn(num[i], c); out_f32[i] = d; }   // 2^-126; NaN compares false
    }
    if (out_u16) out_u16[i] = disp_u16(d);
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
    image_prepare_u8_kernel<false><<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
        img_hwc, out01, out_norm, mean3_host[0], mean3_host[1], mean3_host[2], std3_host[0], std3_host[1], std3_host[2], h, w, H, W, n,
        0);
    return after_launch("image_prepare_u8_kernel");
}

int decnet_image_prepare_u8_shift(const unsigned char *img_hwc, float *out01, float *out_norm, const float *mean3_host,
                                  const float *std3_host, int B, int h, int w, int H, int W, int col_shift, void *stream)
{
    DECNET_REQUIRE(img_hwc && (out01 || out_norm) && mean3_host && std3_host, "null pointer");
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0 && H >= h && W >= w, "padded size %dx%d must cover the image %dx%d", H, W, h, w);
    const long long n = (long long)B * H * W;
    col_shift = std::max(-w, std::min(w, col_shift));                      // beyond +-w every column is black alike
    image_prepare_u8_kernel<true><<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
        img_hwc, out01, out_norm, mean3_host[0], mean3_host[1], mean3_host[2], std3_host[0], std3_host[1], std3_host[2], h, w, H, W, n,
        col_shift);
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

int decnet_disp_add(float *pred, float offset, long long n, void *stream)
{
    DECNET_REQUIRE(pred && (reinterpret_cast<uintptr_t>(pred) & 3) == 0, "pred must be a non-null, 4-byte aligned float pointer");
    DECNET_REQUIRE(n > 0, "empty map (n = %lld)", n);
    const long long head = std::min(n, (long long)(((16 - (reinterpret_cast<uintptr_t>(pred) & 15)) & 15) / 4));
    const long long nvec = (n - head) / 4, threads = nvec + (n - 4 * nvec);
    disp_add_kernel<<<(unsigned)((threads + kBlock - 1) / kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
        pred, offset, head, nvec, n);
    return after_launch("disp_add_kernel");
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
                                                                 row_flags, CheckValid{});
    if (int s = after_launch("lr_check_fill_rows_kernel")) return s;
    lr_fill_empty_rows_kernel<<<(unsigned)rows, kBlock, 0, st>>>(ori_h, ori_w, out_f32, out_u16, row_flags);
    return after_launch("lr_fill_empty_rows_kernel");
}

// The guided fill's stages after the background fill of out_f32 (valid: out_valid), for decnet_lr_check_guided_fill and
// decnet_lr_check_speckle; the callers validate the arguments.
static int guided_stages(const unsigned char *guide, int B, int ori_h, int ori_w, double lambda, double sigma_color,
                         float *out_f32, unsigned short *out_u16, const unsigned char *out_valid, float *scratch, cudaStream_t st)
{
    const long long rows = (long long)B * ori_h, n = rows * ori_w;
    float *table = scratch, *wh = table + kGuideTableFloats, *wv = wh + n, *num = wv + n, *den = num + n, *g = den + n;
    guided_table_kernel<<<(kGuideTable + kBlock - 1) / kBlock, kBlock, 0, st>>>(sigma_color, table);
    if (int s = after_launch("guided_table_kernel")) return s;
    const unsigned pix_grid = (unsigned)((n + kBlock - 1) / kBlock);
    guided_prep_kernel<<<pix_grid, kBlock, 0, st>>>(guide, out_f32, out_valid, table, ori_h, ori_w, n, wh, wv, num, den);
    if (int s = after_launch("guided_prep_kernel")) return s;
    for (int t = 1; t <= kGuideIters; ++t) {
        double q = 1.0;                                                    // 4^(T-t), exact
        for (int k = t; k < kGuideIters; ++k) q *= 4.0;
        const float lt = (float)(lambda * 1.5 * q / 63.0);                 // 63 = 4^T - 1; in the oracle's order
        guided_rows_kernel<<<(unsigned)((rows + kRowTile - 1) / kRowTile), 32, 0, st>>>(wh, num, den, g, lt, rows, ori_w);
        if (int s = after_launch("guided_rows_kernel")) return s;
        guided_cols_kernel<<<(unsigned)(((long long)B * ori_w + kColBlock - 1) / kColBlock), kColBlock, 0, st>>>(
            wv, num, den, g, lt, B, ori_h, ori_w);
        if (int s = after_launch("guided_cols_kernel")) return s;
    }
    guided_compose_kernel<<<pix_grid, kBlock, 0, st>>>(num, den, out_valid, out_f32, out_u16, n);
    return after_launch("guided_compose_kernel");
}

long long decnet_lr_guided_fill_scratch_floats(int B, int ori_h, int ori_w)
{
    return kGuideTableFloats + 5 * (long long)B * ori_h * ori_w;           // table, wh, wv, num, den, g
}

int decnet_lr_check_guided_fill(const float *pred, const unsigned char *guide, int B, int H, int W, int ori_h, int ori_w,
                                float tol, double lambda, double sigma_color, float *out_f32, unsigned short *out_u16,
                                unsigned char *out_valid, unsigned char *row_flags, float *scratch, void *stream)
{
    DECNET_REQUIRE(pred && guide && out_f32 && out_valid && row_flags && scratch,
                   "null prediction, guide, float rows, mask, row flags or scratch");
    DECNET_REQUIRE(B > 0 && ori_h > 0 && ori_w > 0 && ori_h <= H && ori_w <= W, "crop %dx%d outside the %dx%d map", ori_h, ori_w, H, W);
    DECNET_REQUIRE(tol >= 0.f && tol <= 3.402823466e38f, "tolerance must be finite and >= 0");
    DECNET_REQUIRE(lambda >= 0.0 && lambda <= 1.7976931348623157e308, "lambda must be finite and >= 0");
    DECNET_REQUIRE(sigma_color > 0.0 && sigma_color <= 1.7976931348623157e308, "sigma_color must be finite and > 0");
    const long long rows = (long long)B * ori_h;
    DECNET_REQUIRE(rows <= 0x7fffffffLL, "%lld rows exceed the grid", rows);
    if (int s = decnet_lr_check_fill(pred, B, H, W, ori_h, ori_w, tol, out_f32, nullptr, out_valid, row_flags, stream)) return s;
    return guided_stages(guide, B, ori_h, ori_w, lambda, sigma_color, out_f32, out_u16, out_valid, scratch,
                         static_cast<cudaStream_t>(stream));
}

// Speckle planes: val (fp32), label and size (int32), n each, rounded up to 16 bytes; then the guided fill's scratch.
static long long speckle_planes_bytes(long long n) { return (12 * n + 15) / 16 * 16; }

long long decnet_lr_speckle_scratch_bytes(int B, int ori_h, int ori_w, int fill)
{
    const long long n = (long long)B * ori_h * ori_w;
    return speckle_planes_bytes(n) + (fill == 2 ? 4 * decnet_lr_guided_fill_scratch_floats(B, ori_h, ori_w) : 0);
}

int decnet_lr_check_speckle(const float *pred, const unsigned char *guide, int B, int H, int W, int ori_h, int ori_w,
                            float tol, int max_size, float max_diff, int fill, double lambda, double sigma_color,
                            float *out_f32, unsigned short *out_u16, unsigned char *out_valid, unsigned char *row_flags,
                            void *scratch, void *stream)
{
    DECNET_REQUIRE(fill >= 0 && fill <= 2, "fill must be 0 (none), 1 (background) or 2 (guided), got %d", fill);
    DECNET_REQUIRE((guide != nullptr) == (fill == 2), "guide is required for fill 2 (guided) and only for it");
    DECNET_REQUIRE(pred && (out_f32 || out_u16 || out_valid), "null prediction or no output requested");
    DECNET_REQUIRE(fill == 0 || (out_f32 && row_flags), "a fill needs the float rows and row flags");
    DECNET_REQUIRE(fill < 2 || out_valid, "the guided fill needs the mask");
    DECNET_REQUIRE(B > 0 && ori_h > 0 && ori_w > 0 && ori_h <= H && ori_w <= W, "crop %dx%d outside the %dx%d map", ori_h, ori_w, H, W);
    DECNET_REQUIRE(tol >= 0.f && tol <= 3.402823466e38f, "tolerance must be finite and >= 0");
    DECNET_REQUIRE(max_size >= 0, "speckle size must be >= 0, got %d", max_size);
    DECNET_REQUIRE(max_diff >= 0.f && max_diff <= 3.402823466e38f, "speckle range must be finite and >= 0");
    DECNET_REQUIRE(fill < 2 || (lambda >= 0.0 && lambda <= 1.7976931348623157e308), "lambda must be finite and >= 0");
    DECNET_REQUIRE(fill < 2 || (sigma_color > 0.0 && sigma_color <= 1.7976931348623157e308), "sigma_color must be finite and > 0");
    const long long rows = (long long)B * ori_h, n = rows * ori_w;
    DECNET_REQUIRE(n <= 0x7fffffffLL, "%lld pixels exceed the int32 labels", n);
    const long long planes = speckle_planes_bytes(n);
    if (max_size == 0) {                                                   // off: the entries without the filter, as they are
        if (fill == 0) return decnet_lr_check(pred, B, H, W, ori_h, ori_w, tol, out_f32, out_u16, out_valid, stream);
        if (fill == 1) return decnet_lr_check_fill(pred, B, H, W, ori_h, ori_w, tol, out_f32, out_u16, out_valid, row_flags, stream);
        DECNET_REQUIRE(scratch, "null scratch");
        return decnet_lr_check_guided_fill(pred, guide, B, H, W, ori_h, ori_w, tol, lambda, sigma_color, out_f32, out_u16,
                                           out_valid, row_flags, reinterpret_cast<float *>(static_cast<char *>(scratch) + planes),
                                           stream);
    }
    DECNET_REQUIRE(scratch, "null scratch");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    float *val = static_cast<float *>(scratch);
    int *label = reinterpret_cast<int *>(val + n), *size = label + n;
    const long long tx = (ori_w + kTile - 1) / kTile, ty = (ori_h + kTile - 1) / kTile;
    const unsigned tiles = (unsigned)(B * tx * ty);
    speckle_tile_kernel<<<tiles, dim3(kTile, kTileRows), 0, st>>>(pred, B, H, W, ori_h, ori_w, tol, max_diff, val, label, size);
    if (int s = after_launch("speckle_tile_kernel")) return s;
    const long long nv = rows * (tx - 1), edges = nv + B * (ty - 1) * ori_w;
    if (edges > 0) {
        speckle_merge_kernel<<<(unsigned)((edges + kBlock - 1) / kBlock), kBlock, 0, st>>>(val, label, ori_h, ori_w, max_diff, nv,
                                                                                          edges);
        if (int s = after_launch("speckle_merge_kernel")) return s;
    }
    speckle_count_kernel<<<tiles, dim3(kTile, kTileRows), 0, st>>>(label, size, ori_h, ori_w);
    if (int s = after_launch("speckle_count_kernel")) return s;
    if (fill == 0) {
        speckle_apply_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, st>>>(val, label, size, max_size, out_f32, out_u16,
                                                                                      out_valid, n);
        return after_launch("speckle_apply_kernel");
    }
    lr_check_fill_rows_kernel<<<(unsigned)rows, kBlock, 0, st>>>(val, 0, ori_h, ori_w, ori_h, ori_w, 0.f, out_f32,
                                                                 fill == 2 ? nullptr : out_u16, out_valid, row_flags,
                                                                 SpeckleValid{label, size, max_size});
    if (int s = after_launch("lr_check_fill_rows_kernel")) return s;
    lr_fill_empty_rows_kernel<<<(unsigned)rows, kBlock, 0, st>>>(ori_h, ori_w, out_f32, fill == 2 ? nullptr : out_u16, row_flags);
    if (int s = after_launch("lr_fill_empty_rows_kernel")) return s;
    if (fill == 1) return 0;
    return guided_stages(guide, B, ori_h, ori_w, lambda, sigma_color, out_f32, out_u16, out_valid,
                         reinterpret_cast<float *>(static_cast<char *>(scratch) + planes), st);
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
