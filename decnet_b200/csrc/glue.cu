// decnet_b200/csrc/glue.cu -- the HBM-bound glue of the decomposed-matching pipeline (sm_100a):
// cost-volume build, soft-argmin, mask threshold, dynamic-upsampling pack + glue, soft-attention
// pack, sigmoid+blend, disparity warp (+ refinement input pack).  One pass over each operand,
// coalesced along W, no temporaries.  Reference sites: SURVEY.md section 8 rows a2, a4, a6, a8,
// a13, a14 (file:line quoted at each kernel).
#include "common.cuh"
#include <algorithm>
#include <cuda_bf16.h>

namespace decnet {
namespace glue {

constexpr int kBlock = 256;

// The reference normalises pixel coordinates with (size-1)/2 (align_corners=True style,
// submodule.py:497-499) and then samples with grid_sample's DEFAULT align_corners=False,
// whose un-normalisation is ((g+1)*size-1)/2.  Same fp32 operation order here.
__device__ __forceinline__ float sample_coord(float pos_minus_shift, float size) {
    const float g = pos_minus_shift / ((size - 1.0f) / 2.0f) - 1.0f;
    return ((g + 1.0f) * size - 1.0f) / 2.0f;
}

struct Taps {          // 4-tap bilinear with zero padding
    int x0, y0;
    float w00, w01, w10, w11;   // (y0,x0) (y0,x1) (y1,x0) (y1,x1); 0 where the tap is outside
};

__device__ __forceinline__ Taps make_taps(float ix, float iy, int H, int W) {
    Taps t;
    const float fx = floorf(ix), fy = floorf(iy);
    t.x0 = (int)fx; t.y0 = (int)fy;
    const float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.0f - wx1, wy0 = 1.0f - wy1;
    const bool xin0 = t.x0 >= 0 && t.x0 < W, xin1 = t.x0 + 1 >= 0 && t.x0 + 1 < W;
    const bool yin0 = t.y0 >= 0 && t.y0 < H, yin1 = t.y0 + 1 >= 0 && t.y0 + 1 < H;
    t.w00 = (xin0 && yin0) ? wx0 * wy0 : 0.f;
    t.w01 = (xin1 && yin0) ? wx1 * wy0 : 0.f;
    t.w10 = (xin0 && yin1) ? wx0 * wy1 : 0.f;
    t.w11 = (xin1 && yin1) ? wx1 * wy1 : 0.f;
    return t;
}

__device__ __forceinline__ float sample_plane(const float *__restrict__ p, const Taps &t, int H, int W) {
    // clamped addresses are always valid; weights of outside taps are exactly 0
    const int x0 = min(max(t.x0, 0), W - 1), x1 = min(max(t.x0 + 1, 0), W - 1);
    const int y0 = min(max(t.y0, 0), H - 1), y1 = min(max(t.y0 + 1, 0), H - 1);
    float v = 0.f;
    v += __ldg(p + (size_t)y0 * W + x0) * t.w00;
    v += __ldg(p + (size_t)y0 * W + x1) * t.w01;
    v += __ldg(p + (size_t)y1 * W + x0) * t.w10;
    v += __ldg(p + (size_t)y1 * W + x1) * t.w11;
    return v;
}

// ---------------------------------------------------------------------------------------------
// a2: cost volume (GetCostVolume.forward -> get_warped_feats_by_homgrp -> cost_computation_cor,
// submodule.py:532-562, 479-510, 518-522) for the stage-0 candidates d = 0..D-1 (:390):
//   vol[b,c,d,h,w] = (w >= d ? L[b,c,h,w] : 0) * bilinear0(R[b,c], y'(h), x'(w-d))
// LAYOUT 0: fp32 NCDHW [B,C,D,H,W] (the reference's layout, parity / drop-in)
// LAYOUT 1: bf16 NDHWC [B,D,H,W,Cpad] (channels-last, zero-padded to Cpad: the tcgen05 conv input)
// One thread per (b,d,h,w); taps computed once and reused over the channel loop.
// ---------------------------------------------------------------------------------------------
template <int LAYOUT>
__global__ void __launch_bounds__(kBlock)
costvol_kernel(const float *__restrict__ L, const float *__restrict__ R, void *__restrict__ out,
               int B, int C, int H, int W, int D, int Cpad, int row0, int nrows)
{
    // output rows are the window [row0, row0 + nrows) of the H-row volume (row-band mode); rows
    // outside the image are written as zeros (they are the conv's zero padding)
    const long long n = (long long)B * D * nrows * W;
    const long long idx = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (idx >= n) return;
    const int w = (int)(idx % W);
    const int hl = (int)((idx / W) % nrows);
    const int d = (int)((idx / ((long long)W * nrows)) % D);
    const int b = (int)(idx / ((long long)W * nrows * D));
    const int h = row0 + hl;
    const bool in_img = h >= 0 && h < H;
    const int hc = min(max(h, 0), H - 1);
    const float ix = sample_coord((float)w - (float)d, (float)W);
    const float iy = sample_coord((float)hc, (float)H);
    const Taps t = make_taps(ix, iy, H, W);
    const bool left_on = (w >= d) && in_img;
    const size_t plane = (size_t)H * W;
    const float *Lb = L + (size_t)b * C * plane + (size_t)hc * W + w;
    const float *Rb = R + (size_t)b * C * plane;
    if (LAYOUT == 0) {
        float *o = static_cast<float *>(out) + (((size_t)b * C * D + d) * nrows + hl) * W + w;
        for (int c = 0; c < C; ++c) {
            const float r = sample_plane(Rb + (size_t)c * plane, t, H, W);
            const float l = left_on ? __ldg(Lb + (size_t)c * plane) : 0.f;
            o[(size_t)c * D * nrows * W] = l * r;
        }
    } else {
        __nv_bfloat16 *o = static_cast<__nv_bfloat16 *>(out) + (size_t)idx * Cpad;
        for (int c0 = 0; c0 < Cpad; c0 += 8) {
            __align__(16) __nv_bfloat16 v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int c = c0 + k;
                float val = 0.f;
                if (c < C) {
                    const float r = sample_plane(Rb + (size_t)c * plane, t, H, W);
                    const float l = left_on ? __ldg(Lb + (size_t)c * plane) : 0.f;
                    val = l * r;
                }
                v[k] = __float2bfloat16(val);
            }
            *reinterpret_cast<uint4 *>(o + c0) = *reinterpret_cast<const uint4 *>(v);
        }
    }
}

// LAYOUT 1, block-cooperative: one CTA = one (b, d, h) row of the volume.  The NCHW features are read with w fastest
// (coalesced), the products go through a shared-memory tile [w][Cpad] and leave as whole channels-last rows
// (coalesced 16-byte stores).  The per-voxel thread of costvol_kernel<1> walks 224 channels serially with only
// B*D*H*W = 46 080 threads at SceneFlow size (111 us); a thread per (voxel, 8 channels) reads 8 planes apart (144 us).
constexpr int kCvTileW = 64;
__global__ void __launch_bounds__(kBlock)
costvol_bf16_rows_kernel(const float *__restrict__ L, const float *__restrict__ R, __nv_bfloat16 *__restrict__ out,
                         int C, int H, int W, int D, int Cpad, int row0, int nrows)
{
    extern __shared__ __align__(16) unsigned char cv_smem[];
    __nv_bfloat16 *tile = reinterpret_cast<__nv_bfloat16 *>(cv_smem);             // [kCvTileW][Cpad + 2]: odd word stride, conflict-free
    const int ts = Cpad + 2;
    __shared__ Taps taps[kCvTileW];
    const int hl = blockIdx.x % nrows, d = (blockIdx.x / nrows) % D, b = blockIdx.x / (nrows * D);
    const int h = row0 + hl;
    const bool in_img = h >= 0 && h < H;
    const int hc = min(max(h, 0), H - 1);
    const size_t plane = (size_t)H * W;
    const float *Lb = L + (size_t)b * C * plane + (size_t)hc * W;
    const float *Rb = R + (size_t)b * C * plane;
    const float iy = sample_coord((float)hc, (float)H);
    for (int w0 = 0; w0 < W; w0 += kCvTileW) {
        const int wt = min(kCvTileW, W - w0);
        __syncthreads();                                                        // previous tile fully written out
        if (threadIdx.x < wt) taps[threadIdx.x] = make_taps(sample_coord((float)(w0 + threadIdx.x) - (float)d, (float)W), iy, H, W);
        // channel padding of the tile
        for (int i = threadIdx.x; i < wt * (Cpad - C); i += kBlock) tile[(i / (Cpad - C)) * ts + C + i % (Cpad - C)] = __float2bfloat16(0.f);
        __syncthreads();
        // a thread keeps ONE pixel of the tile and walks channels cg, cg + ngrp, ...: the four tap offsets and weights are
        // set up once, every load address is a pointer stepped by ngrp planes (the item-indexed form spent ~180 instructions
        // per sample on divisions, tap clamps and 64-bit address arithmetic); lanes of a warp are neighbouring pixels
        {
            const int ngrp = kBlock / wt;                                        // channel groups (>= 4: wt <= 64)
            const int cg = threadIdx.x / wt, wl = threadIdx.x - cg * wt, w = w0 + wl;
            if (cg < ngrp) {
                const Taps t = taps[wl];
                const int x0 = min(max(t.x0, 0), W - 1), x1 = min(max(t.x0 + 1, 0), W - 1);
                const int y0 = min(max(t.y0, 0), H - 1), y1 = min(max(t.y0 + 1, 0), H - 1);
                const size_t step = (size_t)ngrp * plane;
                const float *q00 = Rb + (size_t)cg * plane + (size_t)y0 * W + x0, *q01 = Rb + (size_t)cg * plane + (size_t)y0 * W + x1;
                const float *q10 = Rb + (size_t)cg * plane + (size_t)y1 * W + x0, *q11 = Rb + (size_t)cg * plane + (size_t)y1 * W + x1;
                const float *ql = Lb + (size_t)cg * plane + w;
                __nv_bfloat16 *tp = tile + wl * ts + cg;
                const bool use_l = w >= d;
                if (in_img) {
#pragma unroll 4
                    for (int c = cg; c < C; c += ngrp) {
                        float v = 0.f;                                          // same summation order as sample_plane()
                        v += __ldg(q00) * t.w00; v += __ldg(q01) * t.w01; v += __ldg(q10) * t.w10; v += __ldg(q11) * t.w11;
                        const float l = use_l ? __ldg(ql) : 0.f;               // l = 0 left of the candidate: keeps NaN/Inf of R
                        *tp = __float2bfloat16(l * v);
                        q00 += step; q01 += step; q10 += step; q11 += step; ql += step; tp += ngrp;
                    }
                } else {
                    for (int c = cg; c < C; c += ngrp) { *tp = __float2bfloat16(0.f); tp += ngrp; }
                }
            }
        }
        __syncthreads();
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + ((((size_t)b * D + d) * nrows + hl) * W + w0) * Cpad);
        const uint32_t *src = reinterpret_cast<const uint32_t *>(tile);
        const int cw = Cpad >> 1, tw2 = ts >> 1;                                   // words per row: output / tile
        for (int i = threadIdx.x; i < wt * cw; i += kBlock) {
            const int wl = i / cw, k = i - wl * cw;
            dst[i] = src[wl * tw2 + k];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// a4: soft-argmin (disparity_regression, submodule.py:766-777): pred = sum_d softmax_d(cost) * d
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
softargmin_kernel(const float *__restrict__ cost, float *__restrict__ pred, int B, int D, int HW)
{
    const long long idx = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (idx >= (long long)B * HW) return;
    const int b = (int)(idx / HW), p = (int)(idx % HW);
    const float *c = cost + (size_t)b * D * HW + p;
    float mx = -INFINITY;
    for (int d = 0; d < D; ++d) mx = fmaxf(mx, __ldg(c + (size_t)d * HW));
    float s0 = 0.f, s1 = 0.f;
    for (int d = 0; d < D; ++d) {
        const float e = expf(__ldg(c + (size_t)d * HW) - mx);
        s0 += e; s1 += e * (float)d;
    }
    pred[idx] = s1 / s0;
}

// ---------------------------------------------------------------------------------------------
// a6: mask selection (SparseDenseNetRefinementMask.py:164-170):
//   m = p > thold ? 1 : (p <= thold ? 0 : p)      (NaN stays NaN)
// for the left and right probability maps in one launch; one CTA per row also emits the number
// of selected pixels of the row for both views (ballot + popc), which the host can use to size
// work and report densities without another pass.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
mask_threshold_kernel(const float *__restrict__ pl, const float *__restrict__ pr, float thold,
                      float *__restrict__ ml, float *__restrict__ mr,
                      int *__restrict__ row_count_l, int *__restrict__ row_count_r, int W)
{
    __shared__ int cnt[2];
    if (threadIdx.x < 2) cnt[threadIdx.x] = 0;
    __syncthreads();
    const size_t m0 = (size_t)blockIdx.x * W;
    int nl = 0, nr = 0;
    for (int w0 = 0; w0 < W; w0 += kBlock) {
        const int w = w0 + threadIdx.x;
        bool sl = false, sr = false;
        if (w < W) {
            const float a = pl[m0 + w], b = pr[m0 + w];
            const float va = a > thold ? 1.f : (a <= thold ? 0.f : a);
            const float vb = b > thold ? 1.f : (b <= thold ? 0.f : b);
            ml[m0 + w] = va; mr[m0 + w] = vb;
            sl = va != 0.f; sr = vb != 0.f;
        }
        nl += __popc(__ballot_sync(0xffffffffu, sl));
        nr += __popc(__ballot_sync(0xffffffffu, sr));
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&cnt[0], nl); atomicAdd(&cnt[1], nr); }
    __syncthreads();
    if (threadIdx.x == 0 && row_count_l) row_count_l[blockIdx.x] = cnt[0];
    if (threadIdx.x == 1 && row_count_r) row_count_r[blockIdx.x] = cnt[1];
}

// ---------------------------------------------------------------------------------------------
// a5 tail, fused: GenerateSparseMask's `(cur - pre) ** 2` (submodule.py:369) as one pass for both views, and
// its last layer -- Conv2d 1x1 3->1 + BN (folded: w[3], b) -> sigmoid -> `> thold` (submodule.py:363-364,
// SparseDenseNetRefinementMask.py:158-170) -- as one pass for both views.  The comparison is done on the
// logit against x* = the smallest float whose torch.sigmoid exceeds thold (found by bisection on the device
// at set-up, model.py), so the mask bits equal `torch.sigmoid(logit) > thold`; NaN logits give NaN like
// mask_threshold_kernel.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
sqdiff_kernel(const float4 *__restrict__ a0, const float4 *__restrict__ b0, float4 *__restrict__ o0,
              const float4 *__restrict__ a1, const float4 *__restrict__ b1, float4 *__restrict__ o1, long long n4)
{
    const float4 *a = blockIdx.y ? a1 : a0, *b = blockIdx.y ? b1 : b0;
    float4 *o = blockIdx.y ? o1 : o0;
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < n4; i += (long long)gridDim.x * kBlock) {
        const float4 x = __ldg(a + i), y = __ldg(b + i);
        const float dx = x.x - y.x, dy = x.y - y.y, dz = x.z - y.z, dw = x.w - y.w;
        o[i] = make_float4(dx * dx, dy * dy, dz * dz, dw * dw);
    }
}

__global__ void __launch_bounds__(kBlock)
sqdiff_scalar_kernel(const float *__restrict__ a0, const float *__restrict__ b0, float *__restrict__ o0,
                     const float *__restrict__ a1, const float *__restrict__ b1, float *__restrict__ o1, long long n)
{
    const float *a = blockIdx.y ? a1 : a0, *b = blockIdx.y ? b1 : b0;
    float *o = blockIdx.y ? o1 : o0;
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < n; i += (long long)gridDim.x * kBlock) {
        const float d = __ldg(a + i) - __ldg(b + i);
        o[i] = d * d;
    }
}

__global__ void __launch_bounds__(kBlock)
detail_head_kernel(const float *__restrict__ xl, const float *__restrict__ xr, float w0, float w1, float w2, float bias,
                   float logit_thold, float *__restrict__ ml, float *__restrict__ mr, long long HW)
{
    const int b = blockIdx.y >> 1;
    const float *x = ((blockIdx.y & 1) ? xr : xl) + (long long)b * 3 * HW;
    float *m = ((blockIdx.y & 1) ? mr : ml) + (long long)b * HW;
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < HW; i += (long long)gridDim.x * kBlock) {
        // same operation order as conv2d_small_kernel<1,P> with a 1x1 kernel: bias, then channels in order
        float v = bias;
        v = fmaf(__ldg(x + i), w0, v);
        v = fmaf(__ldg(x + HW + i), w1, v);
        v = fmaf(__ldg(x + 2 * HW + i), w2, v);
        m[i] = v >= logit_thold ? 1.f : (v < logit_thold ? 0.f : v);
    }
}

// ---------------------------------------------------------------------------------------------
// a8 (input side): DynamicUpsampling's conv input (submodule.py:580):
//   cat(disp.unsqueeze(1), unfold(Lf, k=3, s=3)) -> [B, 1+9C, h, w]
//   ch 0 = disp,  ch 1 + c*9 + ky*3 + kx = Lf[b, c, 3y+ky, 3x+kx]
// One CTA per (b, c, y): the three source rows are read coalesced into shared memory and the nine
// destination rows written coalesced.  blockIdx.y == C handles the disparity plane.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
dynup_pack_kernel(const float *__restrict__ disp, const float *__restrict__ Lf, float *__restrict__ out,
                  int C, int h, int w)
{
    extern __shared__ float rows[];            // [3][3w]
    const int y = blockIdx.x, c = blockIdx.y, b = blockIdx.z;
    const int W3 = 3 * w;
    const size_t oplane = (size_t)h * w;
    float *ob = out + (size_t)b * (9 * C + 1) * oplane + (size_t)y * w;
    if (c == C) {
        for (int x = threadIdx.x; x < w; x += kBlock) ob[x] = disp[((size_t)b * h + y) * w + x];
        return;
    }
    const float *src = Lf + (((size_t)b * C + c) * (3 * h) + 3 * y) * W3;
    for (int i = threadIdx.x; i < 3 * W3; i += kBlock) rows[i] = src[i];
    __syncthreads();
    for (int i = threadIdx.x; i < 9 * w; i += kBlock) {
        const int k = i / w, x = i - k * w;
        const int ky = k / 3, kx = k - ky * 3;
        ob[(size_t)(1 + c * 9 + k) * oplane + x] = rows[ky * W3 + 3 * x + kx];
    }
}

// ---------------------------------------------------------------------------------------------
// a8 (output side): softmax over the 9 taps of each of the 9 sub-pixels, 3x3 gather of the
// replication-padded coarse disparity, weighted sum, pixel-shuffle, x3 (submodule.py:582-589):
//   out[3y+i, 3x+j] = 3 * sum_k softmax_k(logits[(i*3+j)*9 + k]) * disp[clamp(y+ky-1), clamp(x+kx-1)]
// One thread per coarse pixel (81 coalesced channel reads, 9 x 3-wide writes).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
dynup_glue_kernel(const float *__restrict__ logits, const float *__restrict__ disp, float *__restrict__ out,
                  int B, int h, int w)
{
    const long long idx = (long long)blockIdx.x * kBlock + threadIdx.x;
    const long long n = (long long)B * h * w;
    if (idx >= n) return;
    const int x = (int)(idx % w), y = (int)((idx / w) % h), b = (int)(idx / ((long long)w * h));
    const size_t plane = (size_t)h * w;
    const float *db = disp + (size_t)b * plane;
    float nb[9];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int yy = min(max(y + ky - 1, 0), h - 1), xx = min(max(x + kx - 1, 0), w - 1);
            nb[ky * 3 + kx] = __ldg(db + (size_t)yy * w + xx);
        }
    const float *lg = logits + (size_t)b * 81 * plane + (size_t)y * w + x;
    float *ob = out + (size_t)b * 9 * plane;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        float res[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int sub = i * 3 + j;
            float v[9], mx = -INFINITY;
#pragma unroll
            for (int k = 0; k < 9; ++k) { v[k] = __ldg(lg + (size_t)(sub * 9 + k) * plane); mx = fmaxf(mx, v[k]); }
            float s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int k = 0; k < 9; ++k) { const float e = expf(v[k] - mx); s0 += e; s1 += e * nb[k]; }
            res[j] = (s1 / s0) * 3.0f;
        }
        float *o = ob + (size_t)(3 * y + i) * (3 * w) + 3 * x;
        o[0] = res[0]; o[1] = res[1]; o[2] = res[2];
    }
}

// ---------------------------------------------------------------------------------------------
// a8, channels-last variants feeding / draining the TF32 tcgen05 convs (decnet_conv2d_tf32_nhwc):
//   dynup_pack_nhwc : out[b,y,x,ch], ch 0 = disp, ch 1+c*9+ky*3+kx = Lf[b,c,3y+ky,3x+kx], ch >= 1+9C zero
//   dynup_glue_nhwc : logits[b,y,x,sub*9+k] -> same output as dynup_glue_kernel
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
dynup_pack_nhwc_kernel(const float *__restrict__ disp, const float *__restrict__ Lf, float *__restrict__ out,
                       int C, int h, int w, int CP, int TX, int round_tf32, int pad)
{
    // pad = 1: the output is [B, h+2, w+2, CP] with a zero border (decnet_conv2d_tf32_nhwc_halo's layout); blockIdx.y
    // then runs over h+2 rows: the two border rows are zero-filled, interior rows get a zero pixel at both ends
    if (pad) {
        const int yp = blockIdx.y, bb = blockIdx.z, wp = w + 2;
        float4 *row = reinterpret_cast<float4 *>(out + ((size_t)bb * (h + 2) + yp) * wp * CP);
        const int cp4 = CP >> 2;
        if (yp == 0 || yp == h + 1) {
            // every tile zeroes its own span of the border row; tile 0 also the two end pixels
            const int x0 = blockIdx.x * TX;
            for (int i = threadIdx.x; i < min(TX, w - x0) * cp4; i += kBlock) row[(size_t)(x0 + 1) * cp4 + i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (blockIdx.x == 0)
                for (int i = threadIdx.x; i < 2 * cp4; i += kBlock)
                    row[(i < cp4 ? 0 : (size_t)(wp - 1) * cp4) + (i % cp4)] = make_float4(0.f, 0.f, 0.f, 0.f);
            return;
        }
        if (blockIdx.x == 0)
            for (int i = threadIdx.x; i < 2 * cp4; i += kBlock)
                row[(i < cp4 ? 0 : (size_t)(wp - 1) * cp4) + (i % cp4)] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // Block = TX coarse pixels of one row.  Phase 1: the 3C fine-row segments land in shared memory, one warp
    // per segment (coalesced).  Phase 2: channels-last float4 stores; the channel -> (segment, kx) mapping is a
    // per-block table, and the (pixel, channel) cursor advances by add/compare (no divisions per element).
    extern __shared__ float rows[];            // [C*3][3*TX] then int lut[CP]
    const int x0 = blockIdx.x * TX, y = blockIdx.y - pad, b = blockIdx.z;
    const int nx = min(TX, w - x0);
    const int W3 = 3 * w, seg = 3 * TX;
    int *lut = reinterpret_cast<int *>(rows + (size_t)C * 3 * seg);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < C * 3; r += kBlock / 32) {
        const int c = r / 3, ky = r - 3 * c;
        const float *src = Lf + (((size_t)b * C + c) * (3 * h) + 3 * y + ky) * W3 + 3 * x0;
        for (int i = lane; i < 3 * nx; i += 32) rows[r * seg + i] = __ldg(src + i);
    }
    for (int ch = threadIdx.x; ch < CP; ch += kBlock) {
        int v = -1;                            // zero padding
        if (ch == 0) v = -2;                   // the disparity itself
        else if (ch <= 9 * C) {
            const int c = (ch - 1) / 9, k = (ch - 1) - 9 * c, ky = k / 3, kx = k - 3 * ky;
            v = (c * 3 + ky) * seg + kx;
        }
        lut[ch] = v;
    }
    __syncthreads();
    float4 *ob = reinterpret_cast<float4 *>(out + (((size_t)b * (h + 2 * pad) + y + pad) * (w + 2 * pad) + x0 + pad) * CP);
    const float *db = disp + ((size_t)b * h + y) * w + x0;
    const int cp4 = CP >> 2, total4 = nx * cp4;
    int xl = threadIdx.x / cp4, c4 = threadIdx.x - xl * cp4;          // one division per thread
    const int dxl = kBlock / cp4, dc4 = kBlock - dxl * cp4;
    for (int i = threadIdx.x; i < total4; i += kBlock) {
        float o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int l = lut[4 * c4 + e];
            float v = l >= 0 ? rows[l + 3 * xl] : ((l == -2 && disp) ? __ldg(db + xl) : 0.f);
            if (round_tf32) v = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);   // == cvt.rna.tf32
            o[e] = v;
        }
        ob[i] = make_float4(o[0], o[1], o[2], o[3]);
        xl += dxl; c4 += dc4;
        if (c4 >= cp4) { c4 -= cp4; ++xl; }
    }
}

// Channel 0 of a packed tensor (the only channel that depends on the disparity): lets the feature channels be
// packed ahead of time, on another stream, with disp = NULL.
__global__ void __launch_bounds__(kBlock)
dynup_set_disp_nhwc_kernel(const float *__restrict__ disp, float *__restrict__ out, int h, int w, int CP,
                           int round_tf32, int pad, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const int x = (int)(i % w);
    const long long t = i / w;
    const int y = (int)(t % h), b = (int)(t / h);
    float v = __ldg(disp + i);
    if (round_tf32) v = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
    out[(((size_t)b * (h + 2 * pad) + y + pad) * (w + 2 * pad) + x + pad) * CP] = v;
}

// Block = 32 coarse pixels of one row x 9 sub-pixels (288 threads).  The 32 x NP logits are staged through
// shared memory with coalesced float4 loads (a thread-per-pixel walk over its own 324-byte row is
// uncoalesced); thread (i, px, j) then owns fine pixel (3y+i, 3x+j): 9 logits -> softmax -> weighted sum of
// the 3x3 coarse neighbourhood, and the block writes three contiguous 96-float runs.
constexpr int kGluePx = 32;
__global__ void __launch_bounds__(9 * kGluePx)
dynup_glue_nhwc_kernel(const float *__restrict__ logits, const float *__restrict__ disp, float *__restrict__ out,
                       int B, int h, int w, int NP, int pad)
{
    extern __shared__ __align__(16) float lg_s[];          // [32][NP + 1] (odd stride: conflict-free 9-float reads)
    const int x0 = blockIdx.x * kGluePx, y = blockIdx.y, b = blockIdx.z;
    const int nx = min(kGluePx, w - x0);
    const int stride = NP + 1;
    const size_t plane = (size_t)h * w;
    const float *src = logits + (((size_t)b * (h + 2 * pad) + y + pad) * (w + 2 * pad) + x0 + pad) * NP;   // pad: zero-bordered layout
    if ((NP & 3) == 0) {
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        const int np4 = NP >> 2;
        for (int t = threadIdx.x; t < nx * np4; t += 9 * kGluePx) {
            const int px = t / np4, c4 = t - px * np4;
            const float4 v = __ldg(s4 + t);
            float *d = lg_s + px * stride + 4 * c4;
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        }
    } else {
        for (int t = threadIdx.x; t < nx * NP; t += 9 * kGluePx) {
            const int px = t / NP, c = t - px * NP;
            lg_s[px * stride + c] = __ldg(src + t);
        }
    }
    // the 3 x (32 + 2) coarse disparities the block's pixels need (replicate padding), once per block
    __shared__ float nb_s[3][kGluePx + 2];
    if (threadIdx.x < 3 * (kGluePx + 2)) {
        const int ky = threadIdx.x / (kGluePx + 2), kxp = threadIdx.x - ky * (kGluePx + 2);
        const int yy = min(max(y + ky - 1, 0), h - 1), xx = min(max(x0 + kxp - 1, 0), w - 1);
        nb_s[ky][kxp] = __ldg(disp + (size_t)b * plane + (size_t)yy * w + xx);
    }
    __syncthreads();
    const int i = threadIdx.x / (3 * kGluePx), r = threadIdx.x - i * 3 * kGluePx, px = r / 3, j = r - 3 * px;
    if (px >= nx) return;
    const int x = x0 + px;
    float nb[9];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) nb[ky * 3 + kx] = nb_s[ky][px + kx];
    const float *lg = lg_s + px * stride + (i * 3 + j) * 9;
    float v[9], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < 9; ++k) { v[k] = lg[k]; mx = fmaxf(mx, v[k]); }
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) { const float e = expf(v[k] - mx); s0 += e; s1 += e * nb[k]; }
    out[(size_t)b * 9 * plane + (size_t)(3 * y + i) * (3 * w) + 3 * x + j] = (s1 / s0) * 3.0f;
}

// ---------------------------------------------------------------------------------------------
// Layout bridges for the wide (72-channel) refinement layers of the 1/9 level, which run on the zero-bordered
// channels-last TF32 kernel (conv2d_nhwc_tcgen05.cu):
//   nchw_cat_to_nhwc_pad : cat of up to three NCHW sources -> [B, h+2, w+2, CP] (border and channel padding zero;
//                          round_tf32: values rounded to TF32 for the kernel's plain-TF32 mode)
//   nhwc_pad_to_nchw     : interior of [B, h+2, w+2, NP], first C channels -> NCHW [B, C, h, w]
// The tensors are small (52 k pixels at SceneFlow size); one thread per output element.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
nchw_cat_to_nhwc_pad_kernel(const float *__restrict__ s0, const float *__restrict__ s1, const float *__restrict__ s2,
                            int c0, int c1, int c2, float *__restrict__ out, int h, int w, int CP, int round_tf32, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;      // over B*(h+2)*(w+2)*CP
    if (i >= n) return;
    const int c = (int)(i % CP);
    long long p = i / CP;
    const int xp = (int)(p % (w + 2)); p /= (w + 2);
    const int yp = (int)(p % (h + 2));
    const long long b = p / (h + 2);
    float v = 0.f;
    if (xp >= 1 && xp <= w && yp >= 1 && yp <= h && c < c0 + c1 + c2) {
        const long long pix = (long long)(yp - 1) * w + (xp - 1), plane = (long long)h * w;
        if (c < c0) v = __ldg(s0 + (b * c0 + c) * plane + pix);
        else if (c < c0 + c1) v = __ldg(s1 + (b * c1 + (c - c0)) * plane + pix);
        else v = __ldg(s2 + (b * c2 + (c - c0 - c1)) * plane + pix);
        if (round_tf32) v = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
    }
    out[i] = v;
}

// Tiled form of the kernel above for CP % 4 == 0 (the product shapes): a block owns 32 padded pixels of one row; warps read one
// source channel each (32 consecutive pixels: one 128-byte line) into a [32][CP + 1] shared tile, then the block writes the
// 32 x CP floats of the segment, which are contiguous in the channels-last tensor, as float4.  The element-per-thread form read
// 32 different planes per warp load (52 us for 33 MB at the 1/9 level).
__global__ void __launch_bounds__(kBlock)
nchw_cat_to_nhwc_pad_tiled_kernel(const float *__restrict__ s0, const float *__restrict__ s1, const float *__restrict__ s2,
                                  int c0, int c1, int c2, float *__restrict__ out, int h, int w, int CP, int round_tf32)
{
    extern __shared__ float tile[];                        // [32][CP + 1]
    const int xp0 = blockIdx.x * 32, yp = blockIdx.y, b = blockIdx.z;
    const int npx = min(32, w + 2 - xp0), ts = CP + 1, csum = c0 + c1 + c2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool row_in = yp >= 1 && yp <= h;
    const int xp = xp0 + lane;
    const bool px_in = row_in && lane < npx && xp >= 1 && xp <= w;
    const size_t plane = (size_t)h * w, pix = row_in ? (size_t)(yp - 1) * w + (size_t)max(xp - 1, 0) : 0;
    for (int c = warp; c < CP; c += kBlock / 32) {
        float v = 0.f;
        if (px_in && c < csum) {
            const float *src = c < c0 ? s0 + ((size_t)b * c0 + c) * plane
                             : c < c0 + c1 ? s1 + ((size_t)b * c1 + (c - c0)) * plane
                                           : s2 + ((size_t)b * c2 + (c - c0 - c1)) * plane;
            v = __ldg(src + pix);
            if (round_tf32) v = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
        }
        tile[lane * ts + c] = v;
    }
    __syncthreads();
    float4 *ob = reinterpret_cast<float4 *>(out + (((size_t)b * (h + 2) + yp) * (w + 2) + xp0) * CP);
    const int cp4 = CP >> 2, total4 = npx * cp4;
    int px = threadIdx.x / cp4, c4 = threadIdx.x - px * cp4;                  // one division per thread
    const int dpx = kBlock / cp4, dc4 = kBlock - dpx * cp4;
    for (int i = threadIdx.x; i < total4; i += kBlock) {
        const float *t = tile + px * ts + 4 * c4;
        ob[i] = make_float4(t[0], t[1], t[2], t[3]);
        px += dpx; c4 += dc4;
        if (c4 >= cp4) { c4 -= cp4; ++px; }
    }
}

__global__ void __launch_bounds__(kBlock)
nhwc_pad_to_nchw_kernel(const float *__restrict__ in, float *__restrict__ out, int C, int NP, int h, int w, long long n)
{
    const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;      // over B*C*h*w
    if (i >= n) return;
    const int x = (int)(i % w);
    long long p = i / w;
    const int y = (int)(p % h); p /= h;
    const int c = (int)(p % C);
    const long long b = p / C;
    out[i] = __ldg(in + (((b * (h + 2) + y + 1) * (long long)(w + 2)) + x + 1) * NP + c);
}

// ---------------------------------------------------------------------------------------------
// a13 (input side): cat(Lf, dense, sparse, lmask, -var) -> [B, C+4, H, W]
// (SparseDenseNetRefinementMask.py:197).  Flat copy, float4 where aligned.
// ---------------------------------------------------------------------------------------------
// grid.y = output plane (b, c): one source plane -> one destination plane, no index arithmetic per element
template <typename V>
__global__ void __launch_bounds__(kBlock)
attn_pack_kernel(const float *__restrict__ Lf, const float *__restrict__ dense, const float *__restrict__ sparse,
                 const float *__restrict__ lmask, const float *__restrict__ var, float *__restrict__ out,
                 int C, long long HWv)
{
    const int b = blockIdx.y / (C + 4), c = blockIdx.y - b * (C + 4);
    const float *src = c < C ? Lf + ((long long)b * C + c) * HWv * (sizeof(V) / 4)
                             : (c == C ? dense : c == C + 1 ? sparse : c == C + 2 ? lmask : var) + (long long)b * HWv * (sizeof(V) / 4);
    const V *s = reinterpret_cast<const V *>(src);
    V *d = reinterpret_cast<V *>(out + (long long)blockIdx.y * HWv * (sizeof(V) / 4));
    const bool neg = c == C + 3;
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < HWv; i += (long long)gridDim.x * kBlock) {
        V v = __ldg(s + i);
        if (neg) {
            if constexpr (sizeof(V) == 16) { v.x = -v.x; v.y = -v.y; v.z = -v.z; v.w = -v.w; }
            else v = -v;
        }
        d[i] = v;
    }
}

// a13 (output side): m = sigmoid(logit); fused = dense*(1-m) + m*sparse
// (submodule.py:602-604, SparseDenseNetRefinementMask.py:202)
__global__ void __launch_bounds__(kBlock)
blend_kernel(const float *__restrict__ logit, const float *__restrict__ dense, const float *__restrict__ sparse,
             float *__restrict__ soft_mask, float *__restrict__ fused, long long n)
{
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < n; i += (long long)gridDim.x * kBlock) {
        const float m = 1.0f / (1.0f + expf(-logit[i]));
        const float d = dense[i], s = sparse[i];
        if (soft_mask) soft_mask[i] = m;
        fused[i] = d * (1.0f - m) + m * s;
    }
}

// ---------------------------------------------------------------------------------------------
// a14: warp the right features by the (fractional) disparity (Refinement.get_warped_feats_by_homgrp,
// submodule.py:719-745) and, when `packed` is given, build the refinement conv input
// cat(Lf, warped, disp) -> [B, 2C+1, H, W] (:758-759) in the same pass.
// ---------------------------------------------------------------------------------------------
// grid.y = (b, group of CG channels): one thread = one pixel x CG channels, all 5*CG loads independent and
// issued before the first use (the kernel is HBM/L2-latency bound: memory-level parallelism is what matters).
template <int CG>
__global__ void __launch_bounds__(kBlock, 4)
warp_kernel(const float *__restrict__ Lf, const float *__restrict__ Rf, const float *__restrict__ disp,
            float *__restrict__ warped, float *__restrict__ packed, int B, int C, int H, int W,
            int H_total, int row0)
{
    // H rows are the window [row0, row0 + H) of an H_total-row image (row-band mode): the vertical
    // coordinate follows the reference's formula on GLOBAL rows; taps outside the window read 0
    const int groups = (C + CG - 1) / CG;
    const int b = blockIdx.y / groups, c0 = (blockIdx.y - b * groups) * CG;
    const size_t plane = (size_t)H * W;
    const size_t pix = (size_t)blockIdx.x * kBlock + threadIdx.x;
    if (pix >= plane) return;
    const int h = (int)(pix / W), w = (int)(pix - (size_t)h * W);
    const float dv = __ldg(disp + (size_t)b * plane + pix);
    const float ix = sample_coord((float)w - dv, (float)W);
    const float iy = sample_coord((float)(row0 + h), (float)H_total) - (float)row0;
    const Taps t = make_taps(ix, iy, H, W);
    const int x0 = min(max(t.x0, 0), W - 1), x1 = min(max(t.x0 + 1, 0), W - 1);
    const int y0 = min(max(t.y0, 0), H - 1), y1 = min(max(t.y0 + 1, 0), H - 1);
    const size_t o00 = (size_t)y0 * W + x0, o01 = (size_t)y0 * W + x1, o10 = (size_t)y1 * W + x0, o11 = (size_t)y1 * W + x1;
    const float *Rb = Rf + ((size_t)b * C + c0) * plane;
    float v00[CG], v01[CG], v10[CG], v11[CG], lv[CG];
    // four tap pointers stepped by one channel plane: the address arithmetic per load is one 64-bit add (the indexed form cost
    // ~370 of the kernel's 614 instructions per warp: profiles/r02_warp_kernel_ncu.txt)
    const float *q00 = Rb + o00, *q01 = Rb + o01, *q10 = Rb + o10, *q11 = Rb + o11;
    const float *ql = Lf + ((size_t)b * C + c0) * plane + pix;
    const int nch = min(CG, C - c0);
#pragma unroll
    for (int i = 0; i < CG; ++i) {
        const bool ok = i < nch;
        v00[i] = ok ? __ldg(q00) : 0.f;
        v01[i] = ok ? __ldg(q01) : 0.f;
        v10[i] = ok ? __ldg(q10) : 0.f;
        v11[i] = ok ? __ldg(q11) : 0.f;
        lv[i] = (packed && ok) ? __ldg(ql) : 0.f;
        q00 += plane; q01 += plane; q10 += plane; q11 += plane; ql += plane;
    }
    if (packed) {
        float *pb = packed + (size_t)b * (2 * C + 1) * plane + pix;
#pragma unroll
        for (int i = 0; i < CG; ++i)
            if (c0 + i < C) {
                float v = 0.f;                                  // same summation order as sample_plane()
                v += v00[i] * t.w00; v += v01[i] * t.w01; v += v10[i] * t.w10; v += v11[i] * t.w11;
                pb[(size_t)(c0 + i) * plane] = lv[i];
                pb[(size_t)(C + c0 + i) * plane] = v;
            }
        if (c0 == 0) pb[(size_t)(2 * C) * plane] = dv;
    } else {
        float *wb = warped + ((size_t)b * C + c0) * plane + pix;
#pragma unroll
        for (int i = 0; i < CG; ++i) {
            if (i < nch) {
                float v = 0.f;
                v += v00[i] * t.w00; v += v01[i] * t.w01; v += v10[i] * t.w10; v += v11[i] * t.w11;
                *wb = v;
            }
            wb += plane;
        }
    }
}

static int launch_warp(const float *Lf, const float *Rf, const float *disp, float *warped, float *packed,
                       int B, int C, int H, int W, int H_total, int row0, cudaStream_t st, const char *name)
{
    constexpr int CG = 8;
    const long long plane = (long long)H * W;
    const long long gy = (long long)B * ((C + CG - 1) / CG);
    DECNET_REQUIRE(gy <= 65535, "B * ceil(C/8) = %lld exceeds the grid limit", gy);
    warp_kernel<CG><<<dim3((unsigned)((plane + kBlock - 1) / kBlock), (unsigned)gy), kBlock, 0, st>>>(
        Lf, Rf, disp, warped, packed, B, C, H, W, H_total, row0);
    return after_launch(name);
}

// ---------------------------------------------------------------------------------------------
// a7: Haar wavelet lost-detail masks (utils/Wavelet.py:8-123; the reference's filter pickle is
// absent, orthonormal Haar is used -- parity unpinned, see oracle/glue.py).  Per x2 level:
//   haar_analysis_kernel : LL and v = max(|LH|,|HL|,|HH|) per 2x2 block, per-image min/max of v
//   haar_count_kernel    : per image, how many normalised values are <= t_k for the 10 thresholds
//   haar_mask_kernel     : t = first t_k with >= 85 % of the pixels below it (else 1), mask = vn >= t
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
haar_analysis_kernel(const float *__restrict__ x, float *__restrict__ ll, float *__restrict__ v,
                     unsigned int *__restrict__ minmax, int H, int W, int h, int w)
{
    const int b = blockIdx.y;
    const long long n = (long long)h * w;
    float lmin = INFINITY, lmax = 0.f;
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < n; i += (long long)gridDim.x * kBlock) {
        const int xx = (int)(i % w), yy = (int)(i / w);
        const float *p = x + ((size_t)b * H + 2 * yy) * W + 2 * xx;
        const float a = p[0], bb = p[1], c = p[W], d = p[W + 1];
        ll[(size_t)b * n + i] = (a + bb + c + d) * 0.5f;
        const float lh = (a - bb + c - d) * 0.5f, hl = (a + bb - c - d) * 0.5f, hh = (a - bb - c + d) * 0.5f;
        const float m = fmaxf(fmaxf(fabsf(lh), fabsf(hl)), fabsf(hh));
        v[(size_t)b * n + i] = m;
        lmin = fminf(lmin, m); lmax = fmaxf(lmax, m);
    }
    for (int o = 16; o > 0; o >>= 1) {
        lmin = fminf(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    if ((threadIdx.x & 31) == 0) {       // v >= 0: the uint bit pattern orders like the float
        atomicMin(minmax + 2 * b, __float_as_uint(lmin));
        atomicMax(minmax + 2 * b + 1, __float_as_uint(lmax));
    }
}

struct HaarThresholds { float t[10]; };

__global__ void __launch_bounds__(kBlock)
haar_count_kernel(const float *__restrict__ v, const unsigned int *__restrict__ minmax, HaarThresholds th,
                  unsigned int *__restrict__ counts, long long n)
{
    const int b = blockIdx.y;
    const float mn = __uint_as_float(minmax[2 * b]), mx = __uint_as_float(minmax[2 * b + 1]);
    unsigned int c[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) c[k] = 0;
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < n; i += (long long)gridDim.x * kBlock) {
        const float vn = (v[(size_t)b * n + i] - mn) / (mx - mn);
#pragma unroll
        for (int k = 0; k < 10; ++k) c[k] += (vn <= th.t[k]) ? 1u : 0u;
    }
#pragma unroll
    for (int k = 0; k < 10; ++k) {
        unsigned int s = c[k];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((threadIdx.x & 31) == 0 && s) atomicAdd(counts + 10 * b + k, s);
    }
}

__global__ void __launch_bounds__(kBlock)
haar_mask_kernel(const float *__restrict__ v, const unsigned int *__restrict__ minmax,
                 const unsigned int *__restrict__ counts, HaarThresholds th, float *__restrict__ mask, long long n)
{
    const int b = blockIdx.y;
    const float mn = __uint_as_float(minmax[2 * b]), mx = __uint_as_float(minmax[2 * b + 1]);
    float t = 1.0f;
    for (int k = 0; k < 10; ++k)
        if ((float)counts[10 * b + k] / (float)n >= 0.85f) { t = th.t[k]; break; }
    for (long long i = (long long)blockIdx.x * kBlock + threadIdx.x; i < n; i += (long long)gridDim.x * kBlock) {
        const float vn = (v[(size_t)b * n + i] - mn) / (mx - mn);
        mask[(size_t)b * n + i] = (vn >= t) ? 1.f : 0.f;
    }
}

// ---------------------------------------------------------------------------------------------
// a15: skip-stage up-sampling F.interpolate(pred*3, (H, W), mode="bicubic") (SparseDenseNetRefinementMask.py:143-144),
// align_corners=False, A = -0.75, border taps clamped.  Bit-identical to ATen's upsample_bicubic2d_out_frame on CUDA:
// the source index, the coefficients and the 4-tap sums below are ATen's expressions (UpSample.cuh) in the same fp32
// types, so nvcc contracts them into the same FMAs; the scales are (float)in / out, computed on the host as ATen does.
// One thread per output column and a strip of kBicRows output rows: the horizontal pass of an input row depends on the
// column only, so the four rows under the vertical window slide down the strip and each input row is interpolated once
// per column instead of four times; the stores of a warp are one coalesced 128-byte row segment per output row.
// ---------------------------------------------------------------------------------------------
constexpr int kBicRows = 8;

__device__ __forceinline__ float bic_source_index(float scale, int dst_index) {
    return scale * (dst_index + static_cast<float>(0.5)) - static_cast<float>(0.5);
}

__device__ __forceinline__ float bic_conv1(float x, float A) { return ((A + 2) * x - (A + 3)) * x * x + 1; }
__device__ __forceinline__ float bic_conv2(float x, float A) { return ((A * x - 5 * A) * x + 8 * A) * x - 4 * A; }

__device__ __forceinline__ float bic_interp1d(float x0, float x1, float x2, float x3, float t) {
    float coeffs[4];
    const float A = -0.75;
    const float xa = t;
    coeffs[0] = bic_conv2(xa + 1.0, A);
    coeffs[1] = bic_conv1(xa, A);
    const float xb = 1.0 - t;
    coeffs[2] = bic_conv1(xb, A);
    coeffs[3] = bic_conv2(xb + 1.0, A);
    return x0 * coeffs[0] + x1 * coeffs[1] + x2 * coeffs[2] + x3 * coeffs[3];
}

// horizontal pass of input row y (clamped) at the four clamped columns around in_x; v = fl(pred * 3) first
__device__ __forceinline__ float bic_row(const float *__restrict__ in, int y, int h, int w, int in_x, float t_x) {
    const float *row = in + (size_t)max(min(y, h - 1), 0) * w;
    const float v0 = __ldg(row + max(min(in_x - 1, w - 1), 0)) * 3.0f;
    const float v1 = __ldg(row + max(min(in_x + 0, w - 1), 0)) * 3.0f;
    const float v2 = __ldg(row + max(min(in_x + 1, w - 1), 0)) * 3.0f;
    const float v3 = __ldg(row + max(min(in_x + 2, w - 1), 0)) * 3.0f;
    return bic_interp1d(v0, v1, v2, v3, t_x);
}

__global__ void __launch_bounds__(128)
bicubic_up3_kernel(const float *__restrict__ in, float *__restrict__ out, int h, int w, int H, int W,
                   float scale_h, float scale_w)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y0 = blockIdx.y * kBicRows;
    if (x >= W) return;
    const float *src = in + (size_t)blockIdx.z * h * w;
    float *dst = out + (size_t)blockIdx.z * H * W;
    const int y1 = min(y0 + kBicRows, H);
    if (h == H && w == W) {                          // ATen's same-size branch: a copy of pred*3
        for (int y = y0; y < y1; ++y) dst[(size_t)y * W + x] = __ldg(src + (size_t)y * w + x) * 3.0f;
        return;
    }
    const float real_x = bic_source_index(scale_w, x);
    const int in_x = floorf(real_x);
    const float t_x = real_x - in_x;
    // r0..r3: horizontal results of input rows cur-1 .. cur+2 (in_y is non-decreasing along the strip)
    int cur = (int)floorf(bic_source_index(scale_h, y0));
    float r0 = bic_row(src, cur - 1, h, w, in_x, t_x), r1 = bic_row(src, cur, h, w, in_x, t_x);
    float r2 = bic_row(src, cur + 1, h, w, in_x, t_x), r3 = bic_row(src, cur + 2, h, w, in_x, t_x);
    for (int y = y0; y < y1; ++y) {
        const float real_y = bic_source_index(scale_h, y);
        const int in_y = floorf(real_y);
        const float t_y = real_y - in_y;
        if (in_y - cur > 4) cur = in_y - 4;          // down-sampling: skip rows no window covers
        while (cur < in_y) {
            ++cur;
            r0 = r1; r1 = r2; r2 = r3;
            r3 = bic_row(src, cur + 2, h, w, in_x, t_x);
        }
        dst[(size_t)y * W + x] = bic_interp1d(r0, r1, r2, r3, t_y);
    }
}

static inline int grid_for(long long n, int cap = 148 * 16) {
    long long g = (n + kBlock - 1) / kBlock;
    return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace glue
}  // namespace decnet

using namespace decnet;
using namespace decnet::glue;

extern "C" {

int decnet_costvol_fwd(const float *L, const float *R, float *vol, int B, int C, int H, int W, int D, void *stream) {
    DECNET_REQUIRE(L && R && vol, "null pointer");
    DECNET_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && D > 0, "non-positive size");
    const long long n = (long long)B * D * H * W;
    costvol_kernel<0><<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(L, R, vol, B, C, H, W, D, C, 0, H);
    return after_launch("costvol_kernel<f32>");
}

int decnet_costvol_bf16_ndhwc_rows(const float *L, const float *R, void *vol, int B, int C, int Cpad, int H, int W, int D,
                                   int row0, int nrows, void *stream) {
    DECNET_REQUIRE(L && R && vol, "null pointer");
    DECNET_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && D > 0 && nrows > 0, "non-positive size");
    DECNET_REQUIRE(Cpad >= C && Cpad % 8 == 0, "Cpad=%d must be >= C=%d and a multiple of 8", Cpad, C);
    DECNET_REQUIRE((reinterpret_cast<uintptr_t>(vol) & 15u) == 0, "volume must be 16-byte aligned");
    const long long blocks = (long long)B * D * nrows;
    DECNET_REQUIRE(blocks < (1ll << 31), "volume too large for one launch");
    const size_t smem = (size_t)kCvTileW * (Cpad + 2) * sizeof(__nv_bfloat16);
    DECNET_REQUIRE(smem <= 200 * 1024, "Cpad too large");
    if (smem > 48 * 1024)
        DECNET_CUDA(cudaFuncSetAttribute(costvol_bf16_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    costvol_bf16_rows_kernel<<<(unsigned)blocks, kBlock, smem, (cudaStream_t)stream>>>(
        L, R, static_cast<__nv_bfloat16 *>(vol), C, H, W, D, Cpad, row0, nrows);
    return after_launch("costvol_bf16_rows_kernel");
}

int decnet_costvol_bf16_ndhwc(const float *L, const float *R, void *vol, int B, int C, int Cpad, int H, int W, int D,
                              void *stream) {
    return decnet_costvol_bf16_ndhwc_rows(L, R, vol, B, C, Cpad, H, W, D, 0, H, stream);
}

int decnet_softargmin(const float *cost, float *pred, int B, int D, int H, int W, void *stream) {
    DECNET_REQUIRE(cost && pred, "null pointer");
    DECNET_REQUIRE(B > 0 && D > 0 && H > 0 && W > 0, "non-positive size");
    const long long n = (long long)B * H * W;
    softargmin_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(cost, pred, B, D, H * W);
    return after_launch("softargmin_kernel");
}

int decnet_mask_threshold(const float *prob_l, const float *prob_r, float thold, float *mask_l, float *mask_r,
                          int32_t *row_count_l, int32_t *row_count_r, int B, int H, int W, void *stream) {
    DECNET_REQUIRE(prob_l && prob_r && mask_l && mask_r, "null pointer");
    DECNET_REQUIRE(B > 0 && H > 0 && W > 0, "non-positive size");
    mask_threshold_kernel<<<B * H, kBlock, 0, (cudaStream_t)stream>>>(prob_l, prob_r, thold, mask_l, mask_r,
                                                                     row_count_l, row_count_r, W);
    return after_launch("mask_threshold_kernel");
}

int decnet_sqdiff_pair(const float *a0, const float *b0, float *out0, const float *a1, const float *b1, float *out1,
                       long long n, void *stream) {
    DECNET_REQUIRE(a0 && b0 && out0 && a1 && b1 && out1, "null pointer");
    DECNET_REQUIRE(n > 0, "element count must be positive");
    const uintptr_t al = reinterpret_cast<uintptr_t>(a0) | reinterpret_cast<uintptr_t>(b0) | reinterpret_cast<uintptr_t>(out0) |
                         reinterpret_cast<uintptr_t>(a1) | reinterpret_cast<uintptr_t>(b1) | reinterpret_cast<uintptr_t>(out1);
    if ((n & 3) != 0 || (al & 15u) != 0) {      // ragged size or unaligned view: scalar form
        sqdiff_scalar_kernel<<<dim3((unsigned)std::min<long long>((n + kBlock - 1) / kBlock, 148 * 16), 2), kBlock, 0, (cudaStream_t)stream>>>(
            a0, b0, out0, a1, b1, out1, n);
        return after_launch("sqdiff_scalar_kernel");
    }
    const long long n4 = n / 4;
    sqdiff_kernel<<<dim3((unsigned)std::min<long long>((n4 + kBlock - 1) / kBlock, 148 * 16), 2), kBlock, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4 *>(a0), reinterpret_cast<const float4 *>(b0), reinterpret_cast<float4 *>(out0),
        reinterpret_cast<const float4 *>(a1), reinterpret_cast<const float4 *>(b1), reinterpret_cast<float4 *>(out1), n4);
    return after_launch("sqdiff_kernel");
}

int decnet_detail_head(const float *x_l, const float *x_r, const float *w3, float bias, float logit_thold,
                       float *mask_l, float *mask_r, int B, int H, int W, void *stream) {
    DECNET_REQUIRE(x_l && x_r && w3 && mask_l && mask_r, "null pointer");
    DECNET_REQUIRE(B > 0 && 2 * B <= 65535 && H > 0 && W > 0, "bad size");
    const long long HW = (long long)H * W;
    detail_head_kernel<<<dim3((unsigned)std::min<long long>((HW + kBlock - 1) / kBlock, 256), 2 * B), kBlock, 0, (cudaStream_t)stream>>>(
        x_l, x_r, w3[0], w3[1], w3[2], bias, logit_thold, mask_l, mask_r, HW);
    return after_launch("detail_head_kernel");
}

int decnet_dynup_pack(const float *disp, const float *left_fea, float *out, int B, int C, int h, int w, void *stream) {
    DECNET_REQUIRE(disp && left_fea && out, "null pointer");
    DECNET_REQUIRE(B > 0 && C > 0 && h > 0 && w > 0, "non-positive size");
    DECNET_REQUIRE(C + 1 <= 65535 && B <= 65535, "C or B too large for the launch grid");
    const size_t smem = (size_t)9 * w * sizeof(float);
    DECNET_REQUIRE(smem <= 200 * 1024, "row too wide");
    if (smem > 48 * 1024)
        DECNET_CUDA(cudaFuncSetAttribute(dynup_pack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dynup_pack_kernel<<<dim3(h, C + 1, B), kBlock, smem, (cudaStream_t)stream>>>(disp, left_fea, out, C, h, w);
    return after_launch("dynup_pack_kernel");
}

int decnet_dynup_glue(const float *logits, const float *disp, float *out, int B, int h, int w, void *stream) {
    DECNET_REQUIRE(logits && disp && out, "null pointer");
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0, "non-positive size");
    const long long n = (long long)B * h * w;
    dynup_glue_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(logits, disp, out, B, h, w);
    return after_launch("dynup_glue_kernel");
}

int decnet_nchw_cat_to_nhwc_pad(const float *const *srcs, const int *src_channels, int nsrc, float *out,
                                int B, int h, int w, int CP, int round_tf32, void *stream) {
    DECNET_REQUIRE(srcs && src_channels && out, "null pointer");
    DECNET_REQUIRE(nsrc >= 1 && nsrc <= 3 && B > 0 && h > 0 && w > 0, "bad size");
    int c[3] = {0, 0, 0};
    const float *s[3] = {nullptr, nullptr, nullptr};
    int sum = 0;
    for (int i = 0; i < nsrc; ++i) { DECNET_REQUIRE(srcs[i] && src_channels[i] > 0, "source %d", i); c[i] = src_channels[i]; s[i] = srcs[i]; sum += c[i]; }
    DECNET_REQUIRE(CP >= sum, "CP=%d < %d channels", CP, sum);
    const size_t tile_bytes = (size_t)32 * (CP + 1) * sizeof(float);
    if ((CP & 3) == 0 && tile_bytes <= 48 * 1024 && h + 2 <= 65535 && B <= 65535 &&
        (reinterpret_cast<uintptr_t>(out) & 15u) == 0) {
        nchw_cat_to_nhwc_pad_tiled_kernel<<<dim3((w + 2 + 31) / 32, h + 2, B), kBlock, tile_bytes, (cudaStream_t)stream>>>(
            s[0], s[1], s[2], c[0], c[1], c[2], out, h, w, CP, round_tf32);
        return after_launch("nchw_cat_to_nhwc_pad_tiled_kernel");
    }
    const long long n = (long long)B * (h + 2) * (w + 2) * CP;
    nchw_cat_to_nhwc_pad_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(s[0], s[1], s[2], c[0], c[1], c[2],
                                                                                                     out, h, w, CP, round_tf32, n);
    return after_launch("nchw_cat_to_nhwc_pad_kernel");
}

int decnet_nhwc_pad_to_nchw(const float *in_pad, float *out, int B, int C, int NP, int h, int w, void *stream) {
    DECNET_REQUIRE(in_pad && out, "null pointer");
    DECNET_REQUIRE(B > 0 && C > 0 && C <= NP && h > 0 && w > 0, "bad size");
    const long long n = (long long)B * C * h * w;
    nhwc_pad_to_nchw_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(in_pad, out, C, NP, h, w, n);
    return after_launch("nhwc_pad_to_nchw_kernel");
}

int decnet_attn_pack(const float *left_fea, const float *dense, const float *sparse, const float *left_mask,
                     const float *var, float *out, int B, int C, int H, int W, void *stream) {
    DECNET_REQUIRE(dense && sparse && left_mask && var && out, "null pointer");
    DECNET_REQUIRE(B > 0 && C >= 0 && H > 0 && W > 0 && (C == 0 || left_fea), "bad size or null left_fea with C=%d", C);
    const long long HW = (long long)H * W;
    DECNET_REQUIRE((long long)B * (C + 4) <= 65535, "B*(C+4) too large");
    const uintptr_t al = reinterpret_cast<uintptr_t>(left_fea) | reinterpret_cast<uintptr_t>(dense) |
                         reinterpret_cast<uintptr_t>(sparse) | reinterpret_cast<uintptr_t>(left_mask) |
                         reinterpret_cast<uintptr_t>(var) | reinterpret_cast<uintptr_t>(out);
    const dim3 grid_v((unsigned)std::min<long long>((HW / 4 + kBlock - 1) / kBlock, 64), (unsigned)(B * (C + 4)));
    if ((HW & 3) == 0 && (al & 15u) == 0)
        attn_pack_kernel<float4><<<grid_v, kBlock, 0, (cudaStream_t)stream>>>(left_fea, dense, sparse, left_mask, var, out, C, HW / 4);
    else
        attn_pack_kernel<float><<<dim3((unsigned)std::min<long long>((HW + kBlock - 1) / kBlock, 64), (unsigned)(B * (C + 4))),
                                  kBlock, 0, (cudaStream_t)stream>>>(left_fea, dense, sparse, left_mask, var, out, C, HW);
    return after_launch("attn_pack_kernel");
}

int decnet_blend(const float *logit, const float *dense, const float *sparse, float *soft_mask, float *fused,
                 int B, int H, int W, void *stream) {
    DECNET_REQUIRE(logit && dense && sparse && fused, "null pointer");
    DECNET_REQUIRE(B > 0 && H > 0 && W > 0, "non-positive size");
    const long long n = (long long)B * H * W;
    blend_kernel<<<grid_for(n, 148 * 32), kBlock, 0, (cudaStream_t)stream>>>(logit, dense, sparse, soft_mask, fused, n);
    return after_launch("blend_kernel");
}

int decnet_warp_bilinear(const float *right_fea, const float *disp, float *warped, int B, int C, int H, int W, void *stream) {
    DECNET_REQUIRE(right_fea && disp && warped, "null pointer");
    DECNET_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "non-positive size");
    return launch_warp(nullptr, right_fea, disp, warped, nullptr, B, C, H, W, H, 0, (cudaStream_t)stream, "warp_kernel");
}

int decnet_refine_pack_rows(const float *left_fea, const float *right_fea, const float *disp, float *out,
                            int B, int C, int H, int W, int H_total, int row0, void *stream) {
    DECNET_REQUIRE(left_fea && right_fea && disp && out, "null pointer");
    DECNET_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "non-positive size");
    DECNET_REQUIRE(row0 >= 0 && row0 + H <= H_total, "row window [%d,%d) outside the %d-row image", row0, row0 + H, H_total);
    return launch_warp(left_fea, right_fea, disp, nullptr, out, B, C, H, W, H_total, row0, (cudaStream_t)stream, "warp_kernel<pack>");
}

int decnet_refine_pack(const float *left_fea, const float *right_fea, const float *disp, float *out,
                       int B, int C, int H, int W, void *stream) {
    return decnet_refine_pack_rows(left_fea, right_fea, disp, out, B, C, H, W, H, 0, stream);
}

int decnet_haar_level(const float *x, float *ll, float *detail, float *mask, void *workspace,
                      const float *thresholds10, int B, int H, int W, void *stream) {
    DECNET_REQUIRE(x && ll && detail && mask && workspace && thresholds10, "null pointer");
    DECNET_REQUIRE(B > 0 && B <= 65535 && H >= 2 && W >= 2, "bad size B=%d H=%d W=%d", B, H, W);
    const int h = H / 2, w = W / 2;
    const long long n = (long long)h * w;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned int *minmax = static_cast<unsigned int *>(workspace);           // [B][2]
    unsigned int *counts = minmax + 2 * (size_t)B;                            // [B][10]
    HaarThresholds th;
    for (int k = 0; k < 10; ++k) th.t[k] = thresholds10[k];
    // min slots start at +inf bits, max slots and the counters at 0
    DECNET_CUDA(cudaMemsetAsync(workspace, 0, (size_t)B * 12 * sizeof(unsigned int), st));
    DECNET_CUDA(cudaMemset2DAsync(minmax, 2 * sizeof(unsigned int), 0x7f, sizeof(unsigned int), B, st));
    const int gx = grid_for(n, 148 * 4);
    haar_analysis_kernel<<<dim3(gx, B), kBlock, 0, st>>>(x, ll, detail, minmax, H, W, h, w);
    int rc = after_launch("haar_analysis_kernel");
    if (rc) return rc;
    haar_count_kernel<<<dim3(gx, B), kBlock, 0, st>>>(detail, minmax, th, counts, n);
    rc = after_launch("haar_count_kernel");
    if (rc) return rc;
    haar_mask_kernel<<<dim3(gx, B), kBlock, 0, st>>>(detail, minmax, counts, th, mask, n);
    return after_launch("haar_mask_kernel");
}

int decnet_dynup_pack_nhwc(const float *disp, const float *left_fea, float *out, int B, int C, int h, int w, int CP,
                           int round_tf32, int pad, void *stream) {
    DECNET_REQUIRE(pad == 0 || pad == 1, "pad must be 0 or 1");
    DECNET_REQUIRE(left_fea && out, "null pointer");         // disp may be NULL: channel 0 is written as zero
    DECNET_REQUIRE(B > 0 && B <= 65535 && C > 0 && h > 0 && h <= 65535 && w > 0, "bad size");
    DECNET_REQUIRE(CP >= 9 * C + 1, "CP=%d must hold 9*C+1=%d channels", CP, 9 * C + 1);
    int TX = 1200 / C;                            // <= 43 KB of shared memory: 5 blocks per SM
    TX = TX > 128 ? 128 : (TX < 8 ? 8 : (TX & ~7));
    if (TX > w) TX = w;
    DECNET_REQUIRE((CP & 3) == 0, "CP must be a multiple of 4");
    const size_t smem = (size_t)C * 9 * TX * sizeof(float) + (size_t)CP * sizeof(int);
    DECNET_REQUIRE(smem <= 200 * 1024, "C too large");
    if (smem > 48 * 1024)
        DECNET_CUDA(cudaFuncSetAttribute(dynup_pack_nhwc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DECNET_REQUIRE(h + 2 <= 65535, "too many rows");
    dynup_pack_nhwc_kernel<<<dim3((w + TX - 1) / TX, h + 2 * pad, B), kBlock, smem, (cudaStream_t)stream>>>(disp, left_fea, out, C, h, w, CP, TX,
                                                                                                        round_tf32, pad);
    return after_launch("dynup_pack_nhwc_kernel");
}

int decnet_dynup_set_disp_nhwc(const float *disp, float *packed, int B, int h, int w, int CP, int round_tf32, int pad,
                               void *stream) {
    DECNET_REQUIRE(pad == 0 || pad == 1, "pad must be 0 or 1");
    DECNET_REQUIRE(disp && packed, "null pointer");
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0 && CP > 0, "bad size");
    const long long n = (long long)B * h * w;
    dynup_set_disp_nhwc_kernel<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(
        disp, packed, h, w, CP, round_tf32, pad, n);
    return after_launch("dynup_set_disp_nhwc_kernel");
}

int decnet_bicubic_up3(const float *pred, float *out, int B, int h, int w, int H, int W, void *stream) {
    DECNET_REQUIRE(pred && out, "null pointer");
    DECNET_REQUIRE(B > 0 && B <= 65535 && h > 0 && w > 0 && H > 0 && W > 0, "bad size B=%d %dx%d -> %dx%d", B, h, w, H, W);
    const long long strips = ((long long)H + kBicRows - 1) / kBicRows;
    DECNET_REQUIRE(strips <= 65535, "H=%d: too many rows for the launch grid", H);
    // ATen's area_pixel_compute_scale without an explicit scale factor: (float)input_size / output_size
    const float scale_h = (float)h / (float)H, scale_w = (float)w / (float)W;
    bicubic_up3_kernel<<<dim3((W + 127) / 128, (unsigned)strips, B), 128, 0, (cudaStream_t)stream>>>(pred, out, h, w, H, W,
                                                                                                   scale_h, scale_w);
    return after_launch("bicubic_up3_kernel");
}

int decnet_dynup_glue_nhwc(const float *logits, const float *disp, float *out, int B, int h, int w, int NP, int pad, void *stream) {
    DECNET_REQUIRE(pad == 0 || pad == 1, "pad must be 0 or 1");
    DECNET_REQUIRE(logits && disp && out, "null pointer");
    DECNET_REQUIRE(B > 0 && h > 0 && w > 0 && NP >= 81, "bad size");
    DECNET_REQUIRE(h <= 65535 && B <= 65535, "grid limit");
    const size_t smem = (size_t)kGluePx * (NP + 1) * sizeof(float);
    DECNET_REQUIRE(smem <= 48 * 1024, "NP too large");
    dynup_glue_nhwc_kernel<<<dim3((w + kGluePx - 1) / kGluePx, h, B), 9 * kGluePx, smem, (cudaStream_t)stream>>>(logits, disp, out, B, h, w, NP, pad);
    return after_launch("dynup_glue_nhwc_kernel");
}

}  // extern "C"
