/*
 * decnet_b200.h -- C ABI of libdecnet_b200.so (sm_100a).
 *
 * Drop-in boundary for DecNet's decomposed-matching hot path.  Every entry point
 * takes raw DEVICE pointers, explicit sizes and an explicit CUDA stream (passed
 * as void* == cudaStream_t; NULL is the legacy default stream), returns 0 on
 * success or a non-zero code (DECNET_ERR_* or a cudaError_t value offset by
 * DECNET_ERR_CUDA_BASE) and records a message readable through
 * decnet_last_error() (thread-local).  No torch / pybind types appear here.
 *
 * Unless stated otherwise tensors are fp32, contiguous, NCHW ("feats":
 * [B,C,H,W]) or [B,H,W] ("planes"), exactly what the reference's extension
 * receives (reference: modules/SparseMatching/src/SM_kernel.cu:359-376 reads
 * sizes from ref_feas.size(0..3) and data_ptr<float>()).
 *
 * Ownership: the caller allocates every output; the library never allocates
 * user-visible memory and retains no pointer after the call returns (work is
 * only enqueued on `stream`).  The forward entry points write EVERY element of
 * their [B,H,W] outputs (zeros where the left mask is 0), so outputs need not be
 * zero-filled (the reference requires zero-filled outputs:
 * modules/SparseMatching/functions/SpaMat.py:25-27).  The backward entry points
 * keep the reference contract: gradients must arrive zero-filled
 * (functions/SpaMat.py:42-43) and only masked positions are written.
 *
 * Thread safety: no global mutable state except per-device caches guarded by a
 * mutex; safe to call from one host thread per device (the reference is driven
 * by nn.DataParallel worker threads, eval.py:145-146).
 */
#ifndef DECNET_B200_H
#define DECNET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DECNET_ABI_VERSION 2

#define DECNET_OK 0
#define DECNET_ERR_INVALID 1      /* bad argument (null pointer, non-positive size, ...) */
#define DECNET_ERR_UNSUPPORTED 2  /* shape outside what the kernels support          */
#define DECNET_ERR_CUDA_BASE 1000 /* 1000 + cudaError_t                              */

int decnet_abi_version(void);
const char *decnet_last_error(void);
/* Number of SMs / compute capability of the current device (for host-side sizing). */
int decnet_device_info(int *sm_count, int *cc_major, int *cc_minor);
/* Kernel launches issued by this library on the calling thread since the last reset. */
int64_t decnet_launch_count(void);
void decnet_reset_launch_count(void);

/* ------------------------------------------------------------------------- *
 * Sparse matching (SURVEY.md section 8 rows a9-a12).
 *
 * Candidate set of pixel (b,h,w) with lmask != 0:
 *     { d : 0 <= d < min(max_disp, w+1), rmask[b,h,w-d] != 0 }
 *   cost_d   = sum_c L[b,c,h,w] * R[b,c,h,w-d]      (sequential FMA chain over c)
 *   max_cost = max(1e-6, max_d cost_d)
 *   e_d      = expf(cost_d - max_cost);  sum_sim = 1e-6 + sum_d e_d
 *   out      = (1e-6 + sum_d e_d * d) / sum_sim                    (SpaMat)
 *   var      = (1e-6 + sum_d e_d * (d - disp)^2) / sum_sim         (SpaVar)
 * Replaces: sparse_matching_cuda_forward  (modules/SparseMatching/src/SM_cuda.cpp:7-15,
 *           kernels SM_kernel.cu:22-125), sparse_var_cuda_forward
 *           (modules/SparseVar/src/SV_cuda.cpp:7-16, kernels SV_kernel.cu:22-124).
 * ------------------------------------------------------------------------- */
int decnet_spamat_fwd(const float *ref_feas, const float *tar_feas,
                      const float *ref_mask, const float *tar_mask,
                      float *output, float *sum_similarities, float *max_cost,
                      int B, int C, int H, int W, int max_disp, void *stream);

int decnet_spavar_fwd(const float *ref_feas, const float *tar_feas,
                      const float *ref_mask, const float *tar_mask,
                      const float *disparity,
                      float *output, float *sum_similarities, float *max_cost,
                      int B, int C, int H, int W, int max_disp, void *stream);

/* SpaMat followed by SpaVar(disparity = SpaMat output) in ONE pass over the
 * feature rows (what the model does back to back:
 * modules/SparseDenseNetRefinementMask.py:183-192). */
int decnet_spamat_spavar_fwd(const float *ref_feas, const float *tar_feas,
                             const float *ref_mask, const float *tar_mask,
                             float *disp_out, float *var_out,
                             float *sum_similarities, float *max_cost,
                             int B, int C, int H, int W, int max_disp, void *stream);

/* The same fused pass over the rows of SEVERAL pyramid levels in ONE launch (nlev <= 4; arrays of nlev HOST entries, one
 * per level, each with its own B, C, H, W, max_disp): the model runs the op at three levels whose inputs do not depend on each
 * other, and the coarse levels alone are one or two waves of latency.  Give the finest level first. */
int decnet_spamat_spavar_fwd_levels(int nlev, const float *const *ref_feas, const float *const *tar_feas,
                                    const float *const *ref_mask, const float *const *tar_mask,
                                    float *const *disp_out, float *const *var_out,
                                    float *const *sum_similarities, float *const *max_cost,
                                    const int *B, const int *C, const int *H, const int *W, const int *max_disp, void *stream);

/* Replaces sparse_matching_cuda_backward (SM_cuda.cpp:17-27, SM_kernel.cu:143-195,300-355). */
int decnet_spamat_bwd(const float *ref_feas, const float *tar_feas,
                      const float *ref_mask, const float *tar_mask,
                      const float *output, const float *sum_similarities,
                      const float *max_cost, const float *grad_output,
                      float *grad_ref_feas, float *grad_tar_feas,
                      int B, int C, int H, int W, int max_disp, void *stream);

/* Replaces sparse_var_cuda_backward (SV_cuda.cpp:18-30, SV_kernel.cu:142-325). */
int decnet_spavar_bwd(const float *ref_feas, const float *tar_feas,
                      const float *ref_mask, const float *tar_mask,
                      const float *disparity, const float *output,
                      const float *sum_similarities, const float *max_cost,
                      const float *grad_output,
                      float *grad_ref_feas, float *grad_tar_feas, float *grad_disparity,
                      int B, int C, int H, int W, int max_disp, void *stream);

/* Per-pixel candidate count and order-independent 64-bit hash of the candidate
 * set, produced by the SAME compaction code the matching kernels use.  Test hook
 * for the "candidate indices bit-exact" gate. */
int decnet_candidate_signature(const float *ref_mask, const float *tar_mask,
                               int32_t *count, uint64_t *hash,
                               int B, int H, int W, int max_disp, void *stream);

/* Which load path the last spamat/spavar forward on this thread used:
 * 0 = none, 1 = rows staged by cp.async (any W / alignment), 2 = rows staged by TMA,
 * 3 = no staging (sector-gather kernel). */
int decnet_last_sparse_path(void);
/* Force a staged path for the forward ops on this thread: 0 = auto, 1 = cp.async, 2 = TMA. */
void decnet_set_sparse_path(int path);
/* Forward row kernel:
 *   3 = sector-gather kernel (default): only the listed columns are read, straight from global memory into the
 *       compacted operand buffers; one row per CTA, 256 threads, 4 CTAs/SM; any W / alignment (needs path 0);
 *   4 = its software-pipelined form: persistent CTAs, every read issued one row ahead with cp.async;
 *   1 = one row per CTA with the [C,W] rows of both views staged in shared memory (3 CTAs/SM);
 *   2 = the same with persistent CTAs (2 per SM) that put the next row's rows and masks in flight before
 *       evaluating the current row.
 * set: 0 = auto (3; 1 when a staged path is forced or C*H*W >= 2^31), else force; last: what the last forward used. */
int decnet_last_sparse_variant(void);
void decnet_set_sparse_variant(int variant);

/* ------------------------------------------------------------------------- *
 * Coarse dense stage (SURVEY.md section 8 rows a1-a4).
 * ------------------------------------------------------------------------- */

/* Cost volume for the stage-0 candidates d = 0..D-1:
 *   vol[b,c,d,h,w] = (w >= d ? L[b,c,h,w] : 0) * bilinear0(R[b,c], y'(h), x'(w-d))
 * with the reference's coordinate quirk (normalise with (size-1)/2, sample with
 * align_corners=False, zero padding).  Output fp32 NCDHW [B,C,D,H,W].
 * Replaces GetCostVolume.forward / get_warped_feats_by_homgrp / cost_computation_cor
 * (modules/submodule.py:532-562, 479-510, 518-522) + get_disp_samples (:376-390). */
int decnet_costvol_fwd(const float *left_fea, const float *right_fea, float *vol,
                       int B, int C, int H, int W, int D, void *stream);

/* Same volume written as bf16 channels-last [B,D,H,W,Cpad] (Cpad >= C, multiple of 8,
 * channels C..Cpad-1 zero): the input layout of decnet_conv3d_* (tcgen05 implicit GEMM). */
int decnet_costvol_bf16_ndhwc(const float *left_fea, const float *right_fea, void *vol_bf16,
                              int B, int C, int Cpad, int H, int W, int D, void *stream);

/* Row-band variant (single huge pair split across GPUs, SURVEY.md section 8e): writes only the
 * rows [row0, row0+nrows) of the H-row volume -> [B,D,nrows,W,Cpad]; rows outside the image
 * (row0 < 0 or beyond H) are zeros, i.e. the aggregation's zero padding / halo slots. */
int decnet_costvol_bf16_ndhwc_rows(const float *left_fea, const float *right_fea, void *vol_bf16,
                                   int B, int C, int Cpad, int H, int W, int D,
                                   int row0, int nrows, void *stream);

/* pred[b,h,w] = sum_d softmax_d(cost[b,:,h,w]) * d.  Replaces disparity_regression
 * (modules/submodule.py:766-777) for integer candidates 0..D-1. */
int decnet_softargmin(const float *cost, float *pred, int B, int D, int H, int W, void *stream);

/* One Conv3dUnit of the aggregation stack (Conv3d 3x3x3 pad 1 no bias -> BN(eval) -> ReLU
 * [-> + residual], modules/submodule.py:90-123, 650-662) as a bf16 implicit GEMM on tcgen05
 * tensor cores, fp32 accumulation in TMEM.
 *   x        bf16 channels-last [B,D,H,W,cp]           (cp = padded C_in, multiple of 16)
 *   w_packed bf16 [27][np][cp], tap = (kd*3+kh)*3+kw, BN scale folded in, zero padded
 *   bias     fp32 [np] (BN shift), residual bf16 [B,D,H,W,np] or NULL (added AFTER the ReLU)
 *   out_mode 0: out bf16 [B,D,H,W,np];  1: out fp32 [B,D,H,W] = channel 0 (the 216->1 layer)
 * All pointers 16-byte aligned. */
int decnet_conv3d_bf16(const void *x_ndhwc, const void *w_packed, const float *bias,
                       const void *residual, void *out, int out_mode,
                       int B, int D, int H, int W, int cp, int np, int relu, void *stream);

/* Last layer of the aggregation stack (the 216->1 Conv3d, modules/submodule.py:659-662) together with the soft-argmin that
 * follows it (disparity_regression, modules/submodule.py:766-777, called at SparseDenseNetRefinementMask.py:237-239):
 *   cost fp32 [B,D,H,W] = channel 0 of the layer,  pred fp32 [B,H,W] = sum_d softmax_d(cost) * d.
 * When one 128-voxel tile box spans the whole D axis (D <= 8 at every published stage-0 size) the soft-argmin runs in the
 * conv epilogue of the same launch; otherwise decnet_softargmin follows on the same stream.  Both routes give the same bits. */
int decnet_conv3d_bf16_softargmin(const void *x_ndhwc, const void *w_packed, const float *bias, float *cost, float *pred,
                                  int B, int D, int H, int W, int cp, int np, int relu, void *stream);

/* Row-band form (SURVEY.md section 8e, one huge pair split across GPUs): the tensors are a band [B,D,rows+2,W,.] whose
 * rows 0 and rows+1 are halo slots.  The layer computes every owned row from the band (halo rows are inputs) and does NOT
 * store into the halo rows of `out`: they are filled by the neighbouring ranks over NVLink peer memory (decnet_b200/bands.py)
 * or stay zero at the image edge.  out_mode 0 only. */
int decnet_conv3d_bf16_band(const void *x_ndhwc, const void *w_packed, const float *bias, const void *residual,
                            void *out, int B, int D, int H, int W, int cp, int np, int relu, void *stream);

/* 3x3 Conv2d (pad 1, stride 1) + bias [+ ReLU] as a TF32 implicit GEMM on the same tcgen05 kernel
 * (kind::tf32, fp32 operands in shared memory, fp32 accumulation): the 81-channel convs of
 * DynamicUpsampling.weight_learning (modules/submodule.py:571-575), which are GEMM-sized.
 *   x fp32 channels-last [B,H,W,cp] (cp multiple of 8), w_packed fp32 [9][np][cp] (tap = ky*3+kx, BN folded),
 *   bias fp32 [np], out fp32 channels-last [B,H,W,np] (np multiple of 16).  Same precision class as
 *   cuDNN's default TF32 convolutions.
 *   round_out_tf32 != 0 rounds the stored outputs to TF32 (nearest) when they feed another tf32 conv
 *   (the MMA itself truncates; callers should likewise pre-round x and w_packed). */
int decnet_conv2d_tf32_nhwc(const float *x_nhwc, const float *w_packed, const float *bias, float *out,
                            int B, int H, int W, int cp, int np, int relu, int round_out_tf32, void *stream);

/* 3x3 Conv2d (stride 1, padding = dilation) + bias [+ ReLU] on NCHW fp32 tensors as a TF32 implicit GEMM
 * with pixels as the MN-major M dimension (conv2d_tcgen05.cu): the 1..24-channel layers of
 * GenerateSparseMask / SoftAttention / Refinement (modules/submodule.py:347-372, 593-604, 666-762), which the
 * reference runs through cuDNN (TF32 by default).  Operands are rounded to TF32 (nearest) in the kernel.
 *   x fp32 [B,Cin,H,W]; out fp32 [B,Cout,H,W]; bias_padded fp32 [CP] (CP = 4 when Cout <= 4, else Cout rounded up to 8);
 *   w_packed fp32, decnet_conv2d_tf32_packed_floats(Cin,Cout) values laid out as rows of 32:
 *     row = ((kh*nck + chunk)*natoms + atom)*8 + k,  column n  <->  input channel chunk*8+k, GEMM column
 *     atom*32+n = kw*CP + cout  (nck = ceil(Cin/8), natoms = ceil(3*CP/32));
 *     BN folded in, TF32-rounded, zero padded.
 * decnet_conv2d_tf32_supported: 1 when the shape fits (W % 4 == 0, dilation 1..12, 3*CP <= 256,
 * resident weights <= 96 KB). */
int decnet_conv2d_tf32_supported(int Cin, int Cout, int H, int W, int dilation);
int decnet_conv2d_tf32_packed_floats(int Cin, int Cout);
int decnet_conv2d_tf32_nchw(const float *x, const float *w_packed, const float *bias_padded, float *out,
                            int B, int Cin, int Cout, int H, int W, int dilation, int relu, void *stream);
/* Same convolution over the channel concatenation of `nsrc` (1..3) NCHW tensors, without materialising the
 * cat (torch.cat((left, dense, sparse, mask, -var)) before SoftAttention, SparseDenseNetRefinementMask.py:197;
 * cat((left, warped_right, disp)) in Refinement, modules/submodule.py:758-759).  Source i has src_channels[i]
 * channels and occupies ceil(src_channels[i]/8) whole chunks of the packed weights: pack as if the input had
 * sum(8*ceil(C_i/8)) channels with zero weights in each source's padding.
 * w_valid (0 = W): output columns >= w_valid are written as zeros.  Images whose width is not a multiple of 4
 * (KITTI: 1269) run through this kernel as tensors padded on the right to a 16-byte row pitch; the padding is kept
 * at zero layer after layer, and zeros right of the image are exactly the convolution's own padding. */
int decnet_conv2d_tf32_nchw_cat(const float *const *srcs, const int *src_channels, int nsrc, const float *w_packed,
                                const float *bias_padded, float *out, int B, int Cout, int H, int W, int dilation,
                                int relu, int w_valid, void *stream);

/* Precision-selectable forms of the two entry points above (the ones the model calls).
 *   split = 0: plain TF32 (operands rounded to TF32: cuDNN's default convolution precision on a GPU);
 *   split = 1: error-compensated "3xTF32": both operands are split into TF32 hi + lo parts (x: in the kernel; weights:
 *              by the caller, w_packed = the hi rows followed by the lo rows, 2x decnet_conv2d_tf32_packed_floats values)
 *              and every tap issues lo*hi + hi*lo + hi*hi into the same fp32 accumulator.  The result is fp32-class
 *              (~2^-22 relative per product).
 *   split = 2: the same hi/lo decomposition with the two correction products as ONE kind::f16 MMA per tap (the default of
 *              the Python side): the kernel writes [fp16(2^11 * lo(x)) | fp16(x)] (8 + 8 channels) beside the raw tile, the
 *              second half of w_packed holds, per 1 KB block [kh][chunk][n-atom], the MN-major SWIZZLE_64B fp16 operand
 *              [K atom 0: fp16(hi(w) * 2^sw) | K atom 1: fp16(lo(w) * 2^(11+sw))] (8 k x 32 n halves each; its 16-byte units
 *              pre-permuted for the 128B_ATOM_32B TMA map: unit g holds logical unit s64(s128a32(g))), the first half holds
 *              hi(w) * 2^(11+sw), and bias_padded[CP] = 2^-(11+sw) (bias_padded has CP + 4 floats).  sw: any integer that keeps
 *              |w| * 2^sw below 2^15 (decnet_b200/ops.py: _pack_nchw_split16).  Same error budget as split = 1, two MMAs per
 *              tap instead of three.
 * The split modes are those on which the 1e-3 parity gates against the reference's fp32 execution run (the layers the
 * reference computes with F.conv2d: modules/submodule.py:15-49). */
int decnet_conv2d_tc_supported(int Cin, int Cout, int H, int W, int dilation, int split);
int decnet_conv2d_tc_packed_floats(int Cin, int Cout, int split);
int decnet_conv2d_tc_nchw_cat(const float *const *srcs, const int *src_channels, int nsrc, const float *w_packed,
                              const float *bias_padded, float *out, int B, int Cout, int H, int W, int dilation,
                              int relu, int w_valid, int split, void *stream);
/* The same with a single-channel addend [B,H,W] (Cout == 1) added after the activation: the refinement's
 * `disp_map + residual` (modules/submodule.py:761) in the epilogue of its last conv.  addend NULL = the call above. */
int decnet_conv2d_tc_nchw_cat_add(const float *const *srcs, const int *src_channels, int nsrc, const float *w_packed,
                                  const float *bias_padded, const float *addend, float *out, int B, int Cout, int H, int W,
                                  int dilation, int relu, int w_valid, int split, void *stream);

/* Second formulation of the same convolution for C_out <= 8, dilation <= 4 (conv2d_rows_tcgen05.cu): pixels on the
 * GEMM N dimension, block-Toeplitz weights on M, column taps as accumulator column offsets -- the epilogue needs no
 * shuffles and stores 128 bits per thread.  Same sources / output contract as decnet_conv2d_tf32_nchw_cat.
 *   w_compact fp32 [3 kh][3 kw][nck][8 c_out][8 c_in] (nck = sum over sources of ceil(C_i/8); each source padded to
 *   whole 8-channel chunks; BN folded, TF32-rounded, zero padded); bias8 fp32 [8].
 * decnet_conv2d_tf32_rows_supported takes the padded input channel count (8*nck). */
int decnet_conv2d_tf32_rows_supported(int Cin_padded, int Cout, int H, int W, int dilation);
int decnet_conv2d_tf32_rows_nchw_cat(const float *const *srcs, const int *src_channels, int nsrc, const float *w_compact,
                                     const float *bias8, float *out, int B, int Cout, int H, int W, int dilation,
                                     int relu, void *stream);

/* The same TF32 convolution on channels-last tensors that carry a one-pixel ZERO border: x_pad fp32 [B,h+2,w+2,cp],
 * out_pad fp32 [B,h+2,w+2,np] (border written as zeros, so layers chain without a padding pass).  One TMA fill per
 * (row tap, 32-channel chunk) serves the three column taps through row-shifted UMMA descriptors
 * (conv2d_nhwc_tcgen05.cu); weights / bias as for decnet_conv2d_tf32_nhwc. */
int decnet_conv2d_tf32_nhwc_halo(const float *x_pad, const float *w_packed, const float *bias, float *out_pad,
                                 int B, int h, int w, int cp, int np, int relu, int round_out_tf32, void *stream);

/* split = 1: 3xTF32 mode of the same kernel (see decnet_conv2d_tc_nchw_cat): x_pad is plain fp32 (NOT pre-rounded; four
 * converter warps split it into hi + lo tiles in shared memory), w_packed is [18][np][cp] (taps 0-8 the TF32 hi parts of
 * the weights, 9-17 the lo parts), round_out_tf32 should be 0.
 * split = 2 (default of the Python side): the corrections as one K-concatenated kind::f16 MMA per column tap.  Taps 9-17 of
 * w_packed hold, per output channel row and 32-channel chunk of cl channels, the 4*cl bytes
 * [fp16(hi(w) * 2^sw) x cl | fp16(lo(w) * 2^(11+sw)) x cl]; the kernel builds [fp16(2^11 * lo(x)) x cl | fp16(x) x cl]; taps
 * 0-8 are the plain TF32 hi parts; bias has np + 4 floats and bias[np] = 2^-(11+sw), the factor of the correction accumulator
 * (decnet_b200/ops.py: _pack_split_weights).  np <= 96 for the 3x3 form in the split modes (two stages must fit in shared memory).
 * The same holds for the _ldc form and for decnet_gemm_tc_nhwc (taps 0 / 1 instead of 0-8 / 9-17).
 * split = 3 (split16 input; the Python side's default inside the DynamicUpsampling and wide Refinement stacks): x_pad holds
 * "split16" storage, the same 4 bytes per channel, per 32-channel chunk of cl channels the halves
 * [fp16(2^11 * (x - h)) x cl | h x cl] with h = fp16(x), both rounded to nearest and saturating; cp % 16 == 0.  w_packed is
 * [9][np][cp], split = 2's taps 9-17 alone; bias[np] = 2^-(11+sw) and bias[np + 1] = 2^-sw.  Results are fp32-class (the
 * 3xTF32 error budget) for |activations| < 65504; beyond that the stored halves saturate and the results stay finite.
 * round_out is the output's storage format: 0 fp32, 1 fp32 rounded to TF32, 2 split16 (out_pad then holds np channels of
 * split16, as the next split = 3 layer reads them). */
int decnet_conv2d_tc_nhwc_halo(const float *x_pad, const float *w_packed, const float *bias, float *out_pad,
                               int B, int h, int w, int cp, int np, int relu, int round_out, int split, void *stream);

/* Tuning switch (per calling thread): 0 / 1 = one 128-pixel tile per CTA (default); 2 = split-mode launches with at least two
 * tiles per SM and np <= 96 run the pair kernel (two tiles per CTA share every weight stage: 1.7x fewer bytes from L2 per MMA;
 * bit-identical, not faster at the product shapes: DESIGN.md section 3.4); 100 + mask = knock-out timing (results wrong). */
void decnet_conv2d_nhwc_set_variant(int variant);

/* The same kernel writing a channel slice of a wider bordered tensor (row stride ldc floats, np channels from out_pad). */
int decnet_conv2d_tc_nhwc_halo_ldc(const float *x_pad, const float *w_packed, const float *bias, float *out_pad,
                                   int B, int h, int w, int cp, int np, int ldc, int relu, int split, void *stream);

/* GEMM mode of the same kernel (one tap): out[p, 0..np) = act(bias + sum_k x[p, k] * w[n, k]) over P rows of cp channels --
 * the 1x1 convs of the feature extractor, and (behind decnet_im2col3x3) its stride-3, dilated and 1/27-resolution 3x3 convs
 * and the GEMM form of its 216 -> 72 transposed conv (modules/submodule.py:225-241, 272-286, 162-177).
 *   x fp32 [P, cp] (cp multiple of 8, rows 16-byte aligned), w_packed fp32 [1 or 2 (split: hi, then lo / fp16 rows)][np][cp],
 *   bias [np] (split = 2: [np + 4], see decnet_conv2d_tc_nhwc_halo),
 *   out rows of ldc floats (np <= ldc: writes a channel slice of a wider tensor; np <= 128 in split mode).
 *   border_B > 0: the rows are the pixels of a zero-bordered [border_B, border_h+2, border_w+2] tensor; border rows are
 *                 stored as zeros (same pixel index in and out).
 *   dst_h > 0   : the P = B*dst_h*dst_w rows of a flat grid are stored at the interior pixels of a zero-bordered
 *                 [B, dst_h+2, dst_w+2, ldc] tensor (whose border the caller zeroed). */
int decnet_gemm_tc_nhwc(const float *x, const float *w_packed, const float *bias, float *out, long long P, int cp, int np,
                        int ldc, int relu, int split, int border_B, int border_h, int border_w, int dst_h, int dst_w, void *stream);

/* Feature-extractor data movement (featext.cu).
 *   decnet_im2col3x3: out[(b*Ho+yo)*Wo+xo][tap*C + c] = src(b, c, yo*stride + (ky-1)*dil, xo*stride + (kx-1)*dil), zero outside
 *     the logical HxW grid, columns 9C..Kp-1 zero; src is addressed as src[b*sb + c*sc + y*sy + x*sx] (element strides; sc = 1:
 *     channels-last, flat or the interior of a bordered tensor; sx = 1: NCHW).
 *   decnet_deconv3x3s3_shuffle: in [B*h*w, ld_in] with column (ky*3+kx)*Cout + co -> out_pad[b, 3y+ky+1, 3x+kx+1, c_off+co]
 *     of a zero-bordered channels-last [B, 3h+2, 3w+2, ldc] tensor (ConvTranspose2d k 3 s 3 as a GEMM + this shuffle).
 *   decnet_nhwc_to_nchw: channels-last rows of ld floats (pad = 1: interior of a bordered tensor) -> NCHW [B, C, h, w].
 *   decnet_conv3x3s3_nchw: Conv2d(3x3, stride 3, pad 1) + bias [+ ReLU] on NCHW, direct fp32, Cout = 24;
 *     w_packed [Cin][9][Cout]. */
int decnet_im2col3x3(const float *src, float *out, int B, int C, int H, int W, long long sb, long long sc, long long sy,
                     long long sx, int stride, int dilation, int Ho, int Wo, int Kp, void *stream);
int decnet_deconv3x3s3_shuffle(const float *in, float *out_pad, int B, int h, int w, int Cout, int ld_in, int ldc, int c_off,
                               void *stream);
int decnet_nhwc_to_nchw(const float *in, float *out, int B, int C, int ld, int h, int w, int pad, void *stream);
int decnet_conv3x3s3_nchw(const float *x, const float *w_packed, const float *bias, float *out, int B, int Cin, int H, int W,
                          int Cout, int relu, void *stream);

/* Layout bridges around decnet_conv2d_tf32_nhwc_halo for layers whose neighbours are NCHW (the 72-channel refinement
 * layers of the 1/9 level): concatenation of up to three NCHW fp32 sources -> zero-bordered channels-last
 * [B,h+2,w+2,CP] (channel padding zero; format: 0 fp32, 1 rounded to TF32 for the kernel's plain-TF32 mode, 2 split16
 * for its split = 3 mode, CP % 16 == 0), and back: interior / first C channels -> NCHW [B,C,h,w]. */
int decnet_nchw_cat_to_nhwc_pad(const float *const *srcs, const int *src_channels, int nsrc, float *out,
                                int B, int h, int w, int CP, int format, void *stream);
int decnet_nhwc_pad_to_nchw(const float *in_pad, float *out, int B, int C, int NP, int h, int w, void *stream);

/* Profiling hook: when set to a device buffer of 4*SMs int64, every conv3d launch on this thread
 * records per CTA {issuer cycles, cycles blocked on operand barriers, elapsed ns, k-iterations};
 * pass NULL to disable (default). */
void decnet_conv2d_tf32_debug(int flags, void *prof16);   /* tuning only: knock-out mask (1 converters idle, 2 no epilogue, 4 no MMAs) and per-role wait cycles of CTA 0 of conv2d_tcgen05_kernel (16 int64), or NULL */
void decnet_conv2d_nhwc_debug_trace(void *buffer);   /* tuning only: clock64 timeline of CTA 0 of conv2d_nhwc_halo_kernel (2560 int64), or NULL */
void decnet_conv3d_debug_timing(void *dbg_buffer);
/* 0 = auto (single-CTA kernel), 1 = force single-CTA, 2 = CTA-pair kernel (tcgen05 cta_group::2,
 * correct but slower in round 1; kept for tuning).  Per calling thread. */
void decnet_conv3d_set_variant(int variant);

/* ------------------------------------------------------------------------- *
 * Lost-detail mask selection (row a6).
 *   m = p > thold ? 1 : (p <= thold ? 0 : p)  for the left and right maps [B,H,W];
 * row_count_* (optional, [B*H] int32) receive the number of selected pixels per row.
 * Replaces the clone + 4 boolean index_puts of
 * modules/SparseDenseNetRefinementMask.py:164-170. */
int decnet_mask_threshold(const float *prob_l, const float *prob_r, float thold,
                          float *mask_l, float *mask_r,
                          int32_t *row_count_l, int32_t *row_count_r,
                          int B, int H, int W, void *stream);

/* ------------------------------------------------------------------------- *
 * Fusion / up-sampling glue (rows a8, a13, a14).
 * ------------------------------------------------------------------------- */

/* DynamicUpsampling conv input: out[B,1+9C,h,w], ch0 = disp, ch 1+c*9+ky*3+kx =
 * left_fea[b,c,3y+ky,3x+kx]; left_fea is [B,C,3h,3w].  Replaces unfold + cat
 * (modules/submodule.py:580). */
int decnet_dynup_pack(const float *disp, const float *left_fea, float *out,
                      int B, int C, int h, int w, void *stream);

/* DynamicUpsampling output: logits [B,81,h,w] (channel = sub*9+k), disp [B,h,w] ->
 * out [B,3h,3w] = 3 * sum_k softmax_k(logits[sub]) * disp_replicate_pad[y+ky-1, x+kx-1],
 * pixel-shuffled.  Replaces softmax/unfold/mul/sum/pixel_shuffle (submodule.py:581-589). */
int decnet_dynup_glue(const float *logits, const float *disp, float *out,
                      int B, int h, int w, void *stream);

/* Channels-last variants around decnet_conv2d_tf32_nhwc: pack writes [B,h,w,CP] (CP >= 9C+1, padding
 * channels zero), glue reads logits [B,h,w,NP] (NP >= 81, channel = sub*9+k).  pad = 1: both tensors are
 * [B,h+2,w+2,.] with a one-pixel zero border (decnet_conv2d_tf32_nhwc_halo's layout; the pack writes the border).
 * format as for decnet_nchw_cat_to_nhwc_pad (2: split16, CP % 16 == 0). */
int decnet_dynup_pack_nhwc(const float *disp, const float *left_fea, float *out,
                           int B, int C, int h, int w, int CP, int format, int pad, void *stream);
int decnet_dynup_glue_nhwc(const float *logits, const float *disp, float *out,
                           int B, int h, int w, int NP, int pad, void *stream);
/* The feature channels do not depend on the disparity: decnet_dynup_pack_nhwc with disp = NULL writes channel 0 as
 * zero (it can run ahead of the disparity, on another stream) and this fills channel 0 of the interior pixels. */
int decnet_dynup_set_disp_nhwc(const float *disp, float *packed,
                               int B, int h, int w, int CP, int format, int pad, void *stream);

/* Skip-stage up-sampling (row a15; modules/SparseDenseNetRefinementMask.py:143-144): pred fp32 [B,h,w] (contiguous) ->
 * out fp32 [B,H,W] = F.interpolate(pred*3, (H, W), mode="bicubic", align_corners=False), bit for bit what ATen's CUDA
 * kernel returns: v = pred*3 rounded first, source index (h/H)*(y+0.5)-0.5, A = -0.75, clamped border taps, the four
 * rows interpolated along x, then along y.  Any output size (a row band of the map is not an exact x3). */
int decnet_bicubic_up3(const float *pred, float *out, int B, int h, int w, int H, int W, void *stream);

/* Tail of GenerateSparseMask (modules/submodule.py:363-369) for BOTH views in one launch each:
 *   decnet_sqdiff_pair : out_i = (a_i - b_i)^2, i = 0 (left), 1 (right); n elements each
 *   decnet_detail_head : logit = bias + sum_c w3[c] * x[b,c,h,w] (the 3->1 1x1 conv with BN folded; w3 is a HOST
 *                        pointer to 3 floats), mask = logit >= logit_thold ? 1 : 0 (NaN kept), where the caller
 *                        passes logit_thold = the smallest float whose sigmoid exceeds the probability threshold,
 *                        i.e. mask == (sigmoid(logit) > thold) of SparseDenseNetRefinementMask.py:158-170. */
int decnet_sqdiff_pair(const float *a0, const float *b0, float *out0, const float *a1, const float *b1, float *out1,
                       long long n, void *stream);
int decnet_detail_head(const float *x_l, const float *x_r, const float *w3_host, float bias, float logit_thold,
                       float *mask_l, float *mask_r, int B, int H, int W, void *stream);

/* SURVEY.md section 8f rank 3: one pyramid level of the image-space lost-detail detector `detailDetection`
 * (utils/utils.py:447-534, called with scale 3, three levels, thold 0.3 in demo.py:161-162), cv2's float32
 * arithmetic restated on the device.  data fp32 [B,3,H,W] in [0,1] (H, W multiples of 3), down fp32 [B,3,H/3,W/3]
 * (the next level's data), mask fp32 [B,H,W] in {0,1}; scratch holds decnet_detail_level_scratch_floats floats. */
long long decnet_detail_level_scratch_floats(int B, int H, int W);
int decnet_detail_level(const float *data, float *down, float *mask, float *scratch, float thold,
                        int B, int H, int W, void *stream);

/* SURVEY.md section 8f rank 4: the data formats either side of the path.
 *   decnet_image_prepare_u8: uint8 RGB [B,h,w,3] -> top/left zero pad to HxW (demo.py:75-81), out01 = v/255 fp32
 *     [B,3,H,W] (input of detailDetection, demo.py:158-162) and out_norm = (v/255 - mean)/std (demo.py:82-88); either
 *     output may be NULL; mean3 / std3 are HOST pointers.
 *   decnet_image_prepare_u8_shift: decnet_image_prepare_u8 of the image shifted right by col_shift columns: image column
 *     x takes the input's column x - col_shift, and 0 (black) where that lies outside [0, w); any col_shift, negative
 *     included.  Bit for bit the unshifted entry run on the shifted image.  StereoMatcher prepares the right views of a
 *     search range [min_disp, max_disp) with col_shift = min_disp.
 *   decnet_disp_to_u16: clamp(pred*256, 0, 65535) truncated to uint16 and cropped to the last ori_h rows / ori_w
 *     columns (demo.py:191-197; the PNG container is written on the host).
 *   decnet_disp_add: pred[i] = pred[i] + offset in fp32 rounded to nearest (__fadd_rn), in place over n > 0 floats; pred
 *     4-byte aligned, 16-byte vector accesses on its aligned body.  Adds min_disp back to the shifted search's prediction.
 *   decnet_epe_3px: sums3 (device, 3 doubles) = {sum |pred-gt|, #(|err|<3 or <5% gt), #valid} over 0 < gt < max_disp
 *     (modules/loss.py:427-437: epe = sums[0]/sums[2], loss_3 = 100 - 100*sums[1]/sums[2]). */
int decnet_image_prepare_u8(const unsigned char *img_hwc, float *out01, float *out_norm, const float *mean3_host,
                            const float *std3_host, int B, int h, int w, int H, int W, void *stream);
int decnet_image_prepare_u8_shift(const unsigned char *img_hwc, float *out01, float *out_norm, const float *mean3_host,
                                  const float *std3_host, int B, int h, int w, int H, int W, int col_shift, void *stream);
int decnet_disp_to_u16(const float *pred, unsigned short *out, int B, int H, int W, int ori_h, int ori_w, void *stream);
int decnet_disp_add(float *pred, float offset, long long n, void *stream);
int decnet_epe_3px(const float *pred, const float *gt, float max_disp, double *sums3, long long n, void *stream);

/* Left-right consistency check of StereoMatcher (no counterpart in the reference; oracle/lr_check.py is the spec).
 * The reverse disparity of a pair (L, R) is the model run on (mirror(R), mirror(L)), mirror = column flip, cropped like the
 * forward one and mirrored back.
 *   decnet_mirror_swap_u8: out_left[b] = mirror(right[b]), out_right[b] = mirror(left[b]) on uint8 RGB [B,h,w,3] -- the
 *     reverse direction's input.  16-byte accesses when w % 16 == 0 and all pointers are 16-byte aligned, words when
 *     w % 4 == 0 (4-byte aligned), bytes otherwise.
 *   decnet_lr_check: pred fp32 [2B,H,W] padded predictions, images 0..B-1 forward, B..2B-1 the mirrored reverse.  Over the
 *     cropped pixels (the last ori_h rows / ori_w columns), dl = forward, in fp32 without contraction:
 *       u = floor((x - dl) + 0.5);  valid = isfinite(dl) && 0 <= u < ori_w && |dl - dr[u]| <= tol   (NaN dr: invalid)
 *     where dr[u] is the reverse image's padded column W-1-u.  Outputs [B,ori_h,ori_w], each may be NULL (not all):
 *     out_f32 = valid ? dl : 0, out_u16 = valid ? decnet_disp_to_u16's value of dl : 0, out_valid = valid (0 / 1 bytes).
 *   decnet_lr_check_fill: the same check, then background hole filling of the invalid pixels (oracle/lr_fill.py is the
 *     spec), each output a copy of a valid dl.  Row phase: an invalid pixel with valid neighbours L (nearest to the left)
 *     and R (nearest to the right) in its row takes dl[R] if dl[R] < dl[L], else dl[L]; with one of them, its value.
 *     Column phase: a row without a valid pixel takes, column by column, the same rule on the row-phase values of the
 *     nearest rows above and below that have one.  An image without a valid pixel stays 0.  out_f32 and row_flags
 *     [B,ori_h] are required (the column phase reads the float rows; row_flags = the row has a valid pixel); out_u16 =
 *     decnet_disp_to_u16's value of the float output; out_valid is the check's mask, 0 on every filled pixel.  No limit on
 *     ori_w beyond the check's.
 *   decnet_lr_check_guided_fill: decnet_lr_check_fill, then edge-aware filling guided by the left images guide (uint8 RGB
 *     [B,ori_h,ori_w,3]; oracle/lr_guided.py is the spec), in fp32 with every operation rounded separately.  Edge weights
 *     w(k) = (float)exp(-k / sigma_color) in double, k = sum_c |guide_c(p) - guide_c(q)| of neighbours p, q.  Three
 *     iterations t = 1..3 with lam_t = (float)(lambda * 1.5 * 4^(3-t) / 63) (double) each solve every row, then every
 *     column: (I + L) x = f on a line of n pixels, a_i = lam_t * w(k_i) between pixels i and i+1 (a_-1 = a_(n-1) = 0), by
 *     b_i = (1 + a_(i-1)) + a_i, m_i = b_i - a_(i-1) g_(i-1), r_i = 1 / m_i, g_i = a_i r_i, y_i = (f_i + a_(i-1) y_(i-1)) r_i,
 *     x_(n-1) = y_(n-1), x_i = y_i + g_i x_(i+1), for num (starting as valid ? dl : 0) and den (valid ? 1 : 0).  Then an
 *     invalid pixel whose den >= 2^-126 takes num / den; every other pixel keeps its decnet_lr_check_fill value (an image
 *     without a valid pixel stays 0).  lambda must be finite and >= 0 (0: the background fill), sigma_color finite and
 *     > 0.  guide, out_f32, out_valid, row_flags [B,ori_h] and scratch (decnet_lr_guided_fill_scratch_floats floats) are
 *     required; out_u16 = decnet_disp_to_u16's value of the float output; out_valid is the check's mask.  No limit on ori_h
 *     or ori_w beyond the check's.
 *   decnet_lr_check_speckle: the same check, then a speckle filter (oracle/lr_speckle.py is the spec), then fill 0 (none,
 *     as decnet_lr_check), 1 (background, as decnet_lr_check_fill) or 2 (guided, as decnet_lr_check_guided_fill with
 *     lambda and sigma_color) on the filtered mask.  Per image, two valid 4-neighbours (never diagonal) are joined when
 *     |dl_a - dl_b| <= max_diff in fp32; every pixel of a connected region of at most max_size pixels becomes invalid (its
 *     value 0 before the fill).  out_valid is the filtered mask, every output a copy of a valid dl.  max_size must be
 *     >= 0 (0: exactly the entry without the filter), max_diff finite and >= 0, B*ori_h*ori_w < 2^31 (int32 labels).
 *     guide is required for fill 2 and only for it; the other outputs as for that fill's entry.  scratch holds
 *     decnet_lr_speckle_scratch_bytes(B, ori_h, ori_w, fill) bytes, 16-byte aligned.  No other limit on ori_h or ori_w. */
int decnet_mirror_swap_u8(const unsigned char *left, const unsigned char *right, unsigned char *out_left,
                          unsigned char *out_right, int B, int h, int w, void *stream);
int decnet_lr_check(const float *pred, int B, int H, int W, int ori_h, int ori_w, float tol, float *out_f32,
                    unsigned short *out_u16, unsigned char *out_valid, void *stream);
int decnet_lr_check_fill(const float *pred, int B, int H, int W, int ori_h, int ori_w, float tol, float *out_f32,
                         unsigned short *out_u16, unsigned char *out_valid, unsigned char *row_flags, void *stream);
long long decnet_lr_guided_fill_scratch_floats(int B, int ori_h, int ori_w);
int decnet_lr_check_guided_fill(const float *pred, const unsigned char *guide, int B, int H, int W, int ori_h, int ori_w,
                                float tol, double lambda, double sigma_color, float *out_f32, unsigned short *out_u16,
                                unsigned char *out_valid, unsigned char *row_flags, float *scratch, void *stream);
long long decnet_lr_speckle_scratch_bytes(int B, int ori_h, int ori_w, int fill);
int decnet_lr_check_speckle(const float *pred, const unsigned char *guide, int B, int H, int W, int ori_h, int ori_w,
                            float tol, int max_size, float max_diff, int fill, double lambda, double sigma_color,
                            float *out_f32, unsigned short *out_u16, unsigned char *out_valid, unsigned char *row_flags,
                            void *scratch, void *stream);

/* SoftAttention conv input cat(left_fea, dense, sparse, left_mask, -var) -> [B,C+4,H,W]
 * (modules/SparseDenseNetRefinementMask.py:197).  C = 0 (left_fea may be NULL) packs only the four
 * single-channel maps -> [B,4,H,W], the second source of decnet_conv2d_tf32_nchw_cat. */
int decnet_attn_pack(const float *left_fea, const float *dense, const float *sparse,
                     const float *left_mask, const float *var, float *out,
                     int B, int C, int H, int W, void *stream);

/* m = sigmoid(logit); fused = dense*(1-m) + m*sparse; soft_mask may be NULL.
 * Replaces F.sigmoid (submodule.py:604) + the blend (SparseDenseNetRefinementMask.py:202). */
int decnet_blend(const float *logit, const float *dense, const float *sparse,
                 float *soft_mask, float *fused, int B, int H, int W, void *stream);

/* warped[b,c,h,w] = bilinear0(right_fea[b,c], y'(h), x'(w - disp[b,h,w])).
 * Replaces Refinement.get_warped_feats_by_homgrp (modules/submodule.py:719-745). */
int decnet_warp_bilinear(const float *right_fea, const float *disp, float *warped,
                         int B, int C, int H, int W, void *stream);

/* Refinement conv input cat(left_fea, warped, disp) -> [B,2C+1,H,W] in one pass
 * (modules/submodule.py:757-759). */
int decnet_refine_pack(const float *left_fea, const float *right_fea, const float *disp, float *out,
                       int B, int C, int H, int W, void *stream);

/* ------------------------------------------------------------------------- *
 * Haar wavelet lost-detail masks (row a7; utils/Wavelet.py:8-123).  One x2 level:
 *   x [B,1,H,W] -> ll [B,1,H/2,W/2] (next level's input), detail = max(|LH|,|HL|,|HH|),
 *   mask = ((detail-min)/(max-min) >= t), t = first of thresholds10 with >= 85 % of the
 *   pixels below it (else 1.0).  thresholds10 is a HOST array (float32 of
 *   numpy.arange(0,1,.1)+.1).  workspace: device, >= 48*B bytes.
 * The reference's filter bank (wavelet_weights_c2.pkl) is not in the repository:
 * orthonormal Haar is used and parity for this row is UNPINNED. */
int decnet_haar_level(const float *x, float *ll, float *detail, float *mask, void *workspace,
                      const float *thresholds10, int B, int H, int W, void *stream);

/* Row-band variant of decnet_refine_pack: the tensors hold the H rows [row0, row0+H) of an
 * H_total-row image; the vertical sampling coordinate uses GLOBAL rows (the reference's
 * y' = h*H/(H-1) - 1/2 depends on them), taps outside the window read 0. */
int decnet_refine_pack_rows(const float *left_fea, const float *right_fea, const float *disp, float *out,
                            int B, int C, int H, int W, int H_total, int row0, void *stream);

/* ------------------------------------------------------------------------- *
 * Tiny-channel 2-D convolutions of the per-level stacks (SURVEY.md section 8f rank 1;
 * modules/submodule.py:351-364 GenerateSparseMask, :596-600 SoftAttention, :677-716 Refinement).
 *   out[b,co,y,x] = act(bias[co] + sum_{ci,ky,kx} x[b,ci,y+(ky-1)*dil,x+(kx-1)*dil] * w[co,ci,ky,kx]) [+ addend[b,y,x]]
 * NCHW fp32, stride 1, zero padding dil*(k/2), k in {1,3}; BatchNorm(eval) is folded into w / bias
 * by the caller.  w_packed is [Cin][k*k][CoutP] (CoutP = Cout rounded up to 4, zero padded).
 * Supported shapes: decnet_conv2d_small_supported(); `addend` (single-channel outputs only, may be
 * NULL) is added after the activation (Refinement: disp + residual, submodule.py:761). */
int decnet_conv2d_small_supported(int Cin, int Cout, int ksize);
/* 0 = auto (register/L1 kernel), 2 = shared-memory tiled kernel (correct, measured slower in round 1).  Per thread. */
void decnet_conv2d_set_variant(int variant);
int decnet_conv2d_small(const float *x, const float *w_packed, const float *bias, const float *addend, float *out,
                        int B, int Cin, int H, int W, int Cout, int ksize, int dilation, int relu, void *stream);

/* ConvTranspose2d(kernel 3, stride 3) + bias + ReLU (GenerateSparseMask.deconv.0, submodule.py:350-351):
 * x [B,Cin,h,w], w [Cin,Cout,3,3] (PyTorch layout), out [B,Cout,3h,3w]; Cout must be 8. */
int decnet_deconv3x3s3(const float *x, const float *w, const float *bias, float *out,
                       int B, int Cin, int h, int w_in, int Cout, int relu, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DECNET_B200_H */
