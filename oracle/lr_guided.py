"""oracle/lr_guided.py -- TEST INFRASTRUCTURE ONLY.  numpy float32 definition of the edge-aware hole filling that
StereoMatcher's left-right check offers (fill="guided"); decnet_lr_check_guided_fill (decnet_b200/csrc/codec.cu) is held
to it bit for bit.

The rule is modelled on the weighted-least-squares "fast global smoother" (Min et al., 2014, the solver inside OpenCV's
DisparityWLSFilter) used as normalised interpolation: the valid disparities and the validity mask are both smoothed along
the left image, whose colour edges stop the spreading, and an invalid pixel takes their ratio.  This file, not OpenCV, is
the contract; it has not been compared with OpenCV.

  fill_guided   per image of lr_check's (disparity, valid) [B,h,w] and the left image guide uint8 [B,h,w,3], in float32
                with every sum, product and reciprocal rounded separately:
    1. edge weights: neighbours p, q have k = sum_c |I_c(p) - I_c(q)| (0..765, the same for RGB and BGR guides) and the
       weight w(k) = float32(exp(-k / float64(sigma))), from a 766-entry table computed in float64
    2. schedule: T = 3 iterations; iteration t = 1..T uses lam_t = float32(lam * 1.5 * 4^(T-t) / (4^T - 1)) (float64, in
       that order) and solves every row, then every column
    3. one line of n pixels: edge coefficients a_i = float32(lam_t * w(k_i)), i = 0..n-2, a_-1 = a_(n-1) = 0; solve
       (I + lam_t L_w) x = f by the Thomas algorithm with one reciprocal per step (solve_line), for two right-hand sides
       that share the matrix: num, starting as valid ? disp : 0, and den, starting as valid ? 1 : 0
    4. compose: a valid pixel keeps its bits; an invalid pixel whose den is a normal float (>= 2^-126) takes num / den;
       every other invalid pixel (strong edges on every side cut it off, so den is 0 or has lost its precision) keeps
       its oracle.lr_fill.fill_background value, so the output stays dense and an image without a valid pixel stays 0
    -> (float32 filled map, its uint16 image: oracle.codec.disp_to_u16)
lam = 8000 and sigma = 2.6 are OpenCV's filter defaults (lambda 8000, sigma 1.5 on the Euclidean colour distance); on an edge
of equal height in all three channels, 1.5 * sqrt(3) ~ 2.6 on the L1 distance gives the same weight.
"""
import numpy as np

from .codec import disp_to_u16
from .lr_fill import fill_background

F32 = np.float32
ITERS = 3
TABLE = 766                                                                # k = 0..765


def weight_table(sigma):
    """w(k) = float32(exp(-k / float64(sigma))) for k = 0..765."""
    return np.exp(-np.arange(TABLE, dtype=np.float64) / np.float64(sigma)).astype(F32)


def schedule(lam, iters=ITERS):
    """[lam_1, ..., lam_T]: float32(lam * 1.5 * 4^(T-t) / (4^T - 1)), evaluated in float64 in that order."""
    return [F32(np.float64(lam) * 1.5 * 4.0 ** (iters - t) / (4.0 ** iters - 1)) for t in range(1, iters + 1)]


def solve_line(a, rhs):
    """Solve (I + L) x = f along the last axis for each f in rhs, L the path Laplacian of the edge coefficients
    a [..., n-1] (float32, >= 0): the Thomas algorithm, one reciprocal per step, every operation rounded to float32:
        b_i = (1 + a_(i-1)) + a_i,  m_i = b_i - a_(i-1) g_(i-1),  r_i = 1 / m_i,  g_i = a_i r_i,
        y_i = (f_i + a_(i-1) y_(i-1)) r_i;  x_(n-1) = y_(n-1),  x_i = y_i + g_i x_(i+1)
    with a_-1 = a_(n-1) = 0 and g_-1 = y_-1 = 0.  Returns a list of float32 arrays shaped like rhs."""
    rhs = [np.asarray(f, dtype=F32) for f in rhs]
    n = rhs[0].shape[-1]
    a = np.asarray(a, dtype=F32)
    one = F32(1)
    zero = np.zeros(rhs[0].shape[:-1], dtype=F32)
    g = np.empty(rhs[0].shape, dtype=F32)
    ys = [np.empty_like(f) for f in rhs]
    a_prev, g_prev, y_prev = zero, zero, [zero] * len(rhs)
    for i in range(n):
        a_i = a[..., i] if i < n - 1 else zero
        m = ((one + a_prev) + a_i) - a_prev * g_prev
        r = one / m
        g[..., i] = a_i * r
        for y, f, yp in zip(ys, rhs, y_prev):
            y[..., i] = (f[..., i] + a_prev * yp) * r
        a_prev, g_prev, y_prev = a_i, g[..., i], [y[..., i] for y in ys]
    for i in range(n - 2, -1, -1):
        for y in ys:
            y[..., i] = y[..., i] + g[..., i] * y[..., i + 1]
    return ys


def _edges(guide, axis):
    """k between each pixel and its next neighbour along `axis` (1: rows' x, 0: columns' y) of one [h,w,3] image."""
    gi = guide.astype(np.int32)
    return np.abs(np.diff(gi, axis=axis)).sum(-1)


def fill_guided(disp, valid, guide, lam=8000.0, sigma=2.6):
    """Edge-aware hole filling of lr_check's float output `disp` and mask `valid` [B,h,w], guided by the left images
    `guide` uint8 [B,h,w,3] (see the module docstring) -> (filled float32 [B,h,w], filled uint16 [B,h,w])."""
    disp = np.asarray(disp, dtype=F32)
    valid = np.asarray(valid, dtype=bool)
    guide = np.asarray(guide)
    if disp.shape != valid.shape or disp.ndim != 3:
        raise ValueError(f"disp {disp.shape} and valid {valid.shape} must both be [B,h,w]")
    if guide.dtype != np.uint8 or guide.shape != disp.shape + (3,):
        raise ValueError(f"guide must be uint8 {disp.shape + (3,)}, got {guide.dtype} {guide.shape}")
    B, h, w = disp.shape
    table = weight_table(sigma)
    background, _ = fill_background(disp, valid)
    out = np.empty_like(disp)
    for b in range(B):
        wh, wv = table[_edges(guide[b], 1)], table[_edges(guide[b], 0)]   # [h, w-1], [h-1, w]
        num = np.where(valid[b], disp[b], F32(0)).astype(F32)
        den = valid[b].astype(F32)
        for lt in schedule(lam):
            num, den = solve_line(lt * wh, [num, den])
            num, den = (x.T for x in solve_line((lt * wv).T, [num.T, den.T]))
        use = ~valid[b] & (den >= np.finfo(F32).tiny)
        with np.errstate(divide="ignore", invalid="ignore"):
            out[b] = np.where(use, num / den, background[b])                # valid pixels: background keeps their bits
    return out, disp_to_u16(out, h, w)
