"""oracle/lr_speckle.py -- TEST INFRASTRUCTURE ONLY.  numpy / scipy definition of the speckle filter that StereoMatcher's
left-right check runs between the check and the fill (speckle_size, speckle_range); decnet_lr_check_speckle
(decnet_b200/csrc/codec.cu) is held to it bit for bit.

The rule restates OpenCV's cv2.filterSpeckles (StereoSGBM's speckleWindowSize / speckleRange) on a float map with an
explicit mask: a region of at most max_size connected pixels is treated as a mismatch.  This file, not OpenCV, is the
contract; on int16 maps q = 16 * disp with 0 at the invalid pixels it equals cv2.filterSpeckles(q, 0, max_size,
16 * max_diff), which tests/test_lr_speckle_cpu.py checks where OpenCV is installed.

  filter_speckles   per image of lr_check's (disparity, valid) [B,h,w]:
    1. two 4-neighbours (left / right, up / down; never diagonal, never across images) are connected when both are valid
       and abs(float32(a) - float32(b)) <= float32(max_diff): one float32 subtraction and one compare, so +0 and -0 differ
       by 0, and a difference that overflows to inf does not connect
    2. a region is a connected set of valid pixels; every pixel of a region of size <= max_size becomes invalid, with
       disparity 0 (+0.0); every other pixel keeps its bits
    3. max_size = 0 is the identity
    -> (float32 disparity [B,h,w], bool valid [B,h,w])
Every output value is a copy of an input value, so no arithmetic is involved beyond the comparisons.
"""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

F32 = np.float32


def _labels(d, v, max_diff):
    """Connected-component labels of the valid pixels of one [h,w] image (invalid pixels are components of their own)."""
    h, w = d.shape
    idx = np.arange(h * w).reshape(h, w)
    a, b = [], []
    with np.errstate(over="ignore", invalid="ignore"):
        for sl0, sl1 in (((slice(None), slice(None, -1)), (slice(None), slice(1, None))),    # left / right
                         ((slice(None, -1), slice(None)), (slice(1, None), slice(None)))):    # up / down
            ok = v[sl0] & v[sl1] & (np.abs(d[sl0] - d[sl1]) <= max_diff)
            a.append(idx[sl0][ok])
            b.append(idx[sl1][ok])
    a, b = np.concatenate(a), np.concatenate(b)
    graph = coo_matrix((np.ones(a.size, dtype=np.int8), (a, b)), shape=(h * w, h * w))
    return connected_components(graph, directed=False)[1].reshape(h, w)


def filter_speckles(disp, valid, max_size, max_diff):
    """Speckle filter of lr_check's float output `disp` and mask `valid`, both [B,h,w] (see the module docstring)
    -> (float32 disparity, bool valid)."""
    disp = np.asarray(disp, dtype=F32)
    valid = np.asarray(valid, dtype=bool)
    if disp.shape != valid.shape or disp.ndim != 3:
        raise ValueError(f"disp {disp.shape} and valid {valid.shape} must both be [B,h,w]")
    if max_size < 0 or not abs(max_diff) <= np.finfo(F32).max or max_diff < 0:
        raise ValueError(f"max_size must be >= 0 and max_diff finite and >= 0, got {max_size!r}, {max_diff!r}")
    if max_size == 0:
        return disp.copy(), valid.copy()
    keep = np.zeros_like(valid)
    for b in range(disp.shape[0]):
        lab = _labels(disp[b], valid[b], F32(max_diff))
        size = np.bincount(lab[valid[b]], minlength=lab.max() + 1)
        keep[b] = valid[b] & (size[lab] > max_size)
    return np.where(keep, disp, F32(0)).astype(F32), keep
