"""oracle/lr_fill.py -- TEST INFRASTRUCTURE ONLY.  numpy float32 definition of the background hole filling that
StereoMatcher's left-right check offers (fill="background"); decnet_lr_check_fill (decnet_b200/csrc/codec.cu) is held to it
bit for bit.

The rule is modelled on the background interpolation of the KITTI stereo development kit, which fills a submitted map's
missing pixels before scoring it: a pixel the check rejects is occluded in the right view or matches outside it, so it
belongs to the surface behind and takes the smaller disparity of its nearest valid neighbours.  This file, not the devkit,
is the contract.  It has not been compared with the devkit line by line, and its handling of rows without a valid pixel
(step 2) may well differ from it.

  fill_background   per image of lr_check's (disparity, valid) [B,h,w]:
    1. row phase: in a row with a valid pixel, valid pixels keep their value bit for bit; an invalid pixel with nearest
       valid columns L (left) and R (right) takes disp[R] if disp[R] < disp[L] else disp[L] (strict: on equal values,
       -0.0 and +0.0 included, L's bits win); with only R (a leading run) disp[R], with only L (a trailing run) disp[L]
    2. column phase: a row without a valid pixel, in an image with at least one row that has one, takes column by column
       the same rule on the row-phase values of the nearest such rows A (above) and C (below): C's value if strictly less
       than A's, else A's; with only one of them, its value
    3. an image without a valid pixel stays 0
    -> (float32 filled map, its uint16 image: oracle.codec.disp_to_u16, what disp_u16 computes on the device)
Every output value is a copy of a valid input value (finite: the check requires it), so no arithmetic is involved.
"""
import numpy as np

from .codec import disp_to_u16


def _pick(lo_idx, hi_idx, values, n):
    """Per position: the background choice between values[lo_idx] (the nearer neighbour before it; -1 = none) and
    values[hi_idx] (after it; n = none) along axis 0 of `values`, index arrays broadcast over the other axis."""
    lo = np.take_along_axis(values, np.clip(lo_idx, 0, n - 1), axis=0)
    hi = np.take_along_axis(values, np.clip(hi_idx, 0, n - 1), axis=0)
    both = np.where(hi < lo, hi, lo)
    return np.where(lo_idx < 0, hi, np.where(hi_idx >= n, lo, both)).astype(np.float32)


def _nearest(flags):
    """flags [n, m] bool -> (index of the last True strictly before each position along axis 0, -1 if none; index of the
    first True strictly after it, n if none)."""
    n = flags.shape[0]
    idx = np.arange(n)[:, None]
    prev = np.maximum.accumulate(np.where(flags, idx, -1), axis=0)
    nxt = np.minimum.accumulate(np.where(flags, idx, n)[::-1], axis=0)[::-1]
    before = np.vstack([np.full((1, flags.shape[1]), -1), prev[:-1]])
    after = np.vstack([nxt[1:], np.full((1, flags.shape[1]), n)])
    return before, after


def fill_background(disp, valid):
    """Background hole filling of lr_check's float output `disp` and mask `valid`, both [B,h,w] (see the module docstring)
    -> (filled float32 [B,h,w], filled uint16 [B,h,w])."""
    disp = np.asarray(disp, dtype=np.float32)
    valid = np.asarray(valid, dtype=bool)
    if disp.shape != valid.shape or disp.ndim != 3:
        raise ValueError(f"disp {disp.shape} and valid {valid.shape} must both be [B,h,w]")
    B, h, w = disp.shape
    out = np.zeros_like(disp)
    for b in range(B):
        d, v = disp[b], valid[b]
        before, after = _nearest(v.T)                                      # along each row
        rows = np.where(v, d, _pick(before, after, d.T, w).T).astype(np.float32)
        nonempty = v.any(axis=1)
        if not nonempty.any():
            continue                                                       # step 3: stays 0
        above, below = _nearest(np.broadcast_to(nonempty[:, None], (h, w)))
        out[b] = np.where(nonempty[:, None], rows, _pick(above, below, rows, h))
    return out, disp_to_u16(out, h, w)
