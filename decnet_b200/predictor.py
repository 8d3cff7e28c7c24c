"""StereoMatcher: uint8 image pairs in, disparities out -- demo.py's device work (demo.py:144-198) behind one object.

    m = StereoMatcher(state_dict)                 # checkpoint in the reference's layout, or None for seeded weights
    disp = m(left, right)                         # fp32 disparity in pixels, cropped to the input size
    png16 = m(left, right, output="u16")          # demo.py:191-197 (x256, uint16)
    for out in m.stream(pairs, output="u16"): ...
    disp, valid = StereoMatcher(lr_check=1.0)(left, right, return_valid=True)   # left-right check: 0 where it fails
    dense = StereoMatcher(lr_check=1.0, fill="background")(left, right)         # ... and its holes filled
    dense = StereoMatcher(lr_check=1.0, fill="guided")(left, right)             # ... filled along the left image
    dense = StereoMatcher(lr_check=1.0, speckle_size=100, fill="background")(left, right)   # ... speckles removed first
    disp = m(left, right, min_disp=243, max_disp=768)   # search [243, 783) only; min_disp may be negative

Every call of one shape (B, h, w, max_disp) replays one CUDA graph of the whole step: uint8 -> pad / normalise ->
feature extractor (both views, the right one on a forked stream) -> [image-space detail masks] -> decomposed matching.
The graph is captured on the first call of a shape (after one eager run that builds the packed-weight caches), kept in
an LRU cache of `max_graphs` shapes, and re-captured when any weight changed since its capture (the caches are only
checked when Python runs forward, which a replay never does).

With a left-right check (`lr_check` = a tolerance in pixels) the graph also runs the reverse direction: the model on the
mirrored, swapped pair (mirror(right), mirror(left)), whose mirrored-back result is the right view's disparity.  Each
buffer set then holds 2B pairs: the upload fills the first B, ops.mirror_swap_u8 writes the second B inside the graph, and
the unchanged step runs at batch 2B.  ops.lr_check compares the two directions outside the graph, so the tolerance is a
per-call argument that never re-captures.  It keeps the forward disparity where |dl - dr| <= tol at the matched column of
the right view and writes 0 (KITTI's "no value") elsewhere: occluded pixels and matches outside the right image.
fill="background" fills those pixels instead, in the same pass over the predictions (oracle/lr_fill.py): each takes the
smaller disparity of its nearest valid neighbours in the row, because an occluded pixel belongs to the surface behind; a row
without a valid pixel takes the rows above and below.  The mask `valid` stays the check's, so filled pixels are still told
apart from measured ones.  fill="guided" spreads the valid disparities along the left image instead, stopping at its
colour edges (oracle/lr_guided.py: the fast global smoother's row and column solves as normalised interpolation), so the
filled strips follow object outlines rather than one value per row; a pixel that no valid disparity reaches keeps its
background value.  It reads the uploaded left images st.l, on the main stream before the set's `computed` event, so the
next upload into that set cannot overwrite them first.  The fill is also outside the graph: changing it never re-captures
either.

Between the check and the fill, speckle_size > 0 removes speckles (OpenCV's speckleWindowSize / speckleRange, i.e.
cv2.filterSpeckles; oracle/lr_speckle.py): in textureless and repetitive areas, and in occluded strips, some pixels pass
the check by coincidence and form small islands, which either fill would spread as if they were measured.  Valid
4-neighbours whose disparities differ by at most speckle_range join a region, and every region of at most speckle_size
pixels becomes invalid: 0 without a fill, filled with one, False in `valid`.  It runs outside the graph with the check, so
it never re-captures either.

The search range is [min_disp, max_disp) (OpenCV's minDisparity, Middlebury's vmin / vmax; min_disp = 0 by default): only its
width is rounded up to a multiple of 27, D = round_max_disp(max_disp - min_disp), and the range searched is
[min_disp, min_disp + D).  The step runs the unchanged model at width D on (L, shift(R, min_disp)), shift(R, k)[:, x] =
R[:, x - k] with black columns where the source lies outside the image (oracle/disp_range.py), and adds min_disp to the
prediction in fp32: ops.image_prepare_u8(..., col_shift=min_disp) prepares every right view of the graph's batch, the
reverse direction's shift(mirror(L), k) included, and ops.disp_add runs at the end of the graph.  With min_disp = 0 neither
runs and the graph is today's.  The check, the fills and the speckle filter then see true disparities, negative ones
included; output="u16" clamps a negative disparity to 0 (KITTI's "no value").  The start is baked into the graph like
max_disp, so it is part of cache_key.

The capture and the double-buffered loop of `stream()` restate bench.py's `capture` / `pipelined_e2e` on purpose:
bench.py is the fixed measuring stick of the project and does not import the package's public API.
"""
from __future__ import annotations

from collections import OrderedDict, deque

import numpy as np
import torch

from . import ops
from .features import FeatExtNetChannelPlus, extract_pair
from .model import PRECISIONS, DecompMatching, _sig_of

MASKS = ("learned", "image")
OUTPUTS = ("float", "u16")
MULTIPLE = 27                  # demo.py:75-81 pads to multiples of 3**3; demo.py:172-173 rounds max_disp likewise
MIN_SIZE = 1                   # padded to 27 x 27, every level of the pyramid has >= 1 pixel: what the kernels' size checks ask
FE_PREFIX = "feature_extractor."


def round_max_disp(max_disp):
    """max_disp rounded up to a multiple of 27 (demo.py:172-173): 192 -> 216, 768 -> 783."""
    if isinstance(max_disp, bool) or not isinstance(max_disp, (int, np.integer)) or max_disp <= 0:
        raise ValueError(f"max_disp must be a positive integer, got {max_disp!r}")
    return -(-int(max_disp) // MULTIPLE) * MULTIPLE


DISP_LIMIT = 2 ** 24           # |min_disp|, |max_disp| at most this: the offset added to the prediction stays exact in fp32


def disparity_range(min_disp, max_disp):
    """The search range [min_disp, max_disp) as (min_disp, D): the model runs at the width D = max_disp - min_disp rounded up
    to a multiple of 27, so the range searched is [min_disp, min_disp + D).  Host-only; ValueError when either end is not an
    integer (or is a bool) or lies outside [-2**24, 2**24], or when max_disp <= min_disp."""
    for name, v in (("min_disp", min_disp), ("max_disp", max_disp)):
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)):
            raise ValueError(f"{name} must be an integer number of pixels, got {v!r}")
        if not -DISP_LIMIT <= v <= DISP_LIMIT:
            raise ValueError(f"{name} must lie in [-2**24, 2**24] (where the offset stays exact in fp32), got {v!r}")
    if max_disp <= min_disp:
        raise ValueError(f"max_disp must be larger than min_disp, got the range [{min_disp}, {max_disp})")
    return int(min_disp), round_max_disp(int(max_disp) - int(min_disp))


def cache_key(B, h, w, max_disp, masks, precision, lr=False, min_disp=0):
    """What one captured graph is specific to: max_disp is the model's width D; a nonzero min_disp (the right views' shift)
    adds ("min_disp", min_disp); a graph with the left-right check's reverse direction has a trailing "lr"."""
    key = (int(B), int(h), int(w), int(max_disp), masks, precision)
    if min_disp:
        key += (("min_disp", int(min_disp)),)
    return key + ("lr",) if lr else key


def split_state_dict(state_dict, fe_keys, hot_keys):
    """A checkpoint in the reference's layout (`feature_extractor.*` plus the hot-path keys, with or without the
    `module.` prefix of a DataParallel save, demo.py:124-135) -> (extractor dict, hot-path dict).  Strict: a key
    missing from the checkpoint or not belonging to either module raises ValueError naming it."""
    if not hasattr(state_dict, "items"):
        raise ValueError(f"state_dict must be a mapping, got {type(state_dict).__name__}")
    fe, hot = {}, {}
    for k, v in state_dict.items():
        k = k[len("module."):] if k.startswith("module.") else k
        if k.startswith(FE_PREFIX):
            fe[k[len(FE_PREFIX):]] = v
        else:
            hot[k] = v
    unexpected = sorted([FE_PREFIX + k for k in fe if k not in fe_keys] + [k for k in hot if k not in hot_keys])
    missing = sorted([FE_PREFIX + k for k in fe_keys if k not in fe] + [k for k in hot_keys if k not in hot])
    if unexpected:
        raise ValueError(f"unexpected key(s) in state_dict: {', '.join(unexpected[:8])}")
    if missing:
        raise ValueError(f"missing key(s) in state_dict: {', '.join(missing[:8])}")
    return fe, hot


def _kind(x):
    if isinstance(x, np.ndarray):
        return "numpy"
    if isinstance(x, torch.Tensor):
        return "cuda" if x.is_cuda else "cpu"
    raise ValueError(f"images must be numpy arrays or torch tensors, got {type(x).__name__}")


def check_pair(left, right):
    """Validate one pair (host-side only, no device work) -> (kind, batched, B, h, w).  uint8 RGB [h,w,3] or [B,h,w,3];
    both views of the same kind and shape."""
    kl, kr = _kind(left), _kind(right)
    if kl != kr:
        raise ValueError(f"left is a {kl} array, right a {kr} one: give both views the same kind")
    for name, x in (("left", left), ("right", right)):
        if x.dtype != (np.uint8 if kl == "numpy" else torch.uint8):
            raise ValueError(f"{name} must be uint8 RGB, got dtype {x.dtype}")
        if x.ndim not in (3, 4) or x.shape[-1] != 3:
            raise ValueError(f"{name} must be [h,w,3] or [B,h,w,3] RGB, got shape {tuple(x.shape)}")
    if tuple(left.shape) != tuple(right.shape):
        raise ValueError(f"left {tuple(left.shape)} and right {tuple(right.shape)} views differ in shape")
    if kl == "cuda" and left.device != right.device:
        raise ValueError(f"left is on {left.device}, right on {right.device}")
    batched = left.ndim == 4
    B, h, w = (left.shape[0] if batched else 1), left.shape[-3], left.shape[-2]
    if B < 1 or h < MIN_SIZE or w < MIN_SIZE:
        raise ValueError(f"empty input {tuple(left.shape)}: images must be at least {MIN_SIZE}x{MIN_SIZE} pixels "
                         f"(they are padded to multiples of {MULTIPLE}) and a batch at least one pair")
    return kl, batched, int(B), int(h), int(w)


class _Set:
    """One captured graph with its static input / output buffers and pinned host staging.  l, r are the B uploaded pairs;
    with the left-right check they are the first halves of the graph's [2B,h,w,3] inputs xl, xr."""

    def __init__(self, B, h, w, dev, lr=False):
        self.lr = lr
        self.xl = torch.empty(((2 if lr else 1) * B, h, w, 3), dtype=torch.uint8, device=dev)
        self.xr = torch.empty_like(self.xl)
        self.l, self.r = self.xl[:B], self.xr[:B]
        self.host_l = torch.empty((B, h, w, 3), dtype=torch.uint8).pin_memory()
        self.host_r = torch.empty_like(self.host_l).pin_memory()
        self.graph = self.pred = self.sig = None
        self.uploaded = self.computed = None
        self.min_disp = 0                          # the right views' column shift, baked into the graph at its capture


class StereoMatcher:
    """Stereo matcher from uint8 RGB image pairs to disparity (see the module docstring).

    state_dict    reference-layout checkpoint, or None for the seeded random init (params, seed 17)
    max_disp      the exclusive end of the search range; the width max_disp - min_disp is rounded up to a multiple of 27,
                  and m.max_disp is min_disp + that width; a call may override it
    min_disp      the start of the search range, an integer that may be negative (converging rigs, Middlebury's vmin);
                  a call may override it
    masks         "learned": DecompMatching's detectors (use_detail=True, `thold`); "image": demo.py's route,
                  ops.detail_detection of the padded [0,1] images with `detail_thold`, finest level last
    skip_stage_id 3 skips the finest level (bicubic x3 of the 1/3 disparity; Middlebury, demo.sh:5)
    precision     "fp32" (3xTF32 convs) or "tf32"
    max_graphs    shapes whose graphs are kept (least recently used evicted first)
    lr_check      None (off) or the left-right check's tolerance in pixels (a finite number >= 0); a call may override it
    fill          "none" (failing pixels are 0), "background" (failing pixels filled from their valid neighbours in the
                  row) or "guided" (filled along the left image, stopping at its edges); a fill needs a left-right check;
                  a call may override it
    speckle_size  0 (off) or the largest region, in pixels of the input image, that the speckle filter removes after the
                  check and before the fill; needs a left-right check; a call may override it
    speckle_range the largest disparity difference, in pixels, between neighbours of one region (a finite number >= 0);
                  a call may override it
    """

    def __init__(self, state_dict=None, max_disp=192, masks="learned", thold=0.9, detail_thold=0.3, skip_stage_id=4,
                 precision="fp32", device="cuda", max_graphs=4, lr_check=None, fill="none", speckle_size=0,
                 speckle_range=1.0, min_disp=0):
        if masks not in MASKS:
            raise ValueError(f"masks must be one of {MASKS}, got {masks!r}")
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {PRECISIONS}, got {precision!r}")
        if skip_stage_id not in (1, 2, 3, 4):
            raise ValueError(f"skip_stage_id must be 1..4, got {skip_stage_id!r}")
        if isinstance(max_graphs, bool) or not isinstance(max_graphs, int) or max_graphs < 1:
            raise ValueError(f"max_graphs must be a positive integer, got {max_graphs!r}")
        self.lr_check = None if lr_check is None else ops.lr_tolerance(lr_check)
        self.fill = ops.lr_fill(fill)
        self.speckle_size, self.speckle_range = ops.lr_speckle(speckle_size, speckle_range)
        dev = torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"device must be a CUDA device (decnet_b200 has no CPU path), got {device!r}")
        self.min_disp, D = disparity_range(min_disp, max_disp)
        self.max_disp = self.min_disp + D
        self.masks, self.precision, self.detail_thold, self.max_graphs = masks, precision, float(detail_thold), max_graphs
        fe = FeatExtNetChannelPlus(8, precision=precision)
        model = DecompMatching(max_disp=D, skip_stage_id=skip_stage_id, use_detail=masks == "learned",
                               thold=thold, precision=precision)
        self.fe, self.model = fe, model
        self.load_state_dict(state_dict)
        self.dev = dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.fe.to(self.dev)
        self.model.to(self.dev)
        self._graphs = OrderedDict()
        self.captures = 0
        self._cap_stream = self._copy_stream = None

    # ---------------------------------------------------------------------------------------------------------- weights
    def load_state_dict(self, state_dict):
        """Replace the weights (strict, see split_state_dict); None loads the seeded random init."""
        if state_dict is None:
            from .params import make_featext_state, make_hotpath_state
            fe_sd, hot_sd = make_featext_state(17), make_hotpath_state(17)
        else:
            fe_sd, hot_sd = split_state_dict(state_dict, self.fe.state_dict().keys(), self.model.state_dict().keys())
        self.fe.load_state_dict(fe_sd, strict=True)
        self.model.load_state_dict(hot_sd, strict=True)

    def _sig(self):
        return _sig_of(self.fe, self.model)

    # ----------------------------------------------------------------------------------------------------------- graphs
    def clear(self):
        """Drop every captured graph and release its memory pool."""
        for sets in self._graphs.values():
            for st in sets:
                if st.graph is not None:
                    st.graph.reset()
        self._graphs.clear()

    def _forward(self, l, r, min_disp=0):
        """The whole step on the device, for the static inputs l, r -> padded prediction [B,H,W].  A nonzero min_disp
        shifts the right views by min_disp columns as they are prepared and adds min_disp to the prediction."""
        if self.masks == "learned":
            prepare = lambda u8, shift=0: ops.image_prepare_u8(u8, want01=False, col_shift=shift)[1]
            fl, fr = extract_pair(self.fe, l, r, prepare=prepare, prepare_right=lambda u8: prepare(u8, min_disp))
            pred = self.model(fl, fr)[0]
        else:
            l01, lnorm = ops.image_prepare_u8(l)
            r01, rnorm = ops.image_prepare_u8(r, col_shift=min_disp)
            fl, fr = extract_pair(self.fe, lnorm, rnorm)
            lm = ops.detail_detection(l01, 3, self.detail_thold)[::-1]   # finest level last (demo.py:161-162)
            rm = ops.detail_detection(r01, 3, self.detail_thold)[::-1]
            pred = self.model(fl, fr, lm, rm)[0]
        return ops.disp_add(pred, min_disp) if min_disp else pred

    def _step(self, st):
        """What the graph of a set runs: [the reverse direction's inputs, then] the step at the set's batch."""
        if st.lr:
            B = st.l.shape[0]
            ops.mirror_swap_u8(st.l, st.r, st.xl[B:], st.xr[B:])
        return self._forward(st.xl, st.xr, st.min_disp)

    def _capture(self, st, max_disp, min_disp=0):
        """One eager run on a side stream (it rebuilds any stale weight cache), then the capture (bench.py's capture)."""
        if st.graph is not None:
            st.graph.reset()
        if self._cap_stream is None:
            self._cap_stream = torch.cuda.Stream(self.dev)
        side, main = self._cap_stream, torch.cuda.current_stream(self.dev)
        graph = torch.cuda.CUDAGraph()
        st.min_disp = min_disp
        saved, self.model.max_disp = self.model.max_disp, max_disp
        try:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                self._step(st)
                with torch.cuda.graph(graph, stream=side):
                    st.pred = self._step(st)
            main.wait_stream(side)
            torch.cuda.synchronize(self.dev)
        finally:
            self.model.max_disp = saved
        st.graph, st.sig = graph, self._sig()
        self.captures += 1

    def _sets(self, key, n):
        """The first n buffer sets of `key` (LRU bookkeeping, eviction); sets are created empty and captured on use."""
        sets = self._graphs.get(key)
        if sets is None:
            while len(self._graphs) >= self.max_graphs:
                _, old = self._graphs.popitem(last=False)
                for st in old:
                    if st.graph is not None:
                        st.graph.reset()
            sets = self._graphs[key] = []
        self._graphs.move_to_end(key)
        B, h, w = key[:3]
        while len(sets) < n:
            sets.append(_Set(B, h, w, self.dev, lr=key[-1] == "lr"))
        return sets

    def _replay(self, st, max_disp, min_disp=0):
        """Replay, re-capturing first when the set is new or any weight changed since its capture."""
        if st.graph is None or st.sig != self._sig():
            self._capture(st, max_disp, min_disp)
        st.graph.replay()

    # ------------------------------------------------------------------------------------------------------------ calls
    def _result(self, st, h, w, output, tol=None, return_valid=False, fill="none", speckle=(0, 1.0)):
        """Fresh device tensor (never the graph's static buffer) in the requested format, on the current stream; with the
        left-right check (tol) the checked disparity, speckles (size, range) removed, holes filled by `fill`, or
        (disparity, valid) when return_valid."""
        if st.lr:
            out = ops.lr_check(st.pred, h, w, tol, float_out=output == "float", u16_out=output == "u16", valid_out=return_valid,
                               fill=fill, guide=st.l if fill == "guided" else None, speckle_size=speckle[0],
                               speckle_range=speckle[1])
            return out if return_valid else out[0]
        if output == "u16":
            return ops.disp_to_u16(st.pred, h, w)
        H, W = st.pred.shape[-2:]
        return st.pred[:, H - h:, W - w:].clone()                        # demo.py's crop: the last h rows, w columns

    def _range(self, min_disp=None, max_disp=None):
        """The call's search range as (min_disp, width D), either end None for the matcher's, validated on the host."""
        return disparity_range(self.min_disp if min_disp is None else min_disp, self.max_disp if max_disp is None else max_disp)

    def _lr(self, lr_check, return_valid, fill=None):
        """The call's left-right check tolerance (None: off) and fill rule, validated before any device work."""
        fill = None if fill is None else ops.lr_fill(fill)
        tol = self.lr_check if lr_check is None else ops.lr_tolerance(lr_check)
        if return_valid and tol is None:
            raise ValueError("return_valid=True needs a left-right check: give lr_check to the matcher or the call")
        fill = self.fill if fill is None else fill
        if fill != "none" and tol is None:
            raise ValueError(f"fill needs a left-right check: give lr_check to the matcher or the call (fill={fill!r})")
        return tol, fill

    def _speckle(self, tol, speckle_size=None, speckle_range=None):
        """The call's speckle filter (size, range) under the call's tolerance tol, validated before any device work."""
        size = self.speckle_size if speckle_size is None else speckle_size
        rng = self.speckle_range if speckle_range is None else speckle_range
        size, rng = ops.lr_speckle(size, rng)
        if size and tol is None:
            raise ValueError(f"speckle_size needs a left-right check: give lr_check to the matcher or the call "
                             f"(speckle_size={size})")
        return size, rng

    def __call__(self, left, right, output="float", max_disp=None, lr_check=None, return_valid=False, fill=None,
                 speckle_size=None, speckle_range=None, min_disp=None):
        """Disparity of one pair ([h,w,3]), a batch ([B,h,w,3]) or lists of single pairs (any sizes; one batch per
        distinct size, results in input order).  output "float" (pixels) or "u16" (x256, demo.py:191-197); the result
        has the kind of the input (numpy, CPU tensor or CUDA tensor).  lr_check (None: the matcher's) is the left-right
        check's tolerance in pixels; pixels that fail it are 0, or filled from their neighbours with fill="background" or
        along the left image with fill="guided" (None: the matcher's fill).  return_valid: each result is (disparity, bool valid), valid False on filled pixels.
        speckle_size / speckle_range (None: the matcher's) remove speckles between the check and the fill.  min_disp /
        max_disp (None: the matcher's) give the search range [min_disp, max_disp) as for the constructor."""
        if output not in OUTPUTS:
            raise ValueError(f"output must be one of {OUTPUTS}, got {output!r}")
        tol, fill = self._lr(lr_check, return_valid, fill)
        speckle = self._speckle(tol, speckle_size, speckle_range)
        span = self._range(min_disp, max_disp)
        if isinstance(left, (list, tuple)):
            return self._call_list(left, right, output, span, tol, return_valid, fill, speckle)
        kind, batched, B, h, w = check_pair(left, right)
        out = self._run(left, right, kind, B, h, w, output, span, tol, return_valid, fill, speckle)
        return out if batched else _index(out, 0)

    def _call_list(self, lefts, rights, output, span, tol, return_valid, fill, speckle):
        if not isinstance(rights, (list, tuple)) or len(rights) != len(lefts):
            raise ValueError("left and right lists must have the same length")
        groups = OrderedDict()
        for i, (l, r) in enumerate(zip(lefts, rights)):
            kind, batched, B, h, w = check_pair(l, r)
            if batched:
                raise ValueError(f"list item {i}: give single [h,w,3] pairs in a list, got {tuple(l.shape)}")
            groups.setdefault((kind, h, w), []).append(i)
        results = [None] * len(lefts)
        for (kind, h, w), idx in groups.items():
            stack = np.stack if kind == "numpy" else torch.stack
            out = self._run(stack([lefts[i] for i in idx]), stack([rights[i] for i in idx]), kind, len(idx), h, w, output, span,
                            tol, return_valid, fill, speckle)
            for j, i in enumerate(idx):
                results[i] = _index(out, j)
        return results

    def _upload(self, st, left, right, kind):
        """Inputs into the set's static buffers on the current stream: host inputs through its pinned staging."""
        if kind == "cuda":
            st.l.copy_(left)
            st.r.copy_(right)
            return
        if st.uploaded is not None:
            st.uploaded.synchronize()                      # an upload of stream() may still read the staging buffers
        st.host_l.copy_(torch.from_numpy(np.ascontiguousarray(left)) if kind == "numpy" else left)
        st.host_r.copy_(torch.from_numpy(np.ascontiguousarray(right)) if kind == "numpy" else right)
        st.l.copy_(st.host_l, non_blocking=True)
        st.r.copy_(st.host_r, non_blocking=True)

    @torch.no_grad()
    def _run(self, left, right, kind, B, h, w, output, span, tol=None, return_valid=False, fill="none", speckle=(0, 1.0)):
        if kind == "cuda" and left.device != self.dev:
            raise ValueError(f"inputs are on {left.device}, the matcher on {self.dev}")
        k, D = span
        with torch.cuda.device(self.dev):
            st = self._sets(cache_key(B, h, w, D, self.masks, self.precision, tol is not None, k), 1)[0]
            self._upload(st, left, right, kind)
            self._replay(st, D, k)
            out = self._result(st, h, w, output, tol, return_valid, fill, speckle)
            if kind == "cuda":
                return out
            out = _map(lambda t: t.cpu(), out)                            # synchronous: the staging buffers are free again
            return _map(lambda t: t.numpy(), out) if kind == "numpy" else out

    def stream(self, pairs, output="float", max_disp=None, lr_check=None, return_valid=False, fill=None, speckle_size=None,
               speckle_range=None, min_disp=None):
        """Yield the result of each (left, right) of `pairs` in order, software-pipelined over two buffer sets per shape:
        while the graph of item i runs, the copy stream uploads item i+1 into the other set (bench.py's pipelined_e2e).
        Host results are read back through pinned memory and yielded as fresh arrays.  A change of shape drains the
        pipeline and continues with the new shape's sets.  lr_check / return_valid / fill / speckle_size / speckle_range /
        min_disp / max_disp as for a call."""
        if output not in OUTPUTS:
            raise ValueError(f"output must be one of {OUTPUTS}, got {output!r}")
        tol, fill = self._lr(lr_check, return_valid, fill)
        speckle = self._speckle(tol, speckle_size, speckle_range)
        span = self._range(min_disp, max_disp)
        return self._stream(pairs, output, span, tol, return_valid, fill, speckle)   # arguments checked now, not at the first item

    @torch.no_grad()
    def _stream(self, pairs, output, span, tol, return_valid, fill, speckle):
        min_disp, D = span
        with torch.cuda.device(self.dev):
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(self.dev)
            copy, main = self._copy_stream, torch.cuda.current_stream(self.dev)
            pending, key, i = deque(), None, 0
            for left, right in pairs:
                kind, batched, B, h, w = check_pair(left, right)
                if kind == "cuda" and left.device != self.dev:
                    raise ValueError(f"inputs are on {left.device}, the matcher on {self.dev}")
                k = cache_key(B, h, w, D, self.masks, self.precision, tol is not None, min_disp)
                if k != key:
                    while pending:
                        yield self._finish(pending.popleft())
                    key, i = k, 0
                st = self._sets(k, 2)[i & 1]
                i += 1
                if st.uploaded is not None:
                    st.uploaded.synchronize()              # the staging buffers' previous upload has left them
                if kind != "cuda":
                    st.host_l.copy_(torch.from_numpy(np.ascontiguousarray(left)) if kind == "numpy" else left)
                    st.host_r.copy_(torch.from_numpy(np.ascontiguousarray(right)) if kind == "numpy" else right)
                src_l, src_r = (left, right) if kind == "cuda" else (st.host_l, st.host_r)
                if kind == "cuda":
                    copy.wait_stream(main)                 # the caller's tensors are ready on its stream
                    left.record_stream(copy)
                    right.record_stream(copy)
                with torch.cuda.stream(copy):
                    if st.computed is not None:
                        copy.wait_event(st.computed)       # the set's previous replay has read its static inputs
                    st.l.copy_(src_l, non_blocking=True)
                    st.r.copy_(src_r, non_blocking=True)
                    st.uploaded = torch.cuda.Event()
                    st.uploaded.record(copy)
                main.wait_event(st.uploaded)
                self._replay(st, D, min_disp)
                res = self._result(st, h, w, output, tol, return_valid, fill, speckle)
                if kind != "cuda":
                    res = _map(_to_pinned, res)
                st.computed = torch.cuda.Event()
                st.computed.record(main)
                if pending:
                    yield self._finish(pending.popleft())
                pending.append((st.computed, res, kind, batched))
            while pending:
                yield self._finish(pending.popleft())

    @staticmethod
    def _finish(item):
        done, res, kind, batched = item
        done.synchronize()
        if kind == "numpy":
            res = _map(lambda t: t.numpy().copy(), res)
        elif kind == "cpu":
            res = _map(lambda t: t.clone(), res)
        return res if batched else _index(res, 0)


def _map(fn, out):
    """fn over a result: one tensor, or the (disparity, valid) pair of return_valid."""
    return tuple(fn(t) for t in out) if isinstance(out, tuple) else fn(out)


def _index(out, i):
    return _map(lambda t: t[i], out)


def _to_pinned(t):
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    return host
