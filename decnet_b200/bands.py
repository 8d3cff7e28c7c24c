"""Row-band mode: ONE stereo pair (or batch) split across GPUs by image rows (SURVEY.md section 8e,
BASELINE.json configs[3]: Middlebury ~2000x2900, max_disp 768->783, finest stage skipped).

Partition: contiguous bands of the 1/27 grid (shard.coarse_bands); a finer level's band is 3x the
rows.  What crosses a band boundary:

  * a3, 3-D aggregation: every 3x3x3 layer needs +-1 voxel row.  Each rank keeps its band with one
    physical halo row on each side ([B, D, rows+2, W, 224] bf16); after every layer the first/last
    OWNED rows are exchanged with the two neighbours (neighbour-only send/recv, 8 exchanges of
    D*W*224*2 bytes per side: 1.4 MB at Middlebury size); image top/bottom halo rows are zero (the
    conv's padding).  The conv kernel itself is unchanged: it also computes the halo rows, whose
    values are then overwritten by the exchange.
  * stages >= 1: SpaMat/SpaVar, threshold and blend are row-local (no halo).  The 2-D conv stacks
    (a5, a8, a13, a14) run on an EXTENDED band (shard.stage_extension rows of overlap, recomputed
    rather than exchanged layer by layer) with zero padding at its edges; only the owned rows are
    kept.  The previous level's disparity (a few hundred KB) is all-gathered once per level.
  * the bilinear warps use GLOBAL row coordinates (the reference's y' = h*H/(H-1) - 1/2).

Transports: `LocalTransport` runs all ranks in one process (single-GPU test of the decomposition),
`DistTransport` is one process per GPU over torch.distributed send/recv (NCCL; eager only), and
`PeerTransport` is one process per GPU over NVLink PEER MEMORY: the activation buffers of the aggregation and
the per-level disparity maps live in symmetric allocations (torch symmetric memory = CUDA IPC-mapped peer
buffers), every rank STORES its edge rows straight into its neighbours' halo rows and its band into every
rank's full map, and device-side signals order the steps -- no host synchronisation, no collective library call
on the path, so the whole banded step is captured in ONE CUDA graph per rank and replayed.
"""
from __future__ import annotations

import torch

from . import conv3d as c3
from . import ops, shard

# rows (of the level) by which a band is extended; multiples of 3 so that the x3 unfold / deconv of
# the previous level stay aligned:  refinement + attention + 12 (dynamic up-sampling: 4 coarse rows) + 1 (warp)
EXT = {s: -(-(shard.REFINE_HALO[s] + shard.ATTN_HALO + 3 * shard.DYNUP_HALO_COARSE + shard.WARP_HALO) // 3) * 3
       for s in (1, 2, 3)}


class LocalTransport:
    """All ranks live in this process (tensors on one device): exchanges are plain copies."""

    def __init__(self, world):
        self.world = world
        self.ranks_here = list(range(world))

    def exchange_halo(self, xs):
        """xs[rank]: [B, D, rows+2, W, C]; fill every halo row from the neighbour's edge row (zero at the image edge)."""
        snap = {r: (xs[r][:, :, 1].clone(), xs[r][:, :, -2].clone()) for r in xs}
        for r, x in xs.items():
            if r == 0:
                x[:, :, 0].zero_()
            else:
                x[:, :, 0].copy_(snap[r - 1][1])
            if r == self.world - 1:
                x[:, :, -1].zero_()
            else:
                x[:, :, -1].copy_(snap[r + 1][0])

    def all_gather_rows(self, bands):
        """bands[rank]: [B, rows_r, W] -> the full [B, sum rows, W] on every rank."""
        full = torch.cat([bands[r] for r in range(self.world)], dim=1)
        return {r: full for r in bands}


class DistTransport:
    """One process per GPU (torch.distributed, NCCL): neighbour send/recv for the halo rows,
    all_gather for the small disparity maps."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.ranks_here = [self.rank]

    def exchange_halo(self, xs):
        dist = self.dist
        x = xs[self.rank]
        ops_, recv_up, recv_dn = [], None, None
        if self.rank > 0:
            send_up = x[:, :, 1].contiguous()
            recv_up = torch.empty_like(send_up)
            ops_ += [dist.P2POp(dist.isend, send_up, self.rank - 1, self.group),
                     dist.P2POp(dist.irecv, recv_up, self.rank - 1, self.group)]
        if self.rank < self.world - 1:
            send_dn = x[:, :, -2].contiguous()
            recv_dn = torch.empty_like(send_dn)
            ops_ += [dist.P2POp(dist.isend, send_dn, self.rank + 1, self.group),
                     dist.P2POp(dist.irecv, recv_dn, self.rank + 1, self.group)]
        if ops_:
            for req in dist.batch_isend_irecv(ops_):
                req.wait()
        if recv_up is None:
            x[:, :, 0].zero_()
        else:
            x[:, :, 0].copy_(recv_up)
        if recv_dn is None:
            x[:, :, -1].zero_()
        else:
            x[:, :, -1].copy_(recv_dn)

    def all_gather_rows(self, bands):
        dist = self.dist
        mine = bands[self.rank]
        B, rows, W = mine.shape
        if getattr(self, "h_coarse", None):
            # every band is the balanced split of the 1/27 rows scaled to the level: sizes are known without talking
            # (and without a host synchronisation, so the whole step can be captured in a CUDA graph)
            cb = shard.coarse_bands(self.h_coarse, self.world)
            f = rows // (cb[self.rank][1] - cb[self.rank][0])
            all_sizes = [(b - a) * f for a, b in cb]
        else:
            sizes = torch.tensor([rows], device=mine.device, dtype=torch.int64)
            all_sizes = [torch.zeros_like(sizes) for _ in range(self.world)]
            dist.all_gather(all_sizes, sizes, group=self.group)
            all_sizes = [int(s.item()) for s in all_sizes]
        mx = max(all_sizes)
        pad = torch.zeros((B, mx, W), dtype=mine.dtype, device=mine.device)
        pad[:, :rows] = mine
        outs = [torch.empty_like(pad) for _ in range(self.world)]
        dist.all_gather(outs, pad, group=self.group)
        full = torch.cat([o[:, :n] for o, n in zip(outs, all_sizes)], dim=1)
        return {self.rank: full}


class PeerTransport:
    """One process per GPU; halo rows and band gathers are plain device stores into peer memory over NVLink.

    * `conv_buffer(name, shape)`: a symmetric [B, D, rows_max+2, W, C] bf16 allocation (zero-filled once); returns this
      rank's view [B, D, rows+2, W, C].  The aggregation layers write their owned rows into it (decnet_conv3d_bf16_band
      leaves the halo rows alone), `push_halo(name)` then stores the first / last owned row into the down / up halo row of
      the two neighbours' buffers and exchanges one signal with each neighbour: a layer may start once both neighbours'
      rows of the previous layer have landed.  Safe without a second signal: a neighbour can only be one layer ahead after
      it received my rows of the layer before, i.e. after I finished reading the buffer it is about to write into.
    * `all_gather_rows(bands, key)`: every rank stores its band into every rank's symmetric full map, then a device-side
      barrier.
    Everything is stream-ordered kernels / copies: capturable in a CUDA graph (bench.py does)."""

    def __init__(self, h_coarse, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        self.dist, self.symm = dist, symm
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.ranks_here = [self.rank]
        self.h_coarse = h_coarse
        self.bands = shard.coarse_bands(h_coarse, self.world)
        self._conv, self._full, self._chan = {}, {}, 0

    def _alloc(self, shape, dtype, device):
        t = self.symm.empty(*shape, dtype=dtype, device=device)
        t.zero_()
        hdl = self.symm.rendezvous(t, self.group)
        torch.cuda.synchronize(device)
        hdl.barrier(0)
        return t, hdl

    # ---- 3-D aggregation: per-layer halo rows ------------------------------------------------------------------
    def conv_buffer(self, name, B, D, W, C, device):
        if name not in self._conv:
            rows_max = max(b - a for a, b in self.bands)
            t, hdl = self._alloc((B, D, rows_max + 2, W, C), torch.bfloat16, device)
            view = lambda r: hdl.get_buffer(r, (B, D, self.bands[r][1] - self.bands[r][0] + 2, W, C), torch.bfloat16)
            mine = view(self.rank)
            up = view(self.rank - 1) if self.rank > 0 else None
            dn = view(self.rank + 1) if self.rank < self.world - 1 else None
            self._chan += 1
            self._conv[name] = (t, hdl, mine, up, dn, self._chan)
        return self._conv[name][2]

    def push_halo(self, name):
        _, hdl, mine, up, dn, ch = self._conv[name]
        if up is not None:
            up[:, :, -1].copy_(mine[:, :, 1])            # my first owned row -> the up neighbour's bottom halo row
            hdl.put_signal(self.rank - 1, ch)
        if dn is not None:
            dn[:, :, 0].copy_(mine[:, :, -2])            # my last owned row -> the down neighbour's top halo row
            hdl.put_signal(self.rank + 1, ch)
        if up is not None:
            hdl.wait_signal(self.rank - 1, ch)
        if dn is not None:
            hdl.wait_signal(self.rank + 1, ch)

    # ---- per-level disparity maps ---------------------------------------------------------------------------------
    def all_gather_rows(self, bands, key=None):
        mine = bands[self.rank]
        B, rows, W = mine.shape
        f = rows // (self.bands[self.rank][1] - self.bands[self.rank][0])
        H = self.h_coarse * f
        k = (key, B, H, W)
        if k not in self._full:
            t, hdl = self._alloc((B, H, W), torch.float32, mine.device)
            self._chan += 1
            self._full[k] = (t, hdl, [hdl.get_buffer(r, (B, H, W), torch.float32) for r in range(self.world)], self._chan)
        t, hdl, views, ch = self._full[k]
        r0 = self.bands[self.rank][0] * f
        for r in range(self.world):
            views[(self.rank + r) % self.world][:, r0:r0 + rows].copy_(mine)     # staggered: not everyone hits rank 0 first
        hdl.barrier(ch)
        return {self.rank: t}


def _dense_stage_bands(model, left0, right0, D, tr):
    """a2-a4 on row bands with per-layer halo exchange.  Returns {rank: pred band [B, rows, W]}."""
    reg = model.cost_regularizer
    pk = c3.packed_stack(reg)
    u = pk["units"]
    B, C, H0, W = left0.shape
    bands = shard.coarse_bands(H0, tr.world)
    if min(b - a for a, b in bands) < 1:
        raise ValueError(f"{tr.world} bands need at least {tr.world} rows at 1/27 scale, got {H0}")
    vol = {}
    for r in tr.ranks_here:
        r0, r1 = bands[r]
        v = torch.empty((B, D, r1 - r0 + 2, W, pk["cp"]), dtype=torch.bfloat16, device=left0.device)
        ops._call("decnet_costvol_bf16_ndhwc_rows", left0, left0.data_ptr(), right0.data_ptr(), v.data_ptr(),
                  B, C, pk["cp"], H0, W, D, r0 - 1, r1 - r0 + 2)
        vol[r] = v                          # halo rows already exact (computed from the replicated features)

    if isinstance(tr, PeerTransport):
        # peer-memory transport: three symmetric ping-pong buffers; a layer stores its owned rows only, the neighbours store
        # the halo rows (image-edge halo rows stay at their initial zero)
        r = tr.rank
        buf = {n: tr.conv_buffer(n, B, D, W, pk["cp"], left0.device) for n in ("t1", "t2", "o0")}

        def player(i, xin, name, residual=None):
            c3.conv3d_layer(xin, u[i][0], u[i][1], u[i][2], u[i][3], residual=residual, out=buf[name], band=True)
            tr.push_halo(name)
            return buf[name]
        x = player(0, vol[r], "t1")
        o0 = player(1, x, "o0")
        x = player(2, o0, "t1")
        x = player(3, x, "t2")
        x = player(4, x, "t1", residual=o0)
        x = player(5, x, "t2")
        x = player(6, x, "t1")
        cost = c3.conv3d_layer(x, u[7][0], u[7][1], u[7][2], False, out_f32=True)
        return {r: ops.softargmin(cost[:, :, 1:-1].contiguous())}

    def layer(i, xin, residual=None):
        out = {r: c3.conv3d_layer(xin[r], u[i][0], u[i][1], u[i][2], u[i][3],
                                  residual=None if residual is None else residual[r]) for r in tr.ranks_here}
        tr.exchange_halo(out)
        return out
    t1 = layer(0, vol)
    o0 = layer(1, t1)
    t1 = layer(2, o0)
    t2 = layer(3, t1)
    t1 = layer(4, t2, residual=o0)
    t2 = layer(5, t1)
    t1 = layer(6, t2)
    pred = {}
    for r in tr.ranks_here:
        cost = c3.conv3d_layer(t1[r], u[7][0], u[7][1], u[7][2], False, out_f32=True)     # [B, D, rows+2, W]
        pred[r] = ops.softargmin(cost[:, :, 1:-1].contiguous())
    return pred


def _level_stage_band(model, s, l, band, Lf, Rf, prevL, prevR, pred_prev_full, masks, D):
    """Stage s (>= 1) on the extended band [e0, e1); returns the exact owned rows of the new disparity."""
    e0, e1 = band.e0, band.e1
    Lb, Rb = Lf[:, :, e0:e1].contiguous(), Rf[:, :, e0:e1].contiguous()
    c0, c1 = e0 // 3, e1 // 3
    if model.use_detail:
        lm, rm = model.detail_detection[l].masks_pair(Lb, prevL[:, :, c0:c1].contiguous(), Rb,
                                                      prevR[:, :, c0:c1].contiguous(), model.thold)
    else:
        lm, rm = masks[0][l][:, e0:e1].contiguous(), masks[1][l][:, e0:e1].contiguous()
    dense = model.dynamic_upsampling[l](pred_prev_full[:, c0:c1].contiguous(), Lb)
    sparse, var, _, _ = ops.spamat_spavar_forward(Lb, Rb, lm, rm, D)
    x = ops.attn_pack(Lb, dense, sparse, lm, var)
    logit = model.soft_attention[l].logits(x).squeeze(1).contiguous()
    _, fused = ops.blend(logit, dense, sparse, want_mask=False)
    B, C, Hb, W = Lb.shape
    packed = torch.empty((B, 2 * C + 1, Hb, W), dtype=torch.float32, device=Lb.device)
    ops._call("decnet_refine_pack_rows", Lb, Lb.data_ptr(), Rb.data_ptr(), fused.data_ptr(), packed.data_ptr(),
              B, C, Hb, W, Lf.shape[2], e0)
    pred, _ = model.refinement[l].forward_packed(packed, fused, want_residual=False)
    return pred[:, band.r0 - e0: band.r1 - e0].contiguous()


@torch.no_grad()
def forward_bands(model, left_feats, right_feats, transport, left_mask_list=None, right_mask_list=None):
    """Row-band execution of DecompMatching.forward.  `left_feats` / `right_feats` are the FULL
    pyramids, replicated on every rank (each rank only touches its extended bands of the fine levels).
    Returns {rank: full final disparity [B, H, W]} (all-gathered after the last stage)."""
    tr = transport
    H0 = left_feats["stage0"].shape[2]
    tr.h_coarse = H0
    pred = _dense_stage_bands(model, left_feats["stage0"].contiguous(), right_feats["stage0"].contiguous(),
                              model.max_disp // 27, tr)
    gather = (lambda bands, key: tr.all_gather_rows(bands, key)) if isinstance(tr, PeerTransport) else (lambda bands, key: tr.all_gather_rows(bands))
    full = gather(pred, 0)
    for s in range(1, model.num_stage):
        Lf, Rf = left_feats[f"stage{s}"], right_feats[f"stage{s}"]
        if s >= model.skip_stage_id:
            # bicubic x3 (SparseDenseNetRefinementMask.py:143-144): every rank upsamples its coarse band
            # with a 2-row halo and keeps its own rows
            out = {}
            for r in tr.ranks_here:
                b = shard.level_band(H0, tr.world, r, s - 1, 2)
                up = ops.bicubic_skip(full[r][:, b.e0:b.e1].contiguous(), 3 * (b.e1 - b.e0), Lf.shape[3])
                out[r] = up[:, 3 * (b.r0 - b.e0): 3 * (b.r1 - b.e0)].contiguous()
            full = gather(out, s)
            continue
        D = model.max_disp // 3 ** (model.num_stage - s - 1)
        out = {}
        for r in tr.ranks_here:
            band = shard.level_band(H0, tr.world, r, s, EXT[s])
            out[r] = _level_stage_band(model, s, s - 1, band, Lf, Rf, left_feats[f"stage{s - 1}"],
                                       right_feats[f"stage{s - 1}"], full[r],
                                       (left_mask_list, right_mask_list), D)
        full = gather(out, s)
    return full
