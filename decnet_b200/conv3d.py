"""Host side of the tcgen05 3-D aggregation: weight packing (BN folded, bf16 [27][NP][CP]),
activation ping-pong buffers, the 8-layer stack of CostRegNetNoDown (modules/submodule.py:650-662)
and its tensor roofline measurement."""
from __future__ import annotations

import torch

from . import ops


def _pad16(n: int) -> int:
    return (n + 15) // 16 * 16


def pack_unit(unit, cp: int):
    """Conv3dUnit -> (weights bf16 [27][NP][CP] with the BN scale folded in, bias fp32 [NP])."""
    w = unit.conv.weight.detach().float()                      # [Cout, Cin, 3, 3, 3]
    cout, cin = w.shape[:2]
    scale, shift = unit.scale_bias()
    w = w * scale.float().view(-1, 1, 1, 1, 1)
    np_ = _pad16(cout)
    packed = torch.zeros((27, np_, cp), dtype=torch.float32, device=w.device)
    packed[:, :cout, :cin] = w.permute(2, 3, 4, 0, 1).reshape(27, cout, cin)   # tap = (kd*3+kh)*3+kw
    bias = torch.zeros(np_, dtype=torch.float32, device=w.device)
    bias[:cout] = shift.float()
    return packed.to(torch.bfloat16).contiguous(), bias.contiguous(), np_


def packed_stack(reg):
    """Per-module pack, cached on the identity of the module's parameters and BN statistics (model._Cached)."""
    def build():
        cin = reg.conv0[0].conv.weight.shape[1]
        cp = _pad16(cin)
        return {"cp": cp, "units": [pack_unit(u, cp) + (u.relu,) for u in reg.units()]}
    return reg._cached("packed", build)


def conv3d_layer(x, w, bias, np_, relu, residual=None, out=None, out_f32=False, band=False):
    """x bf16 [B,D,H,W,CP] -> bf16 [B,D,H,W,NP] (or fp32 [B,D,H,W] of channel 0 when out_f32).
    band: row-band mode -- rows 0 and H-1 of `out` are halo slots filled by the neighbouring ranks, not stored here."""
    B, D, H, W, cp = x.shape
    if out is None:
        out = (torch.empty((B, D, H, W), dtype=torch.float32, device=x.device) if out_f32
               else torch.empty((B, D, H, W, np_), dtype=torch.bfloat16, device=x.device))
    res = residual.data_ptr() if residual is not None else None
    if band:
        assert not out_f32
        ops._call("decnet_conv3d_bf16_band", x, x.data_ptr(), w.data_ptr(), bias.data_ptr(), res, out.data_ptr(),
                  B, D, H, W, cp, np_, 1 if relu else 0)
    else:
        ops._call("decnet_conv3d_bf16", x, x.data_ptr(), w.data_ptr(), bias.data_ptr(), res, out.data_ptr(),
                  1 if out_f32 else 0, B, D, H, W, cp, np_, 1 if relu else 0)
    return out


def run_stack(reg, vol, with_pred=False):
    """vol bf16 [B,D,H,W,CP] -> regularised cost fp32 [B,D,H,W]; o = conv1(conv0(x)) + conv0(x)."""
    pk = packed_stack(reg)
    u = pk["units"]
    assert vol.shape[-1] == pk["cp"] and all(x[2] == pk["cp"] for x in u[:7]), "channel padding mismatch"
    t1 = conv3d_layer(vol, u[0][0], u[0][1], u[0][2], True)
    o0 = conv3d_layer(t1, u[1][0], u[1][1], u[1][2], True)
    conv3d_layer(o0, u[2][0], u[2][1], u[2][2], True, out=t1)
    t2 = conv3d_layer(t1, u[3][0], u[3][1], u[3][2], True)
    conv3d_layer(t2, u[4][0], u[4][1], u[4][2], True, residual=o0, out=t1)
    conv3d_layer(t1, u[5][0], u[5][1], u[5][2], True, out=t2)
    conv3d_layer(t2, u[6][0], u[6][1], u[6][2], True, out=t1)
    if not with_pred:
        return conv3d_layer(t1, u[7][0], u[7][1], u[7][2], False, out_f32=True)
    # last layer + soft-argmin (a4) in one launch
    B, D, H, W, cp = t1.shape
    cost = torch.empty((B, D, H, W), dtype=torch.float32, device=t1.device)
    pred = torch.empty((B, H, W), dtype=torch.float32, device=t1.device)
    ops._call("decnet_conv3d_bf16_softargmin", t1, t1.data_ptr(), u[7][0].data_ptr(), u[7][1].data_ptr(), cost.data_ptr(),
              pred.data_ptr(), B, D, H, W, cp, u[7][2], 0)
    return pred, cost


def dense_pred(reg, Lf, Rf, D):
    """a2 + a3 + a4: cost volume -> tcgen05 stack -> soft-argmin (in the last layer's epilogue).  (pred [B,H,W], cost)."""
    pk = packed_stack(reg)
    vol = ops.cost_volume_bf16_ndhwc(Lf, Rf, D, pk["cp"])
    return run_stack(reg, vol, with_pred=True)


def dense_cost(reg, Lf, Rf, D):
    """a2 + a3: bf16 channels-last cost volume straight into the tcgen05 stack -> fp32 cost [B,D,H,W]."""
    pk = packed_stack(reg)
    vol = ops.cost_volume_bf16_ndhwc(Lf, Rf, D, pk["cp"])
    return run_stack(reg, vol)


def cost_regularizer_forward(reg, vol_ncdhw):
    """Drop-in path for CostRegNetNoDown.forward([B,C,D,H,W] fp32): repack to bf16 channels-last
    (torch permute/cast: boundary conversion only, the fused route is dense_cost)."""
    pk = packed_stack(reg)
    B, C, D, H, W = vol_ncdhw.shape
    x = torch.zeros((B, D, H, W, pk["cp"]), dtype=torch.bfloat16, device=vol_ncdhw.device)
    x[..., :C] = vol_ncdhw.permute(0, 2, 3, 4, 1)
    return run_stack(reg, x)


def stack_flops(B, D, H, W, cin):
    """Useful (un-padded) FLOPs of the stack: 7 layers cin->cin + one cin->1, zero-padding taps counted
    (SURVEY.md section 8d)."""
    m = B * D * H * W
    return 7 * 2.0 * m * 27 * cin * cin + 2.0 * m * 27 * cin


@torch.no_grad()
def measure_roofline(model, Lf, Rf, D, peaks, iters=10):
    reg = model.cost_regularizer
    pk = packed_stack(reg)
    vol = ops.cost_volume_bf16_ndhwc(Lf, Rf, D, pk["cp"])
    for _ in range(3):
        run_stack(reg, vol)
    torch.cuda.synchronize()
    # the 8 launches are captured in a CUDA graph so that the device time is measured, not the host's
    # launch path (8 ctypes calls + tensor-map lookups per stack)
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run_stack(reg, vol)
        with torch.cuda.graph(graph, stream=side):
            run_stack(reg, vol)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        graph.replay()
    e1.record(); torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3 / iters
    B, _, H, W = Lf.shape
    fl = stack_flops(B, D, H, W, Lf.shape[1])
    ach = fl / t / 1e12
    peak = peaks["bf16_tflops"]
    return {"bound": "tensor", "kernel": "conv3d_tcgen05_kernel x8 (3-D aggregation stack)", "achieved": ach,
            "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
            "peak_source": peaks["source"] + " (cuBLAS bf16 burst)", "useful_flops": fl, "us_per_stack": t * 1e6}
