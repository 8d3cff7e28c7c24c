"""A/B of the channels-last halo conv's two fp32-class input forms at the 13 launches of the benchmarked step (B = 8, SceneFlow):
  fp32   -- split = 2: fp32 activations, converter warps build the fp16 correction tile, TF32 hi taps + fp16 taps of the weights
  split16 -- split = 3: activations stored as split16 by the producer (the route model.py takes), fp16 taps only
Each layer runs as in the step: inner layers write their output in the next layer's input format, the last layer of a stack
writes fp32.  The two forms alternate, ROUNDS rounds of LAUNCHES launches each, timed with CUDA events; the median per launch
is reported.  Prints one line per layer; `ab_halo_split16.py OUT.json` also writes the summary there."""
import json
import statistics
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[2]))
from decnet_b200 import ops

ROUNDS, LAUNCHES = 7, 20
L2_BYTES = 126 * 2 ** 20
B = 8
# (stack, h, w, cin, cout, relu, last): the DynamicUpsampling stacks at 1/27, 1/9, 1/3 and the wide 1/9 Refinement
LAYERS = [("dynup 1/27", 20, 36, 649, 81, True, False), ("dynup 1/27", 20, 36, 81, 81, True, False),
          ("dynup 1/27", 20, 36, 81, 81, False, True),
          ("refine 1/9", 60, 108, 145, 72, True, False), ("refine 1/9", 60, 108, 72, 72, True, False),
          ("refine 1/9", 60, 108, 72, 72, True, False), ("refine 1/9", 60, 108, 72, 36, True, True),
          ("dynup 1/9", 60, 108, 217, 81, True, False), ("dynup 1/9", 60, 108, 81, 81, True, False),
          ("dynup 1/9", 60, 108, 81, 81, False, True),
          ("dynup 1/3", 180, 324, 73, 81, True, False), ("dynup 1/3", 180, 324, 81, 81, True, False),
          ("dynup 1/3", 180, 324, 81, 81, False, True)]


def time_us(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(LAUNCHES):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / LAUNCHES * 1e3


def main():
    assert ops.SPLIT_KIND == 2, "compares against split kind 2 (the default)"
    g = torch.Generator(device="cuda").manual_seed(0)
    rows = []
    for stack, h, w, cin, cout, relu, last in LAYERS:
        x = torch.randn(B, cin, h, w, device="cuda", generator=g)
        wt = torch.randn(cout, cin, 3, 3, device="cuda", generator=g) * (2.0 / (9 * cin)) ** 0.5
        bias = torch.randn(cout, device="cuda", generator=g) * 0.1
        cp8, cp16 = (cin + 7) // 8 * 8, (cin + 15) // 16 * 16
        x_old = ops.nchw_cat_to_nhwc_pad([x], cp8, round_tf32=False)
        x_new = ops.nchw_cat_to_nhwc_pad([x], cp16, split16=True)
        w_old, b_old, np_ = ops.pack_conv2d_tf32_weights(wt, bias, cp8, split=True)
        w_new, b_new, _ = ops.pack_conv2d_tf32_weights(wt, bias, cp16, split=True, split16_in=True)
        old = lambda: ops.conv2d_tf32_nhwc_halo(x_old, w_old, b_old, relu, split=True)
        new = lambda: ops.conv2d_tf32_nhwc_halo(x_new, w_new, b_new, relu, split=True, split16_out=not last)
        want = F.conv2d(x.double(), wt.double(), bias.double(), padding=1)
        want = F.relu(want) if relu else want
        got = ops.conv2d_tf32_nhwc_halo(x_new, w_new, b_new, relu, split=True)[:, 1:-1, 1:-1, :cout].permute(0, 3, 1, 2)
        rel_err = float((got.double() - want).abs().max() / want.abs().max())
        for _ in range(3):
            old(); new()
        t_old, t_new = [], []
        for _ in range(ROUNDS):
            t_old.append(time_us(old))
            t_new.append(time_us(new))
        in_bytes = x_old.numel() * 4
        out_bytes = B * (h + 2) * (w + 2) * np_ * 4
        r = {"stack": stack, "h": h, "w": w, "cin": cin, "cout": cout, "cp_fp32": cp8, "cp_split16": cp16,
             "fp32_us": statistics.median(t_old), "split16_us": statistics.median(t_new),
             "fp32_us_range": [min(t_old), max(t_old)], "split16_us_range": [min(t_new), max(t_new)],
             "input_MB": in_bytes / 1e6, "input_plus_output_exceed_l2": in_bytes + out_bytes > L2_BYTES,
             "split16_rel_err_vs_fp64": rel_err}
        r["ratio"] = r["split16_us"] / r["fp32_us"]
        rows.append(r)
        print(f"{stack:11s} {cin:4d}->{cout:3d} {h}x{w}  fp32 {r['fp32_us']:7.1f} us [{min(t_old):.1f}, {max(t_old):.1f}]  "
              f"split16 {r['split16_us']:7.1f} us [{min(t_new):.1f}, {max(t_new):.1f}]  ratio {r['ratio']:.3f}  "
              f"in+out {'>' if r['input_plus_output_exceed_l2'] else '<='} L2  err {rel_err:.1e}", flush=True)
    tot_old, tot_new = sum(r["fp32_us"] for r in rows), sum(r["split16_us"] for r in rows)
    summary = {"device": torch.cuda.get_device_name(), "B": B, "rounds": ROUNDS, "launches_per_round": LAUNCHES,
               "layers": rows, "sum_fp32_us": tot_old, "sum_split16_us": tot_new}
    print(f"13 launches: fp32 {tot_old:.1f} us, split16 {tot_new:.1f} us, ratio {tot_new / tot_old:.3f}")
    if len(sys.argv) > 1:
        Path(sys.argv[1]).write_text(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
