#!/usr/bin/env python
"""StereoMatcher measurements (one GPU, one process), written as OUT/bench_predictor.json:

  sceneflow_single   one 960x540 pair, max_disp 192, learned masks: host-to-host latency of m(left, right, output="u16")
                     (numpy in / out, p50 / p90 over >= 200 calls), the device time of the graph replay alone (CUDA events),
                     and the host time of the weight-signature check and of the copies either side of the replay
  sceneflow_stream   B = 8 SceneFlow pairs through m.stream() (pinned staging, double-buffered), pairs/s, next to the `e2e`
                     of `python bench.py` run by this script: the matcher is set up as bench.leg_from_images does (seed-17
                     weights, detector mask density calibrated to 0.10 on the same seeded uint8 inputs), so both run one graph
                     of the same work
  middlebury_single  one 2000x2900 pair (padded to 2025x2916), max_disp 768, skip_stage_id 3, masks="image": latency as above
  bicubic_up3        bicubic_up3_kernel against F.interpolate(bicubic) at 675x972 -> 2025x2916: us per launch and the share of
                     the HBM bound (data-sheet 7.7 TB/s; the 23.6 MB output fits the 126 MB L2, so back-to-back launches are not
                     flushed between them)
  *_lr               the same legs with the left-right check (lr_check=1.0: the reverse direction in the same graph at 2B,
                     then lr_check_kernel), measured in the same process, alternating with the plain leg call by call
                     (single pairs) or run by run (stream)
  mirror_swap_u8,    the two kernels of the check at B = 8 SceneFlow pairs: us per launch and the share of the HBM bound on
  lr_check           their algorithmic bytes (mirror: 2 * 2*B*h*w*3; lr_check: 4 + 4 bytes read per pixel plus the outputs),
                     launches rotating over enough buffers (> 300 MB) that each one reads from HBM, not L2
  lr_fill_*          the check fused with background hole filling (decnet_lr_check_fill: lr_check_fill_rows_kernel +
                     lr_fill_empty_rows_kernel) at B = 8 SceneFlow pairs and one Middlebury pair, timed as lr_check_* in the
                     same process beside an lr_check leg of the same shape; bytes: 8 read per pixel, written the float rows
                     (always: the column phase reads them), the requested uint16 / valid outputs and one flag per row
  sceneflow_stream_lr_fill  sceneflow_stream with the check and fill="background", runs alternating with the plain and _lr ones

    python scripts/bench_predictor.py --out DIR
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

HBM_GBS = 7700.0
LR_TOL = 1.0


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit"], info["max_sm_clock"] = (s.strip() for s in r.stdout.strip().split(","))
    except Exception as e:
        info["power_limit"] = f"not read: {type(e).__name__}: {e}"
    return info


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, int(round(q * (len(xs) - 1))))]


def latency(torch, m, left, right, calls, warmup):
    """Host-to-host latency of m(left, right, output="u16") and the parts of one call."""
    for _ in range(warmup):
        m(left, right, output="u16")
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter()
        m(left, right, output="u16")
        ts.append((time.perf_counter() - t0) * 1e3)
    (st,) = m._graphs[next(reversed(m._graphs))]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = max(10, calls // 4)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        st.graph.replay()
    e1.record()
    torch.cuda.synchronize()
    sig_ms = []
    for _ in range(100):
        t0 = time.perf_counter()
        assert m._sig() == st.sig
        sig_ms.append((time.perf_counter() - t0) * 1e3)
    up_ms, down_ms = [], []
    for _ in range(20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m._upload(st, left, right, "numpy")
        torch.cuda.synchronize()
        up_ms.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        m._result(st, left.shape[0], left.shape[1], "u16").cpu().numpy()
        down_ms.append((time.perf_counter() - t0) * 1e3)
    return {"calls": calls, "warmup": warmup, "p50_ms": pct(ts, 0.5), "p90_ms": pct(ts, 0.9), "min_ms": min(ts),
            "replay_device_ms": e0.elapsed_time(e1) / n,
            "signature_check_host_ms": pct(sig_ms, 0.5),
            "upload_host_ms": pct(up_ms, 0.5), "what_upload": "both views into the pinned staging + H2D, synchronised",
            "readback_host_ms": pct(down_ms, 0.5), "what_readback": "disp_to_u16 + D2H into a new numpy array, synchronised"}


def latency_pair(torch, m, left, right, calls, warmup):
    """latency() of the plain call and of the call with the left-right check, alternating call by call."""
    from decnet_b200.predictor import cache_key
    h, w = left.shape[:2]
    legs = {"plain": {}, "lr": {"lr_check": LR_TOL}}
    for kw in legs.values():
        for _ in range(warmup):
            m(left, right, output="u16", **kw)
    ts = {k: [] for k in legs}
    for _ in range(calls):
        for k, kw in legs.items():
            t0 = time.perf_counter()
            m(left, right, output="u16", **kw)
            ts[k].append((time.perf_counter() - t0) * 1e3)
    sets = {k: m._graphs[cache_key(1, h, w, m.max_disp, m.masks, m.precision, k == "lr")][0] for k in legs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = max(10, calls // 8)
    dev_ms = {k: [] for k in legs}
    for _ in range(2):
        for k, st in sets.items():
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n):
                st.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            dev_ms[k].append(e0.elapsed_time(e1) / n)
    out = {}
    for k, st in sets.items():
        tol = legs[k].get("lr_check")
        down = []
        for _ in range(20):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m._result(st, h, w, "u16", tol).cpu().numpy()
            down.append((time.perf_counter() - t0) * 1e3)
        out[k] = {"calls": calls, "warmup": warmup, "p50_ms": pct(ts[k], 0.5), "p90_ms": pct(ts[k], 0.9), "min_ms": min(ts[k]),
                  "replay_device_ms": min(dev_ms[k]), "replay_device_ms_runs": dev_ms[k],
                  "readback_host_ms": pct(down, 0.5),
                  "what_readback": ("lr_check (u16) + D2H" if tol is not None else "disp_to_u16 + D2H") + ", synchronised"}
    out["lr"]["lr_check"] = LR_TOL
    out["lr_over_plain"] = {"p50": out["lr"]["p50_ms"] / out["plain"]["p50_ms"],
                            "replay_device": out["lr"]["replay_device_ms"] / out["plain"]["replay_device_ms"]}
    return out


def kernel_us(torch, fn_of_set, nsets, n=96, reps=5):
    """Device us per launch of fn_of_set(i), rotating i over nsets buffer sets: n launches captured in one CUDA graph (no host
    overhead between them), best of `reps` timed replays."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(nsets):
            fn_of_set(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(n):
            fn_of_set(i % nsets)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = float("inf")
    for _ in range(reps):
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e3 / n)
    g.reset()
    return best


def hbm_share(nbytes, us):
    return {"bytes": nbytes, "hbm_bound_us": nbytes / (HBM_GBS * 1e9) * 1e6,
            "frac_of_hbm_bound": nbytes / (HBM_GBS * 1e9) / (us * 1e-6), "hbm_gbs_assumed": HBM_GBS}


def run_bench_py():
    cmd = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", "20", "--warmup", "5", "--no-cpu-baseline",
           "--no-extras"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, cwd=str(ROOT))
    try:
        line = json.loads(r.stdout.strip().splitlines()[-1])
        return {"command": " ".join(["python", "bench.py"] + cmd[2:]), "e2e": line["e2e"]["value"],
                "value": line["value"], "unit": line["unit"]}
    except Exception as e:
        return {"command": " ".join(cmd[1:]), "error": f"{type(e).__name__}: {e}", "stderr": r.stderr[-2000:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--stream-steps", type=int, default=60)
    args = ap.parse_args()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_predictor.py needs a CUDA device")
    from decnet_b200 import StereoMatcher, ops
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(torch)}
    res["bench_py"] = run_bench_py()

    # 1. one SceneFlow pair
    g = np.random.default_rng(0)
    l1, r1 = (g.integers(0, 256, (540, 960, 3), dtype=np.uint8) for _ in range(2))
    m = StereoMatcher(max_disp=192)
    res["sceneflow_single"] = dict(latency(torch, m, l1, r1, args.calls, 10), shape="540x960 -> 540x972", max_disp=216,
                                   masks="learned")
    res["sceneflow_single_lr"] = dict(latency_pair(torch, m, l1, r1, args.calls, 10), shape="540x960 -> 540x972",
                                      max_disp=216, masks="learned")
    del m
    torch.cuda.empty_cache()

    # 2. B = 8 through stream(), set up as bench.leg_from_images
    from decnet_b200.synthetic import calibrate_mask_density
    B = 8
    m = StereoMatcher(max_disp=192)
    gd = torch.Generator(device=dev).manual_seed(99)
    l8 = torch.randint(0, 256, (B, 540, 960, 3), device=dev, generator=gd, dtype=torch.uint8)
    r8 = torch.randint(0, 256, (B, 540, 960, 3), device=dev, generator=gd, dtype=torch.uint8)
    prep = lambda u8: ops.image_prepare_u8(u8, want01=False)[1]
    dens = calibrate_mask_density(m.model, m.fe(prep(l8)), m.fe(prep(r8)), 0.10)
    pair = (l8.cpu(), r8.cpu())
    for _ in m.stream([pair] * 4, output="u16"):
        pass
    for _ in m.stream([pair] * 4, output="u16", lr_check=LR_TOL):
        pass
    for _ in m.stream([pair] * 4, output="u16", lr_check=LR_TOL, fill="background"):
        pass
    n = args.stream_steps

    def run(**kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in m.stream([pair] * n, output="u16", **kw):
            pass
        return time.perf_counter() - t0
    els = {"plain": [], "lr": [], "lr_fill": []}
    for _ in range(2):                                                   # alternating plain, LR and LR + fill runs
        els["plain"].append(run())
        els["lr"].append(run(lr_check=LR_TOL))
        els["lr_fill"].append(run(lr_check=LR_TOL, fill="background"))
    el = min(els["plain"])
    rate = B * n / el
    rate_lr = B * n / min(els["lr"])
    e2e = res["bench_py"].get("e2e")
    res["sceneflow_stream"] = {"batch": B, "steps": n, "pairs_per_s": rate, "ms_per_step": el / n * 1e3,
                               "left_mask_density": [round(d, 4) for d in dens],
                               "bench_py_e2e_pairs_per_s": e2e if e2e is not None else "not measured",
                               "ratio_to_bench_py_e2e": rate / e2e if e2e else "not measured",
                               "what": "CPU uint8 tensors in -> pinned staging -> H2D on a copy stream -> graph -> disp_to_u16 -> "
                                       "pinned D2H -> new tensor, two buffer sets; host clock over the whole loop; best of two runs"}
    res["sceneflow_stream_lr"] = {"batch": B, "steps": n, "lr_check": LR_TOL, "pairs_per_s": rate_lr,
                                  "ms_per_step": min(els["lr"]) / n * 1e3,
                                  "pairs_per_s_runs": {k: [B * n / e for e in v] for k, v in els.items()},
                                  "lr_over_plain_step_time": rate / rate_lr,
                                  "what": "as sceneflow_stream with the left-right check; runs alternate with the plain ones"}
    rate_fill = B * n / min(els["lr_fill"])
    res["sceneflow_stream_lr_fill"] = {"batch": B, "steps": n, "lr_check": LR_TOL, "fill": "background", "pairs_per_s": rate_fill,
                                       "ms_per_step": min(els["lr_fill"]) / n * 1e3,
                                       "lr_fill_over_lr_step_time": rate_lr / rate_fill,
                                       "what": "as sceneflow_stream_lr with fill=\"background\" (lr_check_fill_rows_kernel + "
                                               "lr_fill_empty_rows_kernel instead of lr_check_kernel); runs alternate with the "
                                               "plain and _lr ones"}
    del m
    torch.cuda.empty_cache()

    # 3. one Middlebury pair, demo.sh's configuration
    lm, rm = (g.integers(0, 256, (2000, 2900, 3), dtype=np.uint8) for _ in range(2))
    m = StereoMatcher(max_disp=768, masks="image", skip_stage_id=3)
    res["middlebury_single"] = dict(latency(torch, m, lm, rm, 30, 3), shape="2000x2900 -> 2025x2916", max_disp=783,
                                    masks="image", skip_stage_id=3)
    res["middlebury_single_lr"] = dict(latency_pair(torch, m, lm, rm, 30, 3), shape="2000x2900 -> 2025x2916",
                                       max_disp=783, masks="image", skip_stage_id=3)
    del m
    torch.cuda.empty_cache()

    # 4. the skip-stage kernel against ATen's
    import torch.nn.functional as F
    x = torch.randn(1, 675, 972, device=dev) * 100
    H, W = 2025, 2916
    assert torch.equal(ops.bicubic_skip(x, H, W), F.interpolate((x * 3).unsqueeze(1), (H, W), mode="bicubic").squeeze(1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def us(fn, n=200):
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / n
    y = torch.empty(1, H, W, device=dev)
    ours = us(lambda: ops._call("decnet_bicubic_up3", x, x.data_ptr(), y.data_ptr(), 1, 675, 972, H, W))
    x3 = (x * 3).unsqueeze(1)
    aten = us(lambda: F.interpolate(x3, (H, W), mode="bicubic"))
    nbytes = 4 * (675 * 972 + H * W)
    res["bicubic_up3"] = {"shape": "1x675x972 -> 1x2025x2916", "us": ours, "aten_interpolate_us": aten,
                          "aten_note": "F.interpolate on pred*3 computed beforehand (the x3 multiply is not timed)",
                          "bytes": nbytes, "hbm_bound_us": nbytes / (HBM_GBS * 1e9) * 1e6,
                          "frac_of_hbm_bound": nbytes / (HBM_GBS * 1e9) / (ours * 1e-6), "hbm_gbs_assumed": HBM_GBS}

    # 5. the left-right check's kernels at B = 8 SceneFlow pairs, rotating over buffer sets larger than L2 together
    B, h, w, H, W, nsets = 8, 540, 960, 540, 972, 8
    img = [[torch.randint(0, 256, (2 * B, h, w, 3), device=dev, dtype=torch.uint8) for _ in range(2)] for _ in range(nsets)]
    ptr = [[t.data_ptr() for t in (a[:B], b[:B], a[B:], b[B:])] for a, b in img]
    t_mirror = kernel_us(torch, lambda i: ops._call("decnet_mirror_swap_u8", img[i][0], *ptr[i], B, h, w), nsets)
    res["mirror_swap_u8"] = dict(hbm_share(2 * 2 * B * h * w * 3, t_mirror), us=t_mirror, shape=f"{B}x{h}x{w}x3, both views",
                                 path="16-byte (w % 16 == 0)", buffer_sets=nsets)
    del img
    preds = [torch.randn(2 * B, H, W, device=dev) * 20 + 40 for _ in range(nsets)]
    for name, out_bytes in (("u16", 2), ("float_valid", 5)):
        outs = [(torch.empty(B, h, w, device=dev) if name == "float_valid" else None,
                 torch.empty(B, h, w, dtype=torch.uint16, device=dev) if name == "u16" else None,
                 torch.empty(B, h, w, dtype=torch.bool, device=dev) if name == "float_valid" else None) for _ in range(nsets)]
        t = kernel_us(torch, lambda i: ops._call("decnet_lr_check", preds[i], preds[i].data_ptr(), B, H, W, h, w, LR_TOL,
                                                 *(o.data_ptr() if o is not None else None for o in outs[i])), nsets)
        res[f"lr_check_{name}"] = dict(hbm_share(B * h * w * (8 + out_bytes), t), us=t, shape=f"pred {2 * B}x{H}x{W} -> {B}x{h}x{w}",
                                       outputs=name, buffer_sets=nsets)
    del preds
    torch.cuda.empty_cache()

    # 6. the check with background hole filling beside the check alone, at B = 8 SceneFlow pairs and one Middlebury pair
    for tag, (B, h, w, H, W, nsets) in (("", (8, 540, 960, 540, 972, 8)), ("_middlebury", (1, 2000, 2900, 2025, 2916, 8))):
        preds = [torch.randn(2 * B, H, W, device=dev) * 20 + 40 for _ in range(nsets)]
        for name, out_bytes in (("u16", 2), ("float_valid", 5)):
            outs = [(torch.empty(B, h, w, device=dev),
                     torch.empty(B, h, w, dtype=torch.uint16, device=dev) if name == "u16" else None,
                     torch.empty(B, h, w, dtype=torch.bool, device=dev) if name == "float_valid" else None,
                     torch.empty(B, h, dtype=torch.uint8, device=dev)) for _ in range(nsets)]
            chk = lambda i: ops._call("decnet_lr_check", preds[i], preds[i].data_ptr(), B, H, W, h, w, LR_TOL,
                                      outs[i][0].data_ptr() if name == "float_valid" else None,
                                      *(o.data_ptr() if o is not None else None for o in outs[i][1:3]))
            fil = lambda i: ops._call("decnet_lr_check_fill", preds[i], preds[i].data_ptr(), B, H, W, h, w, LR_TOL,
                                      *(o.data_ptr() if o is not None else None for o in outs[i]))
            runs = {"check": [], "fill": []}
            for _ in range(2):                                           # alternating, best of each
                runs["check"].append(kernel_us(torch, chk, nsets))
                runs["fill"].append(kernel_us(torch, fil, nsets))
            t_chk, t_fill = min(runs["check"]), min(runs["fill"])
            (valid,) = ops.lr_check(preds[0], h, w, LR_TOL, float_out=False, valid_out=True)
            shape = f"pred {2 * B}x{H}x{W} -> {B}x{h}x{w}"
            if tag:
                res[f"lr_check_{name}{tag}"] = dict(hbm_share(B * h * w * (8 + out_bytes), t_chk), us=t_chk, shape=shape,
                                                    outputs=name, buffer_sets=nsets, us_runs=runs["check"])
            fill_bytes = B * h * w * (8 + 4 + (2 if name == "u16" else 1)) + B * h
            res[f"lr_fill_{name}{tag}"] = dict(hbm_share(fill_bytes, t_fill), us=t_fill, shape=shape, outputs=name,
                                               buffer_sets=nsets, us_runs=runs["fill"], lr_check_us=t_chk,
                                               fill_over_check=t_fill / t_chk,
                                               valid_fraction=float(valid.float().mean()),
                                               what="decnet_lr_check_fill (both kernels) vs decnet_lr_check, alternating")
        del preds
        torch.cuda.empty_cache()
    (out / "bench_predictor.json").write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
