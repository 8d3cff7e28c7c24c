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
    n = args.stream_steps
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in m.stream([pair] * n, output="u16"):
        pass
    el = time.perf_counter() - t0
    rate = B * n / el
    e2e = res["bench_py"].get("e2e")
    res["sceneflow_stream"] = {"batch": B, "steps": n, "pairs_per_s": rate, "ms_per_step": el / n * 1e3,
                               "left_mask_density": [round(d, 4) for d in dens],
                               "bench_py_e2e_pairs_per_s": e2e if e2e is not None else "not measured",
                               "ratio_to_bench_py_e2e": rate / e2e if e2e else "not measured",
                               "what": "CPU uint8 tensors in -> pinned staging -> H2D on a copy stream -> graph -> disp_to_u16 -> "
                                       "pinned D2H -> new tensor, two buffer sets; host clock over the whole loop"}
    del m
    torch.cuda.empty_cache()

    # 3. one Middlebury pair, demo.sh's configuration
    lm, rm = (g.integers(0, 256, (2000, 2900, 3), dtype=np.uint8) for _ in range(2))
    m = StereoMatcher(max_disp=768, masks="image", skip_stage_id=3)
    res["middlebury_single"] = dict(latency(torch, m, lm, rm, 30, 3), shape="2000x2900 -> 2025x2916", max_disp=783,
                                    masks="image", skip_stage_id=3)
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
    (out / "bench_predictor.json").write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
