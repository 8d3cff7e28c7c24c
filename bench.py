#!/usr/bin/env python
"""bench.py -- decomposed-matching hot path throughput (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, one process per GPU)
    python bench.py --impl reference --steps K --warmup W    # reference arm: CPU port on host cores

One "step" = one pass of the hot path (SparseDenseNetRefinementMask.forward after feature
extraction: cost volume -> 3-D aggregation -> soft-argmin, then per level detail masks ->
dynamic up-sampling -> SpaMat/SpaVar -> soft attention + blend -> refinement) over one batch of
synthetic SceneFlow-shaped feature pyramids (540x960 -> 540x972, max_disp "192" -> 216), random-init
weights.  N=1 workload = BASELINE.json configs[1] (batch 8 on one B200); N>1 shards by stereo pair,
no collective on the data path (weak scaling).  Prints ONE JSON line on rank 0.

Keys beyond the base contract:
  value            device-timed, feature pyramids resident in HBM (CUDA graph replay), default precision "fp32" = 3xTF32
  e2e              demo.py's boundary at every N: uint8 image pairs in pinned host memory -> device -> pad / normalise ->
                   feature extractor (both views) -> hot path -> uint16 disparity image -> pinned host memory, every step
  e2e_pyramids     the hot path alone behind host buffers: fp32 feature pyramids (398 MB / step) uploaded every step
  tf32             the same step in the plain-TF32 arithmetic mode (the class cuDNN gives the reference on a GPU)
  roofline         sparse kernel, finest level (+ the three-level aggregate, a density sweep and the reference's own kernels
                   recompiled for sm_100a on the same inputs); roofline_tensor / roofline_conv2d: the other two kernels
  gpu_reference    the UNMODIFIED reference model (PyTorch / cuDNN eager + its CUDA kernels, feature maps given) timed as
                   demo.py:185-189 on the same GPU
  bands            (N > 1) ONE Middlebury pair split into row bands over the N ranks (BASELINE.json configs[3])
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

UNIT = "pairs/s"


def metric_name(workload):
    from decnet_b200.synthetic import WORKLOADS
    H, W, max_disp, _ = WORKLOADS[workload]
    shape = {"sceneflow": "540x960", "kitti": "376x1248", "middlebury": "~2000x2900"}.get(workload, f"{H}x{W}")
    return f"stereo pairs/s @{shape} (decomposed-matching hot path, {workload} shape padded to {H}x{W}, max_disp {max_disp})"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu-leg"])
    ap.add_argument("--workload", default="sceneflow")
    ap.add_argument("--batch", type=int, default=8, help="stereo pairs per GPU per step")
    ap.add_argument("--rho", type=float, default=0.10, help="calibrated lost-detail mask density")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32"],
                    help="arithmetic mode of the 2-D tensor-core convs: fp32 = error-compensated 3xTF32 (parity-gated default), "
                         "tf32 = plain TF32 (what the reference gets from cuDNN on a GPU)")
    ap.add_argument("--mode", default="pairs", choices=["pairs", "bands"],
                    help="pairs: shard by stereo pair (weak scaling); bands: ONE pair split into row bands "
                         "with halo exchange (strong scaling, BASELINE.json configs[3])")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--no-overlap", action="store_true",
                    help="masks + sparse ops on the main stream instead of a forked second stream")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-from-images", action="store_true", help="skip the images -> disparity leg (then e2e = e2e_pyramids)")
    ap.add_argument("--no-extras", action="store_true", help="skip tf32 / gpu_reference / bands / density sweep")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="host time of the bounded CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="our arm: write what the last timed step returned (rank 0's final disparity) as DIR/disparity.npy, "
                         "float32; inputs and weights are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to our arm only")
    return args


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, outputs):
    """Each tensor of `outputs` as out_dir/<name>.npy in float32, all of them together at most DUMP_BYTES.  A tensor larger
    than its share is replaced by a fixed sample of it: the elements at sorted positions drawn without replacement by a
    numpy generator seeded with 0, as a flat array (the same positions in every run with the same arguments)."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // len(outputs) - 1024                    # room for the .npy header
    for name, t in outputs.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            pos = np.sort(np.random.default_rng(0).choice(a.size, share // 4, replace=False))
            a = a.reshape(-1)[pos]
        np.save(out_dir / f"{name}.npy", a)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops", 1590.0),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock / throttle reasons during the timed region: NVML polled every 5 ms from a thread (the region is ~0.1 s long, so
    nvidia-smi's 200 ms loop yields one or two samples); nvidia-smi -lms 200 when pynvml is missing."""

    NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def _nvml_loop(self):
        import pynvml as nv
        h = nv.nvmlDeviceGetHandleByIndex(self.nvml_index)
        self.nvml_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.nvml_stop:
            try:
                self.nvml_rows.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), int(reasons_fn(h))))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        self.nvml_rows, self.nvml_stop, self.nvml_thread, self.nvml_max = [], False, None, None
        try:
            import pynvml as nv
            import torch
            nv.nvmlInit()
            # NVML enumerates physical devices: map the CUDA ordinal through its PCI bus id
            pr = torch.cuda.get_device_properties(self.index)
            bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            self.nvml_index = nv.nvmlDeviceGetIndex(nv.nvmlDeviceGetHandleByPciBusId(bus.encode()))
            self.nvml_thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.nvml_thread.start()
            return
        except Exception:
            self.nvml_thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if getattr(self, "nvml_thread", None) is not None:
            self.nvml_stop = True
            self.nvml_thread.join(timeout=1.0)
            sm = sorted(r[0] for r in self.nvml_rows)
            reasons = sorted({name for r in self.nvml_rows for bit, name in self.NVML_REASONS.items() if r[1] & bit})
            return {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_min_mhz": float(sm[0]) if sm else None,
                    "sm_max_mhz": float(self.nvml_max) if self.nvml_max else None, "reasons": reasons, "samples": len(sm),
                    "source": "NVML, 5 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def bind_to_gpu_numa(local):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off BEFORE any pinned host buffer exists: pinned pages
    are then allocated on that node (first touch), so 8 ranks do not all stream their uploads out of node 0's memory."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        dev = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = Path("/sys/bus/pci/devices") / dev
        cpus = set()
        for part in (base / "local_cpulist").read_text().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        node = int((base / "numa_node").read_text().strip())
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"pci": dev, "numa_node": node, "cpus": len(cpus)}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


# ------------------------------------------------------------------------------------------
# CPU port (oracle) -- used ONLY as the reported cpu_baseline and as the --impl reference arm
# ------------------------------------------------------------------------------------------
def _calibrate_cpu_params(P, left, right, rho, thold):
    """Same one-scalar-per-level calibration as decnet_b200.synthetic.calibrate_mask_density, on the oracle's
    parameter dict: shift the detectors' last BN bias so the learned masks have density `rho`."""
    import math
    import torch
    from oracle import glue as og
    logit_t = math.log(thold / (1.0 - thold))
    pre = left["stage0"]
    for l in range(3):
        cur = left[f"stage{l + 1}"]
        with torch.no_grad():
            lg = og.detail_logits(cur, pre, P, f"detail_detection.{l}")
            q = torch.quantile(lg.flatten()[:: max(1, lg.numel() // 2_000_000)], 1.0 - rho)
        P[f"detail_detection.{l}.conv.1.bn.bias"] = P[f"detail_detection.{l}.conv.1.bn.bias"] + (logit_t - q)
        pre = cur


def _host_threads():
    """All host cores the process may use for the CPU arm, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1
    for its workers): must run before torch / libgomp read the environment."""
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))      # a parent bound to one NUMA node must not confine the CPU arm
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)
    os.environ["MKL_NUM_THREADS"] = str(cores)
    import torch
    torch.set_num_threads(cores)
    return cores


def cpu_port_pairs_per_s(workload, rho, min_seconds=10.0, max_pairs=64, warmup=1, with_features=False):
    """The oracle pipeline (torch-CPU dense/glue + C/OpenMP SpaMat/SpaVar) on all host cores, the same
    configuration as the CUDA arm (learned detectors calibrated to `rho`), one pair per call, repeated
    until `min_seconds` of CPU work.  with_features: every call also runs the CPU restatement of the feature extractor on
    both views (the work our `e2e` leg does on the device).  Returns (pairs/s, cores, seconds, pairs)."""
    cores = _host_threads()
    import torch
    from decnet_b200.params import make_featext_state, make_features, make_hotpath_state
    from decnet_b200.synthetic import WORKLOADS
    from oracle import pipeline as opipe
    H, W, max_disp, skip = WORKLOADS[workload]
    P = make_hotpath_state(17)
    left, right = make_features(1, H, W, seed=17)
    _calibrate_cpu_params(P, left, right, rho, 0.9)
    if with_features:
        from oracle import features as ofe
        fsd = make_featext_state(17)
        g = torch.Generator().manual_seed(3)
        imgs = [torch.randn(1, 3, H, W, generator=g) for _ in range(2)]

    def one_pair():
        with torch.no_grad():
            if with_features:
                fl, fr = ofe.feature_pyramid(imgs[0], fsd), ofe.feature_pyramid(imgs[1], fsd)
                opipe.forward(P, fl, fr, max_disp, use_detail=True, thold=0.9, skip_stage_id=skip)
            else:
                opipe.forward(P, left, right, max_disp, use_detail=True, thold=0.9, skip_stage_id=skip)
    for _ in range(warmup):
        one_pair()
    n, t0 = 0, time.perf_counter()
    while True:
        one_pair()
        n += 1
        el = time.perf_counter() - t0
        if el >= min_seconds or n >= max_pairs:
            break
    return n / el, cores, el, n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # K steps, each a bounded sample (pairs for ~1.5 s of host time, at most the arm's batch)
    v1, cores, el1, n1 = cpu_port_pairs_per_s(args.workload, args.rho, min_seconds=1.5, max_pairs=args.batch,
                                              warmup=max(1, min(args.warmup, 2)))
    steps = max(1, args.steps)
    tot_pairs, tot_s = n1, el1
    for _ in range(steps - 1):
        v, _, el, n = cpu_port_pairs_per_s(args.workload, args.rho, min_seconds=1.5, max_pairs=args.batch, warmup=0)
        tot_pairs += n; tot_s += el
    v = tot_pairs / tot_s
    vf, _, elf, nf = cpu_port_pairs_per_s(args.workload, args.rho, min_seconds=4.0, max_pairs=args.batch, warmup=1, with_features=True)
    sample = (f"{steps} steps x {n1} pair(s) of the {args.workload} workload (learned detectors calibrated to rho={args.rho}), "
              f"torch-CPU dense/glue + C/OpenMP SpaMat/SpaVar oracle, {tot_s:.1f} s")
    line = {"impl": "reference", "metric": metric_name(args.workload), "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": max(1, min(args.warmup, 2)), "ms_per_step": tot_s / steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload} {n1} pair(s)/step on the host cores; the reference's own ops for this "
                                   "path are CUDA-only, so its CPU execution is the oracle port (oracle/)",
                       "max_disp": 216},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "from_images": {"value": vf, "unit": UNIT, "what": "the same port with the CPU restatement of the feature extractor on "
                            f"both views in front (the work of our arm's e2e leg), {nf} pair(s) in {elf:.1f} s"},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
class Env:
    """Rank / device / timing helpers shared by the legs."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py (our arm) needs a CUDA device: there is no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.numa = bind_to_gpu_numa(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world > 1:
            t = self.torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed(self, fn, steps):
        """`steps` calls of fn between barrier + synchronize on both sides, CUDA events on the launching stream, MAX over ranks.
        What the last call returned is kept in self.last."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = None
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        self.barrier()
        self.last = out
        return self.max_over_ranks(e0.elapsed_time(e1))


def capture(torch, fn):
    """fn() eagerly once on a side stream, then captured; returns (graph, static output of fn)."""
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
        with torch.cuda.graph(graph, stream=side):
            out = fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    return graph, out


def pipelined_e2e(env, sets, upload_one, read_back, nsteps):
    """Software-pipelined end-to-end loop over two buffer sets: while the graph of step i runs on set i % 2, the copy
    stream uploads the pinned host inputs of step i+1 into the other set; every step does its full host->device upload and
    its device->host read of the result.  Returns ms (device clock, max over ranks) for `nsteps` steps."""
    torch = env.torch
    copy_stream, main = torch.cuda.Stream(), torch.cuda.current_stream()

    def upload(buf, after):
        with torch.cuda.stream(copy_stream):
            if after is not None:
                copy_stream.wait_event(after)           # the set's previous graph replay has finished
            upload_one(sets[buf])
            ev = torch.cuda.Event(); ev.record(copy_stream)
        return ev

    def run(n):
        computed = [None, None]
        copied = upload(0, None)
        for i in range(n):
            buf = i & 1
            main.wait_event(copied)
            sets[buf]["graph"].replay()
            read_back(sets[buf])
            ev = torch.cuda.Event(); ev.record(main); computed[buf] = ev
            if i + 1 < n:
                copied = upload(1 - buf, computed[1 - buf])
        main.synchronize()

    run(3)
    env.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(nsteps)
    e1.record()
    env.barrier()
    return env.max_over_ranks(e0.elapsed_time(e1))


def leg_from_images(args, env, info, precision):
    """demo.py's device work from the decoded images on (demo.py:144-198): uint8 RGB pairs -> pad / scale / normalise ->
    feature extractor (both views) -> hot path -> 16-bit disparity image, one CUDA graph; device-timed and end to end."""
    torch = env.torch
    from decnet_b200 import ops
    from decnet_b200.features import FeatExtNetChannelPlus, extract_pair
    from decnet_b200.model import DecompMatching
    from decnet_b200.params import make_featext_state, make_hotpath_state
    from decnet_b200.synthetic import calibrate_mask_density
    dev = env.dev
    B, H, W = args.batch, info["H"], info["W"]
    oh, ow = {"sceneflow": (540, 960), "kitti": (376, 1248)}.get(args.workload, (H, W))     # unpadded size (demo.py pads top/left)
    fe = FeatExtNetChannelPlus(8, precision=precision)
    fe.load_state_dict(make_featext_state(17))
    fe = fe.to(dev)
    model = DecompMatching(max_disp=info["max_disp"], skip_stage_id=info["skip_stage_id"], use_detail=True, thold=0.9,
                           precision=precision)
    model.load_state_dict(make_hotpath_state(17))
    model = model.to(dev)
    model.overlap = not args.no_overlap
    g = torch.Generator(device=dev).manual_seed(99 + env.rank)
    sets = [{"l": torch.randint(0, 256, (B, oh, ow, 3), device=dev, generator=g, dtype=torch.uint8),
             "r": torch.randint(0, 256, (B, oh, ow, 3), device=dev, generator=g, dtype=torch.uint8)} for _ in range(2)]
    prep = lambda u8: ops.image_prepare_u8(u8, want01=False)[1]
    dens = calibrate_mask_density(model, fe(prep(sets[0]["l"])), fe(prep(sets[0]["r"])), args.rho)

    def step_eager(st):
        if args.no_overlap:
            fl, fr = fe(prep(st["l"])), fe(prep(st["r"]))
        else:                                            # right view on a forked second stream
            fl, fr = extract_pair(fe, st["l"], st["r"], prepare=prep)
        return ops.disp_to_u16(model(fl, fr)[0], oh, ow)

    for st in sets:
        st["graph"], st["out"] = capture(torch, lambda st=st: step_eager(st))
    for _ in range(3):
        sets[0]["graph"].replay()
    ms = env.timed(lambda: sets[0]["graph"].replay(), args.steps)
    host = {k: sets[0][k].cpu().pin_memory() for k in ("l", "r")}
    host_out = torch.empty((B, oh, ow), dtype=torch.uint16).pin_memory()

    def upload_one(st):
        for k in ("l", "r"):
            st[k].copy_(host[k], non_blocking=True)
    n = max(4, args.steps)
    ms_e2e = pipelined_e2e(env, sets, upload_one, lambda st: host_out.copy_(st["out"], non_blocking=True), n)
    pairs = env.world * B
    return {"what": "uint8 RGB pairs (pinned host) -> device -> pad/scale/normalise -> feature extractor on both views "
                    "(FeatExtNetChannelPlus drop-in) -> hot path -> uint16 disparity image (x256, cropped) -> pinned host; "
                    "one CUDA graph per buffer set, uploads double-buffered on a copy stream",
            "precision": precision, "value": pairs * args.steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / args.steps,
            "e2e": {"value": pairs * n / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / n,
                    "h2d_bytes_per_step": 2 * B * 3 * oh * ow, "d2h_bytes_per_step": B * oh * ow * 2},
            "left_mask_density": [round(d, 4) for d in dens]}


def leg_sparse_roofline(args, env, left, right, info, pk, extras):
    """Roofline of the dominant sparse kernel (fused SpaMat+SpaVar), measured live with CUDA events on the launching
    stream; inputs (370 MB at B=8) exceed the 126 MB L2.  Also: the three-level aggregate, a density sweep, and the
    reference's own kernels (oracle/_ref: SM_kernel.cu / SV_kernel.cu recompiled for sm_100a) on the same inputs."""
    torch = env.torch
    from decnet_b200 import ops
    dev = env.dev
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def level_inputs(s, rho):
        Lf, Rf = left[f"stage{s}"], right[f"stage{s}"]
        Bc, Cc, Hc, Wc = Lf.shape
        g = torch.Generator(device=dev).manual_seed(5 + s)
        pl = torch.rand(Bc, Hc, Wc, device=dev, generator=g)
        pr = torch.rand(Bc, Hc, Wc, device=dev, generator=g)
        ml, mr = ops.mask_threshold(pl, pr, 1.0 - rho)
        return Lf, Rf, ml, mr, info["max_disp"] // 3 ** (3 - s), 4.0 * Bc * Hc * Wc * (2 * Cc + 2 + 4)

    def time_us(fn, n=20, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / n

    top = 3 if info["skip_stage_id"] > 3 else 2
    Lf, Rf, ml, mr, Dc, alg = level_inputs(top, args.rho)
    t_us = time_us(lambda: ops.spamat_spavar_forward(Lf, Rf, ml, mr, Dc))
    ach = alg / (t_us * 1e-6) / 1e9
    roof = {"bound": "hbm", "kernel": "sparse_row_gather_kernel<FUSED> (SpaMat+SpaVar, finest level)",
            "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
            "traffic": None, "traffic_source": "profiles/traffic.json (one ncu --set full capture, not measured in this run)",
            "peak_source": pk["source"] + " (burst copy)", "algorithmic_bytes": alg,
            "us_per_launch": t_us, "mask_density": args.rho}
    tr = ROOT / "profiles" / "traffic.json"
    traffic = {}
    if tr.exists():
        try:
            traffic = json.loads(tr.read_text())
            roof["traffic"] = traffic.get("sparse_row_gather_kernel_bytes_per_launch")
        except Exception:
            pass
    # all levels of the step: what the model launches (ONE kernel over the rows of every level, finest first: the aggregate
    # the 60 % target is about), and each level as a launch of its own beside it
    lv, tot_alg, per = [], 0.0, {}
    for s in range(1, top + 1):
        a = level_inputs(s, args.rho)
        us = time_us(lambda a=a: ops.spamat_spavar_forward(*a[:5]), n=20)
        per[f"1/{3 ** (3 - s)}"] = {"us_alone": round(us, 2), "frac_alone": round(a[5] / (us * 1e-6) / 1e9 / pk["hbm_gbs"], 4)}
        lv.append(a[:5]); tot_alg += a[5]
    tot_us = time_us(lambda: ops.spamat_spavar_forward_levels(lv[::-1]), n=20)
    roof["all_levels"] = {"kernel": "sparse_row_gather_multi_kernel<FUSED>: the rows of all levels in one launch (the product path)",
                          "algorithmic_bytes": tot_alg, "us": round(tot_us, 2),
                          "frac": round(tot_alg / (tot_us * 1e-6) / 1e9 / pk["hbm_gbs"], 4),
                          "us_as_separate_launches": round(sum(v["us_alone"] for v in per.values()), 2), "per_level": per,
                          # DRAM bytes of one launch at the SceneFlow shapes (same ncu capture as `traffic`); null elsewhere
                          "traffic": traffic.get("sparse_row_gather_multi_kernel_bytes_per_launch") if args.workload == "sceneflow" else None}
    if extras:
        sweep = {}
        g = torch.Generator(device=dev).manual_seed(5 + top)
        pl = torch.rand(ml.shape, device=dev, generator=g)
        pr = torch.rand(ml.shape, device=dev, generator=g)
        for rho_s in (0.01, 0.03, args.rho, 0.3):
            mls, mrs = ops.mask_threshold(pl, pr, 1.0 - rho_s)
            us = time_us(lambda: ops.spamat_spavar_forward(Lf, Rf, mls, mrs, Dc), n=10, warm=2)
            sweep[str(rho_s)] = {"gather_us": round(us, 2), "gather_frac": round(alg / (us * 1e-6) / 1e9 / pk["hbm_gbs"], 4)}
        roof["density_sweep"] = sweep
        # the survey's stated bar for a9 / a10: the reference's own kernels recompiled for sm_100a, same inputs, same box
        try:
            from oracle import ref_cuda
            if ref_cuda.available():
                def ref_both():
                    o, _, _ = ref_cuda.spamat_forward(Lf, Rf, ml, mr, Dc, sync=False)
                    ref_cuda.spavar_forward(Lf, Rf, ml, mr, o, Dc, sync=False)
                torch.cuda.synchronize()
                with torch.cuda.stream(torch.cuda.default_stream()):     # the reference launches on the legacy default stream
                    us = time_us(ref_both, n=5, warm=1)
                roof["reference_kernels_us"] = round(us, 1)
                roof["reference_kernels"] = ("SM_kernel.cu + SV_kernel.cu (unmodified, oracle/_ref) SpaMat then SpaVar on the same "
                                             f"inputs: {us / t_us:.0f}x our fused launch")
        except Exception as e:
            roof["reference_kernels_us"] = f"{type(e).__name__}: {e}"
    return roof


def leg_conv2d_roofline(args, env, left, pk):
    """The thin 3x3 Conv2d layers (conv2d_tcgen05_kernel): the 8->8 layer at the finest level in the step's precision;
    algorithmic bytes = input + output once."""
    torch = env.torch
    from decnet_b200 import ops
    try:
        x = left["stage3"]
        Bq, Cq, Hq, Wq = x.shape
        split = args.precision == "fp32"
        if not ops.conv2d_tf32_supported(Cq, 8, Hq, Wq, 1, split):
            return None
        gq = torch.Generator(device=env.dev).manual_seed(7)
        wq = torch.randn(8, Cq, 3, 3, device=env.dev, generator=gq) * 0.1
        wpk, bpk = ops.pack_conv2d_tf32_nchw_weights(wq, torch.zeros(8, device=env.dev), split=split)
        for _ in range(3):
            ops.conv2d_tf32_nchw_cat([x], wpk, bpk, 8, 1, True, split=split)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            ops.conv2d_tf32_nchw_cat([x], wpk, bpk, 8, 1, True, split=split)
        e1.record(); torch.cuda.synchronize()
        t_c = e0.elapsed_time(e1) * 1e-3 / 20
        alg_c = 4.0 * Bq * Hq * Wq * (Cq + 8)
        out = {"bound": "hbm", "kernel": f"conv2d_tcgen05_kernel (3x3, 8->8 channels, finest level, {'hi/lo split, fp32-class' if split else 'TF32'})",
               "achieved": alg_c / t_c / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": alg_c / t_c / 1e9 / pk["hbm_gbs"],
               "traffic": None, "algorithmic_bytes": alg_c, "us_per_launch": t_c * 1e6}
        tr = ROOT / "profiles" / "traffic.json"
        if tr.exists():
            out["traffic"] = json.loads(tr.read_text()).get("conv2d_tcgen05_kernel_bytes_per_launch")
        return out
    except Exception as e:
        return {"bound": "hbm", "note": f"{type(e).__name__}: {e}"}


def leg_gpu_reference(args, env, left, right, info, state):
    """BASELINE.md B4: the UNMODIFIED reference model (staged under baseline/_ref) on this GPU -- its PyTorch / cuDNN layers
    eager (TF32 allowed: PyTorch's default, what demo.py runs) and its own CUDA kernels recompiled for sm_100a (oracle/_ref)
    -- fed the same feature pyramids, timed like demo.py:185-189 (synchronize, wall clock, synchronize)."""
    torch = env.torch
    from oracle import ref_cuda, ref_loader
    if not (ref_loader.available() and ref_cuda.available()):
        return {"unavailable": "reference tree (baseline/_ref) or its compiled kernels (oracle/_ref) not staged"}
    import contextlib
    import io

    class _RefSpaMat:
        @staticmethod
        def sparse_matching_cuda_forward(L, R, ml, mr, out, ssim, mx, D):
            torch.cuda.current_stream().synchronize()            # the reference launches on the legacy default stream
            ref_cuda._lib("spamat").ref_spamat_forward(*map(ref_cuda._p, (L, R, ml, mr, out, ssim, mx)), *L.shape, int(D))
            return 1

    class _RefSpaVar:
        @staticmethod
        def sparse_var_cuda_forward(L, R, ml, mr, disp, out, ssim, mx, D):
            torch.cuda.current_stream().synchronize()
            ref_cuda._lib("spavar").ref_spavar_forward(*map(ref_cuda._p, (L, R, ml, mr, disp.contiguous(), out, ssim, mx)), *L.shape, int(D))
            return 1
    ref_loader.install(_RefSpaMat, _RefSpaVar)
    sys.modules["modules.SparseMatching.functions.SpaMat"].SpaMat = _RefSpaMat
    sys.modules["modules.SparseVar.functions.SpaVar"].SpaVar = _RefSpaVar
    with contextlib.redirect_stdout(io.StringIO()):
        model = ref_loader.build_reference_model(max_disp=info["max_disp"], use_detail=True, thold=0.9,
                                                 skip_stage_id=info["skip_stage_id"])
    missing, unexpected = model.load_state_dict(state, strict=False)          # our arm's weights, detectors calibrated
    assert not unexpected and all(k.startswith("feature_extractor.") for k in missing), (missing[:3], unexpected[:3])
    model = model.to(env.dev).eval()
    feats = iter(())

    class _Given(torch.nn.Module):                               # "feature maps given": the extractor is not on this path
        def forward(self, x):
            return next(feats)
    model.feature_extractor = _Given()
    dummy = [torch.zeros(1, device=env.dev)] * 3
    img = torch.zeros(1, device=env.dev)

    def once():
        nonlocal feats
        feats = iter((left, right))
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            return model(img, img, None, dummy, dummy, is_check=False, is_eval=False)[0]
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        for _ in range(2):
            once()
        ts = []
        for _ in range(5):
            torch.cuda.synchronize(); t0 = time.time()
            once()
            torch.cuda.synchronize(); ts.append(time.time() - t0)
    finally:
        torch.backends.cudnn.benchmark = old
    ts.sort()
    B = left["stage0"].shape[0]
    return {"what": "unmodified reference model (baseline/_ref: PyTorch/cuDNN eager, TF32 allowed as in demo.py; its own "
                    "SpaMat/SpaVar kernels recompiled for sm_100a), feature maps given, timed as demo.py:185-189",
            "value": B / ts[len(ts) // 2], "unit": UNIT, "ms_per_step": ts[len(ts) // 2] * 1e3, "batch": B,
            "note": "same weights as our arm (detectors calibrated to the same mask density)"}


def leg_bands(args, env):
    """BASELINE.json configs[3]: ONE Middlebury pair (2025x2916, D = 783, finest level skipped) split into row bands over
    the ranks.  Halo rows of the 3-D aggregation and the per-level disparity bands are stored straight into the neighbours'
    / every rank's peer memory over NVLink with device-side signals (bands.PeerTransport), so the whole banded step is one
    CUDA graph per rank."""
    torch = env.torch
    from decnet_b200 import bands as _bands
    from decnet_b200.synthetic import build_workload
    model, left, right, info = build_workload("middlebury", 1, seed=17, device=env.dev, rho=args.rho, precision=args.precision)
    h0 = left["stage0"].shape[2]
    transport = _bands.PeerTransport(h0) if env.world > 1 else _bands.LocalTransport(1)
    me = env.rank if env.world > 1 else 0

    def eager():
        return _bands.forward_bands(model, left, right, transport)[me]
    for _ in range(2):
        eager()
    env.barrier()
    launch = "eager"
    step = eager
    if env.world > 1 and not args.no_graph:
        graph, out = capture(torch, eager)
        env.barrier()
        step, launch = graph.replay, "one CUDA graph per rank"
    for _ in range(3):
        step()
    n = 10
    ms = env.timed(step, n)
    model.overlap = not args.no_overlap
    single = None
    if env.rank == 0:                                            # the same pair on one GPU without bands, for the speed-up
        g1, _ = capture(torch, lambda: model(left, right)[0])
        for _ in range(3):
            g1.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            g1.replay()
        e1.record(); torch.cuda.synchronize()
        single = e0.elapsed_time(e1) / n
    env.barrier()
    return {"workload": f"middlebury {info['H']}x{info['W']} padded, max_disp {info['max_disp']}, ONE pair, skip_stage_id 3",
            "ranks": env.world, "ms_per_pair": ms / n, "single_gpu_ms_per_pair": single, "launch": launch,
            "speedup_vs_single_gpu": (single / (ms / n)) if single else None,
            "exchange": "NVLink peer-memory stores: per-layer halo rows of the 3-D aggregation into the neighbours' buffers, each "
                        "level's disparity band into every rank's map; device-side signals, no host synchronisation"}


def run_ours(args):
    env = Env()
    torch, dist = env.torch, env.dist
    from decnet_b200 import _lib
    from decnet_b200.synthetic import build_workload
    world, rank, dev = env.world, env.rank, env.dev
    torch.backends.cudnn.benchmark = True          # only the feature extractor's library layers (e2e leg) use cuDNN
    lib = _lib.lib()
    extras = not args.no_extras

    bands_mode = args.mode == "bands"
    model, left, right, info = build_workload(args.workload, args.batch, seed=17 + (0 if bands_mode else rank),
                                              device=dev, rho=args.rho, precision=args.precision)
    model.overlap = not args.no_overlap
    B = args.batch
    if bands_mode:
        from decnet_b200 import bands as _bands
        transport = _bands.PeerTransport(left["stage0"].shape[2]) if world > 1 else _bands.LocalTransport(1)

        def eager_step():
            return _bands.forward_bands(model, left, right, transport)[rank if world > 1 else 0]
    else:
        def eager_step():
            return model(left, right)[0]

    for _ in range(max(args.warmup, 3)):
        eager_step()
    torch.cuda.synchronize()
    lib.decnet_reset_launch_count()
    eager_step(); torch.cuda.synchronize()
    launches_per_step = int(lib.decnet_launch_count())

    # The step is ~110 launches of our kernels: captured once into a CUDA graph (static input / output buffers) and
    # replayed, so the device is not waiting for the Python launch path.
    use_graph = not args.no_graph and not bands_mode
    sets = None
    if use_graph:
        left2 = {k: v.clone() for k, v in left.items()}
        right2 = {k: v.clone() for k, v in right.items()}
        sets = [{"l": left, "r": right}, {"l": left2, "r": right2}]
        for st in sets:
            st["graph"], st["out"] = capture(torch, lambda st=st: model(st["l"], st["r"])[0])
        ref_out = eager_step()
        sets[0]["graph"].replay()
        assert torch.allclose(sets[0]["out"], ref_out, atol=1e-4, rtol=1e-4), "graph replay differs from eager execution"

        def step():
            sets[0]["graph"].replay()
            return sets[0]["out"]
        for _ in range(3):
            step()
        torch.cuda.synchronize()
    else:
        step = eager_step

    sampler = ClockSampler(env.local)
    if rank == 0:
        sampler.start()
    prof_range = os.environ.get("DECNET_PROFILE_RANGE") == "1"   # ncu --profile-from-start off
    if prof_range:
        torch.cuda.profiler.start()
    ms = env.timed(step, args.steps)
    if prof_range:
        torch.cuda.profiler.stop()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"disparity": env.last})     # before any later leg replays the graph again
    n_units = B if bands_mode else world * B          # bands: all ranks work on the SAME B pairs
    value = n_units * args.steps / (ms * 1e-3)

    # ---- the hot path alone behind host buffers: pinned fp32 feature pyramids -> device every step
    host_l = {k: v.cpu().pin_memory() for k, v in left.items()}
    host_r = {k: v.cpu().pin_memory() for k, v in right.items()}
    host_out = torch.empty((B, info["H"], info["W"]), dtype=torch.float32).pin_memory()
    h2d = sum(v.numel() * 4 for v in host_l.values()) * 2
    if use_graph:
        def upload_one(st):
            for k in host_l:
                st["l"][k].copy_(host_l[k], non_blocking=True)
                st["r"][k].copy_(host_r[k], non_blocking=True)
        pyr_steps = max(4, args.steps // (1 if world == 1 else 2))
        ms_pyr = pipelined_e2e(env, sets, upload_one, lambda st: host_out.copy_(st["out"], non_blocking=True), pyr_steps)
    else:
        dev_l = {k: torch.empty_like(v) for k, v in left.items()}
        dev_r = {k: torch.empty_like(v) for k, v in right.items()}

        def step_e2e():
            for k in host_l:
                dev_l[k].copy_(host_l[k], non_blocking=True)
                dev_r[k].copy_(host_r[k], non_blocking=True)
            out = (_bands.forward_bands(model, dev_l, dev_r, transport)[rank if world > 1 else 0] if bands_mode
                   else model(dev_l, dev_r)[0])
            host_out.copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for _ in range(2):
            step_e2e()
        pyr_steps = max(3, args.steps // 2)
        ms_pyr = env.timed(step_e2e, pyr_steps)
    e2e_pyr = {"value": n_units * pyr_steps / (ms_pyr * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": host_out.numel() * 4, "ms_per_step": ms_pyr / pyr_steps,
               "note": "pinned host fp32 feature pyramids (the reference's interface to this path) -> device on a copy stream, "
                       "double-buffered against the previous step's compute; hot path (CUDA graph); disparity -> pinned host; every "
                       "step.  Bound by the host link: " + f"{h2d / 1e6:.0f} MB up per step"}

    # ---- end to end at demo.py's boundary, every rank: images in, 16-bit disparity out
    from_images = None
    if use_graph and not args.no_from_images:
        try:
            from_images = leg_from_images(args, env, info, args.precision)
        except Exception as e:      # every rank fails or none does (same code, same shapes): no collective is left hanging
            from_images = {"error": f"{type(e).__name__}: {e}"}
    if from_images and "e2e" in from_images:
        e2e = dict(from_images["e2e"])
        e2e["note"] = ("demo.py's boundary: " + from_images["what"] + ".  More work than the reference arm's step (it includes the "
                       "feature extractor); e2e_pyramids is the hot path alone behind host buffers")
    else:
        e2e = dict(e2e_pyr)

    # ---- the same step in the other arithmetic mode (secondary)
    tf32 = None
    if extras and use_graph and args.precision == "fp32":
        try:
            model.set_precision("tf32")
            g2, _ = capture(torch, lambda: model(left, right)[0])
            for _ in range(3):
                g2.replay()
            ms_t = env.timed(lambda: g2.replay(), args.steps)
            tf32 = {"value": n_units * args.steps / (ms_t * 1e-3), "unit": UNIT, "ms_per_step": ms_t / args.steps,
                    "what": "the same hot-path step with the 2-D tensor-core convs in plain TF32 (one MMA per tap): the precision "
                            "class cuDNN gives the reference on a GPU; NOT the parity-gated mode"}
            del g2
        finally:
            model.set_precision(args.precision)

    roof = roof_tensor = roof_conv2d = gpu_ref = None
    if rank == 0:
        pk = peaks()
        roof = leg_sparse_roofline(args, env, left, right, info, pk, extras)
        roof_conv2d = leg_conv2d_roofline(args, env, left, pk)
        try:
            from decnet_b200 import conv3d as c3
            roof_tensor = c3.measure_roofline(model, left["stage0"], right["stage0"], info["max_disp"] // 27, pk)
        except Exception as e:
            roof_tensor = {"bound": "tensor", "note": f"{type(e).__name__}: {e}"}
        if extras and world == 1 and not bands_mode:
            try:
                gpu_ref = leg_gpu_reference(args, env, left, right, info, {k: v.detach().clone() for k, v in model.state_dict().items()})
            except Exception as e:
                gpu_ref = {"error": f"{type(e).__name__}: {e}"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # a fresh process: this one is bound to its GPU's NUMA node and its OpenMP pool was created under that mask
        try:
            r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "cpu-leg", "--workload", args.workload,
                                "--rho", str(args.rho), "--cpu-seconds", str(args.cpu_seconds)], capture_output=True, text=True,
                               timeout=600)
            cpu = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            cpu = {"error": f"{type(e).__name__}: {e}"}

    line = bands = None
    if rank == 0:
        conv_dtype = ("hi/lo operand split (TF32 hi*hi + fp16 corrections, fp32-class) in / f32 acc" if args.precision == "fp32"
                      else "tf32 in / f32 acc")
        line = {"metric": metric_name(args.workload), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong" if bands_mode else "weak", "vs_baseline": None,
                "dtype": f"f32 (sparse / glue kernels); {conv_dtype} (2-D conv stacks, tcgen05); bf16 in / f32 acc (3-D aggregation, tcgen05)",
                "data": "synthetic",
                "config": {"workload": f"{args.workload} {info['H']}x{info['W']} padded, batch {B}/GPU, max_disp {info['max_disp']}, "
                                       "full decomposition pyramid" + (" (BASELINE.json configs[1])" if args.workload == "sceneflow" and B == 8 else ""),
                           "levels": " | ".join(f"1/{27 // 3 ** i} C{c} {info['H'] * 3 ** i // 27}x{info['W'] * 3 ** i // 27} "
                                                f"D{info['max_disp'] * 3 ** i // 27}" for i, c in enumerate((216, 72, 24, 8))),
                           "left_mask_density": info["left_mask_density"], "precision": args.precision,
                           "launch": "CUDA graph replay of the whole step" if use_graph else "eager launches",
                           "streams": "masks + sparse ops on a forked second stream (two graph branches)" if not args.no_overlap else "one stream",
                           "l2": "inputs (400 MB of feature pyramids per step) exceed the 126 MB L2; no flush",
                           "host_numa": env.numa,
                           "parallelism": (f"row bands of one batch over {world} rank(s): per-layer halo rows and per-level disparity "
                                           "bands stored into peer memory over NVLink") if bands_mode
                           else f"by stereo pair, {world} rank(s), no collective"},
                "e2e": e2e, "e2e_pyramids": e2e_pyr,
                "gpu_launches": launches_per_step * args.steps,
                "gpu_launches_per_step": launches_per_step,
                "clocks": clocks, "roofline": roof, "roofline_tensor": roof_tensor, "roofline_conv2d": roof_conv2d,
                "cpu_baseline": cpu, "from_images": from_images, "tf32": tf32, "gpu_reference": gpu_ref, "bands": None}

    # ---- the last leg talks to the other ranks through peer memory: a watchdog guarantees that the line above is printed
    # (without the `bands` object) and that every rank exits even if a peer fails inside it
    if extras and world > 1 and not bands_mode:
        def bail():
            if rank == 0:
                line["bands"] = {"error": "the row-band leg did not finish within 240 s"}
                print(json.dumps(line), flush=True)
            os._exit(0)
        dog = threading.Timer(240.0, bail)
        dog.daemon = True
        dog.start()
        try:
            bands = leg_bands(args, env)
        except Exception as e:
            bands = {"error": f"{type(e).__name__}: {e}"}
        dog.cancel()
        if rank == 0:
            line["bands"] = bands
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        if isinstance(bands, dict) and "error" in bands:
            os._exit(0)                      # a rank failed inside the peer-memory leg: the group cannot be torn down cleanly
        try:
            dist.destroy_process_group()
        except Exception:
            pass


def run_cpu_leg(args):
    """The `cpu_baseline` object of our arm's line (the oracle port on the host cores, bounded sample), as its own process."""
    v, cores, sec, npairs = cpu_port_pairs_per_s(args.workload, args.rho, min_seconds=args.cpu_seconds)
    print(json.dumps({"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                      "sample": f"{npairs} pairs of the same workload (one pair per call, learned detectors calibrated to "
                                f"rho={args.rho}), torch-CPU dense/glue + C/OpenMP SpaMat/SpaVar oracle, {sec:.1f} s"}), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "cpu-leg":
        run_cpu_leg(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
