#!/usr/bin/env python
"""bench.py -- stereo pairs/s of the hot path (StereoJoin -> CBCA -> SGM -> post) on N B200s.

Usage: `python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]`, one JSON
line on stdout from rank 0.  A "step" = one stereo pair (BASELINE.json config 3: 370x1226, d=228,
C=64 features, kitti-slow post-processing with CBCA x4 + 4-direction SGM) through the fused native
pipeline, one pair per GPU per step (pairs shard over GPUs with no collective: weak scaling).

  value      whole-job pairs/s with inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same through the host-buffer C-ABI call (H2D of features+images and D2H of disp inside)
  roofline   the dominant kernel of the step, timed alone with CUDA events on its stream
  cpu_baseline  the CPU oracle (oracle/, a port of the reference) on a bounded sample, rank 0, N=1

`--impl reference` times the reference's OWN implementation of the path: adcensus.cu compiled
unmodified (oracle/_ref/libadcensus_ref.so) and driven in main.lua's order.  The reference has no
CPU path (every op takes torch.CudaTensor), so this arm also runs on the B200 (BASELINE.json
north_star says so); rank 0 only.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json config 3: the configuration the metric is quoted on (default)
    "k228": dict(name="kitti_accurate_370x1226_d228_cbca4_sgm4", H=370, W=1226, D=228, C=64,
                 preset=("kitti", "accurate_cbca4"),
                 desc="kitti slow post-processing, cbca_i1=2 cbca_i2=2, sgm2 (4 directions), LR check, subpixel, "
                      "median5, bilateral"),
    # BASELINE.json config 2 (reported in profiles/, not the driver's bench line)
    "k70": dict(name="kitti_fast_370x1226_d70", H=370, W=1226, D=70, C=64, preset=("kitti", "fast"),
                desc="kitti fast preset (no CBCA), sgm2 (4 directions), LR check, subpixel, median5, bilateral"),
}
WORKLOAD = WORKLOADS["k228"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--stages", action="store_true", help="also print a per-stage timing table to stderr")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--small", action="store_true", help="tiny workload (debug only; not a valid bench line)")
    ap.add_argument("--workload", default="k228", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the disparity maps of the last timed step as DIR/<name>.npy (rank 0); "
                         "the inputs depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(dirname, arrays):
    """`arrays`: name -> tensor, written as float32 .npy files"""
    import numpy as np

    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), t.detach().float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier_sync(world):
    import torch
    import torch.distributed as dist

    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    import torch
    import torch.distributed as dist

    if world == 1:
        return x
    t = torch.tensor([x], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_inputs(cfg, n_pairs, seed0):
    import numpy as np
    import torch

    from mccnn_b200 import synth

    pairs = []
    for i in range(n_pairs):
        p = synth.make_pair(cfg["H"], cfg["W"], cfg["C"], cfg["D"], seed=seed0 + i)
        pairs.append({k: torch.from_numpy(np.ascontiguousarray(p[k])).pin_memory() for k in ("featL", "featR", "imgL", "imgR")})
    return pairs


def algorithmic_bytes(cfg):
    """SURVEY.md 8(d): algorithmic bytes per launch of each kernel of the step"""
    H, W, D, C = cfg["H"], cfg["W"], cfg["D"], cfg["C"]
    V = 4 * D * H * W
    F = 4 * C * H * W
    valid = 4 * H * (D * W - D * (D - 1) // 2)
    return {
        "StereoJoin": 2 * F + 2 * valid,
        "cbca_fast": 2 * V + 32 * H * W,          # per iteration: read V + write V + both images' arms
        "cbca_exact": 2 * V + 32 * H * W,
        "sgm2": 11 * V,                           # documented 4-sweep design: 4 x (read in + RMW out) - 1 read of the zero accumulator
        "transpose_in": 2 * V,
        "transpose_out": 2 * V,
        "argmin": V + 4 * H * W,
    }


def make_config(cfg):
    """`config` of the JSON line: IDENTICAL keys and values in both arms (own, reference)"""
    return {"workload": cfg["name"], "H": cfg["H"], "W": cfg["W"], "D": cfg["D"], "C": cfg["C"], "preset": cfg.get("desc", ""),
            "pairs_per_gpu_per_step": 1, "parallelism": "pairs sharded over GPUs, one process per GPU, no collective",
            "l2": "per-step working set (0.23 GB features + >1.6 GB volumes) exceeds the 126 MB L2; single-kernel timings flush L2 "
                  "with a 256 MB write"}


def time_op(fn, iters, flush):
    """average CUDA-event duration (ms) of fn() on torch's current stream, L2 flushed before each"""
    import torch

    fn()            # untimed: lazy kernel load, pool growth
    evs = []
    for _ in range(iters):
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / len(evs)


def stage_table(cfg, opt, dev_in, iters=5):
    """per-kernel timings at the bench workload through the C ABI, each kernel alone on the stream, L2 flushed, on the
    data layouts the fused pipeline runs them on (pitched (D,H,ld) volumes)"""
    import torch

    from mccnn_b200 import adcensus

    H, W, D, C = cfg["H"], cfg["W"], cfg["D"], cfg["C"]
    ld = (W + 3) // 4 * 4
    dev = dev_in["featL"].device
    flushbuf = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    flush = lambda: flushbuf.fill_(1.0)
    lib = adcensus.lib()
    lib.mccnn_packed_arms_bytes.restype = ctypes.c_size_t
    lib.mccnn_packed_hv_bytes.restype = ctypes.c_size_t
    vp = lambda t_: ctypes.c_void_p(t_.data_ptr())
    fL, fR = dev_in["featL"][None], dev_in["featR"][None]
    iL, iR = dev_in["imgL"][None], dev_in["imgR"][None]
    st = adcensus._stream(fL)
    t = {}
    # StereoJoin: the operator on contiguous outputs (the pipeline launches the same kernel with the row pitch ld)
    vols = torch.full((2, D, H, W), float("nan"), device=dev)
    t["StereoJoin"] = time_op(lambda: adcensus.StereoJoin(fL, fR, vols[0:1], vols[1:2]), iters, flush)
    x0c = torch.empty((1, 4, H, W), device=dev); x1c = torch.empty((1, 4, H, W), device=dev)
    t["cross"] = time_op(lambda: adcensus.cross(iL, x0c, opt.L1, opt.tau1), iters, flush)
    adcensus.cross(iR, x1c, opt.L1, opt.tau1)
    maxarm = max(opt.L1, 2)
    # pitched copy of the left volume
    pin = torch.empty((D, H, ld), device=dev)
    pin[:, :, :W] = vols[0]
    pout = torch.empty_like(pin)
    if opt.cbca_i1 + opt.cbca_i2 > 0:
        hv = torch.empty(lib.mccnn_packed_hv_bytes(H, W), dtype=torch.uint8, device=dev)
        assert lib.mccnn_pack_arms_hv(vp(x0c), vp(x1c), vp(hv), H, W, st) == 0
        t["cbca_fast"] = time_op(lambda: lib.mccnn_cbca_fast_pitched_packed(vp(hv), vp(pin), vp(pout), D, H, W, ld, -1, maxarm, st), iters, flush)
        packed = torch.empty(lib.mccnn_packed_arms_bytes(H, W), dtype=torch.uint8, device=dev)
        assert lib.mccnn_pack_arms(vp(x0c), vp(x1c), vp(packed), H, W, st) == 0
        tmp = torch.empty((1, D, H, W), device=dev)
        t["cbca_exact"] = time_op(lambda: lib.mccnn_cbca_packed(vp(packed), vp(x0c), vp(x1c), vp(vols[0:1]), vp(tmp), D, H, W, -1, maxarm, st),
                                  iters, flush)
    volt = torch.empty((1, H, W, D), device=dev)
    t["transpose_in"] = time_op(lambda: lib.mccnn_transpose_dhw_pitched_to_hwd(vp(pin), vp(volt), D, H, W, ld, st), iters, flush)
    out = torch.zeros_like(volt)

    def sgm():
        out.zero_()
        adcensus.sgm2(iL, iR, volt, out, None, opt.pi1, opt.pi2, opt.tau_so, opt.alpha1, opt.sgm_q1, opt.sgm_q2, -1)

    t_zero = time_op(lambda: out.zero_(), iters, flush)
    t["sgm2"] = time_op(sgm, iters, flush) - t_zero
    t["transpose_out"] = time_op(lambda: lib.mccnn_transpose_hwd_to_dhw_pitched_div4(vp(out), vp(pout), D, H, W, ld, st), iters, flush)
    dmap = torch.empty((1, 1, H, W), device=dev)
    t["argmin"] = time_op(lambda: lib.mccnn_argmin_pitched(vp(pout), vp(dmap), D, H, W, ld, st), iters, flush)
    d = adcensus.argmin(vols[0:1])
    d1 = adcensus.argmin(vols[1:2])
    outl = torch.zeros_like(d)
    t["outlier_detection"] = time_op(lambda: adcensus.outlier_detection(d, d1, outl, D), iters, flush)
    t["interpolate_occlusion"] = time_op(lambda: adcensus.interpolate_occlusion(d, outl), iters, flush)
    t["interpolate_mismatch"] = time_op(lambda: adcensus.interpolate_mismatch(d, outl), iters, flush)
    t["subpixel"] = time_op(lambda: adcensus.subpixel_enchancement(d, vols[0:1], D), iters, flush)
    t["median2d"] = time_op(lambda: adcensus.median2d(d, 5), iters, flush)
    kern = adcensus.gaussian(opt.blur_sigma).to(dev)
    t["mean2d"] = time_op(lambda: adcensus.mean2d(d, kern, opt.blur_t), iters, flush)
    return t


def cpu_baseline(cfg, opt):
    """the CPU oracle (a port: the reference ships no CPU path) on a bounded row band"""
    import numpy as np

    from mccnn_b200 import synth
    from oracle import oracle as orc

    rows = min(cfg["H"], 96)
    p = synth.make_pair(rows, cfg["W"], cfg["C"], cfg["D"], seed=5)
    op = orc.Params(**opt.as_dict())
    orc.lib()
    t0 = time.perf_counter()
    orc.stereo_predict(p["featL"], p["featR"], p["imgL"], p["imgR"], cfg["D"], op)
    dt = time.perf_counter() - t0
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    frac = rows / cfg["H"]
    return {"value": frac / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": "rows 0..%d of one %dx%d d=%d pair (%.1f%% of a pair) in %.1f s, OpenMP oracle; scaled by rows" % (
                rows - 1, cfg["H"], cfg["W"], cfg["D"], 100 * frac, dt)}


def timed_steps(sp, dev_in, disp, K, warm, world, sample_clocks=None):
    """K timed steps (one pair per step) of the fused pipeline through its batch call (mccnn_pipeline_run_batch: the K pairs
    alternate between the pipeline's two lanes), barrier + synchronize on both sides; max over ranks (ms).  The last pair's
    disparity map lands in `disp`."""
    import torch

    tmp = [torch.empty_like(disp), torch.empty_like(disp)]

    def batch(n):
        pairs = [tuple(dev_in[i % 2][k] for k in ("featL", "featR", "imgL", "imgR")) for i in range(n)]
        outs = [disp if i == n - 1 else tmp[i & 1] for i in range(n)]
        sp.run_batch(pairs, outs)

    batch(max(warm, 2))
    barrier_sync(world)
    if sample_clocks is not None:
        sample_clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    batch(K)
    e1.record()
    barrier_sync(world)
    return max_over_ranks(e0.elapsed_time(e1), world)


def load_traffic(workload):
    """DRAM bytes per launch (dram__bytes_read + write) of the kernels of this workload from the committed ncu launch list
    of the same pipeline (profiles/r2_traffic_<workload>.json, written by tools/launch_summary.py --json)"""
    p = os.path.join(ROOT, "profiles", "r2_traffic_%s.json" % workload)
    if os.path.exists(p):
        try:
            return json.load(open(p)), os.path.relpath(p, ROOT)
        except Exception:
            pass
    return {}, None


def rowband_block(rank, world, local):
    """One stereo pair split by row bands over the N ranks (SURVEY.md 8e, BASELINE config 5 at N = 8, the bench pair
    otherwise): CUDA-event time (barrier on both sides, max over ranks), the single-GPU fused pipeline on the same inputs
    (rank 0) and the number of disparity-map pixels that differ from it.  Appended to the bench line at N >= 2 so that the
    driver's scaling run records it; never part of `value`."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from mccnn_b200 import pipeline, rowband, synth

    dev = torch.device("cuda", local)
    if world >= 8:
        H, W, D, C, preset, name = 2000, 3000, 400, 64, ("mb", "fast"), "middlebury_2000x3000_d400_mb_fast"
    else:
        H, W, D, C, preset, name = 370, 1226, 228, 64, ("kitti", "accurate_cbca4"), "kitti_accurate_370x1226_d228_cbca4_sgm4"
    res = {"workload": name, "n_gpus": world, "split": "row bands; halo rows before the CBCA blocks, vertical SGM passes as a "
           "wavefront over column chunks carrying the W x D line state (NCCL send/recv)"}
    try:
        opt = pipeline.make_params(*preset)
        g = torch.Generator(device=dev).manual_seed(7)
        featL = torch.nn.functional.normalize(torch.randn((C, H, W), device=dev, generator=g), dim=0)
        featR = torch.nn.functional.normalize(torch.randn((C, H, W), device=dev, generator=g), dim=0)
        img = synth.natural_image(np.random.default_rng(7), H, W + 16)
        st = lambda x: torch.from_numpy(((x - x.mean()) / x.std(ddof=1)).astype(np.float32)).to(dev)
        imgL, imgR = st(img[:, 16:]).contiguous(), st(img[:, :W]).contiguous()
        ops, comm = rowband.CudaOps(dev), rowband.Comm()
        out = rowband.stereo_predict_rowband(ops, featL, featR, imgL, imgR, D, opt, comm)
        times = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier_sync(world)
            e0.record()
            out = rowband.stereo_predict_rowband(ops, featL, featR, imgL, imgR, D, opt, comm)
            e1.record()
            barrier_sync(world)
            times.append(max_over_ranks(e0.elapsed_time(e1), world))
        res["ms"] = round(min(times), 3)
        if rank == 0:
            sp = pipeline.StereoPipeline(C, D, H, W, opt, device=local, cbca_mode="exact")   # the band driver runs the exact operators
            ref = sp.run(featL, featR, imgL, imgR)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ref = sp.run(featL, featR, imgL, imgR)
            e1.record()
            torch.cuda.synchronize()
            res["single_gpu_ms"] = round(e0.elapsed_time(e1), 3)
            res["speedup"] = round(res["single_gpu_ms"] / res["ms"], 3)
            res["efficiency"] = round(res["single_gpu_ms"] / res["ms"] / world, 3)
            bad = ~((out == ref) | (torch.isnan(out) & torch.isnan(ref)))
            res["mismatches_vs_single_gpu"] = int(bad.sum())
            sp.close()
    except Exception as e:  # the block must never take the bench line down
        res["error"] = "%s: %s" % (type(e).__name__, str(e)[:200])
    return res


def scorer_head_block(local, peaks_path=None):
    """The accurate architecture's scorer head (csrc/scorer_head.cu, SURVEY.md 8f-1) at the bench size: ms per volume pair
    and tensor-core TFLOP/s against the measured dense bf16 peak.  Reported beside the headline, never part of it."""
    import numpy as np
    import torch

    from mccnn_b200 import scorer_head

    dev = torch.device("cuda", local)
    fm, nh2, l2, H, W, D = 112, 384, 4, 370, 1226, 228
    g = torch.Generator(device=dev).manual_seed(0)
    fL = torch.relu(torch.randn((fm, H, W), device=dev, generator=g))
    fR = torch.relu(torch.randn((fm, H, W), device=dev, generator=g))
    rng = np.random.default_rng(0)
    layers, n_in = [], 2 * fm                                   # random-init net_te2 (no trained nets offline)
    for _ in range(l2):
        layers.append(((rng.standard_normal((nh2, n_in)) / np.sqrt(n_in)).astype(np.float32), (0.1 * rng.standard_normal(nh2)).astype(np.float32)))
        n_in = nh2
    layers.append(((rng.standard_normal((1, nh2)) / np.sqrt(nh2)).astype(np.float32), (0.1 * rng.standard_normal(1)).astype(np.float32)))
    head = scorer_head.ScorerHead(layers, device=local)
    rows = H * (D * W - D * (D - 1) // 2)
    flop_row = 2 * (2 * fm * nh2 + (l2 - 1) * nh2 * nh2 + nh2)
    peak = None
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["bf16_tflops_sustained"])
    except Exception:
        pass
    out = {"workload": "kitti slow net_te2 (fm 112, nh2 384, l2 4) at 370x1226 d=228, both volumes", "bound": "tensor"}
    for nterms, key in ((3, "bf16_split_fp32_grade"), (1, "bf16_plain")):
        head.volumes(fL, fR, D, nterms=nterms)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        head.volumes(fL, fR, D, nterms=nterms)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        ach = rows * flop_row * nterms / ms / 1e9
        out[key] = {"ms": round(ms, 2), "useful_tflops": round(rows * flop_row / ms / 1e9, 1), "achieved": round(ach, 1), "unit": "TFLOP/s",
                    "peak": peak, "frac": round(ach / peak, 4) if peak else None,
                    "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peak else None}
    head.close()
    return out


def run_b200(args):
    import torch

    import mccnn_b200  # noqa: F401
    from mccnn_b200 import adcensus, pipeline

    # keep stdout clean for the one JSON line (NCCL / torch may print banners there)
    json_fd = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = dist_setup(args)
    cfg = dict(WORKLOADS[args.workload])
    if args.small:
        cfg.update(name="debug_small", H=64, W=128, D=16)
    opt = pipeline.make_params(*cfg["preset"])
    dev = torch.device("cuda", local)
    adcensus.lib()  # fail loudly if the CUDA library is missing

    pairs = make_inputs(cfg, 2, 1000 + 16 * rank)
    dev_in = [{k: v.to(dev) for k, v in p.items()} for p in pairs]
    sp = pipeline.StereoPipeline(cfg["C"], cfg["D"], cfg["H"], cfg["W"], opt, device=local)
    disp = torch.empty((cfg["H"], cfg["W"]), device=dev)
    K, Wm = args.steps, max(args.warmup, 3)

    # ---- device-resident throughput, default mode (constant-work CBCA, 1e-4 contract) ---------------
    sampler = ClockSampler(local)
    assert sp.cbca_mode == "fast"
    ms_total = timed_steps(sp, dev_in, disp, K, Wm, world, sampler)
    clocks = sampler.stop()
    launches = sp.launches_per_run * K
    disp_fast = disp.clone()

    # ---- same steps in the exact mode (every output bit-identical to the reference) --------------------
    sp.set_cbca_mode("exact")
    ms_exact = timed_steps(sp, dev_in, disp, K, 2, world)
    disp_exact = disp.clone()
    # SURVEY.md 8(d) fast-mode bar on disp.bin: <= 1e-4 on >= (1 - 1e-4) of the pixels
    fast_diff_frac = float(((disp_fast - disp).abs() > 1e-4 * disp.abs().clamp(min=1.0)).float().mean().item())
    sp.set_cbca_mode("fast")

    # ---- end to end through the host-buffer C-ABI call (default mode) --------------------------------------
    # one batch call per timed region: every step's inputs cross PCIe from pinned host memory and every
    # step's disparity map comes back; copies of neighbouring steps overlap the kernels (3 streams)
    host_pairs = [tuple(pairs[i % 2][k] for k in ("featL", "featR", "imgL", "imgR")) for i in range(K)]
    disps_h = [torch.empty((cfg["H"], cfg["W"]), dtype=torch.float32).pin_memory() for _ in range(K)]
    sp.run_host_batch(host_pairs[:2], disps_h[:2])
    barrier_sync(world)
    t0 = time.perf_counter()
    sp.run_host_batch(host_pairs, disps_h)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    barrier_sync(world)
    # single-pair latency through the same boundary (no overlap possible)
    t1 = time.perf_counter()
    sp.run_host(*host_pairs[0], disp=disps_h[0])
    e2e_single_ms = (time.perf_counter() - t1) * 1e3
    F = 4 * cfg["C"] * cfg["H"] * cfg["W"]
    I = 4 * cfg["H"] * cfg["W"]

    # ---- rank 0: the unchanged-main.lua path, per-kernel timings, rooflines ------------------------------------
    out = None
    if rank == 0:
        # op chain: main.lua:929-1082 through the adcensus.* operators one by one (what an unpatched main.lua drives
        # through the Lua face): fill, StereoJoin, cross/cbca with vol:copy, permutes, sgm2, argmin, post
        xb = torch.stack([dev_in[0]["imgL"], dev_in[0]["imgR"]])[:, None].contiguous()
        ft = torch.stack([dev_in[0]["featL"], dev_in[0]["featR"]]).contiguous()
        pipeline.stereo_predict(xb, ft, opt, cfg["D"])
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_chain = 3
        c0.record()
        for _ in range(n_chain):
            pipeline.stereo_predict(xb, ft, opt, cfg["D"])
        c1.record()
        torch.cuda.synchronize()
        chain_ms = c0.elapsed_time(c1) / n_chain
        del xb, ft

        stages = stage_table(cfg, opt, dev_in[0], iters=max(3, min(K, 10)))
        if args.stages:
            for k, v in stages.items():
                sys.stderr.write("%-24s %8.3f ms\n" % (k, v))
        ab = algorithmic_bytes(cfg)
        n_cbca = 2 * (opt.cbca_i1 + opt.cbca_i2)
        peak, peak_src = load_peaks()
        traffic, traffic_src = load_traffic(args.workload if not args.small else "none")

        def roof(name):
            ach = ab[name] / (stages[name] * 1e-3) / 1e9
            return {"kernel": name, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                    "frac": round(ach / peak, 4), "traffic": traffic.get(name), "traffic_source": traffic_src, "peak_source": peak_src,
                    "algorithmic_bytes": ab[name], "ms": round(stages[name], 4)}

        def shares(cb):
            sh = {"StereoJoin": stages["StereoJoin"], "sgm2": 2 * opt.sgm_i * stages["sgm2"],
                  "transpose_in": 2 * opt.sgm_i * stages["transpose_in"], "transpose_out": 2 * opt.sgm_i * stages["transpose_out"],
                  "argmin": 2 * stages["argmin"]}
            if n_cbca:
                sh[cb] = n_cbca * stages[cb]
            return sh

        sh_fast, sh_exact = shares("cbca_fast"), shares("cbca_exact")
        dom_fast, dom_exact = max(sh_fast, key=sh_fast.get), max(sh_exact, key=sh_exact.get)
        out = {
            "metric": "stereo pairs/sec (370x1226 d=%d)" % cfg["D"], "value": round(world * K / (ms_total * 1e-3), 3),
            "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms_total / K, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(cfg),
            "mode": "default: constant-work CBCA (float aggregation within the north star's 1e-4 of the reference, measured ~1e-6; index "
                    "work bit-exact given the volumes); the exact mode (every output bit-identical) is reported under modes.exact",
            "schedule": "one batch call per timed region (mccnn_pipeline_run_batch): pairs alternate between two lanes (two buffer sets / stream sets), inside a lane the two directions of a pair are overlapped on two streams (mccnn_pipeline_set_overlap mode 2)",
            "clocks": clocks,
            "e2e": {"value": round(world * K / e2e_s, 3), "unit": "pairs/s", "h2d_bytes_per_step": 2 * F + 2 * I,
                    "d2h_bytes_per_step": I, "api": "mccnn_pipeline_run_host_batch (host buffers in, host disparity maps out)",
                    "single_pair_latency_ms": round(e2e_single_ms, 3)},
            "gpu_launches": launches,
            "roofline": roof(dom_fast),
            "modes": {
                "fast": {"value": round(world * K / (ms_total * 1e-3), 3), "unit": "pairs/s", "ms_per_step": round(ms_total / K, 4),
                         "roofline": roof(dom_fast), "step_share_ms": {k: round(v, 4) for k, v in sh_fast.items()},
                         "disp_pixels_off_by_more_than_1e-4_vs_exact_frac": fast_diff_frac},
                "exact": {"value": round(world * K / (ms_exact * 1e-3), 3), "unit": "pairs/s", "ms_per_step": round(ms_exact / K, 4),
                          "roofline": roof(dom_exact), "step_share_ms": {k: round(v, 4) for k, v in sh_exact.items()}},
            },
            "roofline_stereojoin": roof("StereoJoin"),
            "roofline_cbca": roof("cbca_fast") if n_cbca else None,
            "roofline_cbca_exact": roof("cbca_exact") if n_cbca else None,
            "roofline_sgm2": roof("sgm2"),
            "op_chain": {"value": round(1e3 / chain_ms, 3), "unit": "pairs/s", "ms_per_pair": round(chain_ms, 3), "n_gpus": 1,
                         "note": "unchanged-main.lua path: adcensus.* operators one by one (exact kernels, Lua-side fill / copy / permute "
                                 "steps included), device-resident, rank 0"},
            "stage_ms": {k: round(v, 4) for k, v in stages.items()},
        }
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(cfg, opt)
        if not args.small:
            try:
                out["scorer_head"] = scorer_head_block(local)
            except Exception as e:
                out["scorer_head"] = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
    sp.close()
    del dev_in
    torch.cuda.empty_cache()
    if world > 1 and not args.small:
        rb = rowband_block(rank, world, local)
        if out is not None:
            out["rowband"] = rb
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        if args.dump_outputs:
            # the headline (default-mode) timed path and the exact mode's, each from its last timed step
            dump_outputs(args.dump_outputs, {"disp": disp_fast, "disp_exact": disp_exact})
        os.write(json_fd, (json.dumps(out) + "\n").encode())


def run_reference(args):
    """The reference's own implementation of the path: adcensus.cu compiled unmodified (oracle/_ref), driven in main.lua's
    order.  It is a GPU implementation (the reference has no CPU path), so under torchrun every rank drives it on its
    own GPU -- like rgs.py:9-14 runs one process per GPU -- and rank 0 prints the aggregate."""
    from oracle import refdriver

    rank = int(os.environ.get("RANK", "0"))
    if not os.path.exists(refdriver.REF_LIB):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libadcensus_ref.so missing (reference tree was not present at build time)"}))
        return
    import torch

    import mccnn_b200  # noqa: F401
    from mccnn_b200 import pipeline

    json_fd = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = dist_setup(args)
    cfg = dict(WORKLOADS[args.workload])
    if args.small:
        cfg.update(name="debug_small", H=64, W=128, D=16)
    opt = pipeline.make_params(*cfg["preset"])
    dev = torch.device("cuda", local)
    pairs = make_inputs(cfg, 2, 1000 + 16 * rank)
    shim = refdriver.ShimLibrary(refdriver.REF_LIB)
    xb = [torch.stack([p["imgL"], p["imgR"]])[:, None].to(dev) for p in pairs]
    ft = [torch.stack([p["featL"], p["featR"]]).to(dev) for p in pairs]
    K, Wm = args.steps, max(args.warmup, 1)
    for i in range(Wm):
        refdriver.stereo_predict(shim, xb[i % 2], ft[i % 2], opt, cfg["D"])
    barrier_sync(world)
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        disp = refdriver.stereo_predict(shim, xb[i % 2], ft[i % 2], opt, cfg["D"])
    e1.record()
    barrier_sync(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world)
    clocks = sampler.stop()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"disp": disp.reshape(cfg["H"], cfg["W"])})
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    v = round(world * K / (ms * 1e-3), 4)
    os.write(json_fd, (json.dumps({
        "impl": "reference", "metric": "stereo pairs/sec (370x1226 d=%d)" % cfg["D"], "value": v, "unit": "pairs/s",
        "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms / K, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(cfg),
        "note": "reference adcensus.cu compiled unmodified for sm_100a (oracle/_ref), driven in main.lua:929-1082 order with torch ops "
                "for the cutorch-side fill/copy/transpose/div; the reference has no CPU path, so its own implementation of the path is "
                "this GPU one, one process per GPU like rgs.py",
        "clocks": clocks,
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": 0, "kind": "reference",
                         "sample": "%d full pairs per GPU on %d B200 (CUDA reference; host cores only launch)" % (K, world)},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }) + "\n").encode())


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
