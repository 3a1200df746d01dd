"""Time the fused pipeline (device-resident inputs) at the bench workload: prints ms per pair.

    python tools/time_pipeline.py [--iters 10] [--exact]
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mccnn_b200  # noqa: E402,F401
from mccnn_b200 import pipeline  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=10)
ap.add_argument("--exact", action="store_true", help="exact (bit-identical) CBCA instead of the default constant-work kernel")
ap.add_argument("--overlap", type=int, default=-1)
ap.add_argument("--preset", default="accurate_cbca4")
ap.add_argument("--D", type=int, default=228)
ap.add_argument("--H", type=int, default=370)
ap.add_argument("--W", type=int, default=1226)
ap.add_argument("--C", type=int, default=64)
ap.add_argument("--batch", action="store_true", help="one mccnn_pipeline_run_batch call for all iterations (lanes: ADCENSUS_LANES)")
a = ap.parse_args()
dev = torch.device("cuda:0")
opt = pipeline.make_params("kitti", a.preset)
g = torch.Generator(device=dev).manual_seed(0)
fL = torch.nn.functional.normalize(torch.randn((a.C, a.H, a.W), device=dev, generator=g), dim=0)
fR = torch.nn.functional.normalize(torch.randn((a.C, a.H, a.W), device=dev, generator=g), dim=0)
iL = torch.randn((a.H, a.W), device=dev, generator=g)
iR = torch.randn((a.H, a.W), device=dev, generator=g)
sp = pipeline.StereoPipeline(a.C, a.D, a.H, a.W, opt, cbca_mode="exact" if a.exact else "fast")
if a.overlap >= 0:
    sp.set_overlap(a.overlap)
for _ in range(3):
    sp.run(fL, fR, iL, iR)
if a.batch:
    sp.run_batch([(fL, fR, iL, iR)] * 4)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
if a.batch:
    sp.run_batch([(fL, fR, iL, iR)] * a.iters)
else:
    for _ in range(a.iters):
        sp.run(fL, fR, iL, iR)
e1.record()
torch.cuda.synchronize()
print("preset=%s lanes=%s cbca=%s overlap=%s ms_per_pair=%.4f launches=%d" % (a.preset, (os.environ.get("ADCENSUS_LANES", "2") if a.batch else "-"), sp.cbca_mode,
                                                                    a.overlap, e0.elapsed_time(e1) / a.iters, sp.launches_per_run))
sp.close()
