"""Fast (constant-work) CBCA against the exact mode at the bench size on a structured synthetic pair: max relative error of
the final left volume and the fraction of disparity-map pixels that differ by more than 1e-4 (the exact mode is
bit-identical to the reference, tests/test_gpu_parity.py)."""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mccnn_b200  # noqa: E402,F401
from mccnn_b200 import pipeline, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--D", type=int, default=228)
ap.add_argument("--H", type=int, default=370)
ap.add_argument("--W", type=int, default=1226)
ap.add_argument("--seed", type=int, default=2)
a = ap.parse_args()
dev = torch.device("cuda:0")
opt = pipeline.make_params("kitti", "accurate_cbca4")
p = synth.make_pair(a.H, a.W, 64, a.D, seed=a.seed)
t = lambda x: torch.from_numpy(x).to(dev)
fL, fR, iL, iR = t(p["featL"]), t(p["featR"]), t(p["imgL"]), t(p["imgR"])
res = {}
for mode in ("exact", "fast"):
    sp = pipeline.StereoPipeline(64, a.D, a.H, a.W, opt, cbca_mode=mode)
    vol = torch.empty((a.D, a.H, a.W), device=dev)
    disp = sp.run(fL, fR, iL, iR, volL=vol)
    torch.cuda.synchronize()
    res[mode] = (disp.clone(), vol)
    sp.close()
de, ve = res["exact"]
df, vf = res["fast"]
nanok = bool((torch.isnan(ve) == torch.isnan(vf)).all())
m = ~torch.isnan(ve)
err = ((vf[m] - ve[m]).abs() / ve[m].abs().clamp(min=1.0))
frac = float(((df - de).abs() > 1e-4 * de.abs().clamp(min=1.0)).float().mean())
print("nan_pattern_ok=%s vol max_rel_err=%.3g mean_rel_err=%.3g disp_frac_off=%.3g"
      % (nanok, float(err.max()), float(err.mean()), frac))
