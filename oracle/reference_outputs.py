"""Stored outputs of the reference's own kernels for the parity tests that need sizes too large to commit -- TEST
INFRASTRUCTURE.

tests/golden/reference_outputs.json holds, per case (inputs named by ``case_key``) and per output (left / right volume,
disparity map), the SHA-256 of the output's float32 bytes after every NaN is replaced by one NaN and -0 by +0 (equal
values or both NaN, what the tests call identical), the element count, and a seeded sample of values that only serves
to say where a mismatch lies.  It also holds the names the reference's ``luaopen_libadcensus`` registers.  A test
compares the pipeline's output with the digest, so the comparison is over every element while the file stays small.

Regenerate (needs oracle/_ref/libadcensus_ref.so, i.e. a build with the reference tree present, and a B200):

    python oracle/reference_outputs.py OUT.json        # then copy OUT.json to tests/golden/reference_outputs.json
"""
import hashlib
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")
SAMPLE = 64
_CHUNK = 1 << 26

# (H, W, C, D, preset, overrides, inputs, directions): the parity tests' cases.  inputs "synth<s>" is
# synth.make_pair(seed=s), "mb<s>" is mb_inputs(seed=s).  directions (-1,) alone: main.lua's 'mb' outside -a predict.
CASES = [
    (48, 100, 32, 24, ("kitti", "slow"), dict(cbca_i2=2), "synth77", (1, -1)),
    (30, 140, 64, 70, ("kitti", "fast"), {}, "synth77", (1, -1)),
    (370, 1226, 64, 70, ("kitti", "fast"), {}, "synth2", (1, -1)),
    (370, 1226, 64, 228, ("kitti", "accurate_cbca4"), {}, "synth2", (1, -1)),
    (370, 1226, 64, 70, ("kitti2015", "slow"), {}, "synth2", (1, -1)),
    (300, 700, 32, 128, ("mb", "slow"), dict(cbca_i2=4), "synth2", (1, -1)),
    (1776, 3000, 64, 400, ("mb", "fast"), {}, "mb3", (-1,)),
]


def case_key(H, W, C, D, preset, over, inputs):
    extra = "".join("_%s=%s" % kv for kv in sorted(over.items()))
    return "%dx%dx%d_d%d_%s_%s%s_%s" % (H, W, C, D, preset[0], preset[1], extra, inputs)


def mb_inputs(H, W, C, dev, seed=3):
    """Middlebury-size inputs generated on the device (numpy would take minutes at 2000 x 3000 x 64): unit-norm random
    features and a standardised natural image pair shifted by 16 pixels."""
    from mccnn_b200 import synth

    g = torch.Generator(device=dev).manual_seed(seed)
    fL = torch.nn.functional.normalize(torch.randn((C, H, W), device=dev, generator=g), dim=0)
    fR = torch.nn.functional.normalize(torch.randn((C, H, W), device=dev, generator=g), dim=0)
    img = synth.natural_image(np.random.default_rng(seed), H, W + 16)
    st = lambda x: torch.from_numpy(((x - x.mean()) / x.std(ddof=1)).astype(np.float32)).to(dev)
    return fL, fR, st(img[:, 16:]).contiguous(), st(img[:, :W]).contiguous()


def canonical_sha256(t):
    """SHA-256 of a float32 tensor's elements in row-major order, NaNs canonical and -0 as +0."""
    h = hashlib.sha256()
    flat = t.detach().reshape(-1)
    for i in range(0, flat.numel(), _CHUNK):
        c = flat[i:i + _CHUNK].float()
        c = torch.where(torch.isnan(c), float("nan"), torch.where(c == 0, 0.0, c))
        h.update(c.cpu().numpy().tobytes())
    return h.hexdigest()


def record(t, seed=0):
    """The stored form of one output."""
    n = t.numel()
    idx = np.sort(np.random.default_rng(seed).integers(0, n, SAMPLE))
    vals = t.detach().reshape(-1)[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()
    return {"numel": n, "sha256": canonical_sha256(t), "sample_index": idx.tolist(),
            "sample_value": [None if math.isnan(v) else float(v) for v in vals]}


_loaded = None


def load():
    global _loaded
    if _loaded is None:
        with open(PATH) as f:
            _loaded = json.load(f)
    return _loaded


def assert_same(got, case, what):
    """`got` equals the reference's output `what` of `case` element for element (equal, or both NaN)."""
    cases = load()["cases"]
    assert case in cases, "no stored reference output for case %s (oracle/reference_outputs.py CASES)" % case
    want = cases[case][what]
    assert got.numel() == want["numel"], "%s: %d elements, the reference has %d" % (what, got.numel(), want["numel"])
    if canonical_sha256(got) == want["sha256"]:
        return
    idx = np.array(want["sample_index"], dtype=np.int64)
    g = got.detach().reshape(-1)[torch.from_numpy(idx).to(got.device)].float().cpu().numpy()
    w = np.array([np.nan if v is None else v for v in want["sample_value"]], dtype=np.float32)
    bad = ~((g == w) | (np.isnan(g) & np.isnan(w)))
    raise AssertionError("%s differs from the reference's (%s); %d of %d sampled elements differ%s" % (
        what, case, int(bad.sum()), len(idx),
        ", first at flat index %s: got %s want %s" % (idx[bad][:5].tolist(), g[bad][:5], w[bad][:5]) if bad.any() else ""))


def main(out_path):
    sys.path.insert(0, ROOT)
    import mccnn_b200  # noqa: F401
    from mccnn_b200 import pipeline, synth
    from oracle import refdriver

    shim = refdriver.ShimLibrary(refdriver.REF_LIB)
    out = {"functions": {t: shim.functions(t) for t in ("adcensus", "nn")}, "cases": {}}
    dev = torch.device("cuda:0")
    for H, W, C, D, preset, over, inputs, directions in CASES:
        opt = pipeline.make_params(*preset, **over)
        if inputs.startswith("mb"):
            fL, fR, iL, iR = mb_inputs(H, W, C, dev, seed=int(inputs[2:]))
        else:
            p = synth.make_pair(H, W, C, D, seed=int(inputs[5:]))
            fL, fR, iL, iR = (torch.from_numpy(p[k]).to(dev) for k in ("featL", "featR", "imgL", "imgR"))
        disp, volL, volR = refdriver.stereo_predict(shim, torch.stack([iL, iR])[:, None], torch.stack([fL, fR]), opt, D,
                                                    want_vols=True, directions=directions)
        del fL, fR, iL, iR
        torch.cuda.synchronize()
        rec = {"left": record(volL), "disp": record(disp)}
        if volR is not None:
            rec["right"] = record(volR)
        key = case_key(H, W, C, D, preset, over, inputs)
        out["cases"][key] = rec
        print(key, {k: v["sha256"][:12] for k, v in rec.items()}, flush=True)
        del disp, volL, volR
        torch.cuda.empty_cache()
    with open(out_path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
