"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the
committed golden fixtures: outputs of the reference's own kernels, as tensors
(tests/golden/pipe_*.npz) and as digests over every element of larger outputs
(tests/golden/reference_outputs.json, oracle/reference_outputs.py).

Bar (BASELINE.json north_star): bit-exact for index / label work; our kernels keep
the reference's fp32 operation order, so the float volumes are required to be
bit-identical too (NaN positions included), which is stricter than the 1e-4 the
north star allows.
"""
import glob
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import mccnn_b200  # noqa: E402,F401
from mccnn_b200 import adcensus, pipeline, synth  # noqa: E402
from oracle import reference_outputs as ro  # noqa: E402


def dev():
    return torch.device("cuda:0")


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev())


def same(a, b, what=""):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else b
    a, b = a.reshape(b.shape), b
    if not np.array_equal(a, b, equal_nan=True):
        bad = ~((a == b) | (np.isnan(a) & np.isnan(b)))
        idx = np.argwhere(bad)[:5]
        raise AssertionError("%s: %d / %d elements differ, first %s: got %s want %s" % (
            what, bad.sum(), bad.size, idx.tolist(), a[bad][:5], b[bad][:5]))


SIZES = [
    # H, W, C, D
    (64, 128, 64, 16),   # BASELINE config 1
    (7, 33, 5, 9),       # ragged, tiny
    (19, 150, 64, 70),   # D = 70 chunking, W not a multiple of anything
    (5, 300, 16, 228),   # D = 228, two disparity chunks
    (3, 40, 128, 33),    # C at the reference limit (adcensus.cu:1460)
]


@pytest.mark.parametrize("H,W,C,D", SIZES)
def test_stereo_join(oracle, H, W, C, D):
    p = synth.make_pair(H, W, C, D, seed=H + W)
    wantL, wantR = oracle.stereo_join(p["featL"], p["featR"], D)
    outL = torch.full((1, D, H, W), float("nan"), device=dev())
    outR = torch.full((1, D, H, W), float("nan"), device=dev())
    adcensus.StereoJoin(cu(p["featL"])[None], cu(p["featR"])[None], outL, outR)
    same(outL, wantL, "StereoJoin left")
    same(outR, wantR, "StereoJoin right")
    # shift convention: outR[d, y, x-d] == outL[d, y, x]  (adcensus.cu:1472-1473)
    oL, oR = outL[0].cpu().numpy(), outR[0].cpu().numpy()
    for d in range(0, D, max(1, D // 5)):
        if d < W:
            assert np.array_equal(oL[d, :, d:], oR[d, :, :W - d])


def test_stereo_join_untouched_entries(oracle):
    """entries with x - d < 0 are not written (caller pre-fills, main.lua:946)"""
    H, W, C, D = 4, 50, 8, 20
    p = synth.make_pair(H, W, C, D, seed=3)
    outL = torch.full((1, D, H, W), 7.0, device=dev())
    outR = torch.full((1, D, H, W), 9.0, device=dev())
    adcensus.StereoJoin(cu(p["featL"])[None], cu(p["featR"])[None], outL, outR)
    oL, oR = outL[0].cpu().numpy(), outR[0].cpu().numpy()
    for d in range(D):
        assert (oL[d, :, :d] == 7.0).all()
        assert (oR[d, :, W - d:] == 9.0).all()


@pytest.mark.parametrize("L1,tau1", [(0, 0.0), (5, 0.13), (14, 0.02), (3, 10.0), (30, 100.0)])
def test_cross(oracle, L1, tau1):
    H, W = 37, 61
    p = synth.make_pair(H, W, 2, 4, seed=L1)
    out = torch.empty((1, 4, H, W), device=dev())
    adcensus.cross(cu(p["imgL"])[None], out, L1, tau1)
    same(out, oracle.cross(p["imgL"], L1, tau1), "cross")


@pytest.mark.parametrize("L1,tau1,direction", [(5, 0.13, -1), (5, 0.13, 1), (14, 0.2, -1), (2, 0.5, 1),
                                               (9, 5.0, -1), (20, 100.0, 1), (0, 0.0, -1)])
def test_cbca(oracle, L1, tau1, direction):
    H, W, C, D = 41, 83, 4, 21
    p = synth.make_pair(H, W, C, D, seed=7)
    volL, volR = oracle.stereo_join(p["featL"], p["featR"], D)
    vol = volL if direction == -1 else volR
    x0c = oracle.cross(p["imgL"], L1, tau1)
    x1c = oracle.cross(p["imgR"], L1, tau1)
    want = oracle.cbca(x0c, x1c, vol, direction)
    out = torch.empty((1, D, H, W), device=dev())
    adcensus.cbca(cu(x0c)[None], cu(x1c)[None], cu(vol)[None], out, direction)
    same(out, want, "cbca")


@pytest.mark.parametrize("H,W,D,direction", [(9, 31, 7, -1), (9, 31, 7, 1), (12, 40, 33, -1), (6, 50, 70, 1),
                                             (5, 260, 228, -1), (4, 300, 300, 1), (8, 20, 64, -1)])
def test_sgm2(oracle, H, W, D, direction):
    p = synth.make_pair(H, W, 4, D, seed=D)
    volL, volR = oracle.stereo_join(p["featL"], p["featR"], D)
    vol = oracle.transpose_dhw_to_hwd(volL if direction == -1 else volR)
    args = (1.32, 24.25, 0.08, 2.0, 3.0, 2.0, direction)
    want = oracle.sgm2(p["imgL"], p["imgR"], vol, *args)
    out = torch.zeros((1, H, W, D), device=dev())
    tmp = torch.empty((W, D), device=dev())
    adcensus.sgm2(cu(p["imgL"])[None], cu(p["imgR"])[None], cu(vol)[None], out, tmp, *args)
    same(out, want, "sgm2")
    # accumulation into a non-zero output (out += val, adcensus.cu:569,616)
    init = np.random.default_rng(0).standard_normal((H, W, D)).astype(np.float32)
    want2 = oracle.sgm2(p["imgL"], p["imgR"], vol, *args, out=init.copy())
    out2 = cu(init)[None].clone()
    adcensus.sgm2(cu(p["imgL"])[None], cu(p["imgR"])[None], cu(vol)[None], out2, None, *args)
    same(out2, want2, "sgm2 accumulate")


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,D,direction", [(11, 37, 20, -1), (10, 45, 70, 1), (7, 300, 228, -1)])
def test_sgm2_bands_equal_whole_image(oracle, H, W, D, direction):
    """mccnn_sgm2_band: horizontal passes on row bands (known-zero accumulator: both directions in one CTA),
    then vertical passes on column bands, must reproduce the whole-image sgm2 bit for bit (the single-GPU
    form of what rowband.py does across GPUs)."""
    from mccnn_b200 import rowband

    p = synth.make_pair(H, W, 4, D, seed=3 * D)
    volL, volR = oracle.stereo_join(p["featL"], p["featR"], D)
    vol = oracle.transpose_dhw_to_hwd(volL if direction == -1 else volR)
    opt = pipeline.make_params("kitti", "fast")
    want = oracle.sgm2(p["imgL"], p["imgR"], vol, opt.pi1, opt.pi2, opt.tau_so, opt.alpha1, opt.sgm_q1, opt.sgm_q2, direction)
    ops = rowband.CudaOps(dev())
    iL, iR, cost = cu(p["imgL"]), cu(p["imgR"]), cu(vol)
    acc = torch.zeros_like(cost)
    for y0, y1 in ((0, H // 3), (H // 3, H)):                       # row bands: right + left
        band = acc[y0:y1].contiguous()
        ops.sgm_band(iL, iR, cost[y0:y1].contiguous(), band, H, W, y0, 0, opt, direction, 3, True)
        acc[y0:y1] = band
    for x0, x1 in ((0, W // 2 + 1), (W // 2 + 1, W)):               # column bands: down + up
        band = acc[:, x0:x1].contiguous()
        ops.sgm_band(iL, iR, cost[:, x0:x1].contiguous(), band, H, W, 0, x0, opt, direction, 12, False)
        acc[:, x0:x1] = band
    same(acc[None], want, "sgm2 by bands")


@pytest.mark.parametrize("H,W,D,direction", [(23, 37, 20, -1), (17, 45, 70, 1), (12, 300, 228, -1)])
def test_sgm2_rows_chained_over_row_bands(oracle, H, W, D, direction):
    """mccnn_sgm2_rows: horizontal passes band by band, then each vertical pass as a chain over three row bands and two
    column chunks with the line state handed from band to band (what rowband.py does across GPUs) == whole-image sgm2"""
    from mccnn_b200 import rowband

    p = synth.make_pair(H, W, 4, D, seed=5 * D)
    volL, volR = oracle.stereo_join(p["featL"], p["featR"], D)
    vol = oracle.transpose_dhw_to_hwd(volL if direction == -1 else volR)
    opt = pipeline.make_params("kitti", "fast")
    want = oracle.sgm2(p["imgL"], p["imgR"], vol, opt.pi1, opt.pi2, opt.tau_so, opt.alpha1, opt.sgm_q1, opt.sgm_q2, direction)
    ops = rowband.CudaOps(dev())
    iL, iR, cost = cu(p["imgL"]), cu(p["imgR"]), cu(vol)
    tab = ops.sgm_tables(iL, iR, D, opt, direction)
    bands = [(0, H // 3), (H // 3, H // 3 + 1), (H // 3 + 1, H)]     # a one-row band in the middle
    costs = [cost[a:b].contiguous() for a, b in bands]
    accs = [torch.full_like(c, float("nan")) for c in costs]         # zero_out: need not be initialised
    for (a, b), c, acc in zip(bands, costs, accs):
        ops.sgm_rows(tab, c, acc, H, a, opt, direction, 3, True, 0, W, None, None)
    chunks = [(0, W // 2 + 1), (W // 2 + 1, W)]
    for sd, order in ((2, [0, 1, 2]), (3, [2, 1, 0])):
        state = None
        for i in order:
            out_state = ops.new_state(W, D, cost) if i != order[-1] else None
            for xa, xb in chunks:
                ops.sgm_rows(tab, costs[i], accs[i], H, bands[i][0], opt, direction, 1 << sd, False, xa, xb, state, out_state)
            state = out_state
    same(torch.cat(accs)[None], want, "sgm2 chained over row bands")


def test_transposes_argmin(oracle):
    D, H, W = 13, 17, 29
    rng = np.random.default_rng(5)
    vol = rng.standard_normal((D, H, W)).astype(np.float32)
    vol[rng.random((D, H, W)) < 0.1] = np.nan
    vol[0] = np.abs(vol[0]) + 5  # d = 0 always valid
    vol[0][np.isnan(vol[0])] = 1.0
    t = adcensus.transpose_dhw_to_hwd(cu(vol)[None])
    same(t, oracle.transpose_dhw_to_hwd(vol), "transpose")
    back = adcensus.transpose_hwd_to_dhw_div4(t)
    same(back, vol / 4, "transpose back /4")
    am = adcensus.argmin(cu(vol)[None])
    same(am, oracle.spatial_argmin(vol) - 1, "argmin")
    out = torch.empty((1, 1, H, W), device=dev())
    adcensus.spatial_argmin(cu(vol)[None], out)
    same(out, oracle.spatial_argmin(vol), "spatial_argmin")
    # ties -> first index
    tie = np.zeros((4, 3, 5), np.float32)
    same(adcensus.argmin(cu(tie)[None]), np.zeros((3, 5), np.float32), "argmin ties")


def test_fill_fix_border(oracle):
    D, H, W = 5, 6, 23
    v = torch.empty((1, D, H, W), device=dev())
    adcensus.fill_nan(v)
    assert torch.isnan(v).all()
    rng = np.random.default_rng(1)
    a = rng.standard_normal((D, H, W)).astype(np.float32)
    for n, direction in [(4, -1), (4, 1), (5, 1), (1, -1)]:
        t = cu(a)[None].clone()
        adcensus.fix_border(t, n, direction)
        same(t, oracle.fix_border(a.copy(), n, direction), "fix_border")
    # odd element counts / unaligned starts for the float4 body of fill_nan
    buf = torch.zeros(1003, device=dev())
    adcensus.fill_nan(buf[1:1000])
    assert torch.isnan(buf[1:1000]).all() and buf[0] == 0 and (buf[1000:] == 0).all()


def _post_inputs(oracle, H=45, W=97, D=24, seed=2):
    p = synth.make_pair(H, W, 8, D, seed=seed)
    opt = pipeline.make_params("kitti", "slow")
    volL, volR = oracle.stereo_join(p["featL"], p["featR"], D)
    dL = oracle.spatial_argmin(volL) - 1
    dR = oracle.spatial_argmin(volR) - 1
    # perturb so that occlusion and mismatch labels both occur
    rng = np.random.default_rng(seed)
    m = rng.random((H, W)) < 0.15
    dL[m] = rng.integers(0, D, size=m.sum())
    return p, opt, volL, dL, dR


def test_post_chain(oracle):
    H, W, D = 45, 97, 24
    p, opt, volL, dL, dR = _post_inputs(oracle, H, W, D)
    want_out = oracle.outlier_detection(dL, dR, D)
    assert set(np.unique(want_out)) == {0.0, 1.0, 2.0}
    outlier = torch.zeros((1, 1, H, W), device=dev())
    adcensus.outlier_detection(cu(dL)[None, None], cu(dR)[None, None], outlier, D)
    same(outlier, want_out, "outlier_detection")
    occ = adcensus.interpolate_occlusion(cu(dL)[None, None], outlier)
    want_occ = oracle.interpolate_occlusion(dL, want_out)
    same(occ, want_occ, "interpolate_occlusion")
    mis = adcensus.interpolate_mismatch(occ, outlier)
    want_mis = oracle.interpolate_mismatch(want_occ, want_out)
    same(mis, want_mis, "interpolate_mismatch")
    sub = adcensus.subpixel_enchancement(mis, cu(volL)[None], D)
    want_sub = oracle.subpixel_enchancement(want_mis, volL, D)
    same(sub, want_sub, "subpixel_enchancement")
    for k in (1, 3, 5, 7, 11):
        same(adcensus.median2d(sub, k), oracle.median2d(want_sub, k), "median2d k=%d" % k)
    med = oracle.median2d(want_sub, 5)
    for sigma, t in [(1.2, 2.0), (5.99, 6.0), (0.4, 100.0)]:
        kern = oracle.gaussian(sigma)
        same(adcensus.gaussian(sigma), kern, "gaussian")
        got = adcensus.mean2d(cu(med)[None, None], cu(kern), t)
        same(got, oracle.mean2d(med, kern, t), "mean2d sigma=%g" % sigma)


def test_normalize_ad_census(oracle):
    rng = np.random.default_rng(9)
    x = rng.standard_normal((2, 7, 11, 19)).astype(np.float32)
    want, wnorm = oracle.normalize_forward(x)
    norm = torch.empty((2, 1, 11, 19), device=dev())
    out = torch.empty((2, 7, 11, 19), device=dev())
    adcensus.Normalize_forward(cu(x), norm, out)
    same(out, want, "Normalize_forward")
    same(norm, wnorm, "Normalize_forward norm")
    a = rng.standard_normal((1, 1, 15, 27)).astype(np.float32)
    b = rng.standard_normal((1, 1, 15, 27)).astype(np.float32)
    for direction in (-1, 1):
        o = torch.empty((1, 6, 15, 27), device=dev())
        adcensus.ad(cu(a), cu(b), o, direction)
        same(o, oracle.ad(a[0, 0], b[0, 0], 6, direction), "ad")
        adcensus.census(cu(a), cu(b), o, direction)
        same(o, oracle.census(a[0], b[0], 6, direction), "census")


@pytest.mark.parametrize("H,W,D,nch", [(15, 27, 6, 1), (40, 300, 70, 1), (9, 140, 150, 3), (21, 131, 17, 3), (5, 7, 9, 2)])
def test_ad_census_b200_kernels(oracle, H, W, D, nch):
    """bit-packed census (popcount of XORed 81-bit descriptors) and the shared-memory AD against the oracle's tap loops
    (adcensus.cu:62-175): bit-identical, borders / D > W / multi-channel included; quantised images force census ties"""
    rng = np.random.default_rng(H * W + nch)
    a = np.round(rng.standard_normal((nch, H, W)) * 3).astype(np.float32) / 3
    b = np.round(rng.standard_normal((nch, H, W)) * 3).astype(np.float32) / 3
    for direction in (-1, 1):
        o = torch.empty((1, D, H, W), device=dev())
        adcensus.census(cu(a)[None], cu(b)[None], o, direction)
        same(o, oracle.census(a, b, D, direction), "census")
        adcensus.ad(cu(a[:1])[None], cu(b[:1])[None], o, direction)
        same(o, oracle.ad(a[0], b[0], D, direction), "ad")


PIPE_CASES = [
    (64, 128, 64, 16, ("kitti", "fast"), {}),
    (64, 128, 64, 16, ("kitti", "slow"), {}),
    (40, 90, 16, 20, ("kitti2015", "slow"), dict(cbca_i2=3)),
    (40, 90, 16, 20, ("mb", "slow"), dict(cbca_i2=2)),
    (33, 70, 8, 12, ("kitti", "accurate_cbca4"), {}),
]


@pytest.mark.parametrize("H,W,C,D,preset,over", PIPE_CASES)
def test_pipeline_vs_oracle(oracle, H, W, C, D, preset, over):
    opt = pipeline.make_params(*preset, **over)
    p = synth.make_pair(H, W, C, D, seed=H * 3 + D)
    want, wL, wR = oracle.stereo_predict(p["featL"], p["featR"], p["imgL"], p["imgR"], D,
                                         oracle.Params(**opt.as_dict()), want_vols=True)
    x_batch = cu(np.stack([p["imgL"], p["imgR"]])[:, None])
    feats = cu(np.stack([p["featL"], p["featR"]]))
    # (a) operator by operator, as main.lua chains them
    d, vL, vR = pipeline.stereo_predict(x_batch, feats, opt, D, want_vols=True)
    same(vL, wL, "left.bin (op chain)")
    same(vR, wR, "right.bin (op chain)")
    same(d, want, "disp.bin (op chain)")
    # (b) the fused native pipeline
    sp = pipeline.StereoPipeline(C, D, H, W, opt, cbca_mode="exact")
    volL = torch.empty((D, H, W), device=dev())
    volR = torch.empty((D, H, W), device=dev())
    disp = sp.run(feats[0], feats[1], x_batch[0, 0], x_batch[1, 0], volL=volL, volR=volR)
    same(volL, wL, "left.bin (fused)")
    same(volR, wR, "right.bin (fused)")
    same(disp, want, "disp.bin (fused)")
    assert sp.launches_per_run > 0
    # (c) host-buffer entry point
    h = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    disp_h = sp.run_host(h(p["featL"]), h(p["featR"]), h(p["imgL"]), h(p["imgR"]))
    same(disp_h, want, "disp.bin (host call)")
    # (d) batched host call: copies of neighbouring pairs overlap the kernels; results stay per pair
    p2 = synth.make_pair(H, W, C, D, seed=H * 3 + D + 1)
    want2 = oracle.stereo_predict(p2["featL"], p2["featR"], p2["imgL"], p2["imgR"], D, oracle.Params(**opt.as_dict()))
    hp = lambda q: (h(q["featL"]), h(q["featR"]), h(q["imgL"]), h(q["imgR"]))
    outs = sp.run_host_batch([hp(p), hp(p2), hp(p), hp(p2), hp(p)])
    for i, o in enumerate(outs):
        same(o, want if i % 2 == 0 else want2, "disp.bin (host batch, pair %d)" % i)
    sp.close()


def _shifted_views(H, W, shift, seed):
    """two views of one textured image, the left one shifted by `shift` pixels, one gain / offset for both"""
    base = synth.natural_image(np.random.default_rng(seed), H, W + shift)
    base = ((base - base.mean()) / base.std(ddof=1)).astype(np.float32)
    return np.ascontiguousarray(base[:, :W]), np.ascontiguousarray(base[:, shift:])


@pytest.mark.gpu
@pytest.mark.parametrize("dataset,arch,H,W,D", [("kitti", "census", 24, 70, 10), ("kitti", "ad", 20, 64, 12),
                                                ("mb", "census", 18, 50, 9), ("mb", "ad", 16, 48, 8)])
def test_pipeline_ad_census_vs_oracle(oracle, dataset, arch, H, W, D):
    """main.lua:932-942: the net-free archs through the same operator chain, bit-identical to the oracle"""
    imgL, imgR = _shifted_views(H, W, 4, seed=H + D)
    opt = pipeline.make_params(dataset, arch)
    want, wantL, wantR = oracle.stereo_predict_chain(imgL, imgR, D, oracle.Params(**opt.as_dict()), arch, want_vols=True)
    xb = cu(np.stack([imgL, imgR])[:, None])
    got, gotL, gotR = pipeline.stereo_predict(xb, None, opt, D, want_vols=True, arch=arch)
    same(gotL, wantL, arch + " left volume")
    same(gotR, wantR, arch + " right volume")
    same(got, want, arch + " disp")


@pytest.mark.gpu
def test_frontend_predict_from_png_files(oracle, tmp_path):
    """frontend.predict: PNG pair -> standardised batch -> census chain -> right.bin, left.bin, disp.bin"""
    from PIL import Image

    from mccnn_b200 import frontend

    H, W, D, shift = 30, 80, 12, 5
    base = synth.natural_image(np.random.default_rng(21), H, W + shift)
    u8 = np.clip((base - base.min()) / (base.max() - base.min()) * 255.0, 0, 255).astype(np.uint8)
    lp, rp = str(tmp_path / "l.png"), str(tmp_path / "r.png")
    Image.fromarray(np.stack([u8[:, :W]] * 3, axis=2)).save(lp)          # colour file: exercises rgb2y
    Image.fromarray(np.ascontiguousarray(u8[:, shift:])).save(rp)
    out = tmp_path / "out"
    disp = frontend.predict(lp, rp, "kitti", "census", disp_max=D, out_dir=str(out))
    batch = frontend.make_batch(lp, rp)
    opt = pipeline.make_params("kitti", "census")
    want, wantL, wantR = oracle.stereo_predict_chain(batch[0, 0], batch[1, 0], D, oracle.Params(**opt.as_dict()),
                                                     "census", want_vols=True)
    same(disp, want, "predict disp")
    assert (np.abs(disp[:, 2 * D:] - shift) < 1.0).mean() > 0.9                 # and it is the right answer
    for name, ref, n in (("right.bin", wantR, D * H * W), ("left.bin", wantL, D * H * W), ("disp.bin", want, H * W)):
        data = np.fromfile(str(out / name), "<f4")
        assert data.size == n
        same(data, ref.ravel(), name)


def test_against_golden(golden_dir):
    files = sorted(glob.glob(os.path.join(golden_dir, "pipe_*.npz")))
    if not files:
        pytest.skip("no golden fixtures committed yet")
    for f in files:
        g = np.load(f)
        H, W, C, D = [int(v) for v in g["meta"]]
        opt = pipeline.Params(**{k: (float(v) if k in ("tau1", "pi1", "pi2", "sgm_q1", "sgm_q2", "alpha1", "tau_so",
                                                        "blur_sigma", "blur_t") else int(v))
                                 for k, v in zip(g["opt_names"], g["opt_values"])})
        x_batch = cu(np.stack([g["imgL"], g["imgR"]])[:, None])
        feats = cu(np.stack([g["featL"], g["featR"]]))
        sp = pipeline.StereoPipeline(C, D, H, W, opt, cbca_mode="exact")
        volL = torch.empty((D, H, W), device=dev())
        disp = sp.run(feats[0], feats[1], x_batch[0, 0], x_batch[1, 0], volL=volL)
        same(disp, g["disp"][0, 0], os.path.basename(f) + " disp")
        outL = torch.full((1, D, H, W), float("nan"), device=dev())
        outR = torch.full((1, D, H, W), float("nan"), device=dev())
        adcensus.StereoJoin(feats[0:1], feats[1:2], outL, outR)
        same(outL, g["sj_left"], os.path.basename(f) + " StereoJoin")
        sp.close()


def test_against_live_reference():
    """the reference's own kernels (adcensus.cu compiled unmodified), through their stored outputs
    (oracle/reference_outputs.py)"""
    for (H, W, C, D, preset, over) in [(48, 100, 32, 24, ("kitti", "slow"), dict(cbca_i2=2)),
                                       (30, 140, 64, 70, ("kitti", "fast"), {})]:
        case = ro.case_key(H, W, C, D, preset, over, "synth77")
        opt = pipeline.make_params(*preset, **over)
        p = synth.make_pair(H, W, C, D, seed=77)
        x_batch = cu(np.stack([p["imgL"], p["imgR"]])[:, None])
        feats = cu(np.stack([p["featL"], p["featR"]]))
        sp = pipeline.StereoPipeline(C, D, H, W, opt, cbca_mode="exact")
        volL = torch.empty((D, H, W), device=dev())
        volR = torch.empty((D, H, W), device=dev())
        disp = sp.run(feats[0], feats[1], x_batch[0, 0], x_batch[1, 0], volL=volL, volR=volR)
        ro.assert_same(volL, case, "left")
        ro.assert_same(volR, case, "right")
        ro.assert_same(disp, case, "disp")
        sp.close()


@pytest.mark.parametrize("H,W,C,D,preset,over", [
    (370, 1226, 64, 228, ("kitti", "accurate_cbca4"), {}),      # BASELINE config 3, the bench workload
    (370, 1226, 64, 70, ("kitti2015", "slow"), {}),             # d = 70 with CBCA x 6 (cbca_i1 = 2, cbca_i2 = 4)
    (300, 700, 32, 128, ("mb", "slow"), dict(cbca_i2=4)),       # Middlebury preset: arms up to 14 pixels (first-generation kernel)
])
def test_full_size_default_mode_against_live_reference(H, W, C, D, preset, over):
    """The pipeline's DEFAULT mode (constant-work CBCA) at BASELINE.json's full size against the reference's own kernels,
    with SURVEY.md 8(d)'s fast-mode thresholds: volumes |a - b| <= 1e-4 * max(1, |b|) with identical NaN pattern; disp.bin
    within 1e-4 on >= (1 - 1e-4) of the pixels.  The reference's outputs are stored as digests (oracle/reference_outputs.py),
    so they are recomputed here by the exact mode and checked against those digests, every element, before the
    comparison."""
    case = ro.case_key(H, W, C, D, preset, over, "synth2")
    opt = pipeline.make_params(*preset, **over)
    p = synth.make_pair(H, W, C, D, seed=2)
    x_batch = cu(np.stack([p["imgL"], p["imgR"]])[:, None])
    feats = cu(np.stack([p["featL"], p["featR"]]))
    sp = pipeline.StereoPipeline(C, D, H, W, opt)
    assert sp.cbca_mode == "fast"
    run = lambda vL, vR: sp.run(feats[0], feats[1], x_batch[0, 0], x_batch[1, 0], volL=vL, volR=vR)
    sp.set_cbca_mode("exact")
    wL, wR = torch.empty((D, H, W), device=dev()), torch.empty((D, H, W), device=dev())
    ref_d = run(wL, wR)
    for got, what in ((wL, "left"), (wR, "right"), (ref_d, "disp")):
        ro.assert_same(got, case, what)
    sp.set_cbca_mode("fast")
    volL = torch.empty((D, H, W), device=dev())
    volR = torch.empty((D, H, W), device=dev())
    disp = run(volL, volR)
    torch.cuda.synchronize()
    for got, ref, what in ((volL, wL, "left.bin"), (volR, wR, "right.bin")):
        assert bool((torch.isnan(got) == torch.isnan(ref)).all()), what + ": NaN pattern differs from the reference"
        ok = torch.isnan(ref) | ((got - ref).abs() <= 1e-4 * ref.abs().clamp(min=1.0))
        err = torch.where(torch.isnan(ref), torch.zeros_like(ref), (got - ref).abs() / ref.abs().clamp(min=1.0)).max().item()
        assert bool(ok.all()), "%s: max relative error %.3g above 1e-4" % (what, err)
    frac = float(((disp - ref_d).abs() > 1e-4 * ref_d.abs().clamp(min=1.0)).float().mean().item())
    assert frac <= 1e-4, "disp.bin: %.3g of the pixels differ by more than 1e-4 (bar 1e-4 of the pixels)" % frac
    sp.close()


def test_middlebury_size_against_live_reference():
    """BASELINE.json config 5 ('mb fast', main.lua:281-293: no CBCA, no LR check, direction -1 only) on ONE GPU against the
    reference's kernels (stored digests, oracle/reference_outputs.py), left.bin and disp.bin bit for bit, at the LARGEST
    height the reference can address: its kernels index the volume with `int` (adcensus.cu:1472 `d * size23 + id`, :560
    etc.), so 2000 x 3000 x 400 = 2.4e9 elements overflows in the reference itself (measured: 2.16e9 elements of its
    left.bin are garbage there).  1776 x 3000 x 400 = 2.13e9 < 2^31 is the same workload per row; the full 2000 rows are
    covered by the test below."""
    import gc

    gc.collect()
    torch.cuda.empty_cache()                                # memory cached by earlier tests counts as used otherwise
    free, _ = torch.cuda.mem_get_info()
    if free < 120e9:
        pytest.skip("needs ~110 GB of device memory")
    H, W, C, D = 1776, 3000, 64, 400
    opt = pipeline.make_params("mb", "fast")
    fL, fR, iL, iR = ro.mb_inputs(H, W, C, dev())
    sp = pipeline.StereoPipeline(C, D, H, W, opt, cbca_mode="exact")
    volL = torch.empty((D, H, W), device=dev())
    disp = sp.run(fL, fR, iL, iR, volL=volL)
    torch.cuda.synchronize()
    sp.close()
    case = ro.case_key(H, W, C, D, ("mb", "fast"), {}, "mb3")
    ro.assert_same(volL, case, "left")
    ro.assert_same(disp, case, "disp")


def test_middlebury_full_size_64bit_indexing():
    """2000 x 3000 x 400 (2.4e9 elements, beyond `int`): the fused pipeline against the operator chain (adcensus.* one by
    one, different kernels for the transposes / SGM layout / arg-min) -- equal bit for bit."""
    import gc

    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < 140e9:
        pytest.skip("needs ~130 GB of device memory")
    H, W, C, D = 2000, 3000, 64, 400
    opt = pipeline.make_params("mb", "fast")
    fL, fR, iL, iR = ro.mb_inputs(H, W, C, dev())
    sp = pipeline.StereoPipeline(C, D, H, W, opt, cbca_mode="exact")
    volL = torch.empty((D, H, W), device=dev())
    disp = sp.run(fL, fR, iL, iR, volL=volL)
    torch.cuda.synchronize()
    sp.close()
    want, wL, _ = pipeline.stereo_predict(torch.stack([iL, iR])[:, None], torch.stack([fL, fR]), opt, D, want_vols=True)
    torch.cuda.synchronize()
    for got, ref, what in ((volL, wL.reshape(D, H, W), "left volume"), (disp, want.reshape(H, W), "disparity map")):
        bad = ~((got == ref) | (torch.isnan(got) & torch.isnan(ref)))
        assert int(bad.sum()) == 0, "%s: %d elements differ between the fused pipeline and the operator chain" % (what, int(bad.sum()))


FULL_SIZE = [
    # BASELINE.json config 2 (KITTI fast, d=70) and config 3 (KITTI accurate, d=228, CBCA x4 + SGM)
    (370, 1226, 64, 70, ("kitti", "fast"), {}),
    (370, 1226, 64, 228, ("kitti", "accurate_cbca4"), {}),
    # Middlebury preset at a moderate size: L1 = 14 (halo 13: the tile kernels of the exact mode), no LR check
    (300, 700, 32, 128, ("mb", "slow"), dict(cbca_i2=4)),
]


@pytest.mark.parametrize("H,W,C,D,preset,over", FULL_SIZE)
def test_full_size_against_live_reference(H, W, C, D, preset, over):
    """BASELINE.json's full sizes: the fused pipeline against the reference's own kernels run in main.lua's order (stored
    digests, oracle/reference_outputs.py) -- left.bin, right.bin and disp.bin bit for bit."""
    opt = pipeline.make_params(*preset, **over)
    p = synth.make_pair(H, W, C, D, seed=2)
    x_batch = cu(np.stack([p["imgL"], p["imgR"]])[:, None])
    feats = cu(np.stack([p["featL"], p["featR"]]))
    sp = pipeline.StereoPipeline(C, D, H, W, opt, cbca_mode="exact")
    volL = torch.empty((D, H, W), device=dev())
    volR = torch.empty((D, H, W), device=dev())
    disp = sp.run(feats[0], feats[1], x_batch[0, 0], x_batch[1, 0], volL=volL, volR=volR)
    torch.cuda.synchronize()
    case = ro.case_key(H, W, C, D, preset, over, "synth2")
    for got, what in ((volL, "left"), (volR, "right"), (disp, "disp")):
        ro.assert_same(got, case, what)
    # size-independent properties of the domain at full size
    d = disp.cpu().numpy()
    assert not np.isnan(d).any() and d.min() >= 0 and d.max() <= D - 1 + 1e-3          # main.lua:1224
    if opt.lr_check:
        assert (np.abs(d - p["gt"]) < 1.0).mean() > 0.6                                # recovers the synthetic GT
    vl = volL[:, H // 2, :].cpu().numpy()
    for dd in range(0, D, 37):                                                         # NaN triangle intact
        assert np.isnan(vl[dd, :dd]).all() and not np.isnan(vl[dd, dd:]).any()
    sp.close()


def test_default_cbca_mode_is_within_tolerance(oracle):
    """The pipeline's DEFAULT CBCA (constant-work, csrc/cbca_tma.cu) is not bit-exact: volumes must agree with the
    oracle within the north star's 1e-4 (they do to ~1e-6), NaN positions exactly, and the final disparity map may
    differ only at isolated near-tie pixels (SURVEY.md 8d: <= 1e-4 on >= (1 - 1e-4) of the pixels is the bar at the
    bench sizes; this small, noisy synthetic pair gets a looser count)."""
    H, W, C, D = 96, 200, 16, 40
    opt = pipeline.make_params("kitti", "accurate_cbca4")
    p = synth.make_pair(H, W, C, D, seed=4)
    want, wL, wR = oracle.stereo_predict(p["featL"], p["featR"], p["imgL"], p["imgR"], D,
                                         oracle.Params(**opt.as_dict()), want_vols=True)
    t = lambda a: cu(a)
    sp = pipeline.StereoPipeline(C, D, H, W, opt)
    assert sp.cbca_mode == "fast"
    volL = torch.empty((D, H, W), device=dev())
    volR = torch.empty((D, H, W), device=dev())
    disp = sp.run(t(p["featL"]), t(p["featR"]), t(p["imgL"]), t(p["imgR"]), volL=volL, volR=volR)
    for got, ref, what in ((volL, wL, "left.bin"), (volR, wR, "right.bin")):
        g = got.cpu().numpy()
        assert np.array_equal(np.isnan(g), np.isnan(ref)), what + ": NaN pattern differs"
        m = ~np.isnan(ref)
        err = np.abs(g[m] - ref[m]) / np.maximum(1.0, np.abs(ref[m]))
        assert err.max() <= 1e-4, "%s: max relative error %.3g above 1e-4" % (what, err.max())
    d = disp.cpu().numpy()
    frac = float((np.abs(d - want) > 1e-4 * np.maximum(1.0, np.abs(want))).mean())
    assert frac < 5e-3, "constant-work CBCA changed %.4f of the disparity map" % frac
    # the exact mode stays bit-identical and selectable
    sp.set_cbca_mode("exact")
    vL = torch.empty((D, H, W), device=dev())
    same(sp.run(t(p["featL"]), t(p["featR"]), t(p["imgL"]), t(p["imgR"]), volL=vL), want, "exact mode after toggling")
    same(vL, wL, "left.bin, exact mode")
    sp.close()


def test_lua_face_through_the_reference_driver(oracle):
    """luaopen_libadcensus of OUR library (shim build), called by the very driver that calls the
    reference's: same 31 names, same positional signatures, same results."""
    from oracle import refdriver

    if not os.path.exists(refdriver.LUAFACE_LIB):
        pytest.skip("oracle/_ref/libadcensus_luaface.so not built")
    ours = refdriver.ShimLibrary(refdriver.LUAFACE_LIB)
    names = ours.functions("adcensus")
    assert len(names) == 31 and ours.functions("nn") == ["SpatialLogSoftMax_updateOutput", "SpatialLogSoftMax_updateGradInput"]
    assert names == ro.load()["functions"]["adcensus"]                                  # adcensus.cu:2061-2096
    H, W, C, D = 36, 80, 16, 18
    opt = pipeline.make_params("kitti2015", "slow", cbca_i2=2)
    p = synth.make_pair(H, W, C, D, seed=5)
    want, wL, wR = oracle.stereo_predict(p["featL"], p["featR"], p["imgL"], p["imgR"], D,
                                         oracle.Params(**opt.as_dict()), want_vols=True)
    x_batch = cu(np.stack([p["imgL"], p["imgR"]])[:, None])
    feats = cu(np.stack([p["featL"], p["featR"]]))
    d, vL, vR = refdriver.stereo_predict(ours, x_batch, feats, opt, D, want_vols=True)
    same(vL, wL, "left.bin (Lua face)")
    same(vR, wR, "right.bin (Lua face)")
    same(d, want, "disp.bin (Lua face)")
    # type errors and out-of-scope names raise Lua errors
    with pytest.raises(refdriver.ShimError, match="torch.CudaTensor expected"):
        ours.call("cross", 1.0, x_batch[0], 5, 0.1)
    with pytest.raises(refdriver.ShimError, match="not implemented"):
        ours.call("Margin2", x_batch[0], x_batch[0], x_batch[0], 0.2, 1)
    with pytest.raises(refdriver.ShimError, match="nil value"):
        ours.call("no_such_function")


def test_error_behaviour():
    """wrong tensor types raise like luaT_checkudata; limits are rejected, not overflowed"""
    with pytest.raises(adcensus.AdcensusError):
        adcensus.cross(torch.zeros(1, 4, 4), torch.zeros(1, 4, 4, 4), 5, 0.1)  # CPU tensors
    a = torch.zeros((1, 129, 2, 8), device=dev())
    o = torch.zeros((1, 4, 2, 8), device=dev())
    with pytest.raises(adcensus.AdcensusError):
        adcensus.StereoJoin(a, a, o, o)  # C > 128 (adcensus.cu:1460)
    with pytest.raises(adcensus.AdcensusError):
        adcensus.median2d(torch.zeros((1, 1, 4, 4), device=dev()), 13)  # > 11 (adcensus.cu:1602)
