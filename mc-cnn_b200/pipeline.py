"""stereo_predict for the 'fast' architecture, from the tower output onwards.

Two faces over the same kernels:

* :func:`stereo_predict` chains the ``adcensus.*`` operator calls exactly as
  main.lua:929-1082 does (same order, same tensors, same Lua-side fill / copy /
  transpose / argmin steps), so it reads like the reference's own driver;
* :class:`StereoPipeline` is the native fused object behind
  ``mccnn_pipeline_*`` (include/adcensus_b200.h): buffers allocated once, one
  stream, no host sync -- what bench.py and a batch driver use.

Hyper-parameter presets are main.lua:70-295 copied as data (SURVEY.md appendix A).
"""
import ctypes

import torch

from . import adcensus


class Params(ctypes.Structure):
    """mccnn_params; field names are main.lua's option names."""

    _fields_ = [
        ("L1", ctypes.c_int),
        ("tau1", ctypes.c_float),
        ("cbca_i1", ctypes.c_int),
        ("cbca_i2", ctypes.c_int),
        ("pi1", ctypes.c_float),
        ("pi2", ctypes.c_float),
        ("sgm_q1", ctypes.c_float),
        ("sgm_q2", ctypes.c_float),
        ("alpha1", ctypes.c_float),
        ("tau_so", ctypes.c_float),
        ("sgm_i", ctypes.c_int),
        ("blur_sigma", ctypes.c_double),
        ("blur_t", ctypes.c_float),
        ("border", ctypes.c_int),
        ("lr_check", ctypes.c_int),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# (dataset, arch) -> stereo-method options, main.lua:70-295.  `border` = (window-1)/2 of the
# feature tower (main.lua:382-391, 923): 4 conv3x3 layers -> 4 (mb: 5 layers -> 5).
PRESETS = {
    ("kitti", "slow"): dict(L1=5, tau1=0.13, cbca_i1=2, cbca_i2=0, pi1=1.32, pi2=24.25, sgm_q1=3, sgm_q2=2,
                            alpha1=2, tau_so=0.08, blur_sigma=5.99, blur_t=6, border=4, lr_check=1),
    ("kitti2015", "slow"): dict(L1=5, tau1=0.03, cbca_i1=2, cbca_i2=4, pi1=2.3, pi2=24.25, sgm_q1=3, sgm_q2=2,
                                alpha1=1.75, tau_so=0.08, blur_sigma=5.99, blur_t=5, border=4, lr_check=1),
    ("mb", "slow"): dict(L1=14, tau1=0.02, cbca_i1=2, cbca_i2=16, pi1=1.3, pi2=13.9, sgm_q1=4.5, sgm_q2=2,
                         alpha1=2.75, tau_so=0.13, blur_sigma=1.67, blur_t=2, border=5, lr_check=0),
    ("kitti", "fast"): dict(L1=0, tau1=0, cbca_i1=0, cbca_i2=0, pi1=4, pi2=55.72, sgm_q1=3, sgm_q2=2.5,
                            alpha1=1.5, tau_so=0.02, blur_sigma=7.74, blur_t=5, border=4, lr_check=1),
    ("kitti2015", "fast"): dict(L1=0, tau1=0, cbca_i1=0, cbca_i2=0, pi1=2.3, pi2=18.38, sgm_q1=3, sgm_q2=2,
                                alpha1=1.25, tau_so=0.08, blur_sigma=4.64, blur_t=5, border=4, lr_check=1),
    ("mb", "fast"): dict(L1=0, tau1=0, cbca_i1=0, cbca_i2=0, pi1=2.3, pi2=24.3, sgm_q1=4, sgm_q2=2,
                         alpha1=1.5, tau_so=0.08, blur_sigma=6, blur_t=2, border=5, lr_check=0),
    # net-free cost volumes (main.lua:146-204): no feature tower, hence no fix_border (border = 0)
    ("kitti", "census"): dict(L1=0, tau1=0.01, cbca_i1=4, cbca_i2=8, pi1=4, pi2=128.0, sgm_q1=3, sgm_q2=3.5,
                              alpha1=1.25, tau_so=1.0, blur_sigma=7.74, blur_t=6, border=0, lr_check=1),
    ("mb", "census"): dict(L1=5, tau1=0.22, cbca_i1=8, cbca_i2=8, pi1=4.0, pi2=32.0, sgm_q1=4, sgm_q2=3,
                           alpha1=1.5, tau_so=1.0, blur_sigma=2.78, blur_t=3, border=0, lr_check=0),
    ("kitti", "ad"): dict(L1=3, tau1=0.03, cbca_i1=0, cbca_i2=4, pi1=0.76, pi2=13.93, sgm_q1=3.5, sgm_q2=2,
                          alpha1=2.5, tau_so=0.01, blur_sigma=7.74, blur_t=6, border=0, lr_check=1),
    ("mb", "ad"): dict(L1=5, tau1=0.36, cbca_i1=0, cbca_i2=4, pi1=0.4, pi2=8.0, sgm_q1=3, sgm_q2=4,
                       alpha1=2.5, tau_so=0.08, blur_sigma=7.74, blur_t=1, border=0, lr_check=0),
    # BASELINE.json config 3 ("KITTI accurate: CBCA x4 + SGM"): kitti slow post-processing with
    # cbca_i1 = cbca_i2 = 2 (SURVEY.md 8d)
    ("kitti", "accurate_cbca4"): dict(L1=5, tau1=0.13, cbca_i1=2, cbca_i2=2, pi1=1.32, pi2=24.25, sgm_q1=3,
                                      sgm_q2=2, alpha1=2, tau_so=0.08, blur_sigma=5.99, blur_t=6, border=4,
                                      lr_check=1),
}


def make_params(dataset="kitti", arch="fast", **overrides):
    d = dict(PRESETS[(dataset, arch)])
    d.setdefault("sgm_i", 1)
    d.update(overrides)
    return Params(**d)


def stereo_predict(x_batch, features, opt, disp_max, want_vols=False, arch="fast", head=None):
    """main.lua:929-1082 through the adcensus.* operators.

    x_batch  (2,1,H,W) standardised images (left, right); arch 'fast': features (2,C,H,W) the tower
    output (unit-norm); arch 'ad' / 'census': the matching cost comes from the images themselves
    (main.lua:932-942), `features` is ignored; arch 'slow' (main.lua:956-981): features (2,fm,H,W) = the accurate
    architecture's tower output and `head` a :class:`mccnn_b200.scorer_head.ScorerHead` (net_te2), which scores every
    disparity into both volumes.  opt a :class:`Params`.
    Returns disp (1,1,H,W) [, left vol, right vol].
    """
    assert x_batch.is_cuda
    H, W = x_batch.size(2), x_batch.size(3)
    dev = x_batch.device
    vols = torch.empty((2, disp_max, H, W), device=dev, dtype=torch.float32)
    adcensus.fill_nan(vols)                                                       # :933 / :939 / :946
    if arch == "ad":
        adcensus.ad(x_batch[0:1], x_batch[1:2], vols[0:1], -1)                    # :934
        adcensus.ad(x_batch[1:2], x_batch[0:1], vols[1:2], 1)                     # :935
    elif arch == "census":
        adcensus.census(x_batch[0:1], x_batch[1:2], vols[0:1], -1)                # :940
        adcensus.census(x_batch[1:2], x_batch[0:1], vols[1:2], 1)                 # :941
    elif arch == "fast":
        assert features is not None and features.is_cuda
        adcensus.StereoJoin(features[0:1], features[1:2], vols[0:1], vols[1:2])   # :947
        adcensus.fix_border(vols[0:1], opt.border, -1)                            # :948
        adcensus.fix_border(vols[1:2], opt.border, 1)                             # :949
    elif arch == "slow":
        assert features is not None and features.is_cuda and head is not None, "arch 'slow' needs the tower output and a ScorerHead"
        vl, vr = head.volumes(features[0].contiguous(), features[1].contiguous(), disp_max)   # :962-979 (both directions at once)
        vols[0:1].copy_(vl)
        vols[1:2].copy_(vr)
        adcensus.fix_border(vols[0:1], opt.border, -1)                            # :981
        adcensus.fix_border(vols[1:2], opt.border, 1)
    else:
        raise ValueError("arch must be 'fast', 'slow', 'ad' or 'census'")

    disp = {}
    out_vols = {}
    vol = None
    for direction in (1, -1):                                                     # :955
        vol = vols[0:1] if direction == -1 else vols[1:2]                         # :986
        x0c = torch.empty((1, 4, H, W), device=dev, dtype=torch.float32)          # :993-996
        x1c = torch.empty((1, 4, H, W), device=dev, dtype=torch.float32)
        adcensus.cross(x_batch[0], x0c, opt.L1, opt.tau1)
        adcensus.cross(x_batch[1], x1c, opt.L1, opt.tau1)
        tmp_cbca = torch.empty_like(vol)
        for _ in range(opt.cbca_i1):                                              # :998-1001
            adcensus.cbca(x0c, x1c, vol, tmp_cbca, direction)
            vol.copy_(tmp_cbca)
        volt = adcensus.transpose_dhw_to_hwd(vol)                                 # :1008
        out = torch.empty_like(volt)
        tmp = torch.empty((W, disp_max), device=dev, dtype=torch.float32)         # :1012
        for _ in range(opt.sgm_i):
            out.zero_()                                                           # :1014
            adcensus.sgm2(x_batch[0], x_batch[1], volt, out, tmp, opt.pi1, opt.pi2, opt.tau_so, opt.alpha1,
                          opt.sgm_q1, opt.sgm_q2, direction)                      # :1015
            volt.copy_(out).div_(4)                                               # :1017
        vol.copy_(adcensus.transpose_hwd_to_dhw_div4(out))                        # :1019-1020
        for _ in range(opt.cbca_i2):                                              # :1035-1038
            adcensus.cbca(x0c, x1c, vol, tmp_cbca, direction)
            vol.copy_(tmp_cbca)
        if want_vols:
            out_vols[direction] = vol.clone()                                     # :1042-1047
        disp[1 if direction == 1 else 2] = adcensus.argmin(vol)                   # :1049-1050

    d = disp[2]
    if opt.lr_check:                                                              # :1054-1066
        outlier = torch.zeros_like(d)
        adcensus.outlier_detection(disp[2], disp[1], outlier, disp_max)
        d = adcensus.interpolate_occlusion(d, outlier)
        d = adcensus.interpolate_mismatch(d, outlier)
    d = adcensus.subpixel_enchancement(d, vol, disp_max)                          # :1068 (left volume)
    d = adcensus.median2d(d, 5)                                                   # :1073
    d = adcensus.mean2d(d, adcensus.gaussian(opt.blur_sigma).to(dev), opt.blur_t)  # :1078
    if want_vols:
        return d, out_vols[-1], out_vols[1]
    return d


class StereoPipeline:
    """Native fused stereo_predict (mccnn_pipeline_*): buffers allocated once per (C,D,H,W)."""

    def __init__(self, C, D, H, W, params, device=0, cbca_mode=None):
        """``cbca_mode``: "fast" (library default) = constant-work aggregation inside the north star's 1e-4 contract
        for float aggregation; "exact" = tap-by-tap sums, volumes bit-identical to the reference."""
        self.C, self.D, self.H, self.W = C, D, H, W
        self.params = params
        self.device = int(device)
        self._h = ctypes.c_void_p()
        rc = adcensus.lib().mccnn_pipeline_create(ctypes.byref(self._h), C, D, H, W, ctypes.byref(params), self.device)
        adcensus._check(rc, "mccnn_pipeline_create")
        if cbca_mode is not None:
            self.set_cbca_mode(cbca_mode)

    def close(self):
        if self._h:
            adcensus.lib().mccnn_pipeline_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_overlap(self, mode=1):
        """Run the two directions concurrently on two streams (mccnn_pipeline_set_overlap); results are unchanged."""
        adcensus._check(adcensus.lib().mccnn_pipeline_set_overlap(self._h, int(mode)), "mccnn_pipeline_set_overlap")

    def set_cbca_mode(self, mode):
        """"fast" / 1: constant-work CBCA (csrc/cbca_tma.cu, ~1e-6 relative to the tap-by-tap sums, bar 1e-4);
        "exact" / 0: bit-identical to the reference (mccnn_pipeline_set_cbca_mode)."""
        m = {"fast": 1, "exact": 0}.get(mode, mode)
        adcensus.lib().mccnn_pipeline_set_cbca_mode(self._h, int(bool(m)))

    @property
    def cbca_mode(self):
        return "fast" if adcensus.lib().mccnn_pipeline_get_cbca_mode(self._h) else "exact"

    def set_fast_cbca(self, on=True):
        """older name of :meth:`set_cbca_mode`"""
        self.set_cbca_mode(1 if on else 0)

    @property
    def device_bytes(self):
        return adcensus.lib().mccnn_pipeline_device_bytes(self._h)

    @property
    def launches_per_run(self):
        return adcensus.lib().mccnn_pipeline_launches_per_run(self._h)

    def run(self, featL, featR, imgL, imgR, disp=None, volL=None, volR=None):
        """Device tensors in, device disparity map out; asynchronous on torch's current stream."""
        n = "mccnn_pipeline_run"
        if disp is None:
            disp = torch.empty((self.H, self.W), device=featL.device, dtype=torch.float32)
        vp = lambda t: adcensus._t(t, 0, n) if t is not None else ctypes.c_void_p(0)
        with torch.cuda.device(featL.device):
            rc = adcensus.lib().mccnn_pipeline_run(self._h, adcensus._t(featL, 1, n), adcensus._t(featR, 2, n),
                                                   adcensus._t(imgL, 3, n), adcensus._t(imgR, 4, n),
                                                   adcensus._t(disp, 5, n), vp(volL), vp(volR),
                                                   adcensus._stream(featL))
        adcensus._check(rc, n)
        return disp

    def run_batch(self, pairs, disps=None):
        """``pairs``: list of (featL, featR, imgL, imgR) DEVICE tensors.  One call for the whole list, ordered on torch's
        current stream as a whole; pairs alternate between two internal lanes (mccnn_pipeline_run_batch) so that the
        post-processing tail of one pair overlaps the volume kernels of the next.  Returns the list of device disparity maps."""
        n = "mccnn_pipeline_run_batch"
        k = len(pairs)
        if disps is None:
            disps = [torch.empty((self.H, self.W), device=pairs[0][0].device, dtype=torch.float32) for _ in range(k)]
        arr = lambda ts, i: (ctypes.c_void_p * k)(*[adcensus._t(t, i, n).value for t in ts])
        with torch.cuda.device(pairs[0][0].device):
            rc = adcensus.lib().mccnn_pipeline_run_batch(
                self._h, k, arr([p[0] for p in pairs], 1), arr([p[1] for p in pairs], 2), arr([p[2] for p in pairs], 3),
                arr([p[3] for p in pairs], 4), arr(disps, 5), adcensus._stream(pairs[0][0]))
        adcensus._check(rc, n)
        return disps

    def run_host(self, featL, featR, imgL, imgR, disp=None):
        """Host (CPU, ideally pinned) float32 tensors in and out; synchronous.  This is the call
        a non-CUDA host (the Lua/FFI side) makes: H2D + pipeline + D2H inside."""
        n = "mccnn_pipeline_run_host"
        for t in (featL, featR, imgL, imgR):
            if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                raise adcensus.AdcensusError("%s: contiguous host float tensors expected" % n)
        if disp is None:
            disp = torch.empty((self.H, self.W), dtype=torch.float32)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        rc = adcensus.lib().mccnn_pipeline_run_host(self._h, p(featL), p(featR), p(imgL), p(imgR), p(disp))
        adcensus._check(rc, n)
        return disp

    def run_host_batch(self, pairs, disps=None):
        """``pairs``: list of (featL, featR, imgL, imgR) host float32 tensors (pinned for overlap).
        H2D of pair i+1 and D2H of pair i-1 overlap the kernels of pair i.  Returns the list of
        host disparity maps (synchronous)."""
        n = "mccnn_pipeline_run_host_batch"
        k = len(pairs)
        for pr in pairs:
            for t in pr:
                if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                    raise adcensus.AdcensusError("%s: contiguous host float tensors expected" % n)
        if disps is None:
            disps = [torch.empty((self.H, self.W), dtype=torch.float32).pin_memory() for _ in range(k)]
        arr = lambda ts: (ctypes.c_void_p * k)(*[t.data_ptr() for t in ts])
        rc = adcensus.lib().mccnn_pipeline_run_host_batch(
            self._h, k, arr([p[0] for p in pairs]), arr([p[1] for p in pairs]), arr([p[2] for p in pairs]),
            arr([p[3] for p in pairs]), arr(disps))
        adcensus._check(rc, n)
        return disps
