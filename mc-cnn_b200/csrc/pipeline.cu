// pipeline.cu -- stereo_predict (main.lua:929-1082, arch 'fast') as one native
// object: every device buffer is allocated once at create time, a run is a fixed
// sequence of kernel launches (no allocation, no host sync) ordered on the caller's
// stream, so a batch driver can keep one pipeline per GPU / per stream busy back to
// back.  By default the two independent directions (main.lua:955) are overlapped:
// direction -1 runs on an internal side stream, started when direction +1 reaches
// its SGM phase, and the HBM-bound permute / SGM phases run on high-priority
// streams, so that they share the GPU with the issue-bound CBCA iterations of the
// other direction (mccnn_pipeline_set_overlap; joined before the LR check).
//
// Stage order, which volume is "left"/"right", the direction loop {+1,-1}, the /4
// and the permutes follow main.lua line by line (cited inline); the kernels are
// the ones behind the adcensus_* C ABI.
#include <initializer_list>
#include <math.h>
#include <new>
#include <stdlib.h>
#include <string.h>

#include "internal.cuh"

// Private volume layout: (D, H, ld), ld = W rounded up to a multiple of 4 floats.  Every row then starts on a
// 16-byte boundary: tensor maps (TMA) can describe the volumes, and 16-byte vector / cp.async accesses along x are
// legal everywhere (the API-facing (D,H,W) tensors with W = 1226 are only 8-byte aligned per row).  The padding
// columns hold unspecified values and are never read as data.
struct mccnn_pipeline {
	int C, D, H, W, ld, device;
	mccnn_params prm;
	long HW, V;       // H*W; elements of one private volume = D*H*ld
	size_t bytes;
	int launches;
	int cbca_mode;    // 1 = constant-work aggregation (default, 1e-4 contract), 0 = exact (bit-identical to the reference)
	size_t tab_bytes;
	// device buffers
	float *vols;      // 2V: [0] left volume, [1] right volume (main.lua:946)
	float *bufA;      // V : CBCA ping-pong
	float *bufC;      // V : SGM accumulator / ping-pong
	float *x0c, *x1c; // 4HW each: cross arms (main.lua:993-996)
	uint32_t *packed; // packed arm lengths of both images: bytes (exact kernels) + H/V words (constant-work kernel)
	int *maxlen;
	float *maps;      // 8HW: disparity maps and stage outputs
	float *gauss;     // ks*ks
	uint8_t *sgmtab;  // SGM penalty-class tables
	int ks;
	// tensor maps of the volume buffers (inputs of the TMA-staged CBCA)
	int ntm;
	const float *tm_ptr[6];
	CUtensorMap tm[6];
	// direction overlap (mccnn_pipeline_set_overlap): the two directions of main.lua:955 are independent
	// until the LR check, so the second one runs on a side stream with its own ping-pong / SGM buffers,
	// started when the first reaches its SGM phase.
	int overlap;      // 0 off, 1 two streams, 2 additionally the SGM phases on high-priority streams
	float *bufA2, *bufC2;
	uint8_t *sgmtab2;
	cudaStream_t side_stream, hi_stream[2];
	cudaEvent_t ev_stagger, ev_join, ev_hi_in[2], ev_hi_out[2];
	// staging for the host-buffer entry points: two slots so that the copy of pair i+1 overlaps
	// the kernels of pair i
	float *h_feat[2], *h_img[2], *h_disp[2];  // device copies per slot: 2F, 2HW, HW
	cudaStream_t own_stream, copy_stream, out_stream;
	cudaEvent_t ev_in[2], ev_free[2], ev_out[2];
	// further lanes of the batch entry points: a chain of twin pipelines (own buffers and streams) taking pairs round-robin, so that the
	// low-occupancy tail of one pair (LR check, interpolation, median, bilateral: ~0.6 ms of small kernels) and the bubbles
	// between its launches run next to the heavy kernels of the next pair
	mccnn_pipeline *twin;
	cudaEvent_t ev_fork, ev_lane;
};

extern "C" int mccnn_pipeline_set_overlap(mccnn_pipeline *p, int mode);

namespace {

int dev_alloc(void **p, size_t bytes, size_t *acc)
{
	cudaError_t e = cudaMalloc(p, bytes);
	if (e != cudaSuccess) return (int)e;
	*acc += bytes;
	return 0;
}

// longest arm cross() can produce for this preset, and the CBCA support radius
int pipe_maxlen(const mccnn_pipeline *p) { return p->prm.L1 > 2 ? p->prm.L1 : 2; }

int add_tensor_map(mccnn_pipeline *p, const float *buf)
{
	const int halo = pipe_maxlen(p) - 1;
	if (halo > adc_cbca_ws_max_halo()) return 0;       // such presets run the exact kernels
	if (p->ntm >= 6) return ADCENSUS_EINVAL;
	int bw, bh;
	adc_cbca_tma_box(halo, &bw, &bh);
	int rc = adc_tma_encode_volume(&p->tm[p->ntm], buf, p->D, p->H, p->W, p->ld, bw, bh);
	if (rc) return rc;
	p->tm_ptr[p->ntm++] = buf;
	return 0;
}

const CUtensorMap *find_tensor_map(const mccnn_pipeline *p, const float *buf)
{
	for (int i = 0; i < p->ntm; i++)
		if (p->tm_ptr[i] == buf) return &p->tm[i];
	return nullptr;
}

struct DeviceGuard {
	int prev;
	explicit DeviceGuard(int dev) { cudaGetDevice(&prev); cudaSetDevice(dev); }
	~DeviceGuard() { cudaSetDevice(prev); }
};

}  // namespace

extern "C" int mccnn_pipeline_create(mccnn_pipeline **out, int C, int D, int H, int W, const mccnn_params *params, int device)
{
	if (!out || !params || C < 1 || D < 1 || H < 1 || W < 1) return ADCENSUS_EINVAL;
	if (C > 128 || D > ADCENSUS_MAX_DISP) return ADCENSUS_ELIMIT;
	if (params->cbca_i1 < 0 || params->cbca_i2 < 0 || params->sgm_i < 0 || params->border < 0 || params->border + 1 > W)
		return ADCENSUS_EINVAL;
	DeviceGuard g(device);
	mccnn_pipeline *p = new (std::nothrow) mccnn_pipeline();
	if (!p) return ADCENSUS_EINVAL;
	memset(p, 0, sizeof(*p));
	p->C = C; p->D = D; p->H = H; p->W = W; p->device = device;
	p->ld = (W + 3) & ~3;
	p->prm = *params;
	p->HW = (long)H * W;
	p->V = (long)D * H * p->ld;
	const char *ex = getenv("ADCENSUS_CBCA_EXACT");
	p->cbca_mode = (ex && atoi(ex)) ? 0 : 1;
	p->tab_bytes = adc_sgm_table_bytes(H, W, D);
	int rc = 0;
	const size_t f = sizeof(float);
	if (!rc) rc = dev_alloc((void **)&p->vols, 2 * p->V * f, &p->bytes);
	if (!rc) rc = dev_alloc((void **)&p->bufA, p->V * f, &p->bytes);
	if (!rc) rc = dev_alloc((void **)&p->bufC, p->V * f, &p->bytes);
	if (!rc) rc = dev_alloc((void **)&p->x0c, 4 * p->HW * f, &p->bytes);
	if (!rc) rc = dev_alloc((void **)&p->x1c, 4 * p->HW * f, &p->bytes);
	if (!rc) rc = dev_alloc((void **)&p->packed, (adc_packed_words(H, W) + adc_packed_hv_words(H, W)) * sizeof(uint32_t), &p->bytes);
	if (!rc) rc = dev_alloc((void **)&p->maxlen, sizeof(int), &p->bytes);
	if (!rc) rc = (int)cudaMemset(p->maxlen, 0, sizeof(int));
	if (!rc) rc = dev_alloc((void **)&p->maps, 8 * p->HW * f, &p->bytes);
	if (!rc) rc = dev_alloc((void **)&p->sgmtab, p->tab_bytes, &p->bytes);
	if (!rc) rc = add_tensor_map(p, p->vols);
	if (!rc) rc = add_tensor_map(p, p->vols + p->V);
	if (!rc) rc = add_tensor_map(p, p->bufA);
	if (!rc) rc = add_tensor_map(p, p->bufC);
	p->ks = mccnn_gaussian(params->blur_sigma, nullptr);
	if (!rc) rc = dev_alloc((void **)&p->gauss, (size_t)p->ks * p->ks * f, &p->bytes);
	if (!rc) {
		float *hk = (float *)malloc((size_t)p->ks * p->ks * f);
		mccnn_gaussian(params->blur_sigma, hk);  // main.lua:1078 gaussian(opt.blur_sigma):cuda()
		rc = (int)cudaMemcpy(p->gauss, hk, (size_t)p->ks * p->ks * f, cudaMemcpyHostToDevice);
		free(hk);
	}
	if (rc) {
		mccnn_pipeline_destroy(p);
		return rc;
	}
	*out = p;
	// Default schedule: the two directions overlapped (mode 2), 6V of volume buffers instead of 4V; if the
	// extra buffers do not fit, the sequential schedule is kept (same results).  ADCENSUS_OVERLAP overrides.
	const char *e = getenv("ADCENSUS_OVERLAP");
	const int mode = e ? atoi(e) : 2;
	rc = mccnn_pipeline_set_overlap(p, mode);
	if (rc && e) {                                     // an explicit request that cannot be met is an error
		*out = nullptr;
		mccnn_pipeline_destroy(p);
		return rc;
	}
	return 0;
}

static void overlap_release(mccnn_pipeline *p);

extern "C" void mccnn_pipeline_destroy(mccnn_pipeline *p)
{
	if (!p) return;
	DeviceGuard g(p->device);
	cudaFree(p->vols); cudaFree(p->bufA); cudaFree(p->bufC); cudaFree(p->x0c); cudaFree(p->x1c);
	cudaFree(p->packed); cudaFree(p->maxlen); cudaFree(p->maps); cudaFree(p->gauss); cudaFree(p->sgmtab);
	for (int k = 0; k < 2; k++) {
		cudaFree(p->h_feat[k]); cudaFree(p->h_img[k]); cudaFree(p->h_disp[k]);
		if (p->ev_in[k]) cudaEventDestroy(p->ev_in[k]);
		if (p->ev_free[k]) cudaEventDestroy(p->ev_free[k]);
		if (p->ev_out[k]) cudaEventDestroy(p->ev_out[k]);
	}
	overlap_release(p);
	if (p->twin) mccnn_pipeline_destroy(p->twin);
	if (p->ev_fork) cudaEventDestroy(p->ev_fork);
	if (p->ev_lane) cudaEventDestroy(p->ev_lane);
	if (p->own_stream) cudaStreamDestroy(p->own_stream);
	if (p->copy_stream) cudaStreamDestroy(p->copy_stream);
	if (p->out_stream) cudaStreamDestroy(p->out_stream);
	delete p;
}

extern "C" size_t mccnn_pipeline_device_bytes(const mccnn_pipeline *p) { return p ? p->bytes : 0; }
// 1 (default) constant-work aggregation within the 1e-4 contract (cbca_tma.cu); 0 exact, bit-identical to the reference
extern "C" void mccnn_pipeline_set_cbca_mode(mccnn_pipeline *p, int mode) { if (p) p->cbca_mode = mode ? 1 : 0; }
extern "C" int mccnn_pipeline_get_cbca_mode(const mccnn_pipeline *p) { return p ? p->cbca_mode : -1; }
extern "C" void mccnn_pipeline_set_fast_cbca(mccnn_pipeline *p, int on) { mccnn_pipeline_set_cbca_mode(p, on); }
static void overlap_release(mccnn_pipeline *p)
{
	const size_t f = sizeof(float);
	if (p->bufA2) { cudaFree(p->bufA2); p->bytes -= p->V * f; }
	if (p->bufC2) { cudaFree(p->bufC2); p->bytes -= p->V * f; }
	if (p->sgmtab2) { cudaFree(p->sgmtab2); p->bytes -= p->tab_bytes; }
	for (int i = 0; i < p->ntm;)                       // forget the maps of the released buffers
		if (p->tm_ptr[i] == p->bufA2 || p->tm_ptr[i] == p->bufC2) {
			p->tm_ptr[i] = p->tm_ptr[p->ntm - 1];
			p->tm[i] = p->tm[p->ntm - 1];
			p->ntm--;
		} else {
			i++;
		}
	p->bufA2 = p->bufC2 = nullptr;
	p->sgmtab2 = nullptr;
	if (p->side_stream) cudaStreamDestroy(p->side_stream);
	if (p->ev_stagger) cudaEventDestroy(p->ev_stagger);
	if (p->ev_join) cudaEventDestroy(p->ev_join);
	p->side_stream = nullptr; p->ev_stagger = nullptr; p->ev_join = nullptr;
	for (int k = 0; k < 2; k++) {
		if (p->hi_stream[k]) cudaStreamDestroy(p->hi_stream[k]);
		if (p->ev_hi_in[k]) cudaEventDestroy(p->ev_hi_in[k]);
		if (p->ev_hi_out[k]) cudaEventDestroy(p->ev_hi_out[k]);
		p->hi_stream[k] = nullptr; p->ev_hi_in[k] = nullptr; p->ev_hi_out[k] = nullptr;
	}
	p->overlap = 0;
}

extern "C" int mccnn_pipeline_set_overlap(mccnn_pipeline *p, int mode)
{
	if (!p || mode < 0 || mode > 2) return ADCENSUS_EINVAL;
	DeviceGuard g(p->device);
	if (mode && !p->side_stream) {
		const size_t f = sizeof(float);
		int rc = 0, lo = 0, hi = 0;
		if (!rc) rc = dev_alloc((void **)&p->bufA2, p->V * f, &p->bytes);
		if (!rc) rc = dev_alloc((void **)&p->bufC2, p->V * f, &p->bytes);
		if (!rc) rc = dev_alloc((void **)&p->sgmtab2, p->tab_bytes, &p->bytes);
		if (!rc) rc = add_tensor_map(p, p->bufA2);
		if (!rc) rc = add_tensor_map(p, p->bufC2);
		if (!rc) rc = (int)cudaDeviceGetStreamPriorityRange(&lo, &hi);   // hi = numerically lowest = greatest priority
		if (!rc) rc = (int)cudaStreamCreateWithPriority(&p->side_stream, cudaStreamNonBlocking, lo);
		for (int k = 0; k < 2 && !rc; k++) {
			rc = (int)cudaStreamCreateWithPriority(&p->hi_stream[k], cudaStreamNonBlocking, hi);
			if (!rc) rc = (int)cudaEventCreateWithFlags(&p->ev_hi_in[k], cudaEventDisableTiming);
			if (!rc) rc = (int)cudaEventCreateWithFlags(&p->ev_hi_out[k], cudaEventDisableTiming);
		}
		if (!rc) rc = (int)cudaEventCreateWithFlags(&p->ev_stagger, cudaEventDisableTiming);
		if (!rc) rc = (int)cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming);
		if (rc) {                                      // leave the pipeline as it was (sequential mode still works)
			overlap_release(p);
			cudaGetLastError();
			return rc;
		}
	}
	p->overlap = mode;
	return 0;
}

extern "C" int mccnn_pipeline_launches_per_run(const mccnn_pipeline *p) { return p ? p->launches : 0; }

#define STEP(call)                 \
	do {                       \
		int rc__ = (call); \
		if (rc__) return rc__; \
	} while (0)

extern "C" int mccnn_pipeline_run(mccnn_pipeline *p, const float *featL, const float *featR,
				  const float *imgL, const float *imgR, float *disp,
				  float *volL, float *volR, adcensus_stream_t stream)
{
	if (!p || !featL || !featR || !imgL || !imgR || !disp) return ADCENSUS_EINVAL;
	DeviceGuard g(p->device);
	cudaStream_t s = adc_stream(stream);
	const int C = p->C, D = p->D, H = p->H, W = p->W, ld = p->ld;
	const long HW = p->HW, V = p->V;
	const mccnn_params &o = p->prm;
	int nl = 0;

	float *volsL = p->vols, *volsR = p->vols + V;
	STEP(adc_fill_invalid(volsL, volsR, D, H, W, ld, s)); nl += 1;                                // main.lua:946 (only what :947 leaves)
	STEP(adc_stereo_join(featL, featR, volsL, volsR, C, D, H, W, ld, /*fast=*/0, s)); nl += 1;    // :947
	STEP(adc_fix_border(volsL, D, H, W, ld, o.border, -1, s));                                    // :948
	STEP(adc_fix_border(volsR, D, H, W, ld, o.border, 1, s)); nl += o.border ? 2 : 0;             // :949

	// cross arms: identical for both directions (main.lua:993-996 recomputes them)
	const int maxlen = pipe_maxlen(p);       // bound on the arm length cross() can produce
	const int ncbca = o.cbca_i1 + o.cbca_i2;
	// fix_border copies column W-n-1 over the border columns: for D > W - n - 1 that column holds NaN at "valid"
	// positions, which only the tap-by-tap generic kernel treats like the reference (NaN only where a tap is NaN)
	const bool nan_in_valid = o.border > 0 && D > W - o.border - 1;
	// constant-work aggregation only for arms <= 5 (the KITTI presets, cbca_ws.cu): with the Middlebury presets' arms of up to
	// 14 pixels the first-generation kernel's float prefixes over 27 x 27 windows reach 1.03e-4 after six iterations (measured,
	// mb slow at 300 x 700 x 128) -- outside the 1e-4 contract -- so those presets run the exact tile kernels in every mode
	const bool tma = p->cbca_mode && !nan_in_valid && maxlen - 1 <= adc_cbca_ws_max_halo();
	uint32_t *hv = p->packed + adc_packed_words(H, W);
	if (ncbca > 0) {
		STEP(adcensus_cross(imgL, p->x0c, H, W, o.L1, o.tau1, s));
		STEP(adcensus_cross(imgR, p->x1c, H, W, o.L1, o.tau1, s)); nl += 2;
		if (tma) {
			STEP(adc_pack_arms_hv(p->x0c, hv, 0, H, W, s));
			STEP(adc_pack_arms_hv(p->x1c, hv, 1, H, W, s)); nl += 2;
		} else if (!nan_in_valid) {
			STEP(adc_pack_arms(p->x0c, p->packed, 0, H, W, p->maxlen, s));
			STEP(adc_pack_arms(p->x1c, p->packed, 1, H, W, p->maxlen, s)); nl += 2;
		}
	}
	auto cbca = [&](const float *in, float *out, int direction, cudaStream_t ds) -> int {        // adcensus.cbca, :999 / :1036
		if (tma) {
			const CUtensorMap *tm = find_tensor_map(p, in);
			if (!tm) return ADCENSUS_EINVAL;
			return adc_cbca_tma(tm, hv, in, out, D, H, W, ld, direction, maxlen - 1, ds);
		}
		return adc_cbca_packed(p->packed, p->x0c, p->x1c, in, out, D, H, W, ld, direction, nan_in_valid ? (1 << 20) : maxlen, ds);
	};

	float *dispR = p->maps, *dispL = p->maps + HW;
	float *final_left = nullptr;
	// One direction of main.lua:955-1051 on stream `ds`: cur/spare ping-pong, acc = SGM accumulator.
	// k = 0: direction +1 (right volume), k = 1: direction -1 (left volume).
	auto run_direction = [&](int k, cudaStream_t ds, float *cur, float *spare, float *acc, uint8_t *tab) -> int {
		const int direction = k == 0 ? 1 : -1;                                                   // :955
		for (int i = 0; i < o.cbca_i1; i++) {                                                    // :998-1001
			STEP(cbca(cur, spare, direction, ds));
			float *t = cur; cur = spare; spare = t; nl += 1;
		}
		if (k == 0 && p->overlap) STEP((int)cudaEventRecord(p->ev_stagger, ds));                 // the other direction may start
		cudaStream_t ss = ds;                                                                    // stream of the SGM phase
		if (p->overlap == 2 && o.sgm_i > 0) {
			ss = p->hi_stream[k];
			STEP((int)cudaEventRecord(p->ev_hi_in[k], ds));
			STEP((int)cudaStreamWaitEvent(ss, p->ev_hi_in[k], 0));
		}
		for (int it = 0; it < o.sgm_i; it++) {                                                   // :1008-1020
			STEP(adc_transpose_dhw_pitched_to_hwd(cur, spare, D, H, W, ld, ss));                 // :1008
			STEP(adc_sgm2(imgL, imgR, spare, acc, tab, H, W, D, o.pi1, o.pi2, o.tau_so, o.alpha1,
				      o.sgm_q1, o.sgm_q2, direction, /*zero_out=*/true, ss));                    // :1014-1016
			STEP(adc_transpose_hwd_to_dhw_pitched_div4(acc, cur, D, H, W, ld, ss));              // :1017-1020
			nl += 7;
		}
		if (ss != ds) {
			STEP((int)cudaEventRecord(p->ev_hi_out[k], ss));
			STEP((int)cudaStreamWaitEvent(ds, p->ev_hi_out[k], 0));
		}
		for (int i = 0; i < o.cbca_i2; i++) {                                                    // :1035-1038
			STEP(cbca(cur, spare, direction, ds));
			float *t = cur; cur = spare; spare = t; nl += 1;
		}
		STEP(adc_argmin_pitched(cur, direction == 1 ? dispR : dispL, D, H, W, ld, ds)); nl += 1; // :1049-1050
		float *dst = direction == 1 ? volR : volL;                                               // :1042-1047
		if (dst) STEP((int)cudaMemcpy2DAsync(dst, (size_t)W * 4, cur, (size_t)ld * 4, (size_t)W * 4, (size_t)D * H,
						     cudaMemcpyDeviceToDevice, ds));
		if (direction == -1) final_left = cur;
		return 0;
	};
	// main.lua:954-955: without the LR check (mb) only direction -1 is consumed, unless the caller asks for the
	// right volume (`-a predict` writes right.bin)
	const bool need_right = o.lr_check || volR;
	if (!need_right) {
		STEP(run_direction(1, s, volsL, p->bufA, p->bufC, p->sgmtab));
	} else if (!p->overlap) {
		// sequential: the right direction's three buffers are dead after its argmin / copy-out
		STEP(run_direction(0, s, volsR, p->bufA, p->bufC, p->sgmtab));
		STEP(run_direction(1, s, volsL, p->bufA, p->bufC, p->sgmtab));
	} else {
		// concurrent: direction -1 on the side stream with its own spare / accumulator / tables,
		// started when direction +1 leaves its first CBCA block
		STEP(run_direction(0, s, volsR, p->bufA, p->bufC, p->sgmtab));
		STEP((int)cudaStreamWaitEvent(p->side_stream, p->ev_stagger, 0));
		STEP(run_direction(1, p->side_stream, volsL, p->bufA2, p->bufC2, p->sgmtab2));
		STEP((int)cudaEventRecord(p->ev_join, p->side_stream));
		STEP((int)cudaStreamWaitEvent(s, p->ev_join, 0));
	}

	float *m = p->maps;
	const float *curd = dispL;                                                                   // disp[2]
	if (o.lr_check) {                                                                            // :1054-1066
		float *outlier = m + 2 * HW;
		STEP(adcensus_outlier_detection(dispL, dispR, outlier, H, W, D, s));                     // :1056
		STEP(adcensus_interpolate_occlusion(curd, outlier, m + 3 * HW, H, W, s));                // :1058
		STEP(adcensus_interpolate_mismatch(m + 3 * HW, outlier, m + 4 * HW, H, W, s));           // :1063
		curd = m + 4 * HW; nl += 3;
	}
	STEP(adc_subpixel(curd, final_left, m + 5 * HW, H, W, ld, D, s));                            // :1068
	STEP(adcensus_median2d(m + 5 * HW, m + 6 * HW, H, W, 5, s));                                 // :1073
	STEP(adcensus_mean2d(m + 6 * HW, p->gauss, disp, H, W, p->ks, o.blur_t, s)); nl += 3;        // :1078
	p->launches = nl;
	return 0;
}

static int host_staging(mccnn_pipeline *p)
{
	if (p->own_stream) return 0;
	const size_t F = (size_t)p->C * p->HW * sizeof(float), I = (size_t)p->HW * sizeof(float);
	int rc = 0;
	for (int k = 0; k < 2 && !rc; k++) {
		if (!rc) rc = dev_alloc((void **)&p->h_feat[k], 2 * F, &p->bytes);
		if (!rc) rc = dev_alloc((void **)&p->h_img[k], 2 * I, &p->bytes);
		if (!rc) rc = dev_alloc((void **)&p->h_disp[k], I, &p->bytes);
		if (!rc) rc = (int)cudaEventCreateWithFlags(&p->ev_in[k], cudaEventDisableTiming);
		if (!rc) rc = (int)cudaEventCreateWithFlags(&p->ev_free[k], cudaEventDisableTiming);
		if (!rc) rc = (int)cudaEventCreateWithFlags(&p->ev_out[k], cudaEventDisableTiming);
	}
	if (!rc) rc = (int)cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking);
	if (!rc) rc = (int)cudaStreamCreateWithFlags(&p->out_stream, cudaStreamNonBlocking);
	if (!rc) rc = (int)cudaStreamCreateWithFlags(&p->own_stream, cudaStreamNonBlocking);
	return rc;
}

// the extra lanes (see struct): a chain of twins created on first use with the same parameters and modes.  ADCENSUS_LANES
// (1..4, default 2) sets the number of lanes; lane 0 is the pipeline itself.
static int batch_lanes(mccnn_pipeline *p, mccnn_pipeline **lane, int want)
{
	static const int lanes_env = getenv("ADCENSUS_LANES") ? atoi(getenv("ADCENSUS_LANES")) : 2;
	int nl = lanes_env < 1 ? 1 : (lanes_env > 4 ? 4 : lanes_env);
	if (nl > want) nl = want;
	lane[0] = p;
	int n = 1;
	for (mccnn_pipeline *q = p; n < nl; n++) {
		if (!q->twin) {
			mccnn_pipeline *t = nullptr;
			if (mccnn_pipeline_create(&t, p->C, p->D, p->H, p->W, &p->prm, p->device)) {
				cudaGetLastError();
				break;                                 // not enough memory for another lane: fewer lanes give the same results
			}
			q->twin = t;
		}
		q = q->twin;
		q->cbca_mode = p->cbca_mode;
		if (q->overlap != p->overlap) mccnn_pipeline_set_overlap(q, p->overlap);
		lane[n] = q;
	}
	return n;
}

// pair number j of lane q from host memory: inputs are copied on q's copy stream into staging slot j % 2 while the lane's
// previous pair computes; the disparity map goes back on q's output stream
// cs: the H2D stream SHARED by the lanes (copies of different lanes would otherwise split the PCIe bandwidth and both arrive late:
// in order, pair i lands one transfer time after pair i - 1)
static int enqueue_host_pair(mccnn_pipeline *q, int j, cudaStream_t cs, const float *featL, const float *featR, const float *imgL, const float *imgR, float *disp)
{
	const size_t F = (size_t)q->C * q->HW * sizeof(float), I = (size_t)q->HW * sizeof(float);
	cudaStream_t ks = q->own_stream, os = q->out_stream;  // kernels, D2H
	const int k = j & 1;
	float *fL = q->h_feat[k], *fR = fL + (size_t)q->C * q->HW;
	float *iL = q->h_img[k], *iR = iL + q->HW;
	if (j >= 2) ADC_CUDA(cudaStreamWaitEvent(cs, q->ev_free[k], 0));   // slot's previous pair consumed
	ADC_CUDA(cudaMemcpyAsync(fL, featL, F, cudaMemcpyHostToDevice, cs));
	ADC_CUDA(cudaMemcpyAsync(fR, featR, F, cudaMemcpyHostToDevice, cs));
	ADC_CUDA(cudaMemcpyAsync(iL, imgL, I, cudaMemcpyHostToDevice, cs));
	ADC_CUDA(cudaMemcpyAsync(iR, imgR, I, cudaMemcpyHostToDevice, cs));
	ADC_CUDA(cudaEventRecord(q->ev_in[k], cs));
	ADC_CUDA(cudaStreamWaitEvent(ks, q->ev_in[k], 0));
	if (j >= 2) ADC_CUDA(cudaStreamWaitEvent(ks, q->ev_out[k], 0));     // slot's previous result copied out
	STEP(mccnn_pipeline_run(q, fL, fR, iL, iR, q->h_disp[k], nullptr, nullptr, ks));
	ADC_CUDA(cudaEventRecord(q->ev_free[k], ks));
	ADC_CUDA(cudaStreamWaitEvent(os, q->ev_free[k], 0));
	ADC_CUDA(cudaMemcpyAsync(disp, q->h_disp[k], I, cudaMemcpyDeviceToHost, os));
	ADC_CUDA(cudaEventRecord(q->ev_out[k], os));
	return 0;
}

// n pairs from host memory (pinned for real overlap): separate H2D / kernel / D2H streams with two staging slots per lane,
// pairs round-robin over the lanes (buffer sets, see batch_lanes).  Returns when every result is in its host buffer.
extern "C" int mccnn_pipeline_run_host_batch(mccnn_pipeline *p, int n, const float *const *featL_host,
					     const float *const *featR_host, const float *const *imgL_host,
					     const float *const *imgR_host, float *const *disp_host)
{
	if (!p || n < 0 || (n > 0 && (!featL_host || !featR_host || !imgL_host || !imgR_host || !disp_host))) return ADCENSUS_EINVAL;
	for (int i = 0; i < n; i++)
		if (!featL_host[i] || !featR_host[i] || !imgL_host[i] || !imgR_host[i] || !disp_host[i]) return ADCENSUS_EINVAL;
	DeviceGuard g(p->device);
	mccnn_pipeline *lane[4];
	const int nl = batch_lanes(p, lane, n > 1 ? n : 1);
	for (int l = 0; l < nl; l++) STEP(host_staging(lane[l]));
	for (int i = 0; i < n; i++)
		STEP(enqueue_host_pair(lane[i % nl], i / nl, p->copy_stream, featL_host[i], featR_host[i], imgL_host[i], imgR_host[i], disp_host[i]));
	for (int l = 0; l < nl; l++) {
		ADC_CUDA(cudaStreamSynchronize(lane[l]->out_stream));
		ADC_CUDA(cudaStreamSynchronize(lane[l]->own_stream));
		ADC_CUDA(cudaStreamSynchronize(lane[l]->copy_stream));
	}
	return 0;
}

// n device-resident pairs, ordered on `stream` as a whole (everything enqueued before the call precedes it, everything after
// it sees all n disparity maps): pairs alternate between the two lanes on their own streams.
extern "C" int mccnn_pipeline_run_batch(mccnn_pipeline *p, int n, const float *const *featL, const float *const *featR,
					const float *const *imgL, const float *const *imgR, float *const *disp, adcensus_stream_t stream)
{
	if (!p || n < 0 || (n > 0 && (!featL || !featR || !imgL || !imgR || !disp))) return ADCENSUS_EINVAL;
	for (int i = 0; i < n; i++)
		if (!featL[i] || !featR[i] || !imgL[i] || !imgR[i] || !disp[i]) return ADCENSUS_EINVAL;
	DeviceGuard g(p->device);
	cudaStream_t s = adc_stream(stream);
	mccnn_pipeline *lane[4];
	const int nl = batch_lanes(p, lane, n > 1 ? n : 1);
	if (nl == 1) {
		for (int i = 0; i < n; i++) STEP(mccnn_pipeline_run(p, featL[i], featR[i], imgL[i], imgR[i], disp[i], nullptr, nullptr, s));
		return 0;
	}
	for (int l = 0; l < nl; l++) {
		STEP(host_staging(lane[l]));                        // creates the lanes' own streams
		if (!lane[l]->ev_lane) ADC_CUDA(cudaEventCreateWithFlags(&lane[l]->ev_lane, cudaEventDisableTiming));
	}
	if (!p->ev_fork) ADC_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
	ADC_CUDA(cudaEventRecord(p->ev_fork, s));
	for (int l = 0; l < nl; l++) ADC_CUDA(cudaStreamWaitEvent(lane[l]->own_stream, p->ev_fork, 0));
	for (int i = 0; i < n; i++) {
		mccnn_pipeline *q = lane[i % nl];
		STEP(mccnn_pipeline_run(q, featL[i], featR[i], imgL[i], imgR[i], disp[i], nullptr, nullptr, q->own_stream));
	}
	for (int l = 0; l < nl; l++) {
		ADC_CUDA(cudaEventRecord(lane[l]->ev_lane, lane[l]->own_stream));
		ADC_CUDA(cudaStreamWaitEvent(s, lane[l]->ev_lane, 0));
	}
	return 0;
}

extern "C" int mccnn_pipeline_run_host(mccnn_pipeline *p, const float *featL_host, const float *featR_host,
				       const float *imgL_host, const float *imgR_host, float *disp_host)
{
	return mccnn_pipeline_run_host_batch(p, 1, &featL_host, &featR_host, &imgL_host, &imgR_host, &disp_host);
}
