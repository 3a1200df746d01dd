/*
 * adcensus_b200.h -- C ABI of libadcensus_b200.so, the B200 (sm_100a) drop-in
 * for the stereo-method hot path of jzbontar/mc-cnn's libadcensus.so.
 *
 * The reference exposes this path only as lua_CFunctions registered into the
 * Lua table `adcensus` (adcensus.cu:2061-2105).  Each `adcensus_<name>` below
 * is the plain-C core that the Lua face (csrc/lua_face.cu,
 * luaopen_libadcensus) -- or any other FFI: cgo, ctypes, JNI -- binds for the
 * Lua function of the same name; arguments are the tensors' raw device
 * pointers plus the sizes the reference reads from the tensors themselves
 * (SURVEY.md 8b).  See INTEGRATION.md for the binding a maintainer adds.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous float32 (the reference
 *     ignores strides: raw THCudaTensor_data + sizes);
 *   - shapes: features (C,H,W); cost volumes (D,H,W); SGM volumes (H,W,D); `*_pitched` entry points take
 *     (D,H,ld) volumes with a row pitch ld (the fused pipeline's private layout);
 *     images / disparity maps (H,W); cross arms (4,H,W);
 *   - `stream` is a cudaStream_t (0 = legacy default stream, what the
 *     reference launches on); all work is asynchronous on it unless noted;
 *   - return 0 on success, a positive cudaError_t, or a negative ADCENSUS_E*
 *     for arguments the kernels cannot handle (the reference's compiled-out
 *     device asserts: C <= 128 adcensus.cu:1460, D <= 400 :574, H <= W for
 *     sgm2's tmp :570).  Nothing here ever falls back to a CPU path.
 *   - no function keeps a pointer after it returns; the library holds no
 *     global mutable state apart from a per-device scratch pool that is
 *     stream-ordered (cudaMallocAsync).
 */
#ifndef ADCENSUS_B200_H
#define ADCENSUS_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADCENSUS_EINVAL (-1)   /* bad size / null pointer / unsupported value */
#define ADCENSUS_ELIMIT (-2)   /* exceeds a documented limit (D, C, ksize ...) */

#define ADCENSUS_MAX_DISP 512      /* sgm2: reference tree-min covers d < 512 (adcensus.cu:579) */
#define ADCENSUS_MAX_MEDIAN 11     /* median2d: float xs[11*11] (adcensus.cu:1582) */

typedef void *adcensus_stream_t;   /* cudaStream_t */

/* "libadcensus_b200 <version>"; replaces adcensus.version (adcensus.cu:2055-2059) */
const char *adcensus_version(void);

/* ---- operators of the hot path (one per Lua function) ------------------- */

/* adcensus.StereoJoin(input_L, input_R, output_L, output_R)  adcensus.cu:1455-1498
 * outL[d,y,x] = outR[d,y,x-d] = -sum_c L[c,y,x]*R[c,y,x-d] for x-d >= 0 (fp32 FMA
 * chain, c ascending); other entries are left untouched (caller pre-fills NaN,
 * main.lua:946). */
int adcensus_StereoJoin(const float *input_L, const float *input_R, float *output_L, float *output_R,
			int C, int D, int H, int W, adcensus_stream_t stream);

/* StereoJoin into PITCHED volumes (D, H, ld), ld % 4 == 0, 16-byte aligned outputs, W even, 8-byte aligned features (else
 * ADCENSUS_EINVAL): 8-byte cp.async operand loads, the left volume leaves through one TMA store per tile.  Same
 * values as adcensus_StereoJoin bit for bit; additionally output_L[d,y,x] = NaN for x < d (the fill of main.lua:946 for
 * the left volume); output_R's entries with x >= W - d are left untouched. */
int mccnn_stereo_join_pitched(const float *input_L, const float *input_R, float *output_L, float *output_R,
			      int C, int D, int H, int W, int ld, adcensus_stream_t stream);

/* adcensus.cross(x0, out, L1, tau1)  adcensus.cu:280-341; out is (4,H,W) */
int adcensus_cross(const float *x0, float *out, int H, int W, int L1, float tau1, adcensus_stream_t stream);

/* adcensus.cbca(x0c, x1c, vol_in, vol_out, direction)  adcensus.cu:343-400
 * vol_in must not alias vol_out.  Fully asynchronous: the longest arm, which sizes the shared-memory tile, stays on
 * the device -- every candidate kernel is launched with a gate on it and the ones out of range return immediately.
 * Precondition shared with the reference's (compiled-out) assert at adcensus.cu:366: vol_in is finite wherever a support can
 * reach, i.e. on x >= d (direction -1) / x < W - d (direction 1) -- for a fix_border'ed volume that means D <= W - border - 1.
 * Under it the result is bit-identical; a NaN inside the valid part spreads to the outputs of the tile rows that walk over it,
 * not only to the supports that contain it. */
int adcensus_cbca(const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
		  int D, int H, int W, int direction, adcensus_stream_t stream);

/* Same with the kernel chosen on the host: the caller states the longest arm cross() can have produced for these arms,
 * max(L1, 2) (main.lua knows opt.L1).  Arms longer than max_arm (<= 14) are CUT at max_arm (a truncated support, never an
 * out-of-bounds read); state the true bound or use adcensus_cbca.  Asynchronous on `stream`. */
int adcensus_cbca_ex(const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
		     int D, int H, int W, int direction, int max_arm, adcensus_stream_t stream);

/* The two halves of adcensus_cbca for callers that aggregate several times with the same arms
 * (main.lua runs cbca_i1 + cbca_i2 iterations per direction): pack both arm tensors once into
 * `packed` (mccnn_packed_arms_bytes(H, W) bytes of device memory), then iterate.  x0c/x1c are still
 * passed to the aggregation for the generic kernel that serves arms longer than 14 pixels. */
size_t mccnn_packed_arms_bytes(int H, int W);
int mccnn_pack_arms(const float *x0c, const float *x1c, void *packed, int H, int W, adcensus_stream_t stream);
int mccnn_cbca_packed(const void *packed, const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
		      int D, int H, int W, int direction, int max_arm, adcensus_stream_t stream);

/* Constant-work aggregation on PITCHED volumes (csrc/cbca_tma.cu): vol_in / vol_out are (D, H, ld) with a row pitch
 * ld >= W, ld % 4 == 0 and 16-byte aligned bases, so that the plane tiles can be staged by TMA.  NOT bit-exact with
 * the reference: every support row's run is a difference of row prefix sums and the rows are combined through
 * running sums down the column (~45 instructions per output instead of ~200, ~1e-6 relative to the tap-by-tap
 * sums, NaN positions identical); it serves the 1e-4 contract of the north star for float aggregation.  x0c / x1c
 * must be cross() outputs with arms of at most max_arm <= 14 pixels, and the volume must be finite on its valid
 * part (D <= W - border - 1 for a fix_border'ed volume).  The padding columns of vol_out are left untouched. */
int mccnn_cbca_fast_pitched(const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
			    int D, int H, int W, int ld, int direction, int max_arm, adcensus_stream_t stream);

/* The two halves of mccnn_cbca_fast_pitched: pack both arm tensors once (mccnn_packed_hv_bytes(H, W) bytes), then iterate. */
size_t mccnn_packed_hv_bytes(int H, int W);
int mccnn_pack_arms_hv(const float *x0c, const float *x1c, void *hv, int H, int W, adcensus_stream_t stream);
int mccnn_cbca_fast_pitched_packed(const void *hv, const float *vol_in, float *vol_out,
				   int D, int H, int W, int ld, int direction, int max_arm, adcensus_stream_t stream);

/* adcensus.sgm2(x0, x1, input, output, tmp, pi1, pi2, tau_so, alpha1, sgm_q1,
 *               sgm_q2, direction)  adcensus.cu:535-697
 * input/output are (H,W,D); output is accumulated into (+=) in the order right,
 * left, down, up.  tmp (>= W*D floats) is the reference's line-state scratch; it
 * is accepted for signature parity and may be NULL (state lives on chip). */
int adcensus_sgm2(const float *x0, const float *x1, const float *input, float *output, float *tmp,
		  int H, int W, int D, float pi1, float pi2, float tau_so, float alpha1,
		  float sgm_q1, float sgm_q2, int direction, adcensus_stream_t stream);

/* Band-wise sgm2 for the row-band / column-band multi-GPU split: x0, x1 are the FULL Ht x Wt images,
 * input/output this GPU's band volume (H,W,D) at image offset (yoff, xoff); pass_mask selects scan
 * directions (bit 0 right, 1 left, 2 down, 3 up; run in that order).  A band must hold whole scanlines
 * of every selected pass (row bands for bits 0-1, column bands for bits 2-3).  zero_out != 0: `output`
 * is known to be zero on entry. */
int mccnn_sgm2_band(const float *x0, const float *x1, const float *input, float *output,
		    int H, int W, int D, int Ht, int Wt, int yoff, int xoff,
		    float pi1, float pi2, float tau_so, float alpha1, float sgm_q1, float sgm_q2,
		    int direction, int pass_mask, int zero_out, adcensus_stream_t stream);

/* Wavefront split of sgm2 over ROW bands (the multi-GPU single-volume path, rowband.py).  Build the penalty-class tables
 * of the image pair once (mccnn_sgm_tables_bytes bytes; classes + the selector words of one `direction`), then run the
 * passes band by band on (H,W,D) band volumes at image row offset yoff: horizontal passes (bits 0-1) are band-local; a
 * vertical pass (bit 2 down or bit 3 up, ONE per call when chained) over the columns [xa, xb) takes the line state of the
 * row before the band from state_in (NULL only where the scan starts at the image border) and leaves the state of the
 * band's last row in state_out: [W][mccnn_sgm_state_pitch(D)] floats.  Same arithmetic and accumulation order as
 * adcensus_sgm2: chained over all bands the result is bit-identical to the whole-image call. */
size_t mccnn_sgm_tables_bytes(int Ht, int Wt, int D);
int mccnn_sgm_state_pitch(int D);
int mccnn_sgm_tables_build(const float *x0, const float *x1, void *tab, int Ht, int Wt, int D, float tau_so,
			   int direction, adcensus_stream_t stream);
int mccnn_sgm2_rows(const void *tab, const float *input, float *output, int H, int W, int D, int Ht, int yoff,
		    float pi1, float pi2, float tau_so, float alpha1, float sgm_q1, float sgm_q2,
		    int direction, int pass_mask, int zero_out, int xa, int xb,
		    const float *state_in, float *state_out, adcensus_stream_t stream);

/* adcensus.outlier_detection(d0, d1, outlier, disp_max)  adcensus.cu:878-918 */
int adcensus_outlier_detection(const float *d0, const float *d1, float *outlier,
			       int H, int W, int disp_max, adcensus_stream_t stream);

/* adcensus.interpolate_occlusion(d0, outlier) -> out  adcensus.cu:1079-1125
 * (the Lua face allocates `out` like new_tensor_like, adcensus.cu:40-45) */
int adcensus_interpolate_occlusion(const float *d0, const float *outlier, float *out,
				   int H, int W, adcensus_stream_t stream);

/* adcensus.interpolate_mismatch(d0, outlier) -> out  adcensus.cu:1001-1077 */
int adcensus_interpolate_mismatch(const float *d0, const float *outlier, float *out,
				  int H, int W, adcensus_stream_t stream);

/* adcensus.subpixel_enchancement(d0, c2, disp_max) -> out  adcensus.cu:1205-1239
 * c2 is the (disp_max,H,W) cost volume */
int adcensus_subpixel_enchancement(const float *d0, const float *c2, float *out,
				   int H, int W, int disp_max, adcensus_stream_t stream);

/* adcensus.median2d(img, kernel_size) -> out  adcensus.cu:1575-1613; odd ksize <= 11 */
int adcensus_median2d(const float *img, float *out, int H, int W, int kernel_size, adcensus_stream_t stream);

/* adcensus.mean2d(img, kernel, alpha2) -> out  adcensus.cu:1241-1282
 * kernel is (ksize,ksize), ksize odd */
int adcensus_mean2d(const float *img, const float *kernel, float *out, int H, int W, int ksize,
		    float alpha2, adcensus_stream_t stream);

/* adcensus.Normalize_forward(input, norm, output)  adcensus.cu:1284-1333
 * input/output (N,C,H,W), norm (N,1,H,W) */
int adcensus_Normalize_forward(const float *input, float *norm, float *output,
			       int N, int C, int H, int W, adcensus_stream_t stream);

/* adcensus.spatial_argmin(input, output)  adcensus.cu:244-278
 * input (N,D,H,W) -> output (N,1,H,W), 1-based, strict <, NaN skipped */
int adcensus_spatial_argmin(const float *input, float *output, int N, int D, int HW, adcensus_stream_t stream);

/* adcensus.ad / adcensus.census  adcensus.cu:62-175 (net-free cost volumes; x0,x1 (nch,H,W)) */
int adcensus_ad(const float *x0, const float *x1, float *out, int D, int H, int W, int direction,
		adcensus_stream_t stream);
int adcensus_census(const float *x0, const float *x1, float *out, int D, int nch, int H, int W,
		    int direction, adcensus_stream_t stream);

/* ---- the Lua-side tensor ops of stereo_predict (cutorch in the reference) - */

/* vols:fill(0/0)  main.lua:946 */
int mccnn_fill_nan(float *p, size_t n, adcensus_stream_t stream);
/* the part of that fill StereoJoin does not overwrite: NaN where x < d (left volume) and x >= W - d
 * (right volume); what the fused pipeline uses instead of filling 2V bytes */
int mccnn_fill_invalid(float *volL, float *volR, int D, int H, int W, adcensus_stream_t stream);
/* fix_border(net, vol, direction)  main.lua:922-927; n = (window-1)/2 */
int mccnn_fix_border(float *vol, int D, int H, int W, int n, int direction, adcensus_stream_t stream);
/* vol:transpose(2,3):transpose(3,4):clone()  main.lua:1008   (D,H,W) -> (H,W,D) */
int mccnn_transpose_dhw_to_hwd(const float *in, float *out, int D, int H, int W, adcensus_stream_t stream);
/* vol:copy(out:transpose(3,4):transpose(2,3)):div(4)  main.lua:1020   (H,W,D) -> (D,H,W), /4 */
int mccnn_transpose_hwd_to_dhw_div4(const float *in, float *out, int D, int H, int W, adcensus_stream_t stream);
/* _, d = torch.min(vol, 2); d:add(-1)  main.lua:1049-1050: 0-based argmin as float,
 * first minimum, NaN skipped (the in-repo statement is spatial_argmin) */
int mccnn_argmin(const float *vol, float *disp, int D, int HW, adcensus_stream_t stream);
/* the same three ops on the fused pipeline's pitched (D, H, ld) volumes: (D,H,ld) -> (H,W,D); (H,W,D) -> (D,H,ld) with /4;
 * first minimum over D */
int mccnn_transpose_dhw_pitched_to_hwd(const float *in, float *out, int D, int H, int W, int ld, adcensus_stream_t stream);
int mccnn_transpose_hwd_to_dhw_pitched_div4(const float *in, float *out, int D, int H, int W, int ld, adcensus_stream_t stream);
int mccnn_argmin_pitched(const float *vol, float *disp, int D, int H, int W, int ld, adcensus_stream_t stream);
/* gaussian(sigma)  main.lua:528-540: HOST helper; returns ksize, fills out (ksize*ksize) if non-NULL */
int mccnn_gaussian(double sigma, float *out_host);

/* ---- fused stereo_predict (main.lua:929-1082, arch 'fast') ---------------- */

typedef struct mccnn_params {
	int L1;
	float tau1;
	int cbca_i1, cbca_i2;
	float pi1, pi2, sgm_q1, sgm_q2, alpha1, tau_so;
	int sgm_i;
	double blur_sigma;
	float blur_t;
	int border;    /* fix_border n (4 for the 4-layer 3x3 tower, main.lua:382-391,923) */
	int lr_check;  /* 1: kitti / kitti2015 (main.lua:1054); 0: mb */
} mccnn_params;

typedef struct mccnn_pipeline mccnn_pipeline;

/* Allocates every device buffer the pipeline needs for (C,D,H,W) on `device`. */
int mccnn_pipeline_create(mccnn_pipeline **out, int C, int D, int H, int W,
			  const mccnn_params *params, int device);
void mccnn_pipeline_destroy(mccnn_pipeline *p);
size_t mccnn_pipeline_device_bytes(const mccnn_pipeline *p);
/* CBCA mode of the pipeline's iterations: 1 (default) = constant-work aggregation (mccnn_cbca_fast_pitched: volumes within
 * the north star's 1e-4 of the reference, measured ~1e-6; disparity map identical except at isolated near-ties);
 * 0 = exact, every output bit-identical to the reference.  ADCENSUS_CBCA_EXACT=1 in the environment makes 0 the default.
 * mccnn_pipeline_set_fast_cbca is the older name of the same switch. */
void mccnn_pipeline_set_cbca_mode(mccnn_pipeline *p, int mode);
int mccnn_pipeline_get_cbca_mode(const mccnn_pipeline *p);
void mccnn_pipeline_set_fast_cbca(mccnn_pipeline *p, int on);
/* opt-in: run the two directions of main.lua:955 concurrently (0 = off: one stream, 4V of volume buffers;
 * 1 = direction -1 on a side stream with its own 2V + tables, started when direction +1 reaches its SGM phase;
 * 2 = additionally the permute / SGM phases on high-priority streams).  Results are identical in every mode
 * (same kernels, same data); only the schedule and the memory footprint change.  Returns 0 or an error. */
int mccnn_pipeline_set_overlap(mccnn_pipeline *p, int mode);
/* number of kernel launches one run issues (for bench.py's gpu_launches) */
int mccnn_pipeline_launches_per_run(const mccnn_pipeline *p);

/* Device-resident inputs: featL/featR (C,H,W) unit-norm tower outputs, imgL/imgR
 * (H,W) standardised images.  disp (H,W) device; volL/volR (D,H,W) device or NULL
 * (what `-a predict` writes to left.bin/right.bin).  Asynchronous on `stream`. */
int mccnn_pipeline_run(mccnn_pipeline *p, const float *featL, const float *featR,
		       const float *imgL, const float *imgR, float *disp,
		       float *volL, float *volR, adcensus_stream_t stream);

/* Host-buffer call (what a non-CUDA caller binds): copies inputs H2D, runs,
 * copies disp back, and returns after the result is in disp_host. */
int mccnn_pipeline_run_host(mccnn_pipeline *p, const float *featL_host, const float *featR_host,
			    const float *imgL_host, const float *imgR_host, float *disp_host);

/* Same for n pairs (arrays of n host pointers each): the H2D copy of pair i+1 and the D2H copy of
 * pair i-1 overlap the kernels of pair i (two staging slots, a copy stream and a compute stream).
 * Host buffers should be pinned for the overlap to materialise.  Returns when all n results are
 * in their host buffers. */
int mccnn_pipeline_run_host_batch(mccnn_pipeline *p, int n, const float *const *featL_host,
				  const float *const *featR_host, const float *const *imgL_host,
				  const float *const *imgR_host, float *const *disp_host);

/* Operator-level calls take their scratch (SGM tables, packed arms) stream-ordered from the device's default memory pool; the
 * library raises that pool's release threshold to 2 GiB (never lowers it) so that repeated calls reuse the memory.
 * adcensus_trim_scratch() hands everything unused back to the driver. */
int adcensus_trim_scratch(void);

/* n device-resident pairs (arrays of n device pointers each), ordered on `stream` as a whole.  Pairs alternate between two
 * lanes (two buffer sets on internal streams, created on first use; ADCENSUS_LANES=1 disables the second lane), so that one
 * pair's low-occupancy post-processing tail overlaps the next pair's volume kernels.  Results identical to n calls of
 * mccnn_pipeline_run. */
int mccnn_pipeline_run_batch(mccnn_pipeline *p, int n, const float *const *featL, const float *const *featR,
			     const float *const *imgL, const float *const *imgR, float *const *disp, adcensus_stream_t stream);

/* ---- the accurate ('slow') architecture's scorer head (csrc/scorer_head.cu) -------------------------------------
 * Replaces the per-disparity loop of main.lua:958-984 over net_te2 (main.lua:688-695: l2 x [SpatialConvolution1_fw,
 * ReLU], SpatialConvolution1_fw(nh2 -> 1), Sigmoid; SpatialConvolution1_fw.lua:11-31 = addmm + bias per pixel) by one
 * fused tcgen05 kernel.  Outside libadcensus.so in the reference (a Lua nn module chain), hence a mccnn_* entry.
 * W[i] (out_i x in_i, row-major) and b[i] (out_i), i = 0 .. l2, DEVICE pointers in net_te2's order: layer 0 is
 * (nh2 x 2 fm), layers 1 .. l2-1 (nh2 x nh2), layer l2 (1 x nh2).  Limits: l2 <= 4, nh2 a multiple of 128 and <= 384,
 * fm a multiple of 8 with 2 fm <= 384 (the kitti / kitti2015 / mb nets: fm 112, nh2 384, l2 3..4). */
typedef struct mccnn_scorer_head mccnn_scorer_head;
int mccnn_scorer_head_create(mccnn_scorer_head **out, int fm, int nh2, int l2, const float *const *W, const float *const *b,
			     int device, adcensus_stream_t stream);
void mccnn_scorer_head_destroy(mccnn_scorer_head *h);
/* featL / featR: (fm, H, W) tower outputs; volL / volR: (D, H, W), either may be NULL.  Writes volL[d, y, x] for x >= d and
 * volR[d, y, x - d] (the same score, main.lua:976); all other entries keep the caller's NaN fill (:962); fix_border (:981)
 * is the caller's next call.  nterms 3: bf16-split operands, fp32-grade (1e-4 contract); 1: plain bf16. */
int mccnn_scorer_head_forward(const mccnn_scorer_head *h, const float *featL, const float *featR, float *volL, float *volR,
			      int H, int W, int D, int nterms, adcensus_stream_t stream);

/* ---- the feature tower in-library (csrc/feature_tower.cu, SURVEY.md 8f-2) ------------------------------------------
 * net_te at test time (main.lua:682-686 arch 'slow', 726-749 arch 'fast'): l1 x cudnn.SpatialConvolution(3x3, stride 1,
 * pad 1) with ReLU between the layers; arch 'fast' ends with Normalize2 (adcensus.cu:1284-1308) instead of a ReLU.
 * W[i] (fm, cin_i, 3, 3) row-major and b[i] (fm), i = 0 .. l1-1, DEVICE pointers (cudnn.SpatialConvolution's weight / bias).
 * Layer 1 (n_in = 1 or 3 planes) is exact fp32; the fm -> fm layers are tcgen05 implicit GEMMs (nterms 3: bf16-split
 * operands, fp32-grade; 1: plain bf16).  Limits: fm a multiple of 16 and <= 128, l1 <= 8. */
typedef struct mccnn_feature_tower mccnn_feature_tower;
int mccnn_feature_tower_create(mccnn_feature_tower **out, int n_in, int fm, int l1, int relu_last, int normalize,
			       const float *const *W, const float *const *b, int device, adcensus_stream_t stream);
void mccnn_feature_tower_destroy(mccnn_feature_tower *h);
/* img (nimg, n_in, H, W) -> out (nimg, fm, H, W); nimg = 2 for x_batch of main.lua:944. */
int mccnn_feature_tower_forward(const mccnn_feature_tower *h, const float *img, float *out, int nimg, int H, int W,
				int nterms, adcensus_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif
