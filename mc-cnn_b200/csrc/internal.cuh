// internal.cuh -- host entry points that one translation unit of libadcensus_b200.so defines and another calls.
// Every file that defines or calls one of them includes this header, so a prototype and its definition cannot drift
// apart unnoticed.  Volumes are (D, H, ld) with row pitch ld >= W unless noted; every call is ordered on stream `s`.
#pragma once

#include "common.cuh"
#include "tma.cuh"

// ---- cross_cbca.cu: exact (bit-identical) aggregation on packed arm lengths
// uint32 words of the packed arms of both images: [image 0 | image 1]
size_t adc_packed_words(int H, int W);
// packs cross() arms `xc` of image `which` (0 or 1) into `pk`, raising *maxlen_dev to the longest arm
int adc_pack_arms(const float *xc, uint32_t *pk, int which, int H, int W, int *maxlen_dev, cudaStream_t s);
// one aggregation pass; maxlen = longest arm of either image (above 14: the tap-by-tap kernel)
int adc_cbca_packed(const uint32_t *pk, const float *x0c, const float *x1c,
		    const float *vol, float *out, int D, int H, int W, int ld, int direction, int maxlen, cudaStream_t s);

// ---- cbca_tma.cu: constant-work aggregation (1e-4 contract); cbca_ws.cu serves support radii up to adc_cbca_ws_max_halo()
// uint32 words of the H/V-packed arms of both images
size_t adc_packed_hv_words(int H, int W);
// packs cross() arms `xc` of image `which` (0 or 1) into the H/V layout
int adc_pack_arms_hv(const float *xc, uint32_t *hv, int which, int H, int W, cudaStream_t s);
// largest support radius (longest arm - 1) cbca_ws.cu is built for
int adc_cbca_ws_max_halo();
// tensor-map box cbca_ws.cu needs for support radius `halo`
void adc_cbca_ws_box(int halo, int *box_w, int *box_h);
// one cbca_ws.cu pass; tm describes `vol` with the box of adc_cbca_ws_box(halo)
int adc_cbca_ws(const CUtensorMap *tm, const uint32_t *hv, const float *vol, float *out, int D, int H, int W, int ld, int direction,
		int halo, cudaStream_t s);
// tensor-map box a volume needs for support radius `halo`
void adc_cbca_tma_box(int halo, int *box_w, int *box_h);
// one constant-work pass; ld % 4 == 0, 16-byte aligned bases, tm describes `vol` with the box of adc_cbca_tma_box(halo)
int adc_cbca_tma(const CUtensorMap *tm, const uint32_t *hv, const float *vol, float *out, int D, int H, int W, int ld, int direction,
		 int halo, cudaStream_t s);

// ---- sgm.cu
// bytes of the penalty-class and selector tables adc_sgm2 needs for an H x W image and D disparities
size_t adc_sgm_table_bytes(int H, int W, int D);
// all four scans over an (H, W, D) volume, accumulated into `out` (zero_out: `out` is known to be zero)
int adc_sgm2(const float *x0, const float *x1, const float *in, float *out, uint8_t *tab, int H, int W, int D,
	     float pi1, float pi2, float tau_so, float alpha1, float q1, float q2, int direction,
	     bool zero_out, cudaStream_t s);

// ---- post.cu
// (D, H, ld) -> (H, W, D)
int adc_transpose_dhw_pitched_to_hwd(const float *in, float *out, int D, int H, int W, int ld, cudaStream_t s);
// (H, W, D) -> (D, H, ld), times 1/4
int adc_transpose_hwd_to_dhw_pitched_div4(const float *in, float *out, int D, int H, int W, int ld, cudaStream_t s);
// NaN where StereoJoin leaves an entry unwritten; either volume may be NULL
int adc_fill_invalid(float *volL, float *volR, int D, int H, int W, int ld, cudaStream_t s);
// fix_border: copies column W-n-1 (direction -1) or n (direction 1) over the n border columns
int adc_fix_border(float *vol, int D, int H, int W, int ld, int n, int direction, cudaStream_t s);
// first minimum over D, 0-based, NaN skipped, into an (H, W) map
int adc_argmin_pitched(const float *vol, float *disp, int D, int H, int W, int ld, cudaStream_t s);
// subpixel_enchancement of disparity map d0 on cost volume c2
int adc_subpixel(const float *d0, const float *c2, float *out, int H, int W, int ld, int disp_max, cudaStream_t s);

// ---- stereo_join.cu; stereo_join_tma.cu
// StereoJoin of (C, H, W) features into (D, H, ldo) volumes; fast = 1 selects the FASTIO kernel
int adc_stereo_join(const float *input_L, const float *input_R, float *output_L, float *output_R,
		    int C, int D, int H, int W, int ldo, int fast, cudaStream_t s);
// 1 when the TMA StereoJoin can run on these buffers
int adc_stereo_join_tma_ok(const float *input_L, const float *input_R, const float *output_L, const float *output_R, int H, int W);
// TMA StereoJoin; ns = register tiles per CTA along the diagonal
int adc_stereo_join_tma(const float *input_L, const float *input_R, float *output_L, float *output_R,
			int C, int D, int H, int W, int ldo, int ns, cudaStream_t s);
