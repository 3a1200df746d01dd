// post.cu -- the H*W-sized stages of the stereo method plus the Lua-side tensor
// ops of stereo_predict, for sm_100a.
//
// Reference: spatial_argmin adcensus.cu:244-278, outlier_detection :878-918,
// interpolate_occlusion :1079-1125, interpolate_mismatch :1001-1077,
// subpixel_enchancement :1205-1239, median2d :1575-1613, mean2d :1241-1282,
// Normalize_forward :1284-1333 (ad / census live in adcensus_cost.cu); Lua side
// main.lua:946 (fill), :922-927 (fix_border), :1008/:1020 (permutes), :1049-1050
// (torch.min).  All of these are bit-exact restatements: index/label work is
// integer, the float expressions keep the reference's operation order (fmaf where
// nvcc contracts the reference's `a += b * c`).
#include "internal.cuh"

namespace {

// ------------------------------------------------------------------ argmin
// 0-based (`base` = 0) or 1-based (`base` = 1) first minimum over D, NaN skipped
// (strict <, init +inf: adcensus.cu:251-259)
__global__ void argmin_kernel(const float *__restrict__ vol, float *__restrict__ out, int D, long HW, long total, float base)
{
	long id = (long)blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= total) return;
	long n = id / HW, p = id % HW;
	const float *v = vol + n * D * HW + p;
	int arg = 0;
	float mn = CUDART_INF_F;
	int d = 0;
	for (; d + 4 <= D; d += 4) {
		float a = ld_stream(v + (long)d * HW), b = ld_stream(v + (long)(d + 1) * HW);
		float c = ld_stream(v + (long)(d + 2) * HW), e = ld_stream(v + (long)(d + 3) * HW);
		if (a < mn) { mn = a; arg = d; }
		if (b < mn) { mn = b; arg = d + 1; }
		if (c < mn) { mn = c; arg = d + 2; }
		if (e < mn) { mn = e; arg = d + 3; }
	}
	for (; d < D; d++) {
		float a = ld_stream(v + (long)d * HW);
		if (a < mn) { mn = a; arg = d; }
	}
	out[id] = (float)arg + base;
}

// ------------------------------------------------------------------ LR check
__global__ void outlier_kernel(const float *__restrict__ d0, const float *__restrict__ d1, float *__restrict__ outlier,
			       int size, int W, int disp_max)
{
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	int x = id % W;
	float v0 = d0[id];
	int d0i = (int)v0;                                              // :883
	float res;
	if (x - d0i < 0) {
		res = 1.0f;
	} else if ((double)fabsf(v0 - d1[id - d0i]) < 1.1) {            // :887
		res = 0.0f;
	} else {
		res = 1.0f;
		int dmax = min(disp_max - 1, x);
		for (int d = 0; d <= dmax; d++)                             // :891-896
			if ((double)fabsf((float)d - d1[id - d]) < 1.1) { res = 2.0f; break; }
	}
	outlier[id] = res;
}

__global__ void interp_occ_kernel(const float *__restrict__ d0, const float *__restrict__ outlier, float *__restrict__ out, int size, int W)
{
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	if (outlier[id] != 1.0f) { out[id] = d0[id]; return; }
	int x = id % W;
	int dx = 0;
	while (x + dx >= 0 && outlier[id + dx] != 0.0f) dx--;           // :1090
	if (x + dx < 0) {
		dx = 0;
		while (x + dx < W && outlier[id + dx] != 0.0f) dx++;        // :1095
	}
	out[id] = (x + dx < W) ? d0[id + dx] : d0[id];
}

// Row form of the same rule (adcensus.cu:1087-1103): instead of every occluded pixel walking its
// row, one block per row records for every column the nearest label-0 pixel to the left and to the
// right (two serial scans over shared memory by two warps), then all threads pick left-else-right.
__global__ void interp_occ_row_kernel(const float *__restrict__ d0, const float *__restrict__ outlier, float *__restrict__ out, int W)
{
	extern __shared__ int occ_smem[];
	int *nl = occ_smem;          // nearest match at or left of x, else -1
	int *nr = occ_smem + W;      // nearest match at or right of x, else W
	float *lab = reinterpret_cast<float *>(occ_smem + 2 * W);
	const long row = (long)blockIdx.x * W;
	for (int x = threadIdx.x; x < W; x += blockDim.x) lab[x] = outlier[row + x];
	__syncthreads();
	if (threadIdx.x == 0) {
		int last = -1;
		for (int x = 0; x < W; x++) { last = lab[x] == 0.0f ? x : last; nl[x] = last; }
	} else if (threadIdx.x == 32) {
		int last = W;
		for (int x = W - 1; x >= 0; x--) { last = lab[x] == 0.0f ? x : last; nr[x] = last; }
	}
	__syncthreads();
	for (int x = threadIdx.x; x < W; x += blockDim.x) {
		float v = d0[row + x];
		if (lab[x] == 1.0f) {
			if (nl[x] >= 0) v = d0[row + nl[x]];          // :1090-1092 found walking left
			else if (nr[x] < W) v = d0[row + nr[x]];      // :1093-1098 else walking right
		}
		out[row + x] = v;
	}
}

__device__ __forceinline__ void sel_sort(float *v, int n)           // adcensus.cu:47-60
{
	for (int i = 0; i < n - 1; i++) {
		int mn = i;
		for (int j = i + 1; j < n; j++)
			if (v[j] < v[mn]) mn = j;
		float t = v[mn]; v[mn] = v[i]; v[i] = t;
	}
}

__global__ void interp_mis_kernel(const float *__restrict__ d0, const float *__restrict__ outlier, float *__restrict__ out, int size, int H, int W)
{
	// 16 directions, adcensus.cu:1003-1020
	const float dirs[32] = {0, 1, -0.5f, 1, -1, 1, -1, 0.5f, -1, 0, -1, -0.5f, -1, -1, -0.5f, -1,
				0, -1, 0.5f, -1, 1, -1, 1, -0.5f, 1, 0, 1, 0.5f, 1, 1, 0.5f, 1};
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	if (outlier[id] != 2.0f) { out[id] = d0[id]; return; }
	float vals[16];
	int n = 0;
	int x = id % W, y = id / W;
	for (int d = 0; d < 16; d++) {
		float dx = dirs[2 * d], dy = dirs[2 * d + 1];
		float xx = x, yy = y;
		int xi = (int)roundf(xx), yi = (int)roundf(yy);
		while (0 <= yi && yi < H && 0 <= xi && xi < W && outlier[yi * W + xi] == 2.0f) {
			xx += dx; yy += dy;
			xi = (int)roundf(xx); yi = (int)roundf(yy);
		}
		if (0 <= yi && yi < H && 0 <= xi && xi < W) vals[n++] = d0[yi * W + xi];
	}
	sel_sort(vals, n);
	out[id] = vals[n / 2];                                           // :1056
}

// c2: (disp_max, H, ld) with row pitch ld >= W (ld == W: contiguous)
__global__ void subpixel_kernel(const float *__restrict__ d0, const float *__restrict__ c2, float *__restrict__ out, int size, int H, int W, int ld, int disp_max)
{
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	int d = (int)d0[id];
	float res = (float)d;
	if (1 <= d && d < disp_max - 1) {
		const long HW = (long)H * ld;
		const long pix = (long)(id / W) * ld + id % W;
		float cn = c2[(long)(d - 1) * HW + pix];
		float cz = c2[(long)d * HW + pix];
		float cp = c2[(long)(d + 1) * HW + pix];
		float denom = 2 * (cp + cn - 2 * cz);                       // :1214
		if ((double)denom > 1e-5)
			res = (float)((double)d - fmin(1.0, fmax(-1.0, (double)((cp - cn) / denom)))); // :1216
	}
	out[id] = res;
}

__global__ void median_kernel(const float *__restrict__ img, float *__restrict__ out, int size, int H, int W, int r)
{
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	int x = id % W, y = id / W;
	float xs[ADCENSUS_MAX_MEDIAN * ADCENSUS_MAX_MEDIAN];
	int n = 0;
	for (int xx = x - r; xx <= x + r; xx++)
		for (int yy = y - r; yy <= y + r; yy++)
			if (0 <= xx && xx < W && 0 <= yy && yy < H) xs[n++] = __ldg(img + yy * W + xx);
	sel_sort(xs, n);
	out[id] = xs[n / 2];                                            // :1592
}

// k = 5 (the only size main.lua uses, :1073): the n/2-th smallest of <= 25 values is found by
// counting, which keeps everything in registers; same order statistic as the sort.
__global__ void median5_kernel(const float *__restrict__ img, float *__restrict__ out, int size, int H, int W)
{
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	int x = id % W, y = id / W;
	float v[25];
	int n = 0;
#pragma unroll
	for (int i = 0; i < 25; i++) {
		int xx = x - 2 + i / 5, yy = y - 2 + i % 5;
		bool ok = 0 <= xx && xx < W && 0 <= yy && yy < H;
		v[i] = ok ? __ldg(img + yy * W + xx) : CUDART_INF_F;        // +inf never below the median slot
		n += ok;
	}
	const int want = n / 2;                                         // rank (0-based) in ascending order
	float res = 0.0f;
#pragma unroll
	for (int i = 0; i < 25; i++) {
		int less = 0, leq = 0;
#pragma unroll
		for (int j = 0; j < 25; j++) {
			less += v[j] < v[i];
			leq += v[j] <= v[i];
		}
		if (less <= want && want < leq) res = v[i];
	}
	out[id] = res;
}

__global__ void mean2d_kernel(const float *__restrict__ img, const float *__restrict__ kernel, float *__restrict__ out,
			      int size, int r, int H, int W, float alpha2)
{
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	int x = id % W, y = id / W;
	const float c = img[id];
	float sum = 0.0f, cnt = 0.0f;
	const int ks = 2 * r + 1;
	for (int xx = x - r; xx <= x + r; xx++) {                       // :1251 (x outer)
		if (xx < 0 || xx >= W) continue;                            // weight index still advances (:1252)
		const float *kcol = kernel + (xx - x + r) * ks;
		int y_lo = max(y - r, 0), y_hi = min(y + r, H - 1);
		for (int yy = y_lo; yy <= y_hi; yy++) {
			float q = __ldg(img + yy * W + xx);
			if (fabsf(q - c) < alpha2) {                            // :1253
				float w = __ldg(kcol + (yy - y + r));
				sum = fmaf(q, w, sum);                              // :1254 (nvcc contracts the reference's +=)
				cnt += w;                                           // :1255
			}
		}
	}
	out[id] = sum / cnt;
}

// Shared-memory form of the same filter: a 32x8 pixel tile plus a halo of r is staged once (NaN
// outside the image: |NaN - c| < alpha2 is false, so those taps drop out exactly like the
// reference's bounds test), the (2r+1)^2 weights too; the tap loop then has no bounds checks and
// keeps the reference's order (x outer, y inner, adcensus.cu:1251-1252) and its fused multiply-add.
constexpr int M2_TX = 32, M2_TY = 8;
__global__ void __launch_bounds__(M2_TX * M2_TY)
mean2d_tile_kernel(const float *__restrict__ img, const float *__restrict__ kernel, float *__restrict__ out,
		   int r, int H, int W, float alpha2)
{
	extern __shared__ float m2_smem[];
	const int ks = 2 * r + 1;
	const int TW = M2_TX + 2 * r, TH = M2_TY + 2 * r;
	float *tile = m2_smem;                  // [TH][TW]
	float *wts = m2_smem + TH * TW;         // [ks][ks], index (dx + r) * ks + (dy + r)
	const int tid = threadIdx.y * M2_TX + threadIdx.x;
	const int x0 = blockIdx.x * M2_TX, y0 = blockIdx.y * M2_TY;
	for (int i = tid; i < TH * TW; i += M2_TX * M2_TY) {
		int ty = i / TW, tx = i - ty * TW;
		int yy = y0 - r + ty, xx = x0 - r + tx;
		tile[i] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(img + yy * W + xx) : adc_nan();
	}
	for (int i = tid; i < ks * ks; i += M2_TX * M2_TY) wts[i] = __ldg(kernel + i);
	__syncthreads();
	const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
	if (x >= W || y >= H) return;
	const float c = tile[(threadIdx.y + r) * TW + threadIdx.x + r];
	float sum = 0.0f, cnt = 0.0f;
	for (int dxx = 0; dxx < ks; dxx++) {                             // :1251 (x outer)
		const float *col = tile + threadIdx.y * TW + threadIdx.x + dxx;
		const float *wcol = wts + dxx * ks;
#pragma unroll 4
		for (int dyy = 0; dyy < ks; dyy++) {
			const float q = col[dyy * TW];
			if (fabsf(q - c) < alpha2) {                             // :1253
				const float w = wcol[dyy];
				sum = fmaf(q, w, sum);                               // :1254
				cnt += w;                                            // :1255
			}
		}
	}
	out[y * W + x] = sum / cnt;
}

// ------------------------------------------------------------------ Normalize
__global__ void normalize_kernel(const float *__restrict__ in, float *__restrict__ norm, float *__restrict__ out, int C, long HW, long total)
{
	long id = (long)blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= total) return;
	long n = id / HW, p = id % HW;
	const float *src = in + n * C * HW + p;
	float sum = 0.0f;
	for (int c = 0; c < C; c++) {
		float v = src[(long)c * HW];
		sum = fmaf(v, v, sum);                                      // :1294
	}
	float nrm = (float)((double)sum + 1e-5);                        // :1296
	norm[id] = nrm;
	float s = sqrtf(nrm);
	float *dst = out + n * C * HW + p;
	for (int c = 0; c < C; c++) dst[(long)c * HW] = src[(long)c * HW] / s; // :1306
}

__global__ void fill_nan_kernel(float4 *p4, size_t n4, float *tail, int ntail)
{
	size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	const float q = adc_nan();
	for (; i < n4; i += (size_t)gridDim.x * blockDim.x) p4[i] = make_float4(q, q, q, q);
	if (blockIdx.x == 0 && threadIdx.x < ntail) tail[threadIdx.x] = q;
}

// NaN only where StereoJoin writes nothing (main.lua:946 fills everything; the op then overwrites the
// rest): left volume x < d, right volume x >= W - d.  One thread per (d, y, t), t < d.
__global__ void fill_invalid_kernel(float *volL, float *volR, int D, int H, int W, int ld)
{
	const int d = blockIdx.y + 1;                  // d = 0 has no invalid entries
	const int n = min(d, W);
	const long HW = (long)H * ld;
	const float q = adc_nan();
	for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < (long)H * n; i += (long)gridDim.x * blockDim.x) {
		const int y = (int)(i / n), t = (int)(i % n);
		if (volL) volL[d * HW + (long)y * ld + t] = q;
		if (volR) volR[d * HW + (long)y * ld + (W - 1 - t)] = q;
	}
}

__global__ void fix_border_kernel(float *vol, long rows, int W, int ld, int n, int direction)
{
	long r = (long)blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= rows) return;
	float *row = vol + r * ld;
	float v = row[direction > 0 ? n : W - n - 1];
	for (int i = 1; i <= n; i++) row[direction > 0 ? i - 1 : W - i] = v;
}

// out[c][r] = in[r][c] (/ div) for an R x Cn row-major matrix.  LONGROWS selects which of the
// two extents rides on gridDim.x (no 65535 limit): false = columns, true = rows.
template <bool LONGROWS>
__global__ void transpose_kernel(const float *__restrict__ in, float *__restrict__ out, long R, long Cn, float div, bool do_div)
{
	__shared__ float t[32][33];
	long c0 = (long)(LONGROWS ? blockIdx.y : blockIdx.x) * 32;
	long r0 = (long)(LONGROWS ? blockIdx.x : blockIdx.y) * 32;
	for (int j = threadIdx.y; j < 32; j += 8) {
		long r = r0 + j, c = c0 + threadIdx.x;
		if (r < R && c < Cn) t[j][threadIdx.x] = in[r * Cn + c];
	}
	__syncthreads();
	for (int j = threadIdx.y; j < 32; j += 8) {
		long c = c0 + j, r = r0 + threadIdx.x;
		if (r < R && c < Cn) {
			float v = t[threadIdx.x][j];
			out[c * R + r] = do_div ? v / div : v;
		}
	}
}

}  // namespace

#define LAUNCH1D(kernel, n, s, ...)                                                   \
	do {                                                                          \
		kernel<<<adc_div_up((long)(n), 256), 256, 0, (s)>>>(__VA_ARGS__);    \
		ADC_CHECK_LAUNCH();                                                   \
	} while (0)

// 64x64 tile, float4 on both sides (R and Cn multiples of 4, 16-byte aligned bases): each thread moves 4 float4 in
// and 4 float4 out; gridDim.x rides the longer extent.
template <bool LONGROWS>
__global__ void __launch_bounds__(256)
transpose64_kernel(const float *__restrict__ in, float *__restrict__ out, long R, long Cn, float div, bool do_div)
{
	__shared__ float t[64][65];
	const long c0 = (long)(LONGROWS ? blockIdx.y : blockIdx.x) * 64;
	const long r0 = (long)(LONGROWS ? blockIdx.x : blockIdx.y) * 64;
	const int tid = threadIdx.x;
#pragma unroll
	for (int i = 0; i < 4; i++) {
		const int idx = tid + 256 * i, row = idx >> 4, c4 = (idx & 15) * 4;
		if (r0 + row < R && c0 + c4 < Cn) {
			const float4 v = *reinterpret_cast<const float4 *>(in + (r0 + row) * Cn + c0 + c4);
			t[row][c4] = v.x; t[row][c4 + 1] = v.y; t[row][c4 + 2] = v.z; t[row][c4 + 3] = v.w;
		}
	}
	__syncthreads();
#pragma unroll
	for (int i = 0; i < 4; i++) {
		const int idx = tid + 256 * i, c = idx >> 4, r4 = (idx & 15) * 4;
		if (c0 + c < Cn && r0 + r4 < R) {
			float4 v = make_float4(t[r4][c], t[r4 + 1][c], t[r4 + 2][c], t[r4 + 3][c]);
			if (do_div) { v.x /= div; v.y /= div; v.z /= div; v.w /= div; }
			*reinterpret_cast<float4 *>(out + (c0 + c) * R + r0 + r4) = v;
		}
	}
}

// Batched tile transpose between a pitched (D, H, ld) volume and the reference's (H, W, D) SGM layout, one image row
// y = blockIdx.z per grid plane:  B[c][r] = A[r][c] (x scale), A[r][c] = in[r * in_rs + y * in_ys + c],
// B[c][r] = out[c * out_rs + y * out_ys + r].  64 x 64 tiles, float4 on both sides when VEC (the contiguous extents are
// multiples of 4 or padded to it: a pitched row may be read / written up to its pitch).
template <bool VEC>
__global__ void __launch_bounds__(256)
transpose_rows_kernel(const float *__restrict__ in, float *__restrict__ out, int R, int Cn, int Rlim, int Clim,
		      long in_rs, long in_ys, long out_rs, long out_ys, float scale)
{
	__shared__ float t[64][65];
	const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
	const long y = blockIdx.z;
	const int tid = threadIdx.x;
	in += y * in_ys;
	out += y * out_ys;
	if (VEC) {
#pragma unroll
		for (int i = 0; i < 4; i++) {
			const int idx = tid + 256 * i, row = idx >> 4, c4 = (idx & 15) * 4;
			if (r0 + row < R && c0 + c4 < Clim) {
				const float4 v = *reinterpret_cast<const float4 *>(in + (long)(r0 + row) * in_rs + c0 + c4);
				t[row][c4] = v.x; t[row][c4 + 1] = v.y; t[row][c4 + 2] = v.z; t[row][c4 + 3] = v.w;
			}
		}
		__syncthreads();
#pragma unroll
		for (int i = 0; i < 4; i++) {
			const int idx = tid + 256 * i, c = idx >> 4, r4 = (idx & 15) * 4;
			if (c0 + c < Cn && r0 + r4 < Rlim) {
				float4 v = make_float4(t[r4][c], t[r4 + 1][c], t[r4 + 2][c], t[r4 + 3][c]);
				v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
				*reinterpret_cast<float4 *>(out + (long)(c0 + c) * out_rs + r0 + r4) = v;
			}
		}
	} else {
		for (int i = tid; i < 64 * 64; i += 256) {
			const int row = i >> 6, c = i & 63;
			if (r0 + row < R && c0 + c < Cn) t[row][c] = in[(long)(r0 + row) * in_rs + c0 + c];
		}
		__syncthreads();
		for (int i = tid; i < 64 * 64; i += 256) {
			const int c = i >> 6, r = i & 63;
			if (c0 + c < Cn && r0 + r < R) out[(long)(c0 + c) * out_rs + r0 + r] = t[r][c] * scale;
		}
	}
}

// (D, H, ld) -> (H, W, D)   main.lua:1008 on the pipeline's pitched volumes
int adc_transpose_dhw_pitched_to_hwd(const float *in, float *out, int D, int H, int W, int ld, cudaStream_t s)
{
	if (H > 65535) return ADCENSUS_ELIMIT;
	const bool vec = (D % 4 == 0) && (ld % 4 == 0) && ((((uintptr_t)in) | ((uintptr_t)out)) % 16 == 0);
	dim3 grid(adc_div_up(W, 64), adc_div_up(D, 64), H);
	const int clim = vec ? ((W + 3) & ~3) : W;     // reads may run into the row padding
	if (vec) transpose_rows_kernel<true><<<grid, 256, 0, s>>>(in, out, D, W, D, clim, (long)H * ld, ld, D, (long)W * D, 1.0f);
	else transpose_rows_kernel<false><<<grid, 256, 0, s>>>(in, out, D, W, D, W, (long)H * ld, ld, D, (long)W * D, 1.0f);
	ADC_CHECK_LAUNCH();
	return 0;
}

// (H, W, D) -> (D, H, ld), x 1/4   main.lua:1017-1020 (x * 0.25f is exactly x / 4)
int adc_transpose_hwd_to_dhw_pitched_div4(const float *in, float *out, int D, int H, int W, int ld, cudaStream_t s)
{
	if (H > 65535) return ADCENSUS_ELIMIT;
	const bool vec = (D % 4 == 0) && (ld % 4 == 0) && ld >= ((W + 3) & ~3) && ((((uintptr_t)in) | ((uintptr_t)out)) % 16 == 0);
	dim3 grid(adc_div_up(D, 64), adc_div_up(W, 64), H);
	const int rlim = vec ? ((W + 3) & ~3) : W;     // writes may run into the row padding
	if (vec) transpose_rows_kernel<true><<<grid, 256, 0, s>>>(in, out, W, D, rlim, D, D, (long)W * D, (long)H * ld, ld, 0.25f);
	else transpose_rows_kernel<false><<<grid, 256, 0, s>>>(in, out, W, D, W, D, D, (long)W * D, (long)H * ld, ld, 0.25f);
	ADC_CHECK_LAUNCH();
	return 0;
}

static int adc_transpose(const float *in, float *out, long R, long Cn, float div, bool do_div, cudaStream_t s)
{
	const bool vec = (R % 4 == 0) && (Cn % 4 == 0) && ((((uintptr_t)in) | ((uintptr_t)out)) % 16 == 0);
	const int tile = vec ? 64 : 32;
	dim3 block = vec ? dim3(256) : dim3(32, 8);
	if (R >= Cn) {
		dim3 grid(adc_div_up(R, tile), adc_div_up(Cn, tile));
		if (grid.y > 65535) return ADCENSUS_ELIMIT;
		if (vec) transpose64_kernel<true><<<grid, block, 0, s>>>(in, out, R, Cn, div, do_div);
		else transpose_kernel<true><<<grid, block, 0, s>>>(in, out, R, Cn, div, do_div);
	} else {
		dim3 grid(adc_div_up(Cn, tile), adc_div_up(R, tile));
		if (grid.y > 65535) return ADCENSUS_ELIMIT;
		if (vec) transpose64_kernel<false><<<grid, block, 0, s>>>(in, out, R, Cn, div, do_div);
		else transpose_kernel<false><<<grid, block, 0, s>>>(in, out, R, Cn, div, do_div);
	}
	ADC_CHECK_LAUNCH();
	return 0;
}

// first minimum over D of a pitched (D, H, ld) volume, 0-based, NaN skipped (main.lua:1049-1050; strict <, init +inf
// like spatial_argmin, adcensus.cu:251-259)
__global__ void argmin_pitched_kernel(const float *__restrict__ vol, float *__restrict__ out, int D, int H, int W, int ld)
{
	const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
	if (x >= W) return;
	const long HW = (long)H * ld;
	const float *v = vol + (long)y * ld + x;
	int arg = 0;
	float mn = CUDART_INF_F;
	int d = 0;
	for (; d + 4 <= D; d += 4) {
		float a = ld_stream(v + (long)d * HW), b = ld_stream(v + (long)(d + 1) * HW);
		float c = ld_stream(v + (long)(d + 2) * HW), e = ld_stream(v + (long)(d + 3) * HW);
		if (a < mn) { mn = a; arg = d; }
		if (b < mn) { mn = b; arg = d + 1; }
		if (c < mn) { mn = c; arg = d + 2; }
		if (e < mn) { mn = e; arg = d + 3; }
	}
	for (; d < D; d++) {
		float a = ld_stream(v + (long)d * HW);
		if (a < mn) { mn = a; arg = d; }
	}
	out[(long)y * W + x] = (float)arg;
}

// ---- pitched (D, H, ld) forms used by the fused pipeline (ld == W: the API-facing contiguous tensors) ----
int adc_argmin_pitched(const float *vol, float *disp, int D, int H, int W, int ld, cudaStream_t s)
{
	if (!vol || !disp || D < 1 || H < 1 || W < 1 || ld < W || H > 65535) return ADCENSUS_EINVAL;
	dim3 grid(adc_div_up(W, 128), H);
	argmin_pitched_kernel<<<grid, 128, 0, s>>>(vol, disp, D, H, W, ld);
	ADC_CHECK_LAUNCH();
	return 0;
}

int adc_subpixel(const float *d0, const float *c2, float *out, int H, int W, int ld, int disp_max, cudaStream_t s)
{
	if (!d0 || !c2 || !out || H < 1 || W < 1 || ld < W || disp_max < 1) return ADCENSUS_EINVAL;
	LAUNCH1D(subpixel_kernel, H * W, s, d0, c2, out, H * W, H, W, ld, disp_max);
	return 0;
}

int adc_fill_invalid(float *volL, float *volR, int D, int H, int W, int ld, cudaStream_t s)
{
	if ((!volL && !volR) || D < 1 || H < 1 || W < 1 || ld < W) return ADCENSUS_EINVAL;   // one of the two may be NULL (skipped)
	if (D == 1) return 0;
	dim3 grid(8, D - 1);
	fill_invalid_kernel<<<grid, 256, 0, s>>>(volL, volR, D, H, W, ld);
	ADC_CHECK_LAUNCH();
	return 0;
}

int adc_fix_border(float *vol, int D, int H, int W, int ld, int n, int direction, cudaStream_t s)
{
	if (!vol || D < 1 || H < 1 || W < 1 || ld < W || n < 0 || n + 1 > W || (direction != 1 && direction != -1)) return ADCENSUS_EINVAL;
	if (n == 0) return 0;
	long rows = (long)D * H;
	LAUNCH1D(fix_border_kernel, rows, s, vol, rows, W, ld, n, direction);
	return 0;
}

extern "C" {

int adcensus_spatial_argmin(const float *input, float *output, int N, int D, int HW, adcensus_stream_t stream)
{
	if (!input || !output || N < 1 || D < 1 || HW < 1) return ADCENSUS_EINVAL;
	long total = (long)N * HW;
	LAUNCH1D(argmin_kernel, total, adc_stream(stream), input, output, D, (long)HW, total, 1.0f);
	return 0;
}

int mccnn_argmin(const float *vol, float *disp, int D, int HW, adcensus_stream_t stream)
{
	if (!vol || !disp || D < 1 || HW < 1) return ADCENSUS_EINVAL;
	LAUNCH1D(argmin_kernel, HW, adc_stream(stream), vol, disp, D, (long)HW, (long)HW, 0.0f);
	return 0;
}

int adcensus_outlier_detection(const float *d0, const float *d1, float *outlier, int H, int W, int disp_max, adcensus_stream_t stream)
{
	if (!d0 || !d1 || !outlier || H < 1 || W < 1 || disp_max < 0) return ADCENSUS_EINVAL;
	LAUNCH1D(outlier_kernel, H * W, adc_stream(stream), d0, d1, outlier, H * W, W, disp_max);
	return 0;
}

int adcensus_interpolate_occlusion(const float *d0, const float *outlier, float *out, int H, int W, adcensus_stream_t stream)
{
	if (!d0 || !outlier || !out || H < 1 || W < 1) return ADCENSUS_EINVAL;
	const size_t smem = 3 * (size_t)W * sizeof(int);
	if (smem <= 48 * 1024) {
		interp_occ_row_kernel<<<H, 128, smem, adc_stream(stream)>>>(d0, outlier, out, W);
		ADC_CHECK_LAUNCH();
	} else {
		LAUNCH1D(interp_occ_kernel, H * W, adc_stream(stream), d0, outlier, out, H * W, W);
	}
	return 0;
}

int adcensus_interpolate_mismatch(const float *d0, const float *outlier, float *out, int H, int W, adcensus_stream_t stream)
{
	if (!d0 || !outlier || !out || H < 1 || W < 1) return ADCENSUS_EINVAL;
	LAUNCH1D(interp_mis_kernel, H * W, adc_stream(stream), d0, outlier, out, H * W, H, W);
	return 0;
}

int adcensus_subpixel_enchancement(const float *d0, const float *c2, float *out, int H, int W, int disp_max, adcensus_stream_t stream)
{
	return adc_subpixel(d0, c2, out, H, W, W, disp_max, adc_stream(stream));
}

int adcensus_median2d(const float *img, float *out, int H, int W, int kernel_size, adcensus_stream_t stream)
{
	if (!img || !out || H < 1 || W < 1 || kernel_size < 1 || kernel_size % 2 != 1) return ADCENSUS_EINVAL;
	if (kernel_size > ADCENSUS_MAX_MEDIAN) return ADCENSUS_ELIMIT;  // adcensus.cu:1602
	if (kernel_size == 5) LAUNCH1D(median5_kernel, H * W, adc_stream(stream), img, out, H * W, H, W);
	else LAUNCH1D(median_kernel, H * W, adc_stream(stream), img, out, H * W, H, W, kernel_size / 2);
	return 0;
}

int adcensus_mean2d(const float *img, const float *kernel, float *out, int H, int W, int ksize, float alpha2, adcensus_stream_t stream)
{
	if (!img || !kernel || !out || H < 1 || W < 1 || ksize < 1 || ksize % 2 != 1) return ADCENSUS_EINVAL;  // :1269
	const int r = ksize / 2;
	const size_t smem = ((size_t)(M2_TY + 2 * r) * (M2_TX + 2 * r) + (size_t)ksize * ksize) * sizeof(float);
	if (smem <= 200 * 1024) {
		if (smem > 48 * 1024) {
			ADC_CUDA(cudaFuncSetAttribute(mean2d_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		}
		dim3 grid(adc_div_up(W, M2_TX), adc_div_up(H, M2_TY)), block(M2_TX, M2_TY);
		mean2d_tile_kernel<<<grid, block, smem, adc_stream(stream)>>>(img, kernel, out, r, H, W, alpha2);
		ADC_CHECK_LAUNCH();
	} else {
		LAUNCH1D(mean2d_kernel, H * W, adc_stream(stream), img, kernel, out, H * W, r, H, W, alpha2);
	}
	return 0;
}

int adcensus_Normalize_forward(const float *input, float *norm, float *output, int N, int C, int H, int W, adcensus_stream_t stream)
{
	if (!input || !norm || !output || N < 1 || C < 1 || H < 1 || W < 1) return ADCENSUS_EINVAL;
	long HW = (long)H * W, total = N * HW;
	LAUNCH1D(normalize_kernel, total, adc_stream(stream), input, norm, output, C, HW, total);
	return 0;
}

int mccnn_fill_nan(float *p, size_t n, adcensus_stream_t stream)
{
	if (!p) return ADCENSUS_EINVAL;
	if (n == 0) return 0;
	// align to 16 bytes for the float4 body
	size_t head = ((16 - ((uintptr_t)p & 15)) & 15) / 4;
	if (head > n) head = n;
	cudaStream_t s = adc_stream(stream);
	if (head) {
		fill_nan_kernel<<<1, 32, 0, s>>>(nullptr, 0, p, (int)head);
		ADC_CHECK_LAUNCH();
	}
	size_t n4 = (n - head) / 4;
	int tail = (int)((n - head) % 4);
	if (n4 || tail) {
		int blocks = (int)((n4 + 255) / 256);
		int cap = adc_num_sms() * 16;
		if (blocks > cap) blocks = cap;
		if (blocks < 1) blocks = 1;
		fill_nan_kernel<<<blocks, 256, 0, s>>>((float4 *)(p + head), n4, p + head + 4 * n4, tail);
		ADC_CHECK_LAUNCH();
	}
	return 0;
}

int mccnn_fill_invalid(float *volL, float *volR, int D, int H, int W, adcensus_stream_t stream)
{
	if (!volL || !volR) return ADCENSUS_EINVAL;
	return adc_fill_invalid(volL, volR, D, H, W, W, adc_stream(stream));
}

int mccnn_fix_border(float *vol, int D, int H, int W, int n, int direction, adcensus_stream_t stream)
{
	return adc_fix_border(vol, D, H, W, W, n, direction, adc_stream(stream));
}

int mccnn_transpose_dhw_to_hwd(const float *in, float *out, int D, int H, int W, adcensus_stream_t stream)
{
	if (!in || !out || in == out || D < 1 || H < 1 || W < 1) return ADCENSUS_EINVAL;
	return adc_transpose(in, out, D, (long)H * W, 1.0f, false, adc_stream(stream));
}

int mccnn_transpose_hwd_to_dhw_div4(const float *in, float *out, int D, int H, int W, adcensus_stream_t stream)
{
	if (!in || !out || in == out || D < 1 || H < 1 || W < 1) return ADCENSUS_EINVAL;
	return adc_transpose(in, out, (long)H * W, D, 4.0f, true, adc_stream(stream));  // exact: x / 4
}

/* pitched (D, H, ld) forms of the Lua-side tensor ops, as the fused pipeline runs them */
int mccnn_transpose_dhw_pitched_to_hwd(const float *in, float *out, int D, int H, int W, int ld, adcensus_stream_t stream)
{
	if (!in || !out || in == out || D < 1 || H < 1 || W < 1 || ld < W) return ADCENSUS_EINVAL;
	return adc_transpose_dhw_pitched_to_hwd(in, out, D, H, W, ld, adc_stream(stream));
}

int mccnn_transpose_hwd_to_dhw_pitched_div4(const float *in, float *out, int D, int H, int W, int ld, adcensus_stream_t stream)
{
	if (!in || !out || in == out || D < 1 || H < 1 || W < 1 || ld < W) return ADCENSUS_EINVAL;
	return adc_transpose_hwd_to_dhw_pitched_div4(in, out, D, H, W, ld, adc_stream(stream));
}

int mccnn_argmin_pitched(const float *vol, float *disp, int D, int H, int W, int ld, adcensus_stream_t stream)
{
	return adc_argmin_pitched(vol, disp, D, H, W, ld, adc_stream(stream));
}

int mccnn_gaussian(double sigma, float *out_host)
{
	// main.lua:528-540, computed in double like Lua numbers, stored as float (:cuda())
	int kr = (int)ceil(sigma * 3);
	int ks = kr * 2 + 1;
	if (out_host)
		for (int i = 0; i < ks; i++)
			for (int j = 0; j < ks; j++) {
				int y = i - kr, x = j - kr;
				out_host[i * ks + j] = (float)exp(-(double)(x * x + y * y) / (2 * sigma * sigma));
			}
	return ks;
}

}  // extern "C"
