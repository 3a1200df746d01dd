// stereo_join.cu -- adcensus.StereoJoin for sm_100a.
//
// Replaces adcensus.cu:1455-1498 (kernel StereoJoin_, one thread per pixel with a
// 512-byte local-memory L cache and C*D scalar R loads).  Per image row the op is
// a banded GEMM,  cost[x][j] = -sum_c L[c][x] * R[c][j]  for 0 <= x - j < D, and it
// is built like one:
//   * a CTA owns (row y, 128 columns x, a chunk of DC = 16*NS - 8 disparities).  In
//     (x, j = x - d) space that chunk is a parallelogram; it is covered by 8x x 16j
//     register tiles laid along the diagonal (16 x-groups, NS tiles each, 6% of the
//     tile entries fall outside the band and are discarded), so the inner loop is a
//     plain outer product: per channel 2 LDS.128 of L + 4 LDS.128 of R for 128 FMAs (64 FFMA2);
//   * operands are stored in shared memory "split-plane" (the low and the high float4
//     of every 8-float group in separate planes), which makes every quarter-warp of
//     an LDS.128 read 128 contiguous bytes: no bank conflicts (the naive layout is
//     2-way conflicted and was shared-memory bound at 16% FMA utilisation);
//   * channel slabs (8 channels x [128 L | 256 R]) stream through a 3-stage cp.async
//     ring, one barrier per slab;
//   * accumulation is the reference's (c ascending, one fused multiply-add per
//     channel into a single accumulator, adcensus.cu:1468-1471) => bit-identical;
//   * the finished tile is staged through shared memory (written along tile
//     diagonals = runs of consecutive x at fixed d) so that both volumes are written
//     as full rows: outL[d][y][x0..] and outR[d][y][x0-d..] are the same 128 floats.
//
// Roofline: 2*C*H*W*4 bytes read + 2*valid*4 bytes written (valid = H*(D*W -
// D(D-1)/2)); at C=64 the FMA work (2*C flop per output) sits at the fp32 ridge
// of the chip, so the kernel is tuned like a GEMM and reported against HBM.
#include <string.h>

#include "internal.cuh"

namespace {

constexpr int SJ_TX = 128;      // x per CTA (16 groups of 8)
constexpr int SJ_CCH = 8;       // channels per pipeline stage
constexpr int SJ_NSTAGE = 3;
constexpr int SJ_ROW = SJ_TX + 2 * SJ_TX;   // floats per channel row: [L 128][R 256]

__device__ __forceinline__ unsigned long long sj_pack2(float lo, float hi)
{
	unsigned long long r;
	asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
	return r;
}
__device__ __forceinline__ void sj_unpack2(unsigned long long v, float &lo, float &hi)
{
	asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long sj_fma2(unsigned long long a, unsigned long long b, unsigned long long c)
{
	unsigned long long d;
	asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
	return d;
}

template <int NS>
struct SJCfg {
	static constexpr int DC = 16 * NS - 8;          // disparities per CTA
	static constexpr int NT = 16 * NS;              // threads
	static constexpr int STAGE = SJ_CCH * SJ_ROW;   // floats
	static constexpr int SMEM_PIPE = SJ_NSTAGE * STAGE * 4;
	static constexpr int SMEM_OUT = DC * SJ_TX * 4;
	static constexpr int SMEM = SMEM_PIPE > SMEM_OUT ? SMEM_PIPE : SMEM_OUT;
};

// split-plane position of element i of a row of NG 8-float groups
__device__ __forceinline__ int split_pos(int i, int NG) { return ((i & 7) >> 2) * (NG * 4) + (i >> 3) * 4 + (i & 3); }

// FASTIO (W even, 8-byte aligned feature bases, outputs pitched with ldo % 4 == 0 and 16-byte aligned):
//   * operand slabs arrive by 8-byte cp.async (feature rows of an even W start on 8-byte boundaries; 16 bytes are
//     not available at W = 1226, which also rules out TMA for the loads: its innermost start must be 16-byte
//     aligned), source pointers advance by one channel plane per copy instead of being recomputed;
//   * the finished tile is staged DENSE in shared memory and the left volume leaves as ONE TMA store of the box
//     {128 x, 1 row, DC disparities} (entries with x < d are set to NaN first: the store then also does the fill of
//     main.lua:946 for the left volume); the right volume's rows start at x0 - d, which is not 16-byte aligned in
//     general, so they are written by the threads as aligned float4.
// The disparity chunk is shifted by one (DTOP) so that the R window starts on an even column.
template <int NS, bool FASTIO>
__global__ void __launch_bounds__(16 * NS, (NS >= 6) ? 3 : 4)
stereo_join_kernel(const __grid_constant__ CUtensorMap tmL, const float *__restrict__ gL, const float *__restrict__ gR,
		   float *__restrict__ outL, float *__restrict__ outR,
		   int C, int D, int H, int W, int ldo)
{
	using Cfg = SJCfg<NS>;
	constexpr int DC = Cfg::DC, NT = Cfg::NT;
	constexpr int DTOP = FASTIO ? DC : DC - 1;           // d - d0 of the tile diagonal xi - ji = 0 at s = 0
	extern __shared__ __align__(128) float smem[];

	const int tid = threadIdx.x;
	const int gx = (tid & 7) + 8 * ((tid >> 3) & 1);    // x group (8 columns); a quarter-warp = 8 consecutive groups
	const int s = tid >> 4;                              // tile index along the diagonal, 0..NS-1
	const int X0 = blockIdx.x * SJ_TX;
	const int y = blockIdx.y;
	const int d0 = blockIdx.z * DC;
	const long HW = (long)H * W;
	const int jbase = X0 - d0 - DTOP;                    // image column of R-window slot 0 (even when FASTIO)

	// ---- fill slots: fixed columns of the channel row per thread -----------------------------
	constexpr int GR = FASTIO ? 2 : 1;                   // floats per copy
	constexpr int NSLOT = (SJ_ROW / GR + NT - 1) / NT;
	const float *src[NSLOT];
	int dst[NSLOT];
	bool ok[NSLOT];
#pragma unroll
	for (int m = 0; m < NSLOT; m++) {
		const int col = (tid + m * NT) * GR;
		const bool isL = col < SJ_TX;
		const int li = isL ? col : col - SJ_TX;          // logical index inside the L row / R window
		const int xc = isL ? X0 + li : jbase + li;       // image column (even when FASTIO: the pair is inside or outside as a whole)
		ok[m] = col < SJ_ROW && xc >= 0 && xc < W;
		src[m] = (isL ? gL : gR) + (long)y * W + (ok[m] ? xc : 0);
		dst[m] = col < SJ_ROW ? (isL ? split_pos(li, 16) : SJ_TX + split_pos(li, 32)) : -1;
	}
	auto issue_stage = [&](int stage_idx, int buf) {
		float *sb = smem + buf * Cfg::STAGE;
		const int c0 = stage_idx * SJ_CCH;
		const float *q[NSLOT];
#pragma unroll
		for (int m = 0; m < NSLOT; m++) q[m] = src[m] + (long)c0 * HW;
#pragma unroll
		for (int cc = 0; cc < SJ_CCH; cc++) {
			const bool cok = c0 + cc < C;
#pragma unroll
			for (int m = 0; m < NSLOT; m++) {
				if (dst[m] >= 0) {
					const unsigned sa = (unsigned)__cvta_generic_to_shared(sb + cc * SJ_ROW + dst[m]);
					const int nbytes = (ok[m] && cok) ? 4 * GR : 0;   // zero-fill outside the image / beyond C
					if (FASTIO)
						asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa), "l"(cok ? q[m] : src[m]), "r"(nbytes));
					else
						asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(sa), "l"(cok ? q[m] : src[m]), "r"(nbytes));
				}
				q[m] += HW;
			}
		}
	};

	// accumulators as packed pairs (ji = 2m, 2m+1) for FFMA2 (fma.rn.f32x2: two independent IEEE
	// fmas per instruction, the pair of R values times one broadcast -L value)
	unsigned long long acc2[8][8];
#pragma unroll
	for (int i = 0; i < 8; i++)
#pragma unroll
		for (int j = 0; j < 8; j++) acc2[i][j] = sj_pack2(0.0f, 0.0f);

	// this tile's disparities: d - d0 = DTOP - 16 s + xi - ji
	const int dtop = d0 + DTOP - 16 * s;                 // d at (xi - ji) = 0
	const bool active = (dtop - 15 < D) && (dtop - 15 < d0 + DC) && (dtop + 7 >= d0);
	const int lofs = gx * 4;                             // float4 slot of this x group in the L planes
	const int rofs = SJ_TX + (gx + 2 * s) * 4;           // first 8-float group of the 16 R columns

	const int nstage = (C + SJ_CCH - 1) / SJ_CCH;
#pragma unroll
	for (int p = 0; p < SJ_NSTAGE - 1; p++) {
		if (p < nstage) issue_stage(p, p);
		asm volatile("cp.async.commit_group;");
	}
	for (int st = 0; st < nstage; st++) {
		asm volatile("cp.async.wait_group %0;" ::"n"(SJ_NSTAGE - 2));
		__syncthreads();                                 // slab st visible; slab st-1's buffer free
		if (st + SJ_NSTAGE - 1 < nstage) issue_stage(st + SJ_NSTAGE - 1, (st + SJ_NSTAGE - 1) % SJ_NSTAGE);
		asm volatile("cp.async.commit_group;");
		if (active) {
			const float *sb = smem + (st % SJ_NSTAGE) * Cfg::STAGE;
#pragma unroll
			for (int cc = 0; cc < SJ_CCH; cc++) {
				const float *row = sb + cc * SJ_ROW;
				float l[8], r[16];
				*reinterpret_cast<float4 *>(&l[0]) = *reinterpret_cast<const float4 *>(row + lofs);
				*reinterpret_cast<float4 *>(&l[4]) = *reinterpret_cast<const float4 *>(row + 64 + lofs);
				*reinterpret_cast<float4 *>(&r[0]) = *reinterpret_cast<const float4 *>(row + rofs);
				*reinterpret_cast<float4 *>(&r[4]) = *reinterpret_cast<const float4 *>(row + 128 + rofs);
				*reinterpret_cast<float4 *>(&r[8]) = *reinterpret_cast<const float4 *>(row + rofs + 4);
				*reinterpret_cast<float4 *>(&r[12]) = *reinterpret_cast<const float4 *>(row + 128 + rofs + 4);
				unsigned long long r2[8];
#pragma unroll
				for (int m = 0; m < 8; m++) r2[m] = sj_pack2(r[2 * m], r[2 * m + 1]);
#pragma unroll
				for (int xi = 0; xi < 8; xi++) {
					const unsigned long long nl = sj_pack2(-l[xi], -l[xi]);
#pragma unroll
					for (int m = 0; m < 8; m++) acc2[xi][m] = sj_fma2(r2[m], nl, acc2[xi][m]);  // adcensus.cu:1470: sum -= l * r
				}
			}
		}
	}
	asm volatile("cp.async.wait_group 0;");
	__syncthreads();                                     // pipeline buffers are reused as the output stage
	float acc[8][16];
#pragma unroll
	for (int i = 0; i < 8; i++)
#pragma unroll
		for (int m = 0; m < 8; m++) sj_unpack2(acc2[i][m], acc[i][2 * m], acc[i][2 * m + 1]);

	// ---- epilogue 1: tile diagonals (fixed d, consecutive x) -> so[dd][x] (split-plane, or dense for FASTIO) ----
	float *so = smem;
#pragma unroll
	for (int t = -15; t <= 7; t++) {                     // t = xi - ji
		const int dd = DTOP - 16 * s + t;                // d - d0
		if (dd < 0 || dd >= DC) continue;
		float *rowp = so + dd * SJ_TX + (FASTIO ? gx * 8 : gx * 4);
#pragma unroll
		for (int h = 0; h < 2; h++) {                    // halves xi = 4h .. 4h+3
			float *hp = rowp + (FASTIO ? h * 4 : h * 64);
			const bool full = (4 * h - t >= 0) && (4 * h + 3 - t <= 15);
			if (full) {
				*reinterpret_cast<float4 *>(hp) =
					make_float4(acc[4 * h][4 * h - t], acc[4 * h + 1][4 * h + 1 - t],
						    acc[4 * h + 2][4 * h + 2 - t], acc[4 * h + 3][4 * h + 3 - t]);
			} else {
#pragma unroll
				for (int e = 0; e < 4; e++) {
					const int xi = 4 * h + e, ji = xi - t;
					if (ji >= 0 && ji <= 15) hp[e] = acc[xi][ji];
				}
			}
		}
	}
	if (FASTIO) fence_proxy_async_smem();                // generic-proxy writes of `so` before the async-proxy (TMA) read
	__syncthreads();

	const int nrows = min(DC, D - d0);
	if constexpr (FASTIO) {
		// ---- epilogue 2 (pitched outputs): left volume = one TMA store, right volume = aligned float4 rows ----
		if (X0 < d0 + DC || X0 + SJ_TX > W) {            // this tile holds entries with x < d or x >= W: they become NaN
			const float q = adc_nan();
			for (int idx = tid; idx < DC * SJ_TX; idx += NT) {
				const int r = idx >> 7, x = X0 + (idx & (SJ_TX - 1));
				if (x < d0 + r || x >= W) so[idx] = q;
			}
			fence_proxy_async_smem();
			__syncthreads();
		}
		if (tid == 0) {
			tma_store_3d(&tmL, so, X0, y, d0);           // outL[d0 .. d0+DC) x row y x [X0, X0+128): clipped at D and W (adcensus.cu:1472)
			tma_store_commit();
		}
		// outR[d][y][x - d] = so[d - d0][x - X0] (adcensus.cu:1473); a row's 128 values span 33 aligned float4 groups
		for (int idx = tid; idx < nrows * 33; idx += NT) {
			const int r = idx / 33, g = idx - r * 33;
			const int d = d0 + r;
			const int q0 = (X0 - d) & ~3;                // first aligned column group touching the row (may be negative)
			const int xp = q0 + 4 * g;                   // output columns xp .. xp+3
			const int xl = xp + d - X0;                  // their tile columns xl .. xl+3 (xl >= -3)
			const float *row = so + r * SJ_TX;
			float v[4];
			bool w[4];
#pragma unroll
			for (int e = 0; e < 4; e++) {
				const int t = xl + e;
				w[e] = t >= 0 && t < SJ_TX && xp + e >= 0 && X0 + t < W;     // inside the tile, x - d >= 0, x < W
				v[e] = w[e] ? row[t] : 0.0f;
			}
			float *dstp = outR + ((long)d * H + y) * ldo + xp;
			if (w[0] && w[1] && w[2] && w[3]) {
				*reinterpret_cast<float4 *>(dstp) = make_float4(v[0], v[1], v[2], v[3]);
			} else {
#pragma unroll
				for (int e = 0; e < 4; e++)
					if (w[e]) dstp[e] = v[e];
			}
		}
		if (tid == 0) tma_store_wait_read();             // the bulk store has read shared memory before the CTA retires
	} else {
		// ---- epilogue 2: full rows of both volumes ------------------------------------------------
		// (NT need not be a multiple of 32: index by thread, consecutive threads -> consecutive x)
		for (int idx = tid; idx < nrows * SJ_TX; idx += NT) {
			const int r = idx >> 7, xl = idx & (SJ_TX - 1);
			const int d = d0 + r;
			const int x = X0 + xl;
			if (x < W && x >= d) {
				const float v = so[r * SJ_TX + split_pos(xl, 16)];
				const long rowbase = ((long)d * H + y) * ldo;   // outputs are (D, H, ldo), ldo >= W
				outL[rowbase + x] = v;       // adcensus.cu:1472
				outR[rowbase + x - d] = v;   // adcensus.cu:1473
			}
		}
	}
}

template <int NS, bool FASTIO>
int launch(const CUtensorMap &tmL, const float *L, const float *R, float *outL, float *outR, int C, int D, int H, int W, int ldo, cudaStream_t s)
{
	using Cfg = SJCfg<NS>;
	static bool attr_done[64] = {false};
	int dev = 0;
	cudaGetDevice(&dev);
	if (!attr_done[dev & 63]) {
		ADC_CUDA(cudaFuncSetAttribute(stereo_join_kernel<NS, FASTIO>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
		attr_done[dev & 63] = true;
	}
	dim3 grid(adc_div_up(W, SJ_TX), H, adc_div_up(D, Cfg::DC));
	stereo_join_kernel<NS, FASTIO><<<grid, Cfg::NT, Cfg::SMEM, s>>>(tmL, L, R, outL, outR, C, D, H, W, ldo);
	ADC_CHECK_LAUNCH();
	return 0;
}

template <bool FASTIO>
int dispatch(int ns, const CUtensorMap &tmL, const float *L, const float *R, float *outL, float *outR, int C, int D, int H, int W, int ldo,
	     cudaStream_t s)
{
	switch (ns) {
	case 1: return launch<1, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	case 2: return launch<2, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	case 3: return launch<3, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	case 4: return launch<4, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	case 5: return launch<5, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	case 6: return launch<6, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	case 7: return launch<7, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	default: return launch<8, FASTIO>(tmL, L, R, outL, outR, C, D, H, W, ldo, s);
	}
}

// D split into equal chunks of at most 120; the smallest tile count that covers one
int sj_ns(int D)
{
	const int nchunk = adc_div_up(D, 120);
	const int dc = adc_div_up(D, nchunk);
	return adc_div_up(dc + 8, 16);
}

}  // namespace

// outputs (D, H, ldo) with row pitch ldo >= W (the fused pipeline's private volumes); features (C, H, W) contiguous.
// The fast load / store path needs W even, 8-byte aligned features and 16-byte aligned outputs with ldo % 4 == 0; it
// writes NaN into the left volume's entries x < d (no separate fill needed there; hence opt-in through `fast`: the
// operator itself leaves them untouched, adcensus.cu:1467) and leaves the right volume's invalid entries untouched.
static int adc_stereo_join_fast_ok(const float *input_L, const float *input_R, const float *output_L, const float *output_R, int W, int ldo)
{
	return (W % 2 == 0) && (ldo % 4 == 0) && ((((uintptr_t)input_L) | ((uintptr_t)input_R)) % 8 == 0) &&
	       ((((uintptr_t)output_L) | ((uintptr_t)output_R)) % 16 == 0);
}

int adc_stereo_join(const float *input_L, const float *input_R, float *output_L, float *output_R,
		    int C, int D, int H, int W, int ldo, int fast, cudaStream_t s)
{
	if (!input_L || !input_R || !output_L || !output_R) return ADCENSUS_EINVAL;
	if (C < 1 || D < 1 || H < 1 || W < 1 || H > 65535 || ldo < W) return ADCENSUS_EINVAL;
	if (C > 128) return ADCENSUS_ELIMIT;  // reference: float L_cache[128] (adcensus.cu:1460-1461)
	const int ns = sj_ns(D);
	if (!fast && adc_stereo_join_tma_ok(input_L, input_R, output_L, output_R, H, W) && (ldo % 4 == 0 || ldo == W))
		return adc_stereo_join_tma(input_L, input_R, output_L, output_R, C, D, H, W, ldo, ns, s);
	if (fast && adc_stereo_join_fast_ok(input_L, input_R, output_L, output_R, W, ldo)) {
		CUtensorMap tmL;
		const uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)D};
		const uint64_t strides[2] = {(uint64_t)ldo * 4, (uint64_t)ldo * 4 * (uint64_t)H};
		const uint32_t box[3] = {(uint32_t)SJ_TX, 1u, (uint32_t)(16 * ns - 8)};
		int rc = adc_tma_encode(&tmL, output_L, 3, dims, strides, box);
		if (rc) return rc;
		return dispatch<true>(ns, tmL, input_L, input_R, output_L, output_R, C, D, H, W, ldo, s);
	}
	CUtensorMap dummy;
	memset(&dummy, 0, sizeof(dummy));
	return dispatch<false>(ns, dummy, input_L, input_R, output_L, output_R, C, D, H, W, ldo, s);
}

extern "C" int adcensus_StereoJoin(const float *input_L, const float *input_R, float *output_L, float *output_R,
				   int C, int D, int H, int W, adcensus_stream_t stream)
{
	return adc_stereo_join(input_L, input_R, output_L, output_R, C, D, H, W, W, /*fast=*/0, adc_stream(stream));
}

// StereoJoin into pitched (D, H, ld) volumes (the fused pipeline's private layout).  Unlike the operator above this
// form also performs the fill of main.lua:946 for the LEFT volume (entries x < d become NaN); the right volume's
// invalid entries (x >= W - d) are left untouched, the caller fills them (mccnn_fill_invalid / adc_fill_invalid).
extern "C" int mccnn_stereo_join_pitched(const float *input_L, const float *input_R, float *output_L, float *output_R,
					 int C, int D, int H, int W, int ld, adcensus_stream_t stream)
{
	if (!input_L || !input_R || !output_L || !output_R || ld < W) return ADCENSUS_EINVAL;
	if (!adc_stereo_join_fast_ok(input_L, input_R, output_L, output_R, W, ld)) return ADCENSUS_EINVAL;
	return adc_stereo_join(input_L, input_R, output_L, output_R, C, D, H, W, ld, /*fast=*/1, adc_stream(stream));
}
