// stereo_join_tma.cu -- adcensus.StereoJoin (adcensus.cu:1455-1498), second generation: TMA-staged feature rows.
//
// Same mathematics and the same diagonal 8x x 16j register tiles as stereo_join.cu (banded GEMM per image row,
// cost[x][j] = -sum_c L[c][x] R[c][j] for 0 <= x - j < D, c ascending into ONE accumulator per output => bit-identical
// to the reference's adcensus.cu:1466-1475), but the operand slabs no longer arrive as 16 predicated 4-/8-byte cp.async per
// thread and stage with their address arithmetic:
//   * the features are a legal 2-D tensor (H*W, C) for TMA when H*W is a multiple of 4 (row stride = a multiple of
//     16 bytes).  What is NOT aligned is the start of an image row (W = 1226: 8 bytes) -- so the tile origin is shifted
//     per row: a CTA owns the 128 columns starting at X0 = 128 bx - ((y W) mod 4), which makes the FLAT index y W + X0 a
//     multiple of 4, and the disparity chunk is anchored so that the right window starts on a multiple of 4 too.  Columns
//     that fall outside the image row read the neighbouring row's data; every entry they touch is discarded (x < 0,
//     x >= W or x - d < 0), exactly the entries the reference does not write;
//   * thread 0 issues two cp.async.bulk.tensor.2d per 8-channel slab ([8][128] left, [8][256] right window,
//     dense rows) into a 4-stage ring behind full / empty mbarriers: no block-wide barrier in the main loop;
//   * dense rows would make the 8-floats-per-thread LDS.128 pairs 2-way bank conflicted (lanes 0-3 and 4-7 of a
//     quarter-warp hit the same banks).  Lanes 4-7 therefore read their two 16-byte halves in the OPPOSITE order (and
//     the four R pieces pairwise swapped): every quarter-warp then covers all 32 banks.  The registers of those lanes hold
//     a fixed permutation of the tile (x offset ^ 4, j offset ^ 4), undone ONCE per CTA by swapping accumulators before
//     the epilogue;
//   * epilogue: the tile is staged dense in shared memory along its diagonals as before, then thread = column walks down
//     the disparities: 128 contiguous bytes per warp and store instruction into each volume, pointers advanced by constant
//     strides (two vectorised variants -- float4 groups aligned to the output address -- measured slower: the realignment
//     selects cost more instructions than the 4-byte stores they saved).
#include <string.h>

#include "internal.cuh"

namespace {

constexpr int ST_TX = 128;       // x per CTA
constexpr int ST_CCH = 8;        // channels per stage
constexpr int ST_NSTG = 4;
constexpr int ST_STAGE_FLOATS = ST_CCH * (ST_TX + 2 * ST_TX);   // [8][128] L block, then [8][256] R block

__device__ __forceinline__ unsigned long long st_pack2(float lo, float hi)
{
	unsigned long long r;
	asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
	return r;
}
__device__ __forceinline__ void st_unpack2(unsigned long long v, float &lo, float &hi)
{
	asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long st_fma2(unsigned long long a, unsigned long long b, unsigned long long c)
{
	unsigned long long d;
	asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
	return d;
}
__device__ __forceinline__ void st_arrive(uint64_t *bar)
{
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tma_smem_addr(bar)) : "memory");
}

template <int NS>
struct STCfg {
	static constexpr int DC = 16 * NS - 8;                  // disparities per CTA
	static constexpr int NCT = ((16 * NS + 31) / 32) * 32;  // threads (whole warps; threads beyond 16 NS idle)
	static constexpr int NT = NCT;                          // thread 0 doubles as the TMA producer (a producer warp would cost the
	                                                        // third CTA per SM: 168 registers x 160 threads)
	static constexpr int SMEM_PIPE = ST_NSTG * ST_STAGE_FLOATS * 4;
	static constexpr int SMEM_OUT = DC * ST_TX * 4;
	static constexpr int OFF_BAR = SMEM_PIPE > SMEM_OUT ? SMEM_PIPE : SMEM_OUT;
	static constexpr int SMEM = OFF_BAR + 2 * ST_NSTG * 8;
};

template <int NS>
__global__ void __launch_bounds__(STCfg<NS>::NT, (NS >= 6) ? 3 : 4)
stereo_join_tma_kernel(const __grid_constant__ CUtensorMap tmL, const __grid_constant__ CUtensorMap tmR,
		       float *__restrict__ outL, float *__restrict__ outR, int C, int D, int H, int W, int ldo)
{
	using Cfg = STCfg<NS>;
	constexpr int DC = Cfg::DC, NCT = Cfg::NCT, DTOP = DC;   // d - d0 of the tile diagonal xi - ji = 0 at s = 0 (a multiple of 8)
	extern __shared__ __align__(128) float st_smem[];
	uint64_t *bar_full = reinterpret_cast<uint64_t *>(reinterpret_cast<unsigned char *>(st_smem) + Cfg::OFF_BAR);
	uint64_t *bar_empty = bar_full + ST_NSTG;

	const int tid = threadIdx.x;
	const int y = blockIdx.y;
	const int d0 = blockIdx.z * DC;
	const int sh = (int)(((long)y * W) & 3);
	const int X0 = blockIdx.x * ST_TX - sh;                // flat index y W + X0 is a multiple of 4
	if (X0 >= W || X0 + ST_TX - 1 < d0) return;            // outside the image row / entirely x < d: nothing to write
	const int jbase = X0 - d0 - DTOP;                       // image column of R-window slot 0
	const int nstage = (C + ST_CCH - 1) / ST_CCH;

	if (tid == 0) {
		for (int s = 0; s < ST_NSTG; s++) {
			mbar_init(&bar_full[s], 1);
			mbar_init(&bar_empty[s], NCT / 32);
		}
		mbar_fence_init();
		tma_prefetch_desc(&tmL);
		tma_prefetch_desc(&tmR);
	}
	__syncthreads();

	const int fL = y * W + X0, fR = y * W + jbase;
	auto issue = [&](int st) {                              // thread 0 only
		const int sl = st % ST_NSTG;
		float *sb = st_smem + sl * ST_STAGE_FLOATS;
		mbar_arrive_expect_tx(&bar_full[sl], ST_STAGE_FLOATS * 4);
		tma_load_2d(sb, &tmL, fL, st * ST_CCH, &bar_full[sl]);                    // [8][128]; channels >= C read as 0
		tma_load_2d(sb + ST_CCH * ST_TX, &tmR, fR, st * ST_CCH, &bar_full[sl]);   // [8][256]
	};
	if (tid == 0)
		for (int st = 0; st < ST_NSTG - 1 && st < nstage; st++) issue(st);

	// -------------------------------------------------------------------- compute threads
	const int gx = (tid & 7) + 8 * ((tid >> 3) & 1);    // x group (8 columns); a quarter-warp = 8 consecutive groups
	const int s = tid >> 4;                              // tile index along the diagonal
	const int hb = (gx >> 2) & 1;                        // lanes 4-7 of a quarter-warp read their halves in the opposite order
	const int lane = tid & 31;

	unsigned long long acc2[8][8];
#pragma unroll
	for (int i = 0; i < 8; i++)
#pragma unroll
		for (int j = 0; j < 8; j++) acc2[i][j] = st_pack2(0.0f, 0.0f);

	// this tile's disparities: d - d0 = DTOP - 16 s + xi - ji
	const int dtop = d0 + DTOP - 16 * s;
	const bool active = s < NS && (dtop - 15 < D) && (dtop - 15 < d0 + DC) && (dtop + 7 >= d0);
	const int lo0 = (2 * gx + hb) * 4, lo1 = (2 * gx + 1 - hb) * 4;                       // float offsets in an L row
	const int cR = 2 * (gx + 2 * s);
	const int ro0 = (cR + hb) * 4, ro1 = (cR + 1 - hb) * 4, ro2 = (cR + 2 + hb) * 4, ro3 = (cR + 3 - hb) * 4;

	for (int st = 0; st < nstage; st++) {
		const int sidx = st % ST_NSTG;
		mbar_wait(&bar_full[sidx], (st / ST_NSTG) & 1);
		if (tid == 0 && st + ST_NSTG - 1 < nstage) {       // refill the slot of slab st - 1 once every warp has released it
			const int nx = st + ST_NSTG - 1;
			if (nx >= ST_NSTG) mbar_wait(&bar_empty[nx % ST_NSTG], ((nx / ST_NSTG) - 1) & 1);
			issue(nx);
		}
		if (active) {
			const float *sb = st_smem + sidx * ST_STAGE_FLOATS;
#pragma unroll
			for (int cc = 0; cc < ST_CCH; cc++) {
				const float *lrow = sb + cc * ST_TX;
				const float *rrow = sb + ST_CCH * ST_TX + cc * 2 * ST_TX;
				float l[8], r[16];
				*reinterpret_cast<float4 *>(&l[0]) = *reinterpret_cast<const float4 *>(lrow + lo0);
				*reinterpret_cast<float4 *>(&l[4]) = *reinterpret_cast<const float4 *>(lrow + lo1);
				*reinterpret_cast<float4 *>(&r[0]) = *reinterpret_cast<const float4 *>(rrow + ro0);
				*reinterpret_cast<float4 *>(&r[4]) = *reinterpret_cast<const float4 *>(rrow + ro1);
				*reinterpret_cast<float4 *>(&r[8]) = *reinterpret_cast<const float4 *>(rrow + ro2);
				*reinterpret_cast<float4 *>(&r[12]) = *reinterpret_cast<const float4 *>(rrow + ro3);
				unsigned long long r2[8];
#pragma unroll
				for (int m = 0; m < 8; m++) r2[m] = st_pack2(r[2 * m], r[2 * m + 1]);
#pragma unroll
				for (int xi = 0; xi < 8; xi++) {
					const unsigned long long nl = st_pack2(-l[xi], -l[xi]);
#pragma unroll
					for (int m = 0; m < 8; m++) acc2[xi][m] = st_fma2(r2[m], nl, acc2[xi][m]);  // adcensus.cu:1470: sum -= l * r
				}
			}
		}
		__syncwarp();
		if (lane == 0) st_arrive(&bar_empty[sidx]);
	}
	asm volatile("bar.sync 1, %0;" ::"n"(NCT) : "memory");   // every compute thread is done with the ring: it becomes the output stage

	// undo the register permutation of the lanes that read in the opposite order: true[a][b] = held[a ^ 4][b ^ 4]
	if (hb) {
#pragma unroll
		for (int a = 0; a < 4; a++)
#pragma unroll
			for (int m = 0; m < 8; m++) {
				const unsigned long long t = acc2[a][m];
				acc2[a][m] = acc2[a + 4][m ^ 2];
				acc2[a + 4][m ^ 2] = t;
			}
	}
	float acc[8][16];
#pragma unroll
	for (int i = 0; i < 8; i++)
#pragma unroll
		for (int m = 0; m < 8; m++) st_unpack2(acc2[i][m], acc[i][2 * m], acc[i][2 * m + 1]);

	// ---- epilogue 1: tile diagonals (fixed d, consecutive x) -> so[dd][x], dense ----
	float *so = st_smem;
	if (s < NS) {
#pragma unroll
		for (int t = -15; t <= 7; t++) {                     // t = xi - ji
			const int dd = DTOP - 16 * s + t;                // d - d0
			if (dd < 0 || dd >= DC) continue;
			float *rowp = so + dd * ST_TX + gx * 8;
#pragma unroll
			for (int h = 0; h < 2; h++) {                    // halves xi = 4h .. 4h+3
				float *hp = rowp + h * 4;
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
	}
	asm volatile("bar.sync 1, %0;" ::"n"(NCT) : "memory");

	// ---- epilogue 2: thread = tile column, walking down the chunk's disparities (adcensus.cu:1472-1473) ----
	// A warp stores 128 contiguous bytes per instruction into each volume; the valid disparities of a column are the
	// prefix d <= x, so the loop needs no per-row test, and both output pointers advance by constant strides.
	const int nrows = min(DC, D - d0);
	for (int xl = tid; xl < ST_TX; xl += NCT) {
		const int x = X0 + xl;
		if (x < 0 || x >= W) continue;
		const int rmax = min(nrows, x - d0 + 1);             // rows with d0 + r <= x
		const float *sp = so + xl;
		const long o = ((long)d0 * H + y) * ldo + x;
		float *pL = outL + o, *pR = outR + o - d0;            // outR[d][y][x - d]
		const long stepL = (long)H * ldo, stepR = stepL - 1;
#pragma unroll 4
		for (int r = 0; r < rmax; r++) {
			const float v = sp[r * ST_TX];
			*pL = v;
			*pR = v;
			pL += stepL;
			pR += stepR;
		}
	}
}

template <int NS>
int launch_tma(const CUtensorMap &tmL, const CUtensorMap &tmR, float *outL, float *outR, int C, int D, int H, int W, int ldo, cudaStream_t s)
{
	using Cfg = STCfg<NS>;
	static bool attr_done[64] = {false};
	int dev = 0;
	cudaGetDevice(&dev);
	if (!attr_done[dev & 63]) {
		ADC_CUDA(cudaFuncSetAttribute(stereo_join_tma_kernel<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
		attr_done[dev & 63] = true;
	}
	dim3 grid(adc_div_up(W + 3, ST_TX), H, adc_div_up(D, Cfg::DC));
	stereo_join_tma_kernel<NS><<<grid, Cfg::NT, Cfg::SMEM, s>>>(tmL, tmR, outL, outR, C, D, H, W, ldo);
	ADC_CHECK_LAUNCH();
	return 0;
}

}  // namespace

// 1 when the TMA kernel can run: H*W a multiple of 4 (tensor-map row stride), 16-byte aligned feature bases and outputs
int adc_stereo_join_tma_ok(const float *input_L, const float *input_R, const float *output_L, const float *output_R, int H, int W)
{
	return (((long)H * W) % 4 == 0) && ((((uintptr_t)input_L) | ((uintptr_t)input_R) | ((uintptr_t)output_L) | ((uintptr_t)output_R)) % 16 == 0);
}

// outputs (D, H, ldo), ldo >= W; features (C, H, W) contiguous.  ns = tiles per CTA along the diagonal (DC = 16 ns - 8).
int adc_stereo_join_tma(const float *input_L, const float *input_R, float *output_L, float *output_R,
			int C, int D, int H, int W, int ldo, int ns, cudaStream_t s)
{
	CUtensorMap tmL, tmR;
	const uint64_t dims[2] = {(uint64_t)H * W, (uint64_t)C};
	const uint64_t strides[1] = {(uint64_t)H * W * 4};
	const uint32_t boxL[2] = {(uint32_t)ST_TX, (uint32_t)ST_CCH}, boxR[2] = {(uint32_t)(2 * ST_TX), (uint32_t)ST_CCH};
	int rc = adc_tma_encode(&tmL, input_L, 2, dims, strides, boxL);
	if (!rc) rc = adc_tma_encode(&tmR, input_R, 2, dims, strides, boxR);
	if (rc) return rc;
	switch (ns) {
	case 1: return launch_tma<1>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	case 2: return launch_tma<2>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	case 3: return launch_tma<3>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	case 4: return launch_tma<4>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	case 5: return launch_tma<5>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	case 6: return launch_tma<6>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	case 7: return launch_tma<7>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	default: return launch_tma<8>(tmL, tmR, output_L, output_R, C, D, H, W, ldo, s);
	}
}
