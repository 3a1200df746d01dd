// feature_tower.cu -- the feature tower of mc-cnn in-library (SURVEY.md 8f-2): l1 x [3x3 convolution, stride 1, zero pad 1]
// with ReLU between the layers (and after the last one for the accurate architecture), optionally followed by Normalize2
// (adcensus.cu:1284-1308: x / sqrt(sum_c x^2 + 1e-5)) -- the producer of StereoJoin's inputs (main.lua:726-749, 897-901,
// 944-951; for arch 'slow' main.lua:682-686).  The reference runs cudnn.SpatialConvolution modules (cross-correlation, no
// kernel flip) with cudnn.benchmark picking the algorithm.
//
// Layer 1 has 1 (grey) or 3 input planes: 9..27 multiply-adds per output, done exactly in fp32 on the CUDA cores.
// Layers 2.. (Cin = fm = 64 / 112) are an implicit GEMM on the tensor cores with the machinery of scorer_head.cu:
//   * tile = 128 consecutive pixels of one image row (MMA M), N = fm output planes (padded to a multiple of 64), K = 9 Cin
//     ordered tap-major (k = tap * Cin + c), tcgen05.mma kind::f16 with bf16-SPLIT operands (three MMAs per K step:
//     hi.whi + lo.whi + hi.wlo, fp32 accumulation in TMEM) => fp32-grade results (~1e-6 relative);
//   * the A operand is built in shared memory by eight warps straight from the (Cin, H, W) activation (coalesced along x,
//     zero outside the image), a few taps at a time (K <= 320 per pass: 164 KB for hi + lo), the passes accumulate into the
//     same TMEM columns;
//   * weights are pre-split into per-K-step slabs and stream from L2 through a 12-slot cp.async.bulk ring;
//   * epilogue: thread = pixel = TMEM lane; + bias, ReLU, and for the last layer of the fast architecture the Normalize2 of
//     Normalize2.lua fused in (sum over the planes in ascending order, like adcensus.cu:1291-1294), stores coalesced along x.
#include <stdlib.h>
#include <string.h>

#include "umma.cuh"

namespace {

constexpr int FT_KA = 320;                         // K of one pass (A operand capacity)
constexpr int FT_ABYTES = (FT_KA / 8) * SH_ACHUNK; // 81920 per hi / lo
constexpr int FT_NMAX = 128, FT_LMAX = 8;
constexpr int FT_SLAB = 2 * FT_NMAX * 16;          // 4096: one K = 16 step of B at N = 128
constexpr int FT_NSLOT = 12;
constexpr int FT_NFEED = 256, FT_NT = FT_NFEED + 64;
constexpr int FT_OFF_AHI = 0, FT_OFF_ALO = FT_ABYTES, FT_OFF_RING = 2 * FT_ABYTES;
constexpr int FT_OFF_BIAS = FT_OFF_RING + FT_NSLOT * FT_SLAB;
constexpr int FT_OFF_BAR = FT_OFF_BIAS + FT_NMAX * 4;
constexpr int FT_OFF_TPTR = FT_OFF_BAR + (2 * FT_NSLOT + 2) * 8;
constexpr int FT_SMEM = FT_OFF_TPTR + 16;
static_assert(FT_SMEM <= 232448, "shared memory budget");

struct FTParams {
	const float *in;                 // (nimg, Cin, H, W)
	float *out;                      // (nimg, fm, H, W)
	const unsigned char *wslabs;     // per K step: [hi slab][lo slab], slab = [2][Np][8] bf16, k = tap * Cin + c
	const float *bias;               // [fm]
	int Cin, fm, Np, H, W, relu, normalize, taps_per_pass;
};

template <int NTERMS>
__global__ void __launch_bounds__(FT_NT, 1)
conv3x3_umma_kernel(const FTParams p)
{
	extern __shared__ __align__(128) unsigned char ft_smem[];
	unsigned char *a_hi = ft_smem + FT_OFF_AHI, *a_lo = ft_smem + FT_OFF_ALO, *ring = ft_smem + FT_OFF_RING;
	float *bias = reinterpret_cast<float *>(ft_smem + FT_OFF_BIAS);
	uint64_t *bar_full = reinterpret_cast<uint64_t *>(ft_smem + FT_OFF_BAR);
	uint64_t *bar_empty = bar_full + FT_NSLOT;
	uint64_t *bar_a = bar_empty + FT_NSLOT, *bar_acc = bar_a + 1;
	uint32_t *tptr = reinterpret_cast<uint32_t *>(ft_smem + FT_OFF_TPTR);

	const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
	const int x0 = blockIdx.x * SH_M, y = blockIdx.y, img = blockIdx.z;
	const int Cin = p.Cin, Np = p.Np, H = p.H, W = p.W;
	const long HW = (long)H * W;
	const int npass = (9 + p.taps_per_pass - 1) / p.taps_per_pass;
	const uint32_t slab_bytes = (uint32_t)Np * 32u;

	if (tid == 0) {
		for (int s = 0; s < FT_NSLOT; s++) {
			mbar_init(&bar_full[s], 1);
			mbar_init(&bar_empty[s], 1);
		}
		mbar_init(bar_a, FT_NFEED);
		mbar_init(bar_acc, 1);
		mbar_fence_init();
	}
	for (int i = tid; i < FT_NMAX; i += FT_NT) bias[i] = i < p.fm ? p.bias[i] : 0.0f;
	if (warp == 9) {
		asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tma_smem_addr(tptr)), "r"(128) : "memory");
		asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
	}
	sh_fence_before();
	__syncthreads();
	sh_fence_after();
	const uint32_t tbase = *tptr;

	if (warp == 8) {
		// ------------------------------------------------------------ weight producer: every K step of the layer, in order
		if (lane == 0) {
			const int nks = 9 * Cin / 16;
			for (unsigned it = 0; it < (unsigned)(nks * (NTERMS == 3 ? 2 : 1)); it++) {
				const int s = it % FT_NSLOT;
				const int ks = NTERMS == 3 ? it >> 1 : it, part = NTERMS == 3 ? it & 1 : 0;
				if (it >= (unsigned)FT_NSLOT) sh_wait(&bar_empty[s], ((it / FT_NSLOT) - 1) & 1);
				mbar_arrive_expect_tx(&bar_full[s], slab_bytes);
				sh_bulk_load(ring + s * FT_SLAB, p.wslabs + ((long)ks * 2 + part) * slab_bytes, slab_bytes, &bar_full[s]);
			}
		}
	} else if (warp == 9) {
		// ------------------------------------------------------------ MMA issuer
		if (lane == 0) {
			const uint32_t a_hi_s = tma_smem_addr(a_hi), a_lo_s = tma_smem_addr(a_lo), ring_s = tma_smem_addr(ring);
			const uint32_t lbo_b = (uint32_t)Np * 16u, idesc = sh_idesc(Np);
			unsigned it = 0;
			int tap0 = 0;
			for (int ps = 0; ps < npass; ps++) {
				const int ntap = min(p.taps_per_pass, 9 - tap0), nks = ntap * Cin / 16;
				sh_wait(bar_a, ps & 1);
				sh_fence_after();
				for (int ks = 0; ks < nks; ks++) {
					const uint32_t acc_on = (ps > 0 || ks > 0) ? 1u : 0u;
					const uint64_t da_hi = sh_desc(a_hi_s + ks * 2 * SH_ACHUNK, SH_ACHUNK, 128);
					const uint64_t da_lo = sh_desc(a_lo_s + ks * 2 * SH_ACHUNK, SH_ACHUNK, 128);
					{
						const int s = it % FT_NSLOT;
						sh_wait(&bar_full[s], (it / FT_NSLOT) & 1);
						sh_fence_after();
						const uint64_t db = sh_desc(ring_s + s * FT_SLAB, lbo_b, 128);
						sh_mma(tbase, da_hi, db, idesc, acc_on);
						if (NTERMS == 3) sh_mma(tbase, da_lo, db, idesc, 1);
						sh_commit(&bar_empty[s]);
						it++;
					}
					if (NTERMS == 3) {
						const int s = it % FT_NSLOT;
						sh_wait(&bar_full[s], (it / FT_NSLOT) & 1);
						sh_fence_after();
						const uint64_t db = sh_desc(ring_s + s * FT_SLAB, lbo_b, 128);
						sh_mma(tbase, da_hi, db, idesc, 1);
						sh_commit(&bar_empty[s]);
						it++;
					}
				}
				sh_commit(bar_acc);
				tap0 += ntap;
			}
		}
	} else {
		// ------------------------------------------------------------ operand builders (8 warps) / epilogue (warps 0-3)
		const int m = (warp & 3) * 32 + lane, hf = warp >> 2;
		const int x = x0 + m;
		const float *src_img = p.in + (long)img * Cin * HW;
		int tap0 = 0;
		for (int ps = 0; ps < npass; ps++) {
			const int ntap = min(p.taps_per_pass, 9 - tap0);
			const int nch = ntap * Cin / 8;                       // 8-wide K chunks of this pass
			if (ps > 0) {                                         // the previous pass's MMAs have read the operand
				sh_wait(bar_acc, (ps - 1) & 1);
				sh_fence_after();
			}
			// chunk kc: tap = tap0 + (8 kc) / Cin, planes c0 .. c0 + 7 (Cin % 8 == 0: a chunk never straddles a tap)
			for (int kc0 = hf * 4; kc0 < nch; kc0 += 8) {          // each half takes alternate groups of 4 chunks
				float v[4][8];
#pragma unroll
				for (int u = 0; u < 4; u++) {
					const int kc = kc0 + u;
					const int k0 = kc * 8, tap = tap0 + k0 / Cin, c0 = k0 % Cin;
					const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
					const bool ok = kc < nch && yy >= 0 && yy < H && xx >= 0 && xx < W;
					const float *src = src_img + (long)c0 * HW + (long)(ok ? yy : 0) * W + (ok ? xx : 0);
#pragma unroll
					for (int e = 0; e < 8; e++) v[u][e] = ok ? __ldg(src + (long)e * HW) : 0.0f;
				}
#pragma unroll
				for (int u = 0; u < 4; u++)
					if (kc0 + u < nch) sh_store8<NTERMS>(a_hi, a_lo, kc0 + u, m, v[u]);
			}
			fence_proxy_async_smem();
			sh_fence_before();
			sh_arrive(bar_a);
			tap0 += ntap;
		}
		// epilogue: warps 0-3, thread = pixel = TMEM lane, all planes (ascending order for the Normalize2 sum)
		if (hf == 0) {
			sh_wait(bar_acc, (npass - 1) & 1);
			sh_fence_after();
			const uint32_t trow = tbase + ((uint32_t)(warp * 32) << 16);
			float scale = 1.0f;
			if (p.normalize) {
				float sum = 0.0f;
				for (int c0 = 0; c0 < Np; c0 += 32) {
					uint32_t r[32];
					sh_tmem_ld32(trow + c0, r);
					sh_tmem_wait(r);
#pragma unroll
					for (int e = 0; e < 32; e++) {
						float z = __uint_as_float(r[e]) + bias[c0 + e];
						if (p.relu) z = fmaxf(z, 0.0f);
						if (c0 + e < p.fm) sum = fmaf(z, z, sum);      // adcensus.cu:1293 (nvcc contracts sum += x * x)
					}
				}
				scale = sqrtf(sum + 1e-5f);                            // :1296, :1305
			}
			float *dst = p.out + (long)img * p.fm * HW + (long)y * W + x;
			for (int c0 = 0; c0 < Np; c0 += 32) {
				uint32_t r[32];
				sh_tmem_ld32(trow + c0, r);
				sh_tmem_wait(r);
#pragma unroll
				for (int e = 0; e < 32; e++) {
					float z = __uint_as_float(r[e]) + bias[c0 + e];
					if (p.relu) z = fmaxf(z, 0.0f);
					if (p.normalize) z = z / scale;
					if (c0 + e < p.fm && x < W) dst[(long)(c0 + e) * HW] = z;
				}
			}
		}
	}
	sh_fence_before();
	__syncthreads();
	if (warp == 9) {
		sh_fence_after();
		asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(128) : "memory");
	}
}

// ---- second form, for Cin = fm <= 64 (the fast architecture): weights RESIDENT, persistent CTAs --------------------------
// The streamed form above is latency-bound (tensor pipe 5 % active at fm = 64: every tile waits for 72 weight slabs and for two
// 40-chunk operand builds).  With 64 planes the whole layer's weights, split, are 147 KB: they stay in shared memory for the
// life of a persistent CTA; the A operand is built one TAP at a time (K = 64: 32 KB for hi + lo) into a double buffer, so the
// eight builder warps (next tap's loads already in flight while the current one is split and stored), the MMA thread and the
// four epilogue warps (two accumulator stages in TMEM) all overlap.
constexpr int F2_NB = 256, F2_NE = 128, F2_NT = F2_NB + F2_NE + 32;      // builders, epilogue, MMA warp
constexpr int F2_WBYTES = 9 * 64 / 16 * 2 * 64 * 32;                       // 147456: 36 K steps x (hi, lo) x [2][64][8] bf16
constexpr int F2_ABUF = 2 * (64 / 8) * SH_ACHUNK;                         // one tap: hi + lo = 32768
constexpr int F2_OFF_A = F2_WBYTES, F2_OFF_BIAS = F2_OFF_A + 2 * F2_ABUF;
constexpr int F2_OFF_BAR = F2_OFF_BIAS + 64 * 4;                           // a_full[2], a_free[2], acc_full[2], acc_free[2]
constexpr int F2_OFF_TPTR = F2_OFF_BAR + 8 * 8;
constexpr int F2_SMEM = F2_OFF_TPTR + 16;
static_assert(F2_SMEM <= 232448, "shared memory budget");

template <int NTERMS>
__global__ void __launch_bounds__(F2_NT, 1)
conv3x3_resident_kernel(const FTParams p, int nimg)
{
	extern __shared__ __align__(128) unsigned char ft_smem[];
	unsigned char *wsm = ft_smem, *abuf = ft_smem + F2_OFF_A;
	float *bias = reinterpret_cast<float *>(ft_smem + F2_OFF_BIAS);
	uint64_t *a_full = reinterpret_cast<uint64_t *>(ft_smem + F2_OFF_BAR), *a_free = a_full + 2;
	uint64_t *acc_full = a_free + 2, *acc_free = acc_full + 2;
	uint32_t *tptr = reinterpret_cast<uint32_t *>(ft_smem + F2_OFF_TPTR);

	const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
	const int H = p.H, W = p.W, Cin = p.Cin, Np = p.Np;           // Cin == 64, Np == 64
	const long HW = (long)H * W;
	const int xt = (W + SH_M - 1) / SH_M;
	const int ntile = nimg * H * xt;
	const int nks_tap = Cin / 16;
	const uint32_t slab = (uint32_t)Np * 32u;

	if (tid == 0) {
		for (int i = 0; i < 2; i++) {
			mbar_init(&a_full[i], F2_NB);
			mbar_init(&a_free[i], 1);
			mbar_init(&acc_full[i], 1);
			mbar_init(&acc_free[i], F2_NE);
		}
		mbar_fence_init();
	}
	{   // the layer's weights: a straight copy of the prepared slabs
		const uint4 *src = reinterpret_cast<const uint4 *>(p.wslabs);
		uint4 *dst = reinterpret_cast<uint4 *>(wsm);
		const int n16 = 9 * nks_tap * 2 * (int)slab / 16;
		for (int i = tid; i < n16; i += F2_NT) dst[i] = __ldg(src + i);
	}
	for (int i = tid; i < 64; i += F2_NT) bias[i] = i < p.fm ? p.bias[i] : 0.0f;
	if (warp == 12) {
		asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tma_smem_addr(tptr)), "r"(128) : "memory");
		asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
	}
	fence_proxy_async_smem();                                  // the weights were written with generic stores
	sh_fence_before();
	__syncthreads();
	sh_fence_after();
	const uint32_t tbase = *tptr;

	if (warp < 8) {
		// ------------------------------------------------------------ operand builders: thread = (pixel m, 4 of the tap's 8 chunks)
		const int m = tid & 127, hf = tid >> 7;
		float nxt[4][8];
		auto load = [&](int tile, int tap, float (&v)[4][8]) {
			const int img = tile / (H * xt), rem = tile - img * (H * xt), y = rem / xt, x = (rem - y * xt) * SH_M + m;
			const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
			const bool ok = tile < ntile && yy >= 0 && yy < H && xx >= 0 && xx < W;
			const float *src = p.in + (long)img * Cin * HW + (long)(hf * 32) * HW + (long)(ok ? yy : 0) * W + (ok ? xx : 0);
#pragma unroll
			for (int u = 0; u < 4; u++)
#pragma unroll
				for (int e = 0; e < 8; e++) v[u][e] = ok ? __ldg(src + (long)(u * 8 + e) * HW) : 0.0f;
		};
		unsigned g = 0;
		int tile = blockIdx.x, tap = 0;
		if (tile < ntile) load(tile, 0, nxt);
		while (tile < ntile) {
			float cur[4][8];
#pragma unroll
			for (int u = 0; u < 4; u++)
#pragma unroll
				for (int e = 0; e < 8; e++) cur[u][e] = nxt[u][e];
			int ntile_i = tile, ntap = tap + 1;                 // the step after this one
			if (ntap == 9) { ntap = 0; ntile_i = tile + gridDim.x; }
			load(ntile_i, ntap, nxt);                           // in flight while this step is split and stored
			const int b = g & 1;
			if (g >= 2) sh_wait(&a_free[b], ((g >> 1) - 1) & 1);
			unsigned char *ah = abuf + b * F2_ABUF, *al = ah + (64 / 8) * SH_ACHUNK;
#pragma unroll
			for (int u = 0; u < 4; u++) sh_store8<NTERMS>(ah, al, hf * 4 + u, m, cur[u]);
			fence_proxy_async_smem();
			sh_fence_before();
			sh_arrive(&a_full[b]);
			g++;
			tile = ntile_i;
			tap = ntap;
		}
	} else if (warp == 12) {
		// ------------------------------------------------------------ MMA issuer
		if (lane == 0) {
			const uint32_t a_s = tma_smem_addr(abuf), w_s = tma_smem_addr(wsm);
			const uint32_t lbo_b = (uint32_t)Np * 16u, idesc = sh_idesc(Np);
			unsigned g = 0, ti = 0;
			for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x, ti++) {
				const int st = ti & 1;
				if (ti >= 2) sh_wait(&acc_free[st], ((ti >> 1) - 1) & 1);
				sh_fence_after();
				for (int tap = 0; tap < 9; tap++, g++) {
					const int b = g & 1;
					sh_wait(&a_full[b], (g >> 1) & 1);
					sh_fence_after();
					for (int ks = 0; ks < nks_tap; ks++) {
						const uint64_t da_hi = sh_desc(a_s + b * F2_ABUF + ks * 2 * SH_ACHUNK, SH_ACHUNK, 128);
						const uint64_t da_lo = sh_desc(a_s + b * F2_ABUF + (64 / 8) * SH_ACHUNK + ks * 2 * SH_ACHUNK, SH_ACHUNK, 128);
						const uint32_t wk = w_s + (uint32_t)(tap * nks_tap + ks) * 2u * slab;
						const uint64_t db_hi = sh_desc(wk, lbo_b, 128), db_lo = sh_desc(wk + slab, lbo_b, 128);
						const uint32_t acc_on = (tap > 0 || ks > 0) ? 1u : 0u;
						sh_mma(tbase + st * 64, da_hi, db_hi, idesc, acc_on);
						if (NTERMS == 3) {
							sh_mma(tbase + st * 64, da_lo, db_hi, idesc, 1);
							sh_mma(tbase + st * 64, da_hi, db_lo, idesc, 1);
						}
					}
					sh_commit(&a_free[b]);
				}
				sh_commit(&acc_full[st]);
			}
		}
	} else {
		// ------------------------------------------------------------ epilogue warps 8-11: thread = pixel = TMEM lane
		const int q = warp & 3, m = q * 32 + lane;
		unsigned ti = 0;
		for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x, ti++) {
			const int st = ti & 1;
			const int img = tile / (H * xt), rem = tile - img * (H * xt), y = rem / xt, x = (rem - y * xt) * SH_M + m;
			sh_wait(&acc_full[st], (ti >> 1) & 1);
			sh_fence_after();
			const uint32_t trow = tbase + ((uint32_t)(q * 32) << 16) + st * 64;
			uint32_t r0[32], r1[32];
			sh_tmem_ld32(trow, r0);
			sh_tmem_ld32(trow + 32, r1);
			sh_tmem_wait(r0);
			sh_tmem_wait(r1);
			sh_fence_before();
			sh_arrive(&acc_free[st]);                             // the accumulator stage is in registers: the MMAs may reuse it
			float z[64];
#pragma unroll
			for (int e = 0; e < 32; e++) {
				z[e] = __uint_as_float(r0[e]) + bias[e];
				z[32 + e] = __uint_as_float(r1[e]) + bias[32 + e];
			}
			if (p.relu) {
#pragma unroll
				for (int e = 0; e < 64; e++) z[e] = fmaxf(z[e], 0.0f);
			}
			if (p.normalize) {
				float sum = 0.0f;
#pragma unroll
				for (int e = 0; e < 64; e++)
					if (e < p.fm) sum = fmaf(z[e], z[e], sum);          // adcensus.cu:1293, planes ascending
				const float scale = sqrtf(sum + 1e-5f);                 // :1296, :1305
#pragma unroll
				for (int e = 0; e < 64; e++) z[e] = z[e] / scale;
			}
			if (x < W) {
				float *dst = p.out + (long)img * p.fm * HW + (long)y * W + x;
#pragma unroll
				for (int e = 0; e < 64; e++)
					if (e < p.fm) dst[(long)e * HW] = z[e];
			}
		}
	}
	sh_fence_before();
	__syncthreads();
	if (warp == 12) {
		sh_fence_after();
		asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(128) : "memory");
	}
}

// first layer (Cin = 1 or 3): exact fp32, thread = pixel, weights in shared memory; planes / rows / columns ascending
__global__ void conv3x3_first_kernel(const float *__restrict__ in, const float *__restrict__ w, const float *__restrict__ b,
				     float *__restrict__ out, int Cin, int fm, int H, int W, int relu)
{
	extern __shared__ float fw[];                         // [fm][Cin * 9] + [fm]
	const int nw = fm * Cin * 9;
	for (int i = threadIdx.x; i < nw + fm; i += blockDim.x) fw[i] = i < nw ? w[i] : b[i - nw];
	__syncthreads();
	const long HW = (long)H * W;
	const long id = (long)blockIdx.x * blockDim.x + threadIdx.x;
	const int img = blockIdx.y;
	if (id >= HW) return;
	const int y = (int)(id / W), x = (int)(id % W);
	float v[27];
	for (int c = 0; c < Cin; c++)
#pragma unroll
		for (int t = 0; t < 9; t++) {
			const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
			v[c * 9 + t] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? in[((long)img * Cin + c) * HW + (long)yy * W + xx] : 0.0f;
		}
	float *dst = out + (long)img * fm * HW + id;
	for (int o = 0; o < fm; o++) {
		float acc = fw[nw + o];
		for (int k = 0; k < Cin * 9; k++) acc = fmaf(fw[o * Cin * 9 + k], v[k], acc);
		dst[(long)o * HW] = relu ? fmaxf(acc, 0.0f) : acc;
	}
}

// weights (fm, Cin, 3, 3) fp32 -> slabs over k = tap * Cin + c: per K step [hi: [2][Np][8] bf16][lo: ...], planes >= fm zero
__global__ void ft_prep_kernel(const float *__restrict__ w, unsigned short *__restrict__ slabs, int fm, int Np, int Cin)
{
	const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= (long)fm * Cin * 9) return;
	const int o = (int)(i / (Cin * 9)), c = (int)((i / 9) % Cin), tap = (int)(i % 9);
	const int k = tap * Cin + c;
	const float v = w[i];
	const unsigned hb = __float_as_uint(v);
	const unsigned hi = (hb + 0x7fffu + ((hb >> 16) & 1u)) >> 16;
	const float r = v - __uint_as_float(hi << 16);
	const unsigned rb = __float_as_uint(r);
	const unsigned lo = (rb + 0x7fffu + ((rb >> 16) & 1u)) >> 16;
	const int ks = k / 16, j = (k / 8) & 1, e = k & 7;
	const long slab = (long)Np * 16;
	const long base = (long)ks * 2 * slab + ((long)j * Np + o) * 8 + e;
	slabs[base] = (unsigned short)hi;
	slabs[base + slab] = (unsigned short)lo;
}

}  // namespace

struct mccnn_feature_tower {
	int n_in, fm, Np, l1, relu_last, normalize, device;
	float *w0, *b0;                     // first layer
	unsigned char *wslabs[FT_LMAX];     // layers 1 .. l1-1
	float *bias[FT_LMAX];
};

// W[i] (fm, cin_i, 3, 3) row-major / b[i] (fm) for i = 0 .. l1-1, DEVICE pointers, the layout of cudnn.SpatialConvolution's
// weight / bias (main.lua:683, 729).  n_in = 1 or 3 input planes; relu_last / normalize: arch 'fast' = (0, 1), 'slow' = (1, 0).
extern "C" int mccnn_feature_tower_create(mccnn_feature_tower **out, int n_in, int fm, int l1, int relu_last, int normalize,
					   const float *const *W, const float *const *b, int device, adcensus_stream_t stream)
{
	if (!out || !W || !b || (n_in != 1 && n_in != 3) || fm < 8 || l1 < 1) return ADCENSUS_EINVAL;
	if (l1 > FT_LMAX || fm > FT_NMAX || (fm % 16)) return ADCENSUS_ELIMIT;
	int prev = 0;
	cudaGetDevice(&prev);
	cudaSetDevice(device);
	cudaStream_t s = adc_stream(stream);
	mccnn_feature_tower *h = (mccnn_feature_tower *)calloc(1, sizeof(*h));
	if (!h) return ADCENSUS_EINVAL;
	h->n_in = n_in; h->fm = fm; h->Np = (fm + 63) / 64 * 64; h->l1 = l1; h->relu_last = relu_last; h->normalize = normalize; h->device = device;
	int rc = (int)cudaMalloc((void **)&h->w0, (size_t)fm * n_in * 9 * sizeof(float));
	if (!rc) rc = (int)cudaMalloc((void **)&h->b0, fm * sizeof(float));
	if (!rc) rc = (int)cudaMemcpyAsync(h->w0, W[0], (size_t)fm * n_in * 9 * sizeof(float), cudaMemcpyDeviceToDevice, s);
	if (!rc) rc = (int)cudaMemcpyAsync(h->b0, b[0], fm * sizeof(float), cudaMemcpyDeviceToDevice, s);
	for (int l = 1; l < l1 && !rc; l++) {
		const size_t bytes = (size_t)(9 * fm / 16) * 2 * h->Np * 32;
		rc = (int)cudaMalloc((void **)&h->wslabs[l], bytes);
		if (!rc) rc = (int)cudaMemsetAsync(h->wslabs[l], 0, bytes, s);
		if (!rc) rc = (int)cudaMalloc((void **)&h->bias[l], fm * sizeof(float));
		if (!rc) rc = (int)cudaMemcpyAsync(h->bias[l], b[l], fm * sizeof(float), cudaMemcpyDeviceToDevice, s);
		if (!rc) {
			ft_prep_kernel<<<adc_div_up((long)fm * fm * 9, 256), 256, 0, s>>>(W[l], (unsigned short *)h->wslabs[l], fm, h->Np, fm);
			rc = (int)cudaPeekAtLastError();
		}
	}
	if (!rc) rc = (int)cudaStreamSynchronize(s);
	cudaSetDevice(prev);
	if (rc) {
		*out = nullptr;
		for (int l = 0; l < FT_LMAX; l++) { cudaFree(h->wslabs[l]); cudaFree(h->bias[l]); }
		cudaFree(h->w0); cudaFree(h->b0);
		free(h);
		return rc;
	}
	*out = h;
	return 0;
}

extern "C" void mccnn_feature_tower_destroy(mccnn_feature_tower *h)
{
	if (!h) return;
	for (int l = 0; l < FT_LMAX; l++) { cudaFree(h->wslabs[l]); cudaFree(h->bias[l]); }
	cudaFree(h->w0); cudaFree(h->b0);
	free(h);
}

// img (nimg, n_in, H, W) -> out (nimg, fm, H, W); nimg = 2 for a stereo pair (x_batch of main.lua:944).  nterms: 3 = bf16-split
// operands (fp32-grade), 1 = plain bf16.  Intermediate activations live in stream-ordered scratch.
extern "C" int mccnn_feature_tower_forward(const mccnn_feature_tower *h, const float *img, float *out, int nimg, int H, int W,
					    int nterms, adcensus_stream_t stream)
{
	if (!h || !img || !out || nimg < 1 || H < 1 || W < 1 || (nterms != 1 && nterms != 3)) return ADCENSUS_EINVAL;
	if (H > 65535 || nimg > 65535) return ADCENSUS_ELIMIT;
	cudaStream_t s = adc_stream(stream);
	const long HW = (long)H * W;
	const size_t act = (size_t)nimg * h->fm * HW * sizeof(float);
	float *buf[2] = {nullptr, nullptr};
	int rc = 0;
	if (h->l1 > 1) rc = adc_scratch_alloc((void **)&buf[0], act, s);
	if (!rc && h->l1 > 2) rc = adc_scratch_alloc((void **)&buf[1], act, s);
	if (rc) return rc;
	// layer 1
	{
		float *dst = h->l1 == 1 ? out : buf[0];
		const int relu = h->l1 > 1 ? 1 : h->relu_last;
		const dim3 grid(adc_div_up(HW, 128), nimg);
		const size_t sm = (size_t)(h->fm * h->n_in * 9 + h->fm) * sizeof(float);
		conv3x3_first_kernel<<<grid, 128, sm, s>>>(img, h->w0, h->b0, dst, h->n_in, h->fm, H, W, relu);
		rc = (int)cudaPeekAtLastError();
	}
	static bool attr3[64] = {false}, attr1[64] = {false};
	int dev = 0;
	cudaGetDevice(&dev);
	for (int l = 1; l < h->l1 && !rc; l++) {
		const bool last = l + 1 == h->l1;
		FTParams p;
		memset(&p, 0, sizeof(p));
		p.in = buf[(l - 1) & 1];
		p.out = last ? out : buf[l & 1];
		p.wslabs = h->wslabs[l]; p.bias = h->bias[l];
		p.Cin = h->fm; p.fm = h->fm; p.Np = h->Np; p.H = H; p.W = W;
		p.relu = last ? h->relu_last : 1;
		p.normalize = last ? h->normalize : 0;
		p.taps_per_pass = FT_KA / h->fm;                       // K of a pass = taps x Cin <= 320
		if (p.taps_per_pass > 9) p.taps_per_pass = 9;
		const dim3 grid(adc_div_up(W, SH_M), H, nimg);
		if (h->fm == 64) {                                         // weights resident, persistent CTAs (the fast architecture)
			static bool attr_r3[64] = {false}, attr_r1[64] = {false};
			const int ntile = nimg * H * adc_div_up(W, SH_M);
			const int nb = ntile < adc_num_sms() ? ntile : adc_num_sms();
			if (nterms == 3) {
				if (!attr_r3[dev & 63]) {
					rc = (int)cudaFuncSetAttribute(conv3x3_resident_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, F2_SMEM);
					attr_r3[dev & 63] = true;
				}
				if (!rc) conv3x3_resident_kernel<3><<<nb, F2_NT, F2_SMEM, s>>>(p, nimg);
			} else {
				if (!attr_r1[dev & 63]) {
					rc = (int)cudaFuncSetAttribute(conv3x3_resident_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, F2_SMEM);
					attr_r1[dev & 63] = true;
				}
				if (!rc) conv3x3_resident_kernel<1><<<nb, F2_NT, F2_SMEM, s>>>(p, nimg);
			}
			if (!rc) rc = (int)cudaPeekAtLastError();
			continue;
		}
		if (nterms == 3) {
			if (!attr3[dev & 63]) {
				rc = (int)cudaFuncSetAttribute(conv3x3_umma_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM);
				attr3[dev & 63] = true;
			}
			if (!rc) conv3x3_umma_kernel<3><<<grid, FT_NT, FT_SMEM, s>>>(p);
		} else {
			if (!attr1[dev & 63]) {
				rc = (int)cudaFuncSetAttribute(conv3x3_umma_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM);
				attr1[dev & 63] = true;
			}
			if (!rc) conv3x3_umma_kernel<1><<<grid, FT_NT, FT_SMEM, s>>>(p);
		}
		if (!rc) rc = (int)cudaPeekAtLastError();
	}
	if (h->l1 == 1 && h->normalize && !rc) rc = ADCENSUS_EINVAL;   // a one-layer tower with Normalize2 is not a net of the reference
	for (int i = 0; i < 2; i++)
		if (buf[i]) {
			const int rc2 = adc_scratch_free(buf[i], s);
			if (!rc) rc = rc2;
		}
	return rc;
}
