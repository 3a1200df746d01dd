// cbca_ws.cu -- constant-work cross-based cost aggregation (adcensus.cbca, adcensus.cu:343-400), second generation:
// warp-specialised, three-stage TMA pipeline, running sums down the column in a per-thread ring.
//
// Same decomposition as cbca_tma.cu -- the run of a support row depends on (d, row, column) only, so with I the
// inclusive prefix of a tile row
//     S(r, x)   = I(r, x + R_ - 1) - I(r, x - L)                                 sum of the run (x - L, x + R_)  (:362-369)
//     out(y, x) = (T(y + Dn - 1, x) - T(y - U, x)) / (N(y + Dn - 1, x) - N(y - U, x))                            (:361, :373)
// with T, N the running sums of S and of the run lengths down the column -- but the work is split by ROLE instead of
// by phase:
//   * one PRODUCER thread keeps three plane tiles in flight (cp.async.bulk.tensor.3d, one box of 144 x (64 + 2R + 1)
//     floats per disparity, zero-filled outside the image) behind full / ready / empty mbarriers;
//   * four PREFIX warps turn each landed tile into row prefixes in place: two tile rows per warp instruction
//     (16 lanes x 9 consecutive columns each, bank-conflict free at the 144-float pitch), two such pairs interleaved
//     (the scan is a chain of dependent adds and shuffles), a 4-step shuffle scan.  The prefixes are centred: one
//     value per tile (its mid pixel) is subtracted first, so that |I| stays a random walk instead of growing with the
//     mean of the plane (less cancellation in the differences); the walkers add it back to every output;
//   * eight WALKER warps: thread = (column, half of the 64 output rows).  A thread walks 32 + 2R tile rows once;
//     per row one LDS of the right image's arms, one packed 16-bit minimum against its own column's arms (registers
//     for the whole disparity chunk), two prefix look-ups -> (S, run length), added as a packed f32x2 to the running
//     (T, N) pair, which goes into a per-thread ring of 16 rows in shared memory.  The output of row y is emitted
//     R rows later as the difference of two ring entries, a reciprocal with one Newton step, one store.
//     No block-wide barrier in the steady state.
// Compared with cbca_tma.cu (32-row tiles, 2 CTAs per SM, prefix and walk as barrier-separated phases): 40 % fewer
// shared-memory wavefronts per output, 64-row tiles (halo overhead 1.25 instead of 1.4 / 1.5), and centred prefixes.
// NOT bit-exact by construction (1e-4 contract; measured ~1e-7).
// Arms up to 5 pixels (R <= 4, the KITTI presets); longer arms stay on cbca_tma.cu / the exact kernels.
#include "internal.cuh"

namespace {

constexpr int WS_TX = 128, WS_TY = 64;
constexpr int WS_HO = 32;                   // output rows per walker thread
constexpr int WS_NWT = WS_TX * (WS_TY / WS_HO);   // walker threads: column x row group
constexpr int WS_NPW = 4;                   // prefix warps
constexpr int WS_NT = WS_NWT + 32 * WS_NPW + 32;  // walkers + prefix warps + one producer warp
constexpr int WS_NST = 3;                   // tile stages
constexpr int WS_RING = 16;                 // rows of (T, N) per walker thread (>= 2R + 2; a power of two: cheap wrap)
constexpr int WS_DCH = 20;                  // max disparities per CTA
constexpr int WS_WW = WS_TX + WS_DCH;       // pitch of the right-image arm windows
constexpr int WS_TWP = 144;                 // tile pitch = TMA box width: 16 lanes x 9 columns, = 16 (mod 32)

template <int R>
struct WSCfg {
	static constexpr int HALO = R + 1;                 // the prefix differences index the first EXCLUDED pixel
	static constexpr int HX = (HALO + 3) & ~3;         // left halo in columns (TMA: 16-byte aligned start along x)
	static constexpr int TH = WS_TY + 2 * R + 1;       // image rows y0 - HALO .. y0 + TY + R - 1
	static constexpr int NWALK = 2 * R + WS_HO;        // rows a thread walks for its WS_HO outputs
	static constexpr int TILE_BYTES = TH * WS_TWP * 4; // bytes one TMA box delivers
	static constexpr int STAGE_BYTES = (TILE_BYTES + 127) & ~127;
	static constexpr int OFF_WINH = WS_NST * STAGE_BYTES;
	static constexpr int OFF_WINV = OFF_WINH + ((TH * WS_WW * 4 + 15) & ~15);
	static constexpr int OFF_MU = OFF_WINV + ((WS_TY * WS_WW * 2 + 15) & ~15);
	static constexpr int OFF_BAR = OFF_MU + 16;
	static constexpr int OFF_RING = OFF_BAR + ((3 * WS_NST * 8 + 15) & ~15);   // [WS_RING][WS_NWT] (T, N) per thread
	static constexpr int SMEM = OFF_RING + WS_RING * WS_NWT * 8;
	static_assert(SMEM <= 232448, "shared memory budget");
	static_assert(WS_RING >= 2 * R + 2, "ring too small");
	static_assert(HX + WS_TX + R <= WS_TWP, "tile pitch too small");
	static_assert(TH <= 256, "TMA box limit");
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tma_smem_addr(bar)) : "memory");
}
__device__ __forceinline__ unsigned long long ws_pack2(float lo, float hi)
{
	unsigned long long r;
	asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
	return r;
}
__device__ __forceinline__ unsigned long long ws_add2(unsigned long long a, unsigned long long b)
{
	unsigned long long d;
	asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
	return d;
}

// planes [da, db) of the tile (x0, y0): out = vol (the entries with x + d * direction outside the image, :353-354), as aligned
// float4 copies with 8 independent loads in flight per thread (rows start 16-byte aligned: x0 % 128 == 0, ld % 4 == 0)
__device__ __forceinline__ void ws_copy_planes(const float *__restrict__ vol, float *__restrict__ out, int da, int db, int x0, int y0,
					       int H, int W, int ld, int tid, int nthreads)
{
	constexpr int Q = WS_TX / 4;                             // float4 per tile row
	const int total = (db - da) * WS_TY * Q;
#pragma unroll 8
	for (int i = tid; i < total; i += nthreads) {
		const int q = i % Q, r = (i / Q) % WS_TY, d = da + i / (Q * WS_TY);
		const int y = y0 + r, x = x0 + 4 * q;
		if (y >= H || x >= W) continue;
		const long idx = ((long)d * H + y) * ld + x;
		if (x + 3 < W) {
			*reinterpret_cast<float4 *>(out + idx) = __ldg(reinterpret_cast<const float4 *>(vol + idx));
		} else {
			for (int e = 0; x + e < W; e++) out[idx + e] = __ldg(vol + idx + e);
		}
	}
}

// Centring: the prefix warps subtract one value per tile (the tile's mid pixel, 0 when that is not finite) before the row
// prefix; the running sums then carry deviations only, and the walkers add the value back to each quotient.
// (Two other ways for an output to gather its rows were measured slower: 2R + 1 predicated add.rn.f32x2, which ptxas
// turns into FADD2 + 2 SEL each, and 2R + 1 fma.rn.f32x2 with 0/1 masks.)
template <int R, int WB>
__global__ void __launch_bounds__(WS_NT, 1)
cbca_ws_kernel(const __grid_constant__ CUtensorMap tmap,
	       const uint32_t *__restrict__ a0h, const uint32_t *__restrict__ a0v,
	       const uint32_t *__restrict__ a1h, const uint32_t *__restrict__ a1v,
	       const float *__restrict__ vol, float *__restrict__ out,
	       int D, int H, int W, int ld, int direction, int dch)
{
	using C = WSCfg<R>;
	constexpr int HALO = C::HALO, HX = C::HX, TH = C::TH, NWALK = C::NWALK, TWP = WS_TWP;
	extern __shared__ __align__(128) unsigned char ws_smem[];
	uint32_t *winH = reinterpret_cast<uint32_t *>(ws_smem + C::OFF_WINH);   // [TH][WS_WW] right-image H words
	uint16_t *winV = reinterpret_cast<uint16_t *>(ws_smem + C::OFF_WINV);   // [WS_TY][WS_WW] right-image U | D << 8
	float *mus = reinterpret_cast<float *>(ws_smem + C::OFF_MU);            // [WS_NST] centre value of the stage's tile
	uint64_t *bar_full = reinterpret_cast<uint64_t *>(ws_smem + C::OFF_BAR);   // TMA landed
	uint64_t *bar_ready = bar_full + WS_NST;                                   // prefixes done
	uint64_t *bar_empty = bar_ready + WS_NST;                                  // walkers done

	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int x0 = blockIdx.x * WS_TX, y0 = blockIdx.y * WS_TY, d0 = blockIdx.z * dch;
	const int dn = min(dch, D - d0);
	const int a1x0 = direction > 0 ? x0 + d0 : x0 - (d0 + dch - 1);   // image column of window column 0

	// disparities whose tile is not entirely inside the invalid triangle form a prefix of the chunk (:353-354)
	int nproc = 0;
	while (nproc < dn && !(direction < 0 ? (x0 + WS_TX - 1 - (d0 + nproc) < 0) : (x0 + d0 + nproc >= W))) nproc++;

	if (nproc == 0) {                                      // the whole chunk lies in the invalid triangle: a plain copy, no staging
		ws_copy_planes(vol, out, d0, d0 + dn, x0, y0, H, W, ld, tid, WS_NT);
		return;
	}
	if (tid == 0) {
#pragma unroll
		for (int s = 0; s < WS_NST; s++) {
			mbar_init(&bar_full[s], 1);
			mbar_init(&bar_ready[s], WS_NPW);
			mbar_init(&bar_empty[s], WS_NWT / 32);
		}
		mbar_fence_init();
		tma_prefetch_desc(&tmap);
	}
	__syncthreads();

	constexpr int W_PROD = WS_NWT / 32 + WS_NPW;       // warp whose lane 0 issues the TMA
	if (warp == W_PROD && lane == 0) {                 // the first tiles fly while the arm windows are staged
#pragma unroll
		for (int s = 0; s < WS_NST; s++)
			if (s < nproc) {
				mbar_arrive_expect_tx(&bar_full[s], C::TILE_BYTES);
				tma_load_3d(ws_smem + s * C::STAGE_BYTES, &tmap, x0 - HX, y0 - HALO, d0 + s, &bar_full[s]);
			}
	}

	// right-image arm windows (once per CTA), 0 outside the image: a warp per window row, lanes along x.  Only the walkers
	// need them: they stage them among themselves (named barrier) while the prefix warps already work on the first tile
	if (warp < WS_NWT / 32) {
		constexpr int NW = WS_NWT / 32, NCH = (WS_WW + 31) / 32;
		for (int r = warp; r < TH; r += NW) {
			const int yy = y0 - HALO + r;
			const bool rowok = yy >= 0 && yy < H;
			const uint32_t *grow = a1h + (long)(rowok ? yy : 0) * W;
#pragma unroll
			for (int m = 0; m < NCH; m++) {
				const int j = lane + 32 * m, xx = a1x0 + j;
				if (j < WS_WW) {
					const bool ok = rowok && xx >= 0 && xx < W;
					const unsigned dst = (unsigned)__cvta_generic_to_shared(winH + r * WS_WW + j);
					const int nbytes = ok ? 4 : 0;
					asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(grow + (ok ? xx : 0)), "r"(nbytes));
				}
			}
		}
		asm volatile("cp.async.commit_group;");
		for (int r = warp; r < WS_TY; r += NW) {
			const int yy = y0 + r;
			const uint32_t *grow = a1v + (long)(yy < H ? yy : 0) * W;
			uint32_t v[NCH];
#pragma unroll
			for (int m = 0; m < NCH; m++) {
				const int xx = a1x0 + lane + 32 * m;
				v[m] = (yy < H && xx >= 0 && xx < W) ? __ldg(grow + xx) : 0u;
			}
#pragma unroll
			for (int m = 0; m < NCH; m++) {
				const int j = lane + 32 * m;
				if (j < WS_WW) winV[r * WS_WW + j] = (uint16_t)(((v[m] >> 8) & 255u) | ((v[m] >> 16) & 0xff00u));   // U | D << 8
			}
		}
		asm volatile("cp.async.wait_group 0;");
		asm volatile("bar.sync 2, %0;" ::"n"(WS_NWT) : "memory");   // windows visible to the walkers
	}

	if (warp == W_PROD) {
		// ---------------------------------------------------------------- producer
		if (lane == 0) {
			for (int dd = WS_NST; dd < nproc; dd++) {
				const int s = dd % WS_NST, k = dd / WS_NST;
				mbar_wait(&bar_empty[s], (k - 1) & 1);          // the walkers are done with plane dd - NST
				mbar_arrive_expect_tx(&bar_full[s], C::TILE_BYTES);
				tma_load_3d(ws_smem + s * C::STAGE_BYTES, &tmap, x0 - HX, y0 - HALO, d0 + dd, &bar_full[s]);
			}
		}
		return;
	}

	if (warp >= WS_NWT / 32) {
		// ---------------------------------------------------------------- prefix warps
		constexpr int EPL = 9;
		static_assert(EPL * 16 == TWP, "two rows per warp: 16 lanes x 9 columns");
		const int pw = warp - WS_NWT / 32;
		const int half = lane >> 4, li = lane & 15;
		for (int dd = 0; dd < nproc; dd++) {
			const int s = dd % WS_NST, d = d0 + dd;
			float *P = reinterpret_cast<float *>(ws_smem + s * C::STAGE_BYTES);
			// does the tile hold entries of the invalid triangle (NaN)?  They never lie inside a run, but a prefix
			// sum would carry them along the row: count them as 0.
			const bool scrub = direction < 0 ? (x0 - HX - d < 0) : (x0 - HX + TWP + d > W);
			mbar_wait(&bar_full[s], (dd / WS_NST) & 1);
			const float m = P[(HALO + WS_TY / 2) * TWP + HX + WS_TX / 2];
			const float mu = (fabsf(m) <= 3.0e38f) ? m : 0.0f;   // finite (NaN and inf fail the compare)
			if (pw == 0 && lane == 0) mus[s] = mu;
			asm volatile("bar.sync 1, %0;" ::"n"(32 * WS_NPW) : "memory");   // every prefix warp has read it before any row is rewritten
			// two independent row pairs per iteration (the scan of one is a chain of dependent adds and shuffles: a single
			// pair per iteration left the prefix warps latency-bound and the walkers waiting for them)
			constexpr int UP = 2;
			for (int pr0 = pw; pr0 < (TH + 1) / 2; pr0 += UP * WS_NPW) {
				float v[UP][EPL];
				float *row[UP];
				bool act[UP];
#pragma unroll
				for (int u = 0; u < UP; u++) {
					const int r = 2 * (pr0 + u * WS_NPW) + half;
					act[u] = r < TH;
					row[u] = P + (act[u] ? r : 0) * TWP + li * EPL;
#pragma unroll
					for (int i = 0; i < EPL; i++) v[u][i] = row[u][i];
				}
#pragma unroll
				for (int u = 0; u < UP; u++) {
#pragma unroll
					for (int i = 0; i < EPL; i++) v[u][i] -= mu;
					if (scrub) {
#pragma unroll
						for (int i = 0; i < EPL; i++) v[u][i] = v[u][i] == v[u][i] ? v[u][i] : 0.0f;
					}
				}
#pragma unroll
				for (int i = 1; i < EPL; i++)
#pragma unroll
					for (int u = 0; u < UP; u++) v[u][i] += v[u][i - 1];
				float incl[UP];
#pragma unroll
				for (int u = 0; u < UP; u++) incl[u] = v[u][EPL - 1];
#pragma unroll
				for (int o = 1; o < 16; o <<= 1) {
					float up[UP];
#pragma unroll
					for (int u = 0; u < UP; u++) up[u] = __shfl_up_sync(0xffffffffu, incl[u], o, 16);
					if (li >= o) {
#pragma unroll
						for (int u = 0; u < UP; u++) incl[u] += up[u];
					}
				}
#pragma unroll
				for (int u = 0; u < UP; u++) {
					const float base = incl[u] - v[u][EPL - 1];
					if (act[u]) {
#pragma unroll
						for (int i = 0; i < EPL; i++) row[u][i] = v[u][i] + base;
					}
				}
			}
			fence_proxy_async_smem();                      // generic writes of this stage before its next TMA refill
			__syncwarp();
			if (lane == 0) mbar_arrive(&bar_ready[s]);
		}
		return;
	}

	// -------------------------------------------------------------------- walkers
	const int c = tid & (WS_TX - 1), h = tid >> 7;      // column, row group (output rows HO h .. HO h + HO - 1)
	const int x = x0 + c;
	const int yb = y0 + WS_HO * h;                       // first output row of this thread
	const int nv = x < W ? max(0, min(WS_HO, H - yb)) : 0;   // output rows of this thread inside the image
	// this thread's own column of the left image's arms: registers for the whole chunk
	uint32_t ah[NWALK], av[WS_HO];
#pragma unroll
	for (int w = 0; w < NWALK; w++) {
		const int yy = yb - HALO + 1 + w;
		ah[w] = (x < W && yy >= 0 && yy < H) ? __ldg(a0h + (long)yy * W + x) : 0u;
	}
#pragma unroll
	for (int k = 0; k < WS_HO; k++) {
		const int yy = yb + k;
		av[k] = (x < W && yy < H) ? __ldg(a0v + (long)yy * W + x) : 0u;
	}

	for (int dd = 0; dd < nproc; dd++) {
		const int d = d0 + dd, s = dd % WS_NST;
		const float *P = reinterpret_cast<const float *>(ws_smem + s * C::STAGE_BYTES);
		const int sh = d * direction;
		const int xs = x + sh;
		const bool valid_col = x < W && xs >= 0 && xs < W;
		const int off = (x0 + sh) - a1x0;                 // window column of tile column 0
		mbar_wait(&bar_ready[s], (dd / WS_NST) & 1);
		const float mu = mus[s];

		// column walk: relative row rr <-> tile row 32h + rr <-> image row yb - HALO + rr
		const char *Pc = reinterpret_cast<const char *>(P + (WS_HO * h) * TWP + c + HX);   // own pixel's prefix entry, relative row 0
		const uint32_t *wh = winH + (WS_HO * h) * WS_WW + c + off;
		const uint16_t *wv = winV + (WS_HO * h) * WS_WW + c + off;
		char *po = reinterpret_cast<char *>(out + ((long)d * H + yb) * ld + x);
		const long ldb = (long)ld * 4;
		const int nst = valid_col ? nv : 0;                          // rows this thread stores from the walk
		constexpr int RROW = WS_NWT * 8;                             // ring row pitch in bytes
		char *rgb = reinterpret_cast<char *>(ws_smem + C::OFF_RING) + tid * 8;
		unsigned long long run = ws_pack2(0.0f, 0.0f);
		*reinterpret_cast<unsigned long long *>(rgb) = run;          // relative row 0: the excluded row of output 0
		// rows in batches of WB: all the shared-memory reads of a batch are issued before its arithmetic
#pragma unroll
		for (int b0 = 1; b0 <= NWALK; b0 += WB) {
			uint32_t hw[WB], vw[WB];
			float ph[WB], pl[WB];
#pragma unroll
			for (int i = 0; i < WB; i++) {
				const int rr = b0 + i;
				if (rr <= NWALK) {
					hw[i] = __vminu2(ah[rr - 1], wh[rr * WS_WW]);   // min of lengths = (max of left ends, min of right ends), :362-363
					if (rr >= 2 * R + 1) {
						const int k = rr - 2 * R - 1;
						vw[i] = __vminu2(av[k], __byte_perm((uint32_t)wv[k * WS_WW], 0u, 0x1404));   // :359-360
					}
				}
			}
#pragma unroll
			for (int i = 0; i < WB; i++) {
				const int rr = b0 + i;
				if (rr <= NWALK) {
					const int L4 = hw[i] & 0xffffu, R4 = hw[i] >> 16;
					const char *pr = Pc + rr * (TWP * 4);
					ph[i] = *reinterpret_cast<const float *>(pr + R4);
					pl[i] = *reinterpret_cast<const float *>(pr - L4);
				}
			}
#pragma unroll
			for (int i = 0; i < WB; i++) {
				const int rr = b0 + i;
				if (rr > NWALK) continue;
				const int L4 = hw[i] & 0xffffu, R4 = hw[i] >> 16;
				// run length L + R_ - 1 = (L4 + R4) / 4 as a float without a conversion: (2^23 + m) / 4 - 2^21, all exact
				const float nf = fmaf(__int_as_float(0x4B000000 + L4 + R4), 0.25f, -2097152.0f);   // :368
				const float S = ph[i] - pl[i];                         // sum of the run (x - L, x + R_), :364-367
				run = ws_add2(run, ws_pack2(S, nf));
				*reinterpret_cast<unsigned long long *>(rgb + (rr % WS_RING) * RROW) = run;
				if (rr >= 2 * R + 1) {
					const int k = rr - 2 * R - 1;                    // output row yb + k = relative row HALO + k = k + R + 1
					const unsigned U8 = vw[i] & 0xffffu, D8 = vw[i] >> 16;   // U << 8, Dn << 8
					constexpr int RB = WS_RING * RROW;
					constexpr int SC = RROW / 256;                 // U8 = U << 8: U8 * SC = U * RROW
					const int rk = HALO + k;
					// rows y - U + 1 .. y + Dn - 1 (:361): run(rk + Dn - 1) - run(rk - U); the ring index wraps only
					// where the (compile-time) row position says it can
					const int sb = (rk - 1) % WS_RING, sb2 = rk % WS_RING;
					int oh = D8 * SC + sb * RROW;
					if (sb + R + 1 >= WS_RING) oh &= RB - 1;
					int ol = sb2 * RROW - U8 * SC;
					if (sb2 - R - 1 < 0) ol = (ol + RB) & (RB - 1);
					const float2 a = *reinterpret_cast<const float2 *>(rgb + oh), b = *reinterpret_cast<const float2 *>(rgb + ol);
					const float T = a.x - b.x, N = a.y - b.y;
					float rc;
					asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(N));   // count >= 1
					float q = T * rc;
					q = fmaf(fmaf(-q, N, T), rc, q);                     // one Newton step: T / N to the last bit or so (:373)
					q += mu;
					asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.s32 p, %2, %3;\n\t@p st.global.f32 [%0], %1;\n\t}" ::"l"(po), "f"(q), "r"(k), "r"(nst)
						     : "memory");
					po += ldb;
				}
			}
		}
		if (!valid_col && nv > 0) {                        // x + d*direction outside the image: plain copy, keeps NaN (:353-354)
			const long idx0 = ((long)d * H + yb) * ld + x;
#pragma unroll 8
			for (int k = 0; k < nv; k++) out[idx0 + (long)k * ld] = __ldg(vol + idx0 + (long)k * ld);
		}
		// the walkers only READ the stage: the mbarrier release / acquire orders those reads before the refill (the
		// proxy fence is needed after generic WRITES, i.e. in the prefix warps; here it would also wait for the
		// thread's global stores to drain, once per plane)
		__syncwarp();
		if (lane == 0) mbar_arrive(&bar_empty[s]);
	}
	if (nproc < dn) {                                      // planes entirely inside the invalid triangle: plain copy
		ws_copy_planes(vol, out, d0 + nproc, d0 + dn, x0, y0, H, W, ld, tid, WS_NWT);
	}
}

template <int R, int WB>
int launch_ws(const CUtensorMap &tm, const uint32_t *hv, const float *vol, float *out, int D, int H, int W, int ld, int direction,
	      cudaStream_t s)
{
	using C = WSCfg<R>;
	static bool attr_done[64] = {false};
	int dev = 0;
	cudaGetDevice(&dev);
	if (!attr_done[dev & 63]) {
		ADC_CUDA(cudaFuncSetAttribute(cbca_ws_kernel<R, WB>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
		attr_done[dev & 63] = true;
	}
	const int dch = adc_div_up(D, adc_div_up(D, WS_DCH));   // equal chunks (19 x 12 at D = 228)
	const long HW = (long)H * W;
	dim3 grid(adc_div_up(W, WS_TX), adc_div_up(H, WS_TY), adc_div_up(D, dch));
	cbca_ws_kernel<R, WB><<<grid, WS_NT, C::SMEM, s>>>(tm, hv, hv + 2 * HW, hv + HW, hv + 3 * HW, vol, out, D, H, W, ld, direction, dch);
	ADC_CHECK_LAUNCH();
	return 0;
}

}  // namespace

// ---- internal entry points (cbca_tma.cu dispatches here for short arms) ------------------------------
int adc_cbca_ws_max_halo() { return 4; }

void adc_cbca_ws_box(int halo, int *box_w, int *box_h)
{
	*box_w = WS_TWP;
	*box_h = halo <= 1 ? WSCfg<1>::TH : WSCfg<4>::TH;
}

// hv: packed arms (adc_pack_arms_hv); tm: tensor map of `vol` with the box of adc_cbca_ws_box(halo)
int adc_cbca_ws(const CUtensorMap *tm, const uint32_t *hv, const float *vol, float *out, int D, int H, int W, int ld, int direction,
		int halo, cudaStream_t s)
{
	if (halo <= 1) return launch_ws<1, 6>(*tm, hv, vol, out, D, H, W, ld, direction, s);
	if (halo <= 4) return launch_ws<4, 4>(*tm, hv, vol, out, D, H, W, ld, direction, s);
	return ADCENSUS_ELIMIT;
}
