// cbca_tma.cu -- cross-based cost aggregation with CONSTANT WORK PER PIXEL (adcensus.cbca, adcensus.cu:343-400)
// for sm_100a: TMA-staged plane tiles, prefix sums along x, one column walk per thread.
// This is the first generation.  Arms of up to 5 pixels go to the second generation (cbca_ws.cu, faster and more
// accurate); this kernel is kept as the constant-work path for arms of 6-14 pixels behind mccnn_cbca_fast_pitched*.
//
// The reference gathers up to (2*L1-1)^2 taps per output.  The run of a support row depends on (d, row,
// column) only, not on which output row uses it, so with I = inclusive prefix of the tile row
//     S(r, x)   = I(r, x + R_ - 1) - I(r, x - L)                  sum of the run (x - L, x + R_)  (:362-369)
//     out(y, x) = (T(y + Dn - 1, x) - T(y - U, x)) / (N(y + Dn - 1, x) - N(y - U, x))           (:361, :373)
// where T, N are the running sums of S and of the run lengths down the column.  That is ~45 instructions
// per output instead of ~200 for the tap-by-tap order, which makes the kernel HBM-bound territory (2V bytes
// per iteration).  NOT bit-exact by construction: it serves the north star's 1e-4 bar for float aggregation
// (measured ~1e-6 relative; prefixes are local to a 32 x 128 tile + halo, which bounds the cancellation).
// The bit-exact kernels stay in cross_cbca.cu and remain selectable.
//
// Per CTA: a 32 x 128 pixel tile, a chunk of `dch` disparities.
//   * the plane tile (+halo, zero-filled outside the image; its first column 16-byte aligned, which the TMA
//     requires of the innermost coordinate) of every disparity arrives by ONE TMA box
//     (cp.async.bulk.tensor.3d on the (W, H, D) view of the pitched volume), double-buffered on two
//     mbarriers: plane d + 2 streams in while d + 1 is processed;
//   * row prefix sums in place: a warp per row, five consecutive columns per lane, lane totals combined by a
//     shuffle scan (one read and one write of the tile, bank-conflict free);
//   * thread = (column, half of the output rows): it walks 2R + 16 tile rows once; per row one LDS of the
//     right image's arms (window staged once per CTA), one VIMNMX.U16x2 against its own column's arms
//     (registers), two prefix lookups, and the running (T, N) pair goes into a per-thread shared-memory
//     ring of 2R + 2 rows; the output of row y is emitted R rows later from two ring reads.
// Arms are pre-packed per image into H words (4L | 4(R-1) << 16) and V words (U << 8 | D << 24), lengths
// relative to the pixel, so "max of left ends / min of right ends" is one packed 16-bit minimum.
#include "internal.cuh"

namespace {

constexpr int CT_TX = 128, CT_TY = 32, CT_NT = 256, CT_HO = CT_TY / 2;
constexpr int CT_WB = 4;                   // rows per walk batch
constexpr int CT_DCH = 20;                 // disparities per CTA (window width); the per-CTA staging of the arm windows is amortised over them
constexpr int CT_WW = CT_TX + CT_DCH;      // pitch of the right-image arm windows

template <int R>
struct CTCfg {
	static constexpr int HALO = R + 1;                 // the prefix differences index the first EXCLUDED pixel
	static constexpr int HX = (HALO + 3) & ~3;         // left halo in columns: TMA needs a 16-byte aligned start along x
	static constexpr int TH = CT_TY + 2 * R + 1;       // image rows y0 - HALO .. y0 + TY + R - 1
	static constexpr int TWMIN = HX + CT_TX + R;       // image columns x0 - HX .. x0 + TX + R - 1
	static constexpr int SEG = 20;                     // the tile pitch is a multiple of 20 floats (16-byte rows for TMA, 5 per lane for the row scan)
	static constexpr int NSEG = (TWMIN + SEG - 1) / SEG;
	static constexpr int TWP = NSEG * SEG;             // tile pitch = TMA box width (160 floats)
	static constexpr int RING = 32;                    // >= 2R + 2 rows of (T, N) per thread
	static constexpr int NWALK = 2 * R + CT_HO;        // rows a thread walks for its 16 outputs
	static constexpr int TILE_BYTES = TH * TWP * 4;    // = bytes one TMA box delivers
	static constexpr int STAGE_BYTES = (TILE_BYTES + 127) & ~127;
	static constexpr int OFF_RING = 2 * STAGE_BYTES;
	static constexpr int OFF_WINH = OFF_RING + RING * CT_NT * 8;
	static constexpr int OFF_WINV = OFF_WINH + TH * CT_WW * 4;
	static constexpr int OFF_BAR = OFF_WINV + ((CT_TY * CT_WW * 2 + 15) & ~15);
	static constexpr int SMEM = OFF_BAR + 16;
	static_assert(RING >= 2 * R + 2, "ring too small");
	static_assert(TWP <= 256 && TH <= 256, "TMA box limits");
};

template <int R>
__global__ void __launch_bounds__(CT_NT, (CTCfg<R>::SMEM <= 112 * 1024) ? 2 : 1)
cbca_tma_kernel(const __grid_constant__ CUtensorMap tmap,
		const uint32_t *__restrict__ a0h, const uint32_t *__restrict__ a0v,
		const uint32_t *__restrict__ a1h, const uint32_t *__restrict__ a1v,
		const float *__restrict__ vol, float *__restrict__ out,
		int D, int H, int W, int ld, int direction, int dch)
{
	using C = CTCfg<R>;
	constexpr int HALO = C::HALO, HX = C::HX, TH = C::TH, TWP = C::TWP, RING = C::RING, NWALK = C::NWALK;
	extern __shared__ __align__(128) unsigned char ct_smem[];
	float2 *ring = reinterpret_cast<float2 *>(ct_smem + C::OFF_RING);       // [RING][CT_NT] (T, N) per thread
	uint32_t *winH = reinterpret_cast<uint32_t *>(ct_smem + C::OFF_WINH);   // [TH][CT_WW] right-image H words
	uint16_t *winV = reinterpret_cast<uint16_t *>(ct_smem + C::OFF_WINV);   // [CT_TY][CT_WW] right-image U | D << 8
	uint64_t *bars = reinterpret_cast<uint64_t *>(ct_smem + C::OFF_BAR);

	const int tid = threadIdx.x;
	const int c = tid & (CT_TX - 1), h = tid >> 7;      // column, half (output rows 16h .. 16h + 15)
	const int x0 = blockIdx.x * CT_TX, y0 = blockIdx.y * CT_TY, d0 = blockIdx.z * dch;
	const int dn = min(dch, D - d0);
	const int a1x0 = direction > 0 ? x0 + d0 : x0 - (d0 + dch - 1);   // image column of window column 0
	const int x = x0 + c;
	const int yb = y0 + CT_HO * h;                       // first output row of this thread
	const int nv = x < W ? max(0, min(CT_HO, H - yb)) : 0;   // output rows of this thread inside the image

	// disparities whose tile is not entirely inside the invalid triangle form a prefix of the chunk (:353-354)
	int nproc = 0;
	while (nproc < dn && !(direction < 0 ? (x0 + CT_TX - 1 - (d0 + nproc) < 0) : (x0 + d0 + nproc >= W))) nproc++;

	if (tid == 0) {
		mbar_init(&bars[0], 1);
		mbar_init(&bars[1], 1);
		mbar_fence_init();
		tma_prefetch_desc(&tmap);
	}
	__syncthreads();
	if (tid == 0) {
#pragma unroll
		for (int s = 0; s < 2; s++)
			if (s < nproc) {
				mbar_arrive_expect_tx(&bars[s], C::TILE_BYTES);
				tma_load_3d(ct_smem + s * C::STAGE_BYTES, &tmap, x0 - HX, y0 - HALO, d0 + s, &bars[s]);
			}
	}

	// right-image arm windows (once per CTA), 0 outside the image: a warp per window row, lanes along x.  The H words
	// go straight to shared memory (cp.async, zero-filled outside the image; waited for before the first walk), the V
	// words are narrowed to U | D << 8 on the way.
	{
		const int lane = tid & 31, warp = tid >> 5;
		constexpr int NW = CT_NT / 32, NCH = (CT_WW + 31) / 32;
		for (int r = warp; r < TH; r += NW) {
			const int yy = y0 - HALO + r;
			const bool rowok = yy >= 0 && yy < H;
			const uint32_t *grow = a1h + (long)(rowok ? yy : 0) * W;
#pragma unroll
			for (int m = 0; m < NCH; m++) {
				const int j = lane + 32 * m, xx = a1x0 + j;
				if (j < CT_WW) {
					const bool ok = rowok && xx >= 0 && xx < W;
					const unsigned dst = (unsigned)__cvta_generic_to_shared(winH + r * CT_WW + j);
					const int nbytes = ok ? 4 : 0;
					asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(grow + (ok ? xx : 0)), "r"(nbytes));
				}
			}
		}
		asm volatile("cp.async.commit_group;");
		for (int r = warp; r < CT_TY; r += NW) {
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
				if (j < CT_WW) winV[r * CT_WW + j] = (uint16_t)(((v[m] >> 8) & 255u) | ((v[m] >> 16) & 0xff00u));   // U | D << 8
			}
		}
	}
	// this thread's own column of the left image's arms: registers for the whole chunk
	uint32_t ah[NWALK], av[CT_HO];
#pragma unroll
	for (int w = 0; w < NWALK; w++) {
		const int yy = yb - HALO + 1 + w;
		ah[w] = (x < W && yy >= 0 && yy < H) ? __ldg(a0h + (long)yy * W + x) : 0u;
	}
#pragma unroll
	for (int k = 0; k < CT_HO; k++) {
		const int yy = yb + k;
		av[k] = (x < W && yy < H) ? __ldg(a0v + (long)yy * W + x) : 0u;
	}

	for (int dd = 0; dd < nproc; dd++) {
		const int d = d0 + dd, s = dd & 1;
		float *P = reinterpret_cast<float *>(ct_smem + s * C::STAGE_BYTES);
		const int sh = d * direction;
		const int xs = x + sh;
		const bool valid_col = x < W && xs >= 0 && xs < W;
		const int off = (x0 + sh) - a1x0;                 // window column of tile column 0
		// does the tile hold entries of the invalid triangle (NaN)?  They never lie inside a run, but a
		// prefix sum would carry them along the row: count them as 0.
		const bool clean = direction < 0 ? (x0 - HX - d < 0) : (x0 + CT_TX + R + d >= W);
		mbar_wait(&bars[s], (dd >> 1) & 1);

		// 1. inclusive prefix of every tile row, in place: a warp per row, a lane owns EPL consecutive columns (stride-5 word
		// accesses are bank-conflict free), lane totals combined by a shuffle scan -- one read and one write of the tile
		{
			constexpr int EPL = 5, NLN = TWP / EPL;
			static_assert(TWP % EPL == 0 && NLN <= 32, "row does not fit one warp");
			const int lane = tid & 31;
			for (int r = tid >> 5; r < TH; r += CT_NT / 32) {
				float *row = P + r * TWP + lane * EPL;
				float v[EPL];
#pragma unroll
				for (int i = 0; i < EPL; i++) v[i] = lane < NLN ? row[i] : 0.0f;
				if (clean) {
#pragma unroll
					for (int i = 0; i < EPL; i++) v[i] = v[i] == v[i] ? v[i] : 0.0f;
				}
#pragma unroll
				for (int i = 1; i < EPL; i++) v[i] += v[i - 1];
				float incl = v[EPL - 1];
#pragma unroll
				for (int o = 1; o < 32; o <<= 1) {
					const float up = __shfl_up_sync(0xffffffffu, incl, o);
					if (lane >= o) incl += up;
				}
				const float base = incl - v[EPL - 1];
				if (lane < NLN) {
#pragma unroll
					for (int i = 0; i < EPL; i++) row[i] = v[i] + base;
				}
			}
		}
		if (dd == 0) asm volatile("cp.async.wait_group 0;");   // the arm windows of this chunk have landed
		__syncthreads();

		// 2. column walk: relative row rr <-> tile row 16h + rr <-> image row yb - HALO + rr.
		// H words hold 4L | 4(R-1) << 16 (byte offsets into the prefix row), V words U << 8 | (D << 8) << 16
		// (x 8 = byte offsets into the ring, whose rows are CT_NT * 8 = 2048 bytes apart); the ring carries
		// (4T, 4N): the factor drops out of the quotient.
		const char *Pc = reinterpret_cast<const char *>(P + (CT_HO * h) * TWP + c + HX);   // own pixel's prefix entry, relative row 0
		const uint32_t *wh = winH + (CT_HO * h) * CT_WW + c + off;
		const uint16_t *wv = winV + (CT_HO * h) * CT_WW + c + off;
		char *rgb = reinterpret_cast<char *>(ring + tid);
		constexpr int RROW = CT_NT * 8, RMASK = RING * RROW - 1;
		char *po = reinterpret_cast<char *>(out + ((long)d * H + yb) * ld + x);
		const long ldb = (long)ld * 4;
		const int nst = valid_col ? nv : 0;                          // rows this thread stores from the walk
		float T = 0.0f;
		int N = 0;
		*reinterpret_cast<float2 *>(rgb) = make_float2(0.0f, __int_as_float(0));   // relative row 0: the excluded row of output 0
		// rows in batches of CT_WB: all the shared-memory reads of a batch are issued before its (short) serial part, so that
		// their latency overlaps (the kernel is latency-, not bandwidth-bound at 16 warps per SM)
#pragma unroll
		for (int b0 = 1; b0 <= NWALK; b0 += CT_WB) {
			uint32_t hw[CT_WB], vw[CT_WB];
			float ph[CT_WB], pl[CT_WB];
#pragma unroll
			for (int i = 0; i < CT_WB; i++) {
				const int rr = b0 + i;
				if (rr <= NWALK) {
					hw[i] = __vminu2(ah[rr - 1], wh[rr * CT_WW]);   // min of lengths = (max of left ends, min of right ends), :362-363
					if (rr >= 2 * R + 1) {
						const int k = rr - 2 * R - 1;
						vw[i] = __vminu2(av[k], __byte_perm((uint32_t)wv[k * CT_WW], 0u, 0x1404));   // :359-360
					}
				}
			}
#pragma unroll
			for (int i = 0; i < CT_WB; i++) {
				const int rr = b0 + i;
				if (rr <= NWALK) {
					const int L4 = hw[i] & 0xffffu, R4 = hw[i] >> 16;
					const char *pr = Pc + rr * (TWP * 4);
					ph[i] = *reinterpret_cast<const float *>(pr + R4);
					pl[i] = *reinterpret_cast<const float *>(pr - L4);
				}
			}
#pragma unroll
			for (int i = 0; i < CT_WB; i++) {
				const int rr = b0 + i;
				if (rr > NWALK) continue;
				const int L4 = hw[i] & 0xffffu, R4 = hw[i] >> 16;
				T = fmaf(ph[i] - pl[i], 4.0f, T);                    // + 4 x sum of the run (x - L, x + R_), :364-367
				N += L4 + R4;                                        // + 4 x its length, :368
				*reinterpret_cast<float2 *>(rgb + (rr & (RING - 1)) * RROW) = make_float2(T, __int_as_float(N));
				if (rr >= 2 * R + 1) {
					constexpr int M = RING - 1;
					const int k = rr - 2 * R - 1;                    // output row yb + k = relative row HALO + k
					const int rk = HALO + k;
					const int U8 = vw[i] & 0xffffu, D8 = vw[i] >> 16;
					// rows y - U + 1 .. y + Dn - 1 (:361): T(rk + Dn - 1) - T(rk - U); the ring index wraps only
					// where the (compile-time) row position says it can
					int oh = D8 * 8 + (((rk - 1) & M) * RROW);
					if (((rk - 1) & M) + R + 1 > M) oh &= RMASK;
					int ol = ((rk & M) * RROW) - U8 * 8;
					if ((rk & M) - R - 1 < 0) ol = (ol + RING * RROW) & RMASK;
					const float2 a = *reinterpret_cast<const float2 *>(rgb + oh), b = *reinterpret_cast<const float2 *>(rgb + ol);
					const float cnt = (float)(__float_as_int(a.y) - __float_as_int(b.y));
					float rc;
					asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(cnt));   // count >= 1; 1-ulp reciprocal, inside the 1e-4 contract
					const float res = (a.x - b.x) * rc;                       // :373
					asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.s32 p, %2, %3;\n\t@p st.global.f32 [%0], %1;\n\t}" ::"l"(po), "f"(res), "r"(k), "r"(nst)
						     : "memory");
					po += ldb;
				}
			}
		}
		if (!valid_col && nv > 0) {                        // x + d*direction outside the image: plain copy, keeps NaN (:353-354)
			const long idx0 = ((long)d * H + yb) * ld + x;
			for (int k = 0; k < nv; k++) out[idx0 + (long)k * ld] = __ldg(vol + idx0 + (long)k * ld);
		}
		fence_proxy_async_smem();                          // generic-proxy accesses (the in-place prefix) before the TMA refill
		__syncthreads();                                   // every reader of this stage is done
		if (tid == 0 && dd + 2 < nproc) {
			mbar_arrive_expect_tx(&bars[s], C::TILE_BYTES);
			tma_load_3d(P, &tmap, x0 - HX, y0 - HALO, d + 2, &bars[s]);
		}
	}
	for (int dd = nproc; dd < dn; dd++) {                  // tiles entirely inside the invalid triangle: plain copy
		const int d = d0 + dd;
#pragma unroll
		for (int k = 0; k < CT_HO; k++) {
			const int y = yb + k;
			const long idx = ((long)d * H + y) * ld + x;
			if (y < H && x < W) out[idx] = __ldg(vol + idx);
		}
	}
}

// H word = 4L | 4(R-1) << 16, V word = U << 8 | (D << 8) << 16 (lengths relative to the pixel, pre-scaled to the byte
// offsets the kernel adds; a packed 16-bit minimum of two words is still the pair of minima)
__global__ void pack_arms_hv_kernel(const float *__restrict__ xc, uint32_t *__restrict__ hw, uint32_t *__restrict__ vw, int H, int W)
{
	const int id = blockIdx.x * blockDim.x + threadIdx.x;
	const int HW = H * W;
	if (id >= HW) return;
	const int x = id % W, y = id / W;
	int l = x - (int)xc[id];
	int r = (int)xc[HW + id] - x;
	int u = y - (int)xc[2 * HW + id];
	int d = (int)xc[3 * HW + id] - y;
	l = min(max(l, 0), 255); r = min(max(r, 1), 255);
	u = min(max(u, 0), 255); d = min(max(d, 0), 255);
	hw[id] = (uint32_t)(4 * l) | ((uint32_t)(4 * (r - 1)) << 16);
	vw[id] = ((uint32_t)u << 8) | ((uint32_t)d << 24);
}

template <int R>
int launch_tma(const CUtensorMap &tm, const uint32_t *hv, const float *vol, float *out, int D, int H, int W, int ld, int direction,
	       cudaStream_t s)
{
	using C = CTCfg<R>;
	static bool attr_done[64] = {false};
	int dev = 0;
	cudaGetDevice(&dev);
	if (!attr_done[dev & 63]) {
		ADC_CUDA(cudaFuncSetAttribute(cbca_tma_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
		attr_done[dev & 63] = true;
	}
	const long HW = (long)H * W;
	dim3 grid(adc_div_up(W, CT_TX), adc_div_up(H, CT_TY), adc_div_up(D, CT_DCH));
	cbca_tma_kernel<R><<<grid, CT_NT, C::SMEM, s>>>(tm, hv, hv + 2 * HW, hv + HW, hv + 3 * HW, vol, out, D, H, W, ld, direction, CT_DCH);
	ADC_CHECK_LAUNCH();
	return 0;
}

}  // namespace

// ---- internal entry points (pipeline.cu) ---------------------------------------------------------
// hv buffer layout (uint32 words, HW = H*W): [H words image 0 | H words image 1 | V words image 0 | V words image 1]
size_t adc_packed_hv_words(int H, int W) { return 4 * (size_t)H * W; }

int adc_pack_arms_hv(const float *xc, uint32_t *hv, int which, int H, int W, cudaStream_t s)
{
	const long HW = (long)H * W;
	pack_arms_hv_kernel<<<adc_div_up(HW, 256), 256, 0, s>>>(xc, hv + which * HW, hv + (2 + which) * HW, H, W);
	ADC_CHECK_LAUNCH();
	return 0;
}

// largest support radius (longest arm - 1) the constant-work kernel is instantiated for
static int adc_cbca_tma_max_halo() { return 13; }

// box of the tensor map a volume needs for support radius `halo` (= longest arm - 1)
void adc_cbca_tma_box(int halo, int *box_w, int *box_h)
{
	if (halo <= adc_cbca_ws_max_halo()) adc_cbca_ws_box(halo, box_w, box_h);
	else if (halo <= 8) { *box_w = CTCfg<8>::TWP; *box_h = CTCfg<8>::TH; }
	else { *box_w = CTCfg<13>::TWP; *box_h = CTCfg<13>::TH; }
}

// vol/out: (D, H, ld) with ld % 4 == 0 and 16-byte aligned bases; tm: tensor map of `vol` with the box of `halo`
int adc_cbca_tma(const CUtensorMap *tm, const uint32_t *hv, const float *vol, float *out, int D, int H, int W, int ld, int direction,
		 int halo, cudaStream_t s)
{
	if (halo <= adc_cbca_ws_max_halo()) return adc_cbca_ws(tm, hv, vol, out, D, H, W, ld, direction, halo, s);
	if (halo <= 8) return launch_tma<8>(*tm, hv, vol, out, D, H, W, ld, direction, s);
	if (halo <= 13) return launch_tma<13>(*tm, hv, vol, out, D, H, W, ld, direction, s);
	return ADCENSUS_ELIMIT;
}

// ---- public: one aggregation pass on pitched volumes ---------------------------------------------
// Constant-work aggregation (1e-4 contract, not bit-exact).  vol_in / vol_out are (D, H, ld) with ld >= W,
// ld % 4 == 0, 16-byte aligned; x0c / x1c are cross() outputs (4,H,W) with arms of at most max_arm <= 14 pixels.
extern "C" int mccnn_cbca_fast_pitched(const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
				       int D, int H, int W, int ld, int direction, int max_arm, adcensus_stream_t stream)
{
	if (!x0c || !x1c || !vol_in || !vol_out || vol_in == vol_out) return ADCENSUS_EINVAL;
	if (D < 1 || H < 1 || W < 1 || ld < W || (ld & 3) || (direction != 1 && direction != -1) || max_arm < 1) return ADCENSUS_EINVAL;
	if ((((uintptr_t)vol_in) | ((uintptr_t)vol_out)) & 15) return ADCENSUS_EINVAL;
	if (max_arm - 1 > adc_cbca_tma_max_halo()) return ADCENSUS_ELIMIT;
	cudaStream_t s = adc_stream(stream);
	CUtensorMap tm;
	int bw, bh;
	adc_cbca_tma_box(max_arm - 1, &bw, &bh);
	int rc = adc_tma_encode_volume(&tm, vol_in, D, H, W, ld, bw, bh);
	if (rc) return rc;
	uint32_t *hv = nullptr;
	rc = adc_scratch_alloc((void **)&hv, adc_packed_hv_words(H, W) * sizeof(uint32_t), s);
	if (rc) return rc;
	rc = adc_pack_arms_hv(x0c, hv, 0, H, W, s);
	if (!rc) rc = adc_pack_arms_hv(x1c, hv, 1, H, W, s);
	if (!rc) rc = adc_cbca_tma(&tm, hv, vol_in, vol_out, D, H, W, ld, direction, max_arm - 1, s);
	int rc2 = adc_scratch_free(hv, s);
	return rc ? rc : rc2;
}

// The two halves of mccnn_cbca_fast_pitched for callers that aggregate several times with the same arms (main.lua runs
// cbca_i1 + cbca_i2 iterations per direction): pack once into `hv` (mccnn_packed_hv_bytes(H, W) bytes), then iterate.
extern "C" size_t mccnn_packed_hv_bytes(int H, int W) { return adc_packed_hv_words(H, W) * sizeof(uint32_t); }

extern "C" int mccnn_pack_arms_hv(const float *x0c, const float *x1c, void *hv, int H, int W, adcensus_stream_t stream)
{
	if (!x0c || !x1c || !hv || H < 1 || W < 1) return ADCENSUS_EINVAL;
	int rc = adc_pack_arms_hv(x0c, (uint32_t *)hv, 0, H, W, adc_stream(stream));
	if (!rc) rc = adc_pack_arms_hv(x1c, (uint32_t *)hv, 1, H, W, adc_stream(stream));
	return rc;
}

extern "C" int mccnn_cbca_fast_pitched_packed(const void *hv, const float *vol_in, float *vol_out,
					      int D, int H, int W, int ld, int direction, int max_arm, adcensus_stream_t stream)
{
	if (!hv || !vol_in || !vol_out || vol_in == vol_out) return ADCENSUS_EINVAL;
	if (D < 1 || H < 1 || W < 1 || ld < W || (ld & 3) || (direction != 1 && direction != -1) || max_arm < 1) return ADCENSUS_EINVAL;
	if ((((uintptr_t)vol_in) | ((uintptr_t)vol_out)) & 15) return ADCENSUS_EINVAL;
	if (max_arm - 1 > adc_cbca_tma_max_halo()) return ADCENSUS_ELIMIT;
	CUtensorMap tm;
	int bw, bh;
	adc_cbca_tma_box(max_arm - 1, &bw, &bh);
	int rc = adc_tma_encode_volume(&tm, vol_in, D, H, W, ld, bw, bh);
	if (rc) return rc;
	return adc_cbca_tma(&tm, (const uint32_t *)hv, vol_in, vol_out, D, H, W, ld, direction, max_arm - 1, adc_stream(stream));
}
