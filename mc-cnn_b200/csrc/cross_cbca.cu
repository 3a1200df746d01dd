// cross_cbca.cu -- adcensus.cross and adcensus.cbca for sm_100a.
//
// cross (adcensus.cu:280-341): per pixel, the four exclusive arm end-points.
// Tiny (4*H*W outputs, <= L1 steps each); one thread per (arm, pixel).
//
// cbca (adcensus.cu:343-400): cross-based cost aggregation.  The reference does
// up to (2*L1-1)^2 scattered global loads per output plus 4 float arm loads per
// support row.  Here:
//   * the float arm coordinates of both images are packed once per call into one
//     32-bit word per pixel (4 arm LENGTHS as bytes).  In relative form the
//     support of output (d,y,x) with xs = x + d*direction is
//         rows  y - min(U0(y,x),U1(y,xs)) < yy < y + min(D0(y,x),D1(y,xs))
//         cols  x - min(L0(yy,x),L1(yy,xs)) < xx < x + min(R0(yy,x),R1(yy,xs))
//     so one __vminu4 of two packed words replaces 4 loads + 2 max/min + 2 cvt;
//   * a CTA owns a 16x64 pixel tile and loops over a chunk of disparities; the
//     packed arms of the tile (left image) and of the shifted window (right image)
//     are loaded into shared memory once per CTA, the volume plane tile (+halo)
//     once per disparity (shared-memory line stencil), so every tap is an LDS;
//   * taps are summed in the reference's order (rows outer, columns inner, one
//     fp32 accumulator, adcensus.cu:361-370) => bit-identical volumes.
// Roofline: read V + write V (V = 4*D*H*W bytes) per iteration; this exact-order
// version is bound by shared-memory/FADD issue (one dependent FADD per tap), not
// by HBM -- see DESIGN.md.
#include <stdlib.h>

#include "internal.cuh"

namespace {

// ------------------------------------------------------------------ cross
__global__ void cross_kernel(const float *__restrict__ img, float *__restrict__ out, int H, int W, int L1, float tau1)
{
	long id = (long)blockIdx.x * blockDim.x + threadIdx.x;
	long HW = (long)H * W;
	if (id >= 4 * HW) return;
	int x = (int)(id % W);
	int y = (int)((id / W) % H);
	int dir = (int)(id / HW);
	int dx = dir == 0 ? -1 : (dir == 1 ? 1 : 0);
	int dy = dir == 2 ? -1 : (dir == 3 ? 1 : 0);
	float c = __ldg(img + (long)y * W + x);
	int xx = x + dx, yy = y + dy;
	for (;; xx += dx, yy += dy) {
		if (xx < 0 || xx >= W || yy < 0 || yy >= H) break;            // :307
		int dist = max(abs(xx - x), abs(yy - y));
		if (dist == 1) continue;                                       // :310
		if (fabsf(c - __ldg(img + (long)yy * W + xx)) >= tau1) break;  // :315
		if (dist >= L1) break;                                         // :318
	}
	out[id] = dir <= 1 ? xx : yy;                                      // :320
}

// ------------------------------------------------------------------ arm packing
// word = L | R<<8 | U<<16 | D<<24 with L = x - left end-point etc. (all >= 1 for arms made by cross)
// clamp > 0: lengths are cut at `clamp` (the caller's stated longest arm): the window / tile kernels size their shared-memory
// walks by it, so an understated bound gives a truncated support instead of an out-of-bounds read
__global__ void pack_arms_kernel(const float *__restrict__ xc, uint32_t *__restrict__ packed, int H, int W, int *maxlen, int clamp)
{
	int id = blockIdx.x * blockDim.x + threadIdx.x;
	int HW = H * W;
	int m = 0;
	if (id < HW) {
		int x = id % W, y = id / W;
		int l = x - (int)xc[id];
		int r = (int)xc[HW + id] - x;
		int u = y - (int)xc[2 * HW + id];
		int d = (int)xc[3 * HW + id] - y;
		m = max(max(l, r), max(u, d));
		int lo = min(min(l, r), min(u, d));
		if (lo < 0) m = 1 << 20;  // not a cross() output: force the generic kernel
		const int hi = clamp > 0 ? min(clamp, 255) : 255;
		l = min(max(l, 0), hi); r = min(max(r, 0), hi);
		u = min(max(u, 0), hi); d = min(max(d, 0), hi);
		packed[id] = (uint32_t)l | ((uint32_t)r << 8) | ((uint32_t)u << 16) | ((uint32_t)d << 24);
	}
	m = __reduce_max_sync(0xffffffffu, m);
	if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(maxlen, m);
}

// packed fp32 pairs for FFMA2 (sm_100a): two independent round-to-nearest fmas per instruction
__device__ __forceinline__ unsigned long long adc_pack2(float lo, float hi)
{
	unsigned long long r;
	asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
	return r;
}
__device__ __forceinline__ void adc_unpack2(unsigned long long v, float &lo, float &hi)
{
	asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long adc_fma2(unsigned long long a, unsigned long long b, unsigned long long c)
{
	unsigned long long d;
	asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
	return d;
}

// ------------------------------------------------------------------ cbca, fixed-window column strips
// (arms up to 5 pixels: every KITTI preset, main.lua:86-113,207-262)
//
// A thread owns ONE column and NVT = 16 consecutive output rows of one disparity plane and walks
// the NVT + 2R tile rows covering all their supports once.  Per tile row it loads the 2R+1 window
// columns and the row's combined horizontal arms (L, R_), and masks the window ONCE: slots outside
// the run (x - L, x + R_) become +0.0f (one compare + one select per slot, shared by every output
// that uses this row).  Every output whose vertical arm may contain the row then accumulates
// acc = fmaf(wm[k], q, acc) (two outputs per FFMA2, see the kernel body) in column order with q in {0.0f, 1.0f} (row inside its vertical arm,
// adcensus.cu:361): no predicates (nine live outputs per row would spill the 7 predicate registers).
// Exactness: fmaf(w, 1, acc) is acc + w (one rounding of the same real number); fmaf(w, 0, acc)
// adds +-0.0f to an accumulator that is never -0.0f (it starts at +0.0f and a sum is -0.0f only
// if both operands are) => acc unchanged.  (Moving the masks to FADD.SAT/FMUL on the FMA pipe and
// the arm minima to VIMNMX.U16x2 was measured slower: 1.15 ms vs 1.02 ms with scalar FFMA; the
// FFMA2 pairing took 1.02 ms to 0.92 ms.)  The order of the real
// additions per output is rows ascending, columns ascending => bit-identical to adcensus.cu:361-370.
// The masks are selects, so NaNs of the invalid triangle (never inside a run) are dropped; the
// accumulation itself needs finite values inside the runs, i.e. a volume that is finite on its
// valid part (the reference asserts !isnan there, adcensus.cu:366).
// No data-dependent loop, no divergence; stores are 32 consecutive columns per warp instruction.
constexpr int CW_TX = 128, CW_NVT = 16, CW_TY = 2 * CW_NVT, CW_DCH_MAX = 24, CW_NT = 256;

template <int R>
struct CWCfg {
	static constexpr int TH = CW_TY + 2 * R;
	static constexpr int TWP = CW_TX + 2 * R + 1;               // odd pitch: conflict-free column walks
	static constexpr int A1W = CW_TX + CW_DCH_MAX;             // right-image arm window for up to CW_DCH_MAX disparities
	// two plane-tile buffers (double-buffered)
	static constexpr int SMEM = (TH * CW_TX + TH * A1W + TH * CW_TX + 2 * TH * TWP) * 4;
};

// vol / out: (D, H, ld) with row pitch ld >= W (ld == W for the API-facing contiguous tensors)
template <int R>
__global__ void __launch_bounds__(CW_NT, 2)
cbca_win_kernel(const uint32_t *__restrict__ a0g, const uint32_t *__restrict__ a1g,
		const float *__restrict__ vol, float *__restrict__ out, int D, int H, int W, int ld, int direction, int dch,
		const int *__restrict__ gate, int gate_lo, int gate_hi)
{
	// device-side kernel selection (adcensus_cbca): run only if the longest arm, known on the device, is in this kernel's range
	if (gate && (*gate < gate_lo || *gate > gate_hi)) return;
	using Cfg = CWCfg<R>;
	constexpr int TH = Cfg::TH, TWP = Cfg::TWP, A1W = Cfg::A1W;
	extern __shared__ __align__(16) uint32_t cw_smem[];
	uint32_t *sa0 = cw_smem;                       // [TH][CW_TX]  left-image packed arms (L | R<<8 | U<<16 | D<<24) of the tile
	uint32_t *sa1 = sa0 + TH * CW_TX;              // [TH][A1W]    right-image packed arms, shifted window
	uint32_t *scomb = sa1 + TH * A1W;              // [TH][CW_TX]  byte-wise minimum of both for the current d
	float *svbuf = reinterpret_cast<float *>(scomb + TH * CW_TX);  // 2 x [TH][TWP] volume plane tile + halo

	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int x0 = blockIdx.x * CW_TX, y0 = blockIdx.y * CW_TY, d0 = blockIdx.z * dch;   // dch <= CW_DCH_MAX disparities per CTA
	const int dn = min(dch, D - d0);
	const int a1x0 = direction > 0 ? x0 + d0 : x0 - (d0 + dch - 1);
	const long HW = (long)H * ld;                  // elements per plane

	const int cx = 32 * (warp & 3) + lane;         // this thread's tile column
	const int ry = CW_NVT * (warp >> 2);           // first of its NVT output rows (tile-relative)
	const int x = x0 + cx;
	constexpr int NW = CW_NT / 32;

	// packed arms: one warp per tile row, lanes along x (no index division anywhere)
	for (int r = warp; r < TH; r += NW) {
		const int yy = y0 - R + r;
		const bool rowok = yy >= 0 && yy < H;
#pragma unroll
		for (int m = 0; m < CW_TX / 32; m++) {
			int c = lane + 32 * m, xx = x0 + c;
			sa0[r * CW_TX + c] = (rowok && xx < W) ? __ldg(a0g + yy * W + xx) : 0u;
		}
#pragma unroll
		for (int m = 0; m < (A1W + 31) / 32; m++) {
			int c = lane + 32 * m, xx = a1x0 + c;
			if (c < A1W) sa1[r * A1W + c] = (rowok && xx >= 0 && xx < W) ? __ldg(a1g + yy * W + xx) : 0u;
		}
	}

	// Disparities whose whole tile lies inside the invalid triangle (x + d*direction outside the image
	// for every column) form a suffix of the chunk: plain copy, adcensus.cu:353-354, handled last.
	int nproc = 0;
	while (nproc < dn && !(direction < 0 ? (x0 + CW_TX - 1 - (d0 + nproc) < 0) : (x0 + d0 + nproc >= W))) nproc++;

	// volume plane tile (+halo) of disparity d into `buf`: cp.async, 4-byte granules (rows of W floats
	// are only 4-byte aligned), zero-filled outside the image
	auto issue_tile = [&](int d, float *buf) {
		const float *plane = vol + (long)d * HW;
		for (int r = warp; r < TH; r += NW) {
			const int yy = y0 - R + r;
			const bool rowok = yy >= 0 && yy < H;
			const float *grow = plane + (long)(rowok ? yy : 0) * ld;
#pragma unroll
			for (int m = 0; m < (TWP + 31) / 32; m++) {
				const int c = lane + 32 * m, xx = x0 - R + c;
				if (c < TWP) {
					const bool ok = rowok && xx >= 0 && xx < W;
					const unsigned dst = (unsigned)__cvta_generic_to_shared(buf + r * TWP + c);
					const int nbytes = ok ? 4 : 0;
					asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(grow + (ok ? xx : 0)), "r"(nbytes));
				}
			}
		}
	};
	// the tile of disparity dd+1 streams into the other buffer while dd is aggregated
	constexpr int PD = 1;
	if (nproc > 0) {
		issue_tile(d0, svbuf);
		asm volatile("cp.async.commit_group;");
	}
	for (int dd = 0; dd < nproc; dd++) {
		const int d = d0 + dd;
		const int off = (x0 + d * direction) - a1x0;   // sa1 column of tile column 0
		const int xs = x + d * direction;
		const bool valid_col = x < W && xs >= 0 && xs < W;
		float *sv = svbuf + (PD ? (dd & 1) : 0) * TH * TWP;
		__syncthreads();                               // previous plane consumed; arms visible
		if (PD == 1) {
			if (dd + 1 < nproc) issue_tile(d + 1, svbuf + ((dd + 1) & 1) * TH * TWP);
		} else {
			issue_tile(d, sv);
		}
		asm volatile("cp.async.commit_group;");
		// combined arms of this disparity: byte-wise min of the left arms at x and the right arms at x + d*dir
		for (int r = warp; r < TH; r += NW) {
#pragma unroll
			for (int m = 0; m < CW_TX / 32; m++) {
				const int c = lane + 32 * m;
				scomb[r * CW_TX + c] = __vminu4(sa0[r * CW_TX + c], sa1[r * A1W + c + off]);
			}
		}
		asm volatile("cp.async.wait_group %0;" ::"n"(PD));
		__syncthreads();
		// Outputs are accumulated in PAIRS (rows 2j, 2j+1) with the packed FFMA2 of sm_100a
		// (fma.rn.f32x2: two independent IEEE fmas per instruction): {acc[2j], acc[2j+1]} +=
		// {q[2j], q[2j+1]} * wm[k].  A row touches 2R+1 outputs = R+1 pairs, so a slot costs R+1
		// instructions instead of 2R+1; the pair member outside the range gets q = 0 (acc unchanged).
		int U[CW_NVT], Dn[CW_NVT];
		unsigned long long acc2[CW_NVT / 2], cnt2[CW_NVT / 2];
#pragma unroll
		for (int oy = 0; oy < CW_NVT; oy++) {
			const uint32_t c = scomb[(ry + oy + R) * CW_TX + cx];
			U[oy] = (c >> 16) & 255;
			Dn[oy] = c >> 24;
		}
#pragma unroll
		for (int j = 0; j < CW_NVT / 2; j++) acc2[j] = cnt2[j] = adc_pack2(0.0f, 0.0f);

#pragma unroll
		for (int ri = 0; ri < CW_NVT + 2 * R; ri++) {
			const float *wrow = sv + (ry + ri) * TWP + cx;     // window column k of this thread: image column x - R + k
			const uint32_t c = scomb[(ry + ri) * CW_TX + cx];
			const int L = c & 255, Rr = (c >> 8) & 255;
			const float LRf = (float)(L + Rr - 1);             // taps of this row's run (:364-369), exact in fp32
			const unsigned long long LR2 = adc_pack2(LRf, LRf);
			unsigned long long wm2[2 * R + 1];
#pragma unroll
			for (int k = 0; k <= 2 * R; k++) {
				// slot inside the run (x - L, x + Rr) (:362-364) keeps its value, the others become +0.0f
				const float v = wrow[k];
				const float w = k < R ? (L > R - k ? v : 0.0f) : (k > R ? (Rr > k - R ? v : 0.0f) : (L > 0 ? v : 0.0f));
				wm2[k] = adc_pack2(w, w);
			}
#pragma unroll
			for (int j = 0; j < CW_NVT / 2; j++) {
				// row offset from the centre rows of outputs 2j and 2j+1
				const int dlo = ri - 2 * j - R, dhi = dlo - 1;
				const bool inlo = dlo >= -R && dlo <= R, inhi = dhi >= -R && dhi <= R;
				if (!inlo && !inhi) continue;
				// 1.0f for a row inside the output's vertical arm (:361); the centre row iff the output is valid
				const float qlo = inlo && (dlo < 0 ? U[2 * j] > -dlo : Dn[2 * j] > dlo) ? 1.0f : 0.0f;
				const float qhi = inhi && (dhi < 0 ? U[2 * j + 1] > -dhi : Dn[2 * j + 1] > dhi) ? 1.0f : 0.0f;
				const unsigned long long q2 = adc_pack2(qlo, qhi);
#pragma unroll
				for (int k = 0; k <= 2 * R; k++) acc2[j] = adc_fma2(q2, wm2[k], acc2[j]);   // :364-367
				cnt2[j] = adc_fma2(q2, LR2, cnt2[j]);                                          // :368
			}
		}
#pragma unroll
		for (int oy = 0; oy < CW_NVT; oy++) {
			const int y = y0 + ry + oy;
			if (y >= H || x >= W) continue;
			float alo, ahi, clo, chi;
			adc_unpack2(acc2[oy / 2], alo, ahi);
			adc_unpack2(cnt2[oy / 2], clo, chi);
			float res = valid_col ? ((oy & 1) ? ahi / chi : alo / clo)                     // :373
					      : sv[(ry + oy + R) * TWP + cx + R];                      // :353-354 (keeps NaN)
			out[(long)d * HW + (long)y * ld + x] = res;
		}
	}
	for (int dd = nproc; dd < dn; dd++) {              // tiles entirely inside the invalid triangle
		const int d = d0 + dd;
		const float *plane = vol + (long)d * HW;
#pragma unroll
		for (int oy = 0; oy < CW_NVT; oy++) {
			const int y = y0 + ry + oy;
			if (y < H && x < W) out[(long)d * HW + (long)y * ld + x] = __ldg(plane + (long)y * ld + x);
		}
	}
}

// ------------------------------------------------------------------ cbca, shared-memory tile with run loops
// (arms of 6..14 pixels, e.g. the Middlebury presets)
constexpr int CB_TX = 64, CB_TY = 16, CB_DCH = 16, CB_NT = 256;

template <int R>  // halo = longest arm - 1
__global__ void __launch_bounds__(CB_NT)
cbca_loop_kernel(const uint32_t *__restrict__ a0g, const uint32_t *__restrict__ a1g,
		 const float *__restrict__ vol, float *__restrict__ out, int D, int H, int W, int ld, int direction,
		 const int *__restrict__ gate, int gate_lo, int gate_hi)
{
	if (gate && (*gate < gate_lo || *gate > gate_hi)) return;
	constexpr int TH = CB_TY + 2 * R;          // tile rows incl. halo
	constexpr int TW = CB_TX + 2 * R;          // volume tile columns incl. halo
	constexpr int A1W = CB_TX + CB_DCH;        // right-image arm window columns
	__shared__ uint32_t sa0[TH][CB_TX];
	__shared__ uint32_t sa1[TH][A1W];
	__shared__ float sv[TH][TW + 1];

	const int tid = threadIdx.x;
	const int x0 = blockIdx.x * CB_TX, y0 = blockIdx.y * CB_TY, d0 = blockIdx.z * CB_DCH;
	const int dn = min(CB_DCH, D - d0);
	// column of the right image that sa1[.][0] holds: xs = x + d*direction spans
	// [x0 + dlo, x0 + CB_TX - 1 + dhi] with (dlo,dhi) = (d0,d0+dn-1)*direction sorted
	const int a1x0 = direction > 0 ? x0 + d0 : x0 - (d0 + CB_DCH - 1);

	for (int i = tid; i < TH * CB_TX; i += CB_NT) {
		int r = i / CB_TX, c = i % CB_TX;
		int yy = y0 - R + r, xx = x0 + c;
		sa0[r][c] = (yy >= 0 && yy < H && xx < W) ? a0g[yy * W + xx] : 0u;
	}
	for (int i = tid; i < TH * A1W; i += CB_NT) {
		int r = i / A1W, c = i % A1W;
		int yy = y0 - R + r, xx = a1x0 + c;
		sa1[r][c] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? a1g[yy * W + xx] : 0u;
	}

	const int lx = tid % CB_TX;                // 0..63
	const int ly = tid / CB_TX;                // 0..3 ; rows ly, ly+4, ly+8, ly+12
	const int x = x0 + lx;
	const long HW = (long)H * ld;              // elements per plane

	for (int dd = 0; dd < dn; dd++) {
		const int d = d0 + dd;
		const float *plane = vol + (long)d * HW;
		__syncthreads();  // previous plane consumed (and arms visible on the first pass)
		for (int i = tid; i < TH * TW; i += CB_NT) {
			int r = i / TW, c = i % TW;
			int yy = y0 - R + r, xx = x0 - R + c;
			sv[r][c] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(plane + (long)yy * ld + xx) : 0.0f;
		}
		__syncthreads();
		const int xs = x + d * direction;
		const int c1 = xs - a1x0;              // column in sa1
#pragma unroll
		for (int k = 0; k < CB_TY / 4; k++) {
			const int y = y0 + ly + 4 * k;
			if (x >= W || y >= H) continue;
			const int r = ly + 4 * k + R;      // tile row of y
			float res;
			if (xs < 0 || xs >= W) {
				res = sv[r][lx + R];           // adcensus.cu:353-354 (keeps NaN)
			} else {
				uint32_t mc = __vminu4(sa0[r][lx], sa1[r][c1]);
				int up = (mc >> 16) & 255, dn_ = mc >> 24;
				float sum = 0.0f;
				int cnt = 0;
				for (int rr = r - up + 1; rr < r + dn_; rr++) {           // :361
					uint32_t m = __vminu4(sa0[rr][lx], sa1[rr][c1]);
					int lo = lx + R - (int)(m & 255) + 1;                  // :362
					int hi = lx + R + (int)((m >> 8) & 255);               // :363 (exclusive)
					const float *row = sv[rr];
					for (int cc = lo; cc < hi; cc++) sum += row[cc];       // :364-369
					cnt += hi - lo;
				}
				res = sum / (float)cnt;                                    // :373
			}
			out[(long)d * HW + (long)y * ld + x] = res;
		}
	}
}

// ------------------------------------------------------------------ cbca, generic (any arm length)
// Same arithmetic straight from global memory; used when an arm is longer than the
// largest shared-memory halo or the arms are not integer cross() outputs.
__global__ void cbca_generic_kernel(const float *__restrict__ x0c, const float *__restrict__ x1c,
				    const float *__restrict__ vol, float *__restrict__ out,
				    long size, int H, int W, int ld, int direction,
				    const int *__restrict__ gate, int gate_lo, int gate_hi)
{
	if (gate && (*gate < gate_lo || *gate > gate_hi)) return;
	long id = (long)blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= size) return;
	long HW = (long)H * W;
	int x = (int)(id % W);
	int y = (int)((id / W) % H);
	int d = (int)(id / HW);
	int xs = x + d * direction;
	const long prow = ((long)d * H) * ld;      // plane offset in the (D, H, ld) volumes
	if (xs < 0 || xs >= W) { out[prow + (long)y * ld + x] = vol[prow + (long)y * ld + x]; return; }
	float sum = 0.0f;
	int cnt = 0;
	int yy_s = (int)fmaxf(x0c[2 * HW + (long)y * W + x], x1c[2 * HW + (long)y * W + xs]);
	int yy_t = (int)fminf(x0c[3 * HW + (long)y * W + x], x1c[3 * HW + (long)y * W + xs]);
	for (int yy = yy_s + 1; yy < yy_t; yy++) {
		int xx_s = (int)fmaxf(x0c[(long)yy * W + x], x1c[(long)yy * W + xs] - d * direction);
		int xx_t = (int)fminf(x0c[HW + (long)yy * W + x], x1c[HW + (long)yy * W + xs] - d * direction);
		for (int xx = xx_s + 1; xx < xx_t; xx++) {
			sum += __ldg(vol + prow + (long)yy * ld + xx);
			cnt++;
		}
	}
	out[prow + (long)y * ld + x] = sum / (float)cnt;
}

template <int R>
int launch_win(const uint32_t *a0, const uint32_t *a1, const float *vol, float *out, int D, int H, int W, int ld, int direction, cudaStream_t s,
	       const int *gate = nullptr, int gate_lo = 0, int gate_hi = 0)
{
	using Cfg = CWCfg<R>;
	constexpr int SMEM = Cfg::SMEM;
	static bool attr_done[64] = {false};
	int dev = 0;
	cudaGetDevice(&dev);
	if (!attr_done[dev & 63]) {
		ADC_CUDA(cudaFuncSetAttribute(cbca_win_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
		attr_done[dev & 63] = true;
	}
	// disparities per CTA.  Measured at 370x1226x228: 4..12 -> 1.01-1.04 ms, 16 -> 1.01 ms, 19 (whole
	// waves) -> 1.08 ms: the kernel is issue-bound and balances dynamically, so the chunk size hardly
	// matters; 10 keeps the per-chunk re-staging of the packed arms (L2 traffic only) small.
	constexpr int dch = 10;
	static_assert(dch <= CW_DCH_MAX, "arm window too narrow");
	dim3 grid(adc_div_up(W, CW_TX), adc_div_up(H, CW_TY), adc_div_up(D, dch));
	cbca_win_kernel<R><<<grid, CW_NT, SMEM, s>>>(a0, a1, vol, out, D, H, W, ld, direction, dch, gate, gate_lo, gate_hi);
	return 0;
}

template <int R>
void launch_tile(const uint32_t *a0, const uint32_t *a1, const float *vol, float *out, int D, int H, int W, int ld, int direction, cudaStream_t s,
		 const int *gate = nullptr, int gate_lo = 0, int gate_hi = 0)
{
	dim3 grid(adc_div_up(W, CB_TX), adc_div_up(H, CB_TY), adc_div_up(D, CB_DCH));
	cbca_loop_kernel<R><<<grid, CB_NT, 0, s>>>(a0, a1, vol, out, D, H, W, ld, direction, gate, gate_lo, gate_hi);
}

}  // namespace

// ---- internal entry points shared with pipeline.cu -------------------------
// packed buffer layout (uint32 words, HW = H*W): [image 0 | image 1]
size_t adc_packed_words(int H, int W) { return 2 * (size_t)H * W; }

static int pack_arms(const float *xc, uint32_t *pk, int which, int H, int W, int *maxlen_dev, int clamp, cudaStream_t s)
{
	const long HW = (long)H * W;
	pack_arms_kernel<<<adc_div_up(HW, 256), 256, 0, s>>>(xc, pk + which * HW, H, W, maxlen_dev, clamp);
	ADC_CHECK_LAUNCH();
	return 0;
}

int adc_pack_arms(const float *xc, uint32_t *pk, int which, int H, int W, int *maxlen_dev, cudaStream_t s)
{
	return pack_arms(xc, pk, which, H, W, maxlen_dev, 0, s);
}

// Exact (bit-identical) aggregation.  maxlen = longest arm (distance to the exclusive end-point) of either
// image; vol / out are (D, H, ld) with ld >= W (ld == W: the API-facing contiguous tensors).
int adc_cbca_packed(const uint32_t *pk, const float *x0c, const float *x1c,
		    const float *vol, float *out, int D, int H, int W, int ld, int direction, int maxlen, cudaStream_t s)
{
	const long HW = (long)H * W;
	const uint32_t *a0 = pk, *a1 = pk + HW;
	int halo = maxlen - 1;
	if (halo <= 1) {
		int rc = launch_win<1>(a0, a1, vol, out, D, H, W, ld, direction, s);
		if (rc) return rc;
	} else if (halo <= 4) {
		int rc = launch_win<4>(a0, a1, vol, out, D, H, W, ld, direction, s);
		if (rc) return rc;
	}
	else if (halo <= 8) launch_tile<8>(a0, a1, vol, out, D, H, W, ld, direction, s);
	else if (halo <= 13) launch_tile<13>(a0, a1, vol, out, D, H, W, ld, direction, s);
	else {
		long size = (long)D * H * W;
		cbca_generic_kernel<<<adc_div_up(size, 256), 256, 0, s>>>(x0c, x1c, vol, out, size, H, W, ld, direction, nullptr, 0, 0);
	}
	ADC_CHECK_LAUNCH();
	return 0;
}

// Public split of adcensus_cbca for callers that aggregate several times with the same arms (main.lua
// runs cbca_i1 + cbca_i2 iterations per direction): pack both arm tensors once, then iterate.
extern "C" int mccnn_pack_arms(const float *x0c, const float *x1c, void *packed, int H, int W, adcensus_stream_t stream)
{
	if (!x0c || !x1c || !packed || H < 1 || W < 1) return ADCENSUS_EINVAL;
	cudaStream_t s = adc_stream(stream);
	uint32_t *pk = (uint32_t *)packed;
	const long HW = (long)H * W;
	int *maxlen_dev = (int *)(pk + adc_packed_words(H, W));
	int rc = (int)cudaMemsetAsync(maxlen_dev, 0, sizeof(int), s);
	if (!rc) rc = adc_pack_arms(x0c, pk, 0, H, W, maxlen_dev, s);
	if (!rc) rc = adc_pack_arms(x1c, pk, 1, H, W, maxlen_dev, s);
	return rc;
}

extern "C" size_t mccnn_packed_arms_bytes(int H, int W) { return (adc_packed_words(H, W) + 1) * sizeof(uint32_t); }

extern "C" int mccnn_cbca_packed(const void *packed, const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
				 int D, int H, int W, int direction, int max_arm, adcensus_stream_t stream)
{
	if (!packed || !x0c || !x1c || !vol_in || !vol_out || vol_in == vol_out) return ADCENSUS_EINVAL;
	if (D < 1 || H < 1 || W < 1 || (direction != 1 && direction != -1) || max_arm < 1) return ADCENSUS_EINVAL;
	const uint32_t *pk = (const uint32_t *)packed;
	return adc_cbca_packed(pk, x0c, x1c, vol_in, vol_out, D, H, W, W, direction, max_arm, adc_stream(stream));
}

extern "C" int adcensus_cross(const float *x0, float *out, int H, int W, int L1, float tau1, adcensus_stream_t stream)
{
	if (!x0 || !out || H < 1 || W < 1) return ADCENSUS_EINVAL;
	long n = 4L * H * W;
	cross_kernel<<<adc_div_up(n, 256), 256, 0, adc_stream(stream)>>>(x0, out, H, W, L1, tau1);
	ADC_CHECK_LAUNCH();
	return 0;
}

extern "C" int adcensus_cbca_ex(const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
				int D, int H, int W, int direction, int max_arm, adcensus_stream_t stream)
{
	if (!x0c || !x1c || !vol_in || !vol_out || vol_in == vol_out) return ADCENSUS_EINVAL;
	if (D < 1 || H < 1 || W < 1 || (direction != 1 && direction != -1) || max_arm < 1) return ADCENSUS_EINVAL;
	cudaStream_t s = adc_stream(stream);
	long HW = (long)H * W;
	uint32_t *packed = nullptr;
	int rc = adc_scratch_alloc((void **)&packed, (adc_packed_words(H, W) + 1) * sizeof(uint32_t), s);
	if (rc) return rc;
	int *maxlen_dev = (int *)(packed + adc_packed_words(H, W));
	rc = (int)cudaMemsetAsync(maxlen_dev, 0, sizeof(int), s);
	const int clamp = max_arm <= 14 ? max_arm : 0;            // beyond 14 the generic kernel reads the float arms themselves
	if (!rc) rc = pack_arms(x0c, packed, 0, H, W, maxlen_dev, clamp, s);
	if (!rc) rc = pack_arms(x1c, packed, 1, H, W, maxlen_dev, clamp, s);
	if (!rc) rc = adc_cbca_packed(packed, x0c, x1c, vol_in, vol_out, D, H, W, W, direction, max_arm, s);
	int rc2 = adc_scratch_free(packed, s);
	return rc ? rc : rc2;
}

extern "C" int adcensus_cbca(const float *x0c, const float *x1c, const float *vol_in, float *vol_out,
			     int D, int H, int W, int direction, adcensus_stream_t stream)
{
	if (!x0c || !x1c || !vol_in || !vol_out || vol_in == vol_out) return ADCENSUS_EINVAL;
	if (D < 1 || H < 1 || W < 1 || (direction != 1 && direction != -1)) return ADCENSUS_EINVAL;
	cudaStream_t s = adc_stream(stream);
	const long HW = (long)H * W;
	uint32_t *packed = nullptr;
	int rc = adc_scratch_alloc((void **)&packed, (adc_packed_words(H, W) + 1) * sizeof(uint32_t), s);
	if (rc) return rc;
	int *maxlen_dev = (int *)(packed + adc_packed_words(H, W));
	rc = (int)cudaMemsetAsync(maxlen_dev, 0, sizeof(int), s);
	if (!rc) rc = adc_pack_arms(x0c, packed, 0, H, W, maxlen_dev, s);
	if (!rc) rc = adc_pack_arms(x1c, packed, 1, H, W, maxlen_dev, s);
	if (!rc) {
		// The longest arm is only known on the device.  Instead of reading it back (a host synchronisation per call),
		// every candidate kernel is launched with a gate on that device value; the ones out of range return at once.
		const uint32_t *a0 = packed, *a1 = packed + HW;
		rc = launch_win<1>(a0, a1, vol_in, vol_out, D, H, W, W, direction, s, maxlen_dev, 0, 2);
		if (!rc) rc = launch_win<4>(a0, a1, vol_in, vol_out, D, H, W, W, direction, s, maxlen_dev, 3, 5);
		if (!rc) {
			launch_tile<8>(a0, a1, vol_in, vol_out, D, H, W, W, direction, s, maxlen_dev, 6, 9);
			launch_tile<13>(a0, a1, vol_in, vol_out, D, H, W, W, direction, s, maxlen_dev, 10, 14);
			const long size = (long)D * H * W;
			cbca_generic_kernel<<<adc_div_up(size, 256), 256, 0, s>>>(x0c, x1c, vol_in, vol_out, size, H, W, W, direction, maxlen_dev, 15, 1 << 30);
			rc = (int)cudaPeekAtLastError();
		}
	}
	int rc2 = adc_scratch_free(packed, s);
	return rc ? rc : rc2;
}
