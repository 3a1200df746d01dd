// sgm.cu -- adcensus.sgm2 for sm_100a.
//
// Replaces adcensus.cu:535-697: the reference launches one kernel per scan step
// (2*(W+H) = 3192 launches at 370x1226), each block re-reading the previous
// step's line state from global `tmp` and tree-reducing the min over D in shared
// memory.  Here one launch does a whole direction:
//   * ONE WARP PER SCANLINE keeps the line state L_r(p-r, .) in registers for the
//     entire scan; lane l owns the K consecutive disparities l*K .. l*K+K-1;
//   * the min over D is a K-element register tree + one `redux.sync.min.f32`
//     (CREDUX, sm_100a) instead of a shared-memory tree with 9 barriers;
//   * the d-1 / d+1 neighbours are registers (one shuffle each at lane borders);
//   * the cost vectors of the next PF pixels stream into a per-warp shared-memory
//     ring with cp.async (16-byte granules, each lane fetching exactly the
//     elements it will consume, so no barrier is needed), which keeps ~PF*2 KB per
//     warp in flight and hides HBM latency behind the serial recurrence;
//   * the P1/P2 selection (adcensus.cu:586-605) is table driven: a pre-pass
//     classifies |I(p) - I(p-r)| against tau_so once per image / scan axis into
//     byte tables (padded by D columns of the out-of-image class, D2 = 10).
//     Horizontal scans stage the two class rows of their image row in shared
//     memory and slide a register window of class bytes by one byte per step;
//     vertical scans fetch one pre-compared selector word per lane and step
//     (sgm_sel_kernel) through the cp.async ring;
//   * the two horizontal directions of a row run in ONE CTA (sgm_hpair_kernel)
//     when the accumulator is known to be zero, meeting at the row's midpoint.
//
// Arithmetic is the reference's, expression for expression (adds, fminf, IEEE
// divisions; nothing contractible), and `out` is accumulated in the reference's
// direction order (right, left, down, up) => bit-identical results for volumes
// whose valid disparities form a prefix per pixel (what StereoJoin / ad / census
// produce).  Padding slots d >= D are carried as NaN, which fminf ignores exactly
// like the reference's `d + 1 < size3` guard.
//
// Layout: input/output (H,W,D) like the reference (INDEX, adcensus.cu:531-533).
// Algorithmic traffic per call: 4 passes x (read input + read-modify-write
// output) = 12V bytes (V = 4*D*H*W); 11V when the caller guarantees a zeroed
// output (pipeline), because the first pass then skips the read.
#include "internal.cuh"

namespace {

struct SgmParams {
	float pi1, pi2, tau_so, alpha1, q1, q2;
	int direction;
	// band support: the volume (H,W,D) handed to a pass may be a row band or a column band of the
	// image; its pixel (y, x) is image pixel (yoff + y, xoff + x) of the Ht x Wt image the class
	// tables were built from.  Bands never cut a scanline of the pass they are used for.
	int Ht, Wt, yoff, xoff;
	// vertical scans over a ROW band of the image (wavefront split, rowband.py): the line state L_r(p - r, .) of the
	// row before the band enters through state_in and leaves through state_out ([line][32*K] floats; NULL: the scan
	// starts / ends at the image border); line0 .. line1: the scanlines (columns) of this launch
	const float *state_in;
	float *state_out;
	int line0, line1;
};

// ---------------------------------------------------------------- penalty class tables
// class of a colour difference against tau_so: 0 (< tau), 2 (> tau), 1 otherwise (== tau or NaN):
// exactly the three branches of adcensus.cu:596-605.
__device__ __forceinline__ uint8_t sgm_class(float diff, float tau)
{
	return diff < tau ? 0 : (diff > tau ? 2 : 1);
}

// tab layout: 4 planes [h0, v0, h1, v1], each H rows of pitch Wp = W + 2*pad bytes, image column
// j at byte pad + j.  h: |I[y][j] - I[y][j-1]|, v: |I[y][j] - I[y-1][j]|; entries whose
// neighbour is outside the image, and the padding, hold the class of D2 = 10 (adcensus.cu:591).
// Plane 0/1 from x0 (D1, always in range where used), plane 2/3 from x1 (D2).
__global__ void sgm_class_kernel(const float *__restrict__ x0, const float *__restrict__ x1, uint8_t *__restrict__ tab,
				 int H, int W, int pad, float tau)
{
	const int Wp = W + 2 * pad;
	const long plane = (long)H * Wp;
	long id = (long)blockIdx.x * blockDim.x + threadIdx.x;
	if (id >= plane) return;
	int y = (int)(id / Wp), j = (int)(id % Wp) - pad;
	const uint8_t oob = sgm_class(10.0f, tau);
	uint8_t h0 = oob, v0 = oob, h1 = oob, v1 = oob;
	if (j >= 0 && j < W) {
		long p = (long)y * W + j;
		if (j >= 1) {
			h0 = sgm_class(fabsf(x0[p] - x0[p - 1]), tau);
			h1 = sgm_class(fabsf(x1[p] - x1[p - 1]), tau);
		}
		if (y >= 1) {
			v0 = sgm_class(fabsf(x0[p] - x0[p - W]), tau);
			v1 = sgm_class(fabsf(x1[p] - x1[p - W]), tau);
		}
	}
	tab[id] = h0;
	tab[plane + id] = v0;
	tab[2 * plane + id] = h1;
	tab[3 * plane + id] = v1;
}

// Vertical scans: per (table row ty, band column x, lane) one word that already holds the outcome of
// the class comparisons of adcensus.cu:596-605 for the lane's K slots: bit k = (D2 class of slot k ==
// D1 class), bits 16-17 = D1 class.  Every step of a vertical scan is a new table row, so this word
// is the only class data a lane fetches per step (through the cp.async ring, like the costs).
__host__ __device__ inline size_t sgm_sel_offset(int Ht, int Wp) { return ((size_t)4 * Ht * Wp + 16 + 255) & ~(size_t)255; }

// block (32 lanes, 8 columns), grid (ceil(W / 8), Ht).  K % 4 == 0: the lane's K class bytes are read as
// K/4+1 aligned words and compared four at a time (classes are 0..2, so a byte of the xor with the D1
// class is zero iff neither of its two low bits is set).
template <int K>
__global__ void sgm_sel_kernel(const uint8_t *__restrict__ tab, unsigned *__restrict__ sel, int Ht, int W, int Wp, int pad,
			       int xoff, int ddir)
{
	const int lane = threadIdx.x, xb = blockIdx.x * 8 + threadIdx.y, ty = blockIdx.y;
	if (xb >= W) return;
	const long plane = (long)Ht * Wp;
	const long col = (long)ty * Wp + pad + xoff + xb;
	const unsigned c1 = __ldg(tab + plane + col);                // v0: D1 class (:587)
	const uint8_t *q = tab + 3 * plane + col + (long)lane * K * ddir;   // v1: D2 classes (:588-594), slot k at q[k * ddir]
	unsigned w = 0;
	if constexpr (K % 4 == 0) {
		const uintptr_t lo = (uintptr_t)(ddir > 0 ? q : q - (K - 1));
		const unsigned *al = reinterpret_cast<const unsigned *>(lo & ~(uintptr_t)3);
		const int sh = (int)(lo & 3) * 8;
		unsigned raw[K / 4 + 1];
#pragma unroll
		for (int i = 0; i <= K / 4; i++) raw[i] = __ldg(al + i);
#pragma unroll
		for (int i = 0; i < K / 4; i++) {
			const unsigned x = __funnelshift_r(raw[i], raw[i + 1], sh) ^ (c1 * 0x01010101u);
			const unsigned e = ~(x | (x >> 1)) & 0x01010101u;    // bit 8b set iff byte b equals c1
			w |= ((e * 0x00204081u) >> 21 & 0xfu) << (4 * i);      // gather bits 0, 8, 16, 24 -> 0..3 (ascending address)
		}
		if (ddir < 0) w = __brev(w) >> (32 - K);                 // slot k sits at the k-th address from the top
	} else {
		for (int k = 0; k < K; k++) w |= (unsigned)(__ldg(q + k * ddir) == c1) << k;
	}
	sel[((long)ty * W + xb) * 32 + lane] = w | (c1 << 16);
}

// ---------------------------------------------------------------- helpers
__device__ __forceinline__ float warp_min_f32(float v)
{
	float r;
	asm("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));  // NaN inputs are skipped
	return r;
}

__device__ __forceinline__ void cp_async16(float *smem_dst, const float *gsrc)
{
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void cp_async4(float *smem_dst, const float *gsrc)
{
	asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}

template <int K, bool VEC>
__device__ __forceinline__ void issue_vec(float *slot, const float *g, int dbase, int D)
{
	if constexpr (VEC) {
#pragma unroll
		for (int k = 0; k < K; k += 4)
			if (dbase + k < D) cp_async16(slot + k, g + k);
	} else {
#pragma unroll
		for (int k = 0; k < K; k++)
			if (dbase + k < D) cp_async4(slot + k, g + k);
	}
}

template <int K>
__device__ __forceinline__ void read_slot(float (&r)[K], const float *slot)
{
	if constexpr (K % 4 == 0) {
#pragma unroll
		for (int k = 0; k < K; k += 4) {
			float4 v = *reinterpret_cast<const float4 *>(slot + k);
			r[k] = v.x; r[k + 1] = v.y; r[k + 2] = v.z; r[k + 3] = v.w;
		}
	} else {
#pragma unroll
		for (int k = 0; k < K; k++) r[k] = slot[k];
	}
}

template <int K, bool VEC>
__device__ __forceinline__ void store_vec(const float (&r)[K], float *p, int dbase, int D)
{
	if constexpr (VEC) {
#pragma unroll
		for (int k = 0; k < K; k += 4)
			if (dbase + k < D) *reinterpret_cast<float4 *>(p + k) = make_float4(r[k], r[k + 1], r[k + 2], r[k + 3]);
	} else {
#pragma unroll
		for (int k = 0; k < K; k++)
			if (dbase + k < D) p[k] = r[k];
	}
}

// ---------------------------------------------------------------- one scan direction
// copy `nbytes` table bytes starting at `row` into shared memory with aligned word loads; returns
// the shared-memory address of row[0].  Reads at most 3 bytes before / after the range (inside the
// table, see adc_sgm_table_bytes).
__device__ __forceinline__ const uint8_t *sgm_stage_row(unsigned *dst, const uint8_t *row, int nbytes, int tid, int nthreads)
{
	const uintptr_t a = (uintptr_t)row;
	const unsigned *al = reinterpret_cast<const unsigned *>(a & ~(uintptr_t)3);
	const int mis = (int)(a & 3);
	const int nw = (mis + nbytes + 3) >> 2;
	for (int i = tid; i < nw; i += nthreads) dst[i] = __ldg(al + i);
	return reinterpret_cast<const uint8_t *>(dst) + mis;
}

__device__ __forceinline__ void cp_async4u(unsigned *smem_dst, const unsigned *gsrc)
{
	asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}

// State of one warp scanning one line.  SD: 0 right, 1 left, 2 down, 3 up (adcensus.cu:541-565).
//
// Penalty classes (D1: one byte per step; D2: the bytes at K consecutive table columns per lane):
//  horizontal scans: the CTA stages the two class rows of its image row in shared memory once; the
//    K bytes of step s+1 are those of step s moved by one slot, so each lane keeps them in a
//    register window that is shifted by one byte per step, with ONE byte read from shared memory;
//  vertical scans: every step is a new table row; a lane fetches ONE pre-compared selector word
//    (sgm_sel_kernel) per step through the same cp.async ring as the cost vectors, PF steps ahead.
//    (Class bytes loaded one step ahead with plain loads were the top stall: they queue behind the
//    streaming traffic and never hit L1.)
template <int K, bool VEC, int SD, int PF>
struct SgmScan {
	static constexpr int VSZ = 32 * K;             // floats per cost vector slot (padded to 32*K)
	static constexpr int dx = SD == 0 ? 1 : (SD == 1 ? -1 : 0);
	static constexpr int dy = SD == 2 ? 1 : (SD == 3 ? -1 : 0);
	static constexpr int tshift_x = dx < 0 ? 1 : 0;
	static constexpr int tshift_y = dy < 0 ? 1 : 0;
	static constexpr bool HORIZ = SD < 2;
	static constexpr int NWD = (K + 3) / 4;        // class window registers, 4 slots each
	static constexpr int CRING_WORDS = HORIZ ? 0 : PF * 32;   // selector ring, per warp

	const float *in;
	float *out;
	float *ring;                                   // this lane's K floats of slot 0: [PF][2][VSZ] (in, out)
	int lane, dbase, D, W, ddir;
	long pix_step;
	float P1f, P2f, P1s, P2s, P1m, P2m, P1f_a, P1s_a, P1m_a;
	int x, y;                                      // pixel of the NEXT step to execute
	long base;
	float prev[K];
	unsigned cw[NWD], c1c;                         // classes of the step being executed; byte k%4 of cw[k/4] = slot k
	// horizontal
	const uint8_t *p1, *pe;                        // shared-memory class rows: D1 of pixel xs at p1[xs], entering D2 byte at pe[xs]
	unsigned nw[NWD], qn, c1n;                     // window / D1 class of the next step, byte entering the step after
	int xl;
	bool up;
	// vertical
	unsigned *cring;                               // this lane's word of slot 0: [PF][32]
	const unsigned *selp;                          // selector word of the next step to execute
	long cstep;                                    // selector words per step (+-32*W)
	unsigned selw;                                 // selector word of the step being executed

	// srow1 / srow2: (horizontal) shared-memory copies of the D1 / D2 class rows of this line, at
	// image column 0 of the band.  cring_: (vertical) this warp's class ring.
	__device__ __forceinline__ void init(const uint8_t *tab, const float *in_, float *out_, float *ring_, unsigned *cring_,
					      const uint8_t *srow1, const uint8_t *srow2, int H, int W_, int D_,
					      int pad, const SgmParams &prm, int line)
	{
		in = in_; out = out_; ring = ring_;
		lane = threadIdx.x & 31;
		dbase = lane * K;
		D = D_;
		W = W_;
		ddir = prm.direction;
		// adcensus.cu:595-605 and :609/:612, same expressions
		P1f = prm.pi1; P2f = prm.pi2;
		P1s = prm.pi1 / (prm.q1 * prm.q2); P2s = prm.pi2 / (prm.q1 * prm.q2);
		P1m = prm.pi1 / prm.q1; P2m = prm.pi2 / prm.q1;
		P1f_a = P1f / prm.alpha1; P1s_a = P1s / prm.alpha1; P1m_a = P1m / prm.alpha1;
		x = SD == 0 ? 0 : (SD == 1 ? W - 1 : line);
		y = SD == 2 ? 0 : (SD == 3 ? H - 1 : line);
		pix_step = (long)(dy * W + dx) * D;
		base = ((long)y * W + x) * D + dbase;
		// NaN in the padding slots of the ring (never overwritten)
#pragma unroll
		for (int s = 0; s < PF * 2; s++)
#pragma unroll
			for (int k = 0; k < K; k++) ring[s * VSZ + k] = adc_nan();
		// The stored difference at (y, j) pairs pixel j with its left / upper neighbour, so scans
		// that look right / down (dx = -1, dy = -1) read the entry one further (tshift).
		if constexpr (HORIZ) {
			// step 0 uses no penalties; prepare step 1 = pixel x + dx
			const int xs = clampx(x + dx);
			p1 = srow1 + tshift_x;
			const uint8_t *r2 = srow2 + tshift_x;
			up = dx * ddir < 0;                        // slot k of the next step = slot k-1 of this one
			pe = r2 + (dbase + (up ? 0 : K - 1)) * ddir;
#pragma unroll
			for (int i = 0; i < NWD; i++) nw[i] = 0;
#pragma unroll
			for (int k = 0; k < K; k++) nw[k / 4] |= (unsigned)r2[xs + (dbase + k) * ddir] << (8 * (k & 3));   // :588-594
			c1n = p1[xs];                              // :587
			qn = pe[clampx(xs + dx)];
			xl = xs + dx;
		} else {
			const int Wp = prm.Wt + 2 * pad;
			cring = cring_;
			cstep = (long)dy * W * 32;
			selp = reinterpret_cast<const unsigned *>(tab + sgm_sel_offset(prm.Ht, Wp)) +
			       ((long)(y + prm.yoff + tshift_y) * W + x) * 32 + lane;       // step 0 (never fetched)
		}
	}

	__device__ __forceinline__ int clampx(int xs) const { return min(max(xs, 0), W - 1); }

	// vertical: start the copy of the selector word of the step `ahead` steps after the next one
	__device__ __forceinline__ void cls_issue(int slot, int ahead) { cp_async4u(cring + slot * 32, selp + ahead * cstep); }

	// classes of the step about to execute -> (c1c, cw)
	__device__ __forceinline__ void cls_take(int slot)
	{
		if constexpr (HORIZ) {
#pragma unroll
			for (int i = 0; i < NWD; i++) cw[i] = nw[i];
			c1c = c1n;
			constexpr unsigned topmask = (1u << (8 * ((K - 1) & 3))) - 1u;   // bytes below the top slot of the last word
			if (up) {
#pragma unroll
				for (int i = NWD - 1; i > 0; i--) nw[i] = __funnelshift_l(nw[i - 1], nw[i], 8);
				nw[0] = (nw[0] << 8) | qn;
			} else {
#pragma unroll
				for (int i = 0; i < NWD - 1; i++) nw[i] = __funnelshift_r(nw[i], nw[i + 1], 8);
				nw[NWD - 1] = ((nw[NWD - 1] >> 8) & topmask) | (qn << (8 * ((K - 1) & 3)));
			}
			c1n = p1[clampx(xl)];
			qn = pe[clampx(xl + dx)];
			xl += dx;
		} else {
			selw = cring[slot * 32];
			c1c = (selw >> 16) & 3u;
		}
	}

	// steps [s_begin, s_end) of the scan; use_out: read-modify-write the accumulator (else it is
	// known to hold zeros).  Streams the cost (and accumulator) vectors of the next PF pixels into
	// the shared-memory ring with cp.async; every lane fetches exactly the elements it consumes.
	// carried: the scan continues a line whose state is already in `prev` (vertical wavefront): step 0 is an ordinary step
	__device__ __forceinline__ void run(int s_begin, int s_end, bool use_out, bool carried = false)
	{
#pragma unroll
		for (int u = 0; u < PF; u++) {
			if (s_begin + u < s_end) {
				issue_vec<K, VEC>(ring + (u * 2) * VSZ, in + base + u * pix_step, dbase, D);
				if (use_out) issue_vec<K, VEC>(ring + (u * 2 + 1) * VSZ, out + base + u * pix_step, dbase, D);
				if constexpr (!HORIZ)
					if (s_begin + u >= 1 || carried) cls_issue(u, u);
			}
			asm volatile("cp.async.commit_group;");
		}
		int slot = 0;
#pragma unroll 1
		for (int s = s_begin; s < s_end; s++) {
			float *rs = ring + slot * (2 * VSZ);
			const int cslot = slot;
			slot = slot + 1 == PF ? 0 : slot + 1;
			asm volatile("cp.async.wait_group %0;" ::"n"(PF - 1));
			float cin[K], cout[K];
			read_slot<K>(cin, rs);
			if (use_out) read_slot<K>(cout, rs + VSZ);

			float val[K];
			if (s == 0 && !carried) {                       // adcensus.cu:567-572
#pragma unroll
				for (int k = 0; k < K; k++) val[k] = cin[k];
			} else {
				float mt[K];
#pragma unroll
				for (int k = 0; k < K; k++) mt[k] = prev[k];
#pragma unroll
				for (int w = K / 2; w > 0; w >>= 1)
#pragma unroll
					for (int k = 0; k < w; k++) mt[k] = fminf(mt[k], mt[k + w]);
				const float m = warp_min_f32(mt[0]);            // :579-584
				float left = __shfl_up_sync(0xffffffffu, prev[K - 1], 1);
				float right = __shfl_down_sync(0xffffffffu, prev[0], 1);
				if (lane == 0) left = adc_nan();                // d - 1 < 0 (:608)
				if (lane == 31) right = adc_nan();

				cls_take(cslot);
				// penalties when the D2 class equals the D1 class (both < tau or both > tau), else middle
				const unsigned c1 = c1c;
				const bool c1lt = c1 == 0;
				const float P1e = c1 == 1 ? P1m : (c1lt ? P1f : P1s);
				const float P2e = c1 == 1 ? P2m : (c1lt ? P2f : P2s);
				const float P1ae = c1 == 1 ? P1m_a : (c1lt ? P1f_a : P1s_a);
				unsigned xw[NWD];
#pragma unroll
				for (int i = 0; i < NWD; i++) xw[i] = HORIZ ? cw[i] ^ (c1 * 0x01010101u) : 0u;
#pragma unroll
				for (int k = 0; k < K; k++) {
					const bool eq = HORIZ ? (xw[k / 4] & (0xffu << (8 * (k & 3)))) == 0 : (selw >> k) & 1u;
					const float P1 = eq ? P1e : P1m, P2 = eq ? P2e : P2m, P1a = eq ? P1ae : P1m_a;
					const float pm = k > 0 ? prev[k - 1] : left;
					const float pp = k < K - 1 ? prev[k + 1] : right;
					float cost = fminf(prev[k], m + P2);                               // :607
					cost = fminf(cost, pm + (SD == 2 ? P1a : P1));                     // :609
					cost = fminf(cost, pp + (SD == 3 ? P1a : P1));                     // :612
					val[k] = cin[k] + cost - m;                                        // :615
				}
			}
			float o[K];
#pragma unroll
			for (int k = 0; k < K; k++) {
				o[k] = (use_out ? cout[k] : 0.0f) + val[k];                            // :569 / :616
				prev[k] = val[k];                                                      // :570 / :617
			}
			store_vec<K, VEC>(o, out + base, dbase, D);
			// refill this ring slot with step s + PF (its values are in registers by now)
			if (s + PF < s_end) {
				issue_vec<K, VEC>(rs, in + base + PF * pix_step, dbase, D);
				if (use_out) issue_vec<K, VEC>(rs + VSZ, out + base + PF * pix_step, dbase, D);
				if constexpr (!HORIZ) cls_issue(cslot, PF);
			}
			asm volatile("cp.async.commit_group;");
			base += pix_step;
			x += dx;
			y += dy;
			if constexpr (!HORIZ) {
				selp += cstep;
			}
		}
		asm volatile("cp.async.wait_group 0;");
	}
};

// shared-memory bytes of one staged class row (horizontal scans)
__host__ __device__ inline int sgm_row_bytes(int Wt, int pad) { return (Wt + 2 * pad + 8 + 15) & ~15; }

// One launch = one direction: one warp per scanline.  ZERO: output known to be 0 on entry.
template <int K, bool VEC, int SD, bool ZERO, int PF, int WPB>
__global__ void __launch_bounds__(32 * WPB)
sgm_pass_kernel(const uint8_t *__restrict__ tab, const float *__restrict__ in, float *__restrict__ out,
		int H, int W, int D, int pad, SgmParams prm)
{
	extern __shared__ __align__(16) float sgm_smem[];
	using Scan = SgmScan<K, VEC, SD, PF>;
	const int wib = threadIdx.x >> 5;
	const int lane = threadIdx.x & 31;
	const int line = prm.line0 + blockIdx.x * WPB + wib;
	if (line >= prm.line1) return;                 // whole warp
	float *ring = sgm_smem + (size_t)wib * PF * 2 * Scan::VSZ;
	unsigned *extra = reinterpret_cast<unsigned *>(sgm_smem + (size_t)WPB * PF * 2 * Scan::VSZ);
	const uint8_t *s1 = nullptr, *s2 = nullptr;
	unsigned *cring = nullptr;
	if constexpr (SD < 2) {
		const int Wp = prm.Wt + 2 * pad, RB = sgm_row_bytes(prm.Wt, pad);
		const long plane = (long)prm.Ht * Wp;
		const int ty = min(max(line + prm.yoff, 0), prm.Ht - 1);
		unsigned *rows = extra + (size_t)wib * (2 * RB / 4);
		s1 = sgm_stage_row(rows, tab + (long)ty * Wp, Wp, lane, 32) + pad + prm.xoff;                      // plane 0
		s2 = sgm_stage_row(rows + RB / 4, tab + 2 * plane + (long)ty * Wp, Wp, lane, 32) + pad + prm.xoff;   // plane 2
		__syncwarp();
	} else {
		cring = extra + (size_t)wib * Scan::CRING_WORDS + lane;
	}
	Scan sc;
	sc.init(tab, in, out, ring + lane * K, cring, s1, s2, H, W, D, pad, prm, line);
	bool carried = false;
	if constexpr (SD >= 2) {
		if (prm.state_in) {                            // line state of the row before this band
			carried = true;
#pragma unroll
			for (int k = 0; k < K; k++) sc.prev[k] = prm.state_in[(long)line * Scan::VSZ + lane * K + k];
		}
	}
	sc.run(0, SD < 2 ? W : H, !ZERO, carried);
	if constexpr (SD >= 2) {
		if (prm.state_out) {
#pragma unroll
			for (int k = 0; k < K; k++) prm.state_out[(long)line * Scan::VSZ + lane * K + k] = sc.prev[k];
		}
	}
}

// Both horizontal directions of one image row in ONE CTA (two warps), for an accumulator that is
// known to be zero on entry: warp 0 scans right, warp 1 scans left, concurrently (a horizontal
// scan is 1226 strictly serial steps on only 370 lines, so a single direction leaves most SM
// sub-partitions idle).  The reference's accumulation order out = (0 + right) + left is kept:
// in the half of the row a scan reaches FIRST it stores 0 + v; after a block barrier at the
// crossing point it adds its v to what the other scan stored.  For the left scan that is
// (0 + right) + left literally; for the right scan it is (0 + right) + (0 + left), and
// (0 + a) + b == (0 + b) + a holds in IEEE arithmetic (0 + a only canonicalises -0, + commutes).
template <int K, bool VEC, int PF>
__global__ void __launch_bounds__(64)
sgm_hpair_kernel(const uint8_t *__restrict__ tab, const float *__restrict__ in, float *__restrict__ out,
		 int H, int W, int D, int pad, SgmParams prm)
{
	extern __shared__ __align__(16) float sgm_smem[];
	const int line = blockIdx.x;
	const int wib = threadIdx.x >> 5;
	const int M = W / 2;                           // columns [0, M) are reached first by the right scan
	float *ring = sgm_smem + (size_t)wib * PF * 2 * 32 * K + (threadIdx.x & 31) * K;
	// the two scans share the class rows of the line
	const int Wp = prm.Wt + 2 * pad, RB = sgm_row_bytes(prm.Wt, pad);
	const long plane = (long)prm.Ht * Wp;
	const int ty = min(max(line + prm.yoff, 0), prm.Ht - 1);
	unsigned *rows = reinterpret_cast<unsigned *>(sgm_smem + (size_t)2 * PF * 2 * 32 * K);
	const uint8_t *s1 = sgm_stage_row(rows, tab + (long)ty * Wp, Wp, threadIdx.x, 64) + pad + prm.xoff;
	const uint8_t *s2 = sgm_stage_row(rows + RB / 4, tab + 2 * plane + (long)ty * Wp, Wp, threadIdx.x, 64) + pad + prm.xoff;
	__syncthreads();
	if (wib == 0) {
		SgmScan<K, VEC, 0, PF> sc;
		sc.init(tab, in, out, ring, nullptr, s1, s2, H, W, D, pad, prm, line);
		sc.run(0, M, false);
		__syncthreads();
		sc.run(M, W, true);
	} else {
		SgmScan<K, VEC, 1, PF> sc;
		sc.init(tab, in, out, ring, nullptr, s1, s2, H, W, D, pad, prm, line);
		sc.run(0, W - M, false);                   // columns W-1 .. M
		__syncthreads();
		sc.run(W - M, W, true);                    // columns M-1 .. 0
	}
}

constexpr int SGM_SMEM_MAX = 160 * 1024;

// done: one flag array per kernel instantiation (the caller's static)
template <typename Kern>
int sgm_allow_smem(Kern kern, int smem, bool *done)
{
	if (smem > SGM_SMEM_MAX) return ADCENSUS_ELIMIT;
	int dev = 0;
	cudaGetDevice(&dev);
	if (!done[dev & 63]) {
		ADC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SGM_SMEM_MAX));
		done[dev & 63] = true;
	}
	return 0;
}

template <int K, bool VEC, int SD, bool ZERO>
int launch_pass(const uint8_t *tab, const float *in, float *out, int H, int W, int D, int pad,
		const SgmParams &prm, cudaStream_t s)
{
	constexpr int PF = K >= 16 ? 6 : 8;
	// horizontal scans have few, long lines: one warp per CTA spreads them over all SMs
	constexpr int WPB = SD < 2 ? 1 : 4;
	using Scan = SgmScan<K, VEC, SD, PF>;
	const int smem = WPB * (PF * 2 * Scan::VSZ * 4 + Scan::CRING_WORDS * 4 + (SD < 2 ? 2 * sgm_row_bytes(prm.Wt, pad) : 0));
	auto kern = sgm_pass_kernel<K, VEC, SD, ZERO, PF, WPB>;
	static bool done[64] = {false};
	int rc = sgm_allow_smem(kern, smem, done);
	if (rc) return rc;
	const int nlines = prm.line1 - prm.line0;
	if (nlines <= 0) return 0;
	kern<<<adc_div_up(nlines, WPB), 32 * WPB, smem, s>>>(tab, in, out, H, W, D, pad, prm);
	ADC_CHECK_LAUNCH();
	return 0;
}

template <int K, bool VEC>
int launch_hpair(const uint8_t *tab, const float *in, float *out, int H, int W, int D, int pad,
		 const SgmParams &prm, cudaStream_t s)
{
	constexpr int PF = K >= 16 ? 6 : 8;
	const int smem = 2 * PF * 2 * 32 * K * 4 + 2 * sgm_row_bytes(prm.Wt, pad);
	auto kern = sgm_hpair_kernel<K, VEC, PF>;
	static bool done[64] = {false};
	int rc = sgm_allow_smem(kern, smem, done);
	if (rc) return rc;
	kern<<<H, 64, smem, s>>>(tab, in, out, H, W, D, pad, prm);
	ADC_CHECK_LAUNCH();
	return 0;
}

// pass_mask bit i = run scan direction i (0 right, 1 left, 2 down, 3 up), always in that order
template <int K, bool VEC>
int launch_all(const uint8_t *tab, const float *in, float *out, int H, int W, int D, int pad,
	       const SgmParams &prm, bool zero_out, int pass_mask, cudaStream_t s)
{
	int rc = 0;
	SgmParams ph = prm, pv = prm;                     // horizontal scans: every row; vertical: the caller's column range (default all)
	ph.line0 = 0; ph.line1 = H; ph.state_in = nullptr; ph.state_out = nullptr;
	if (pv.line1 <= pv.line0) { pv.line0 = 0; pv.line1 = W; }
	if ((pass_mask & 3) == 3 && zero_out && W >= 2) {
		rc = launch_hpair<K, VEC>(tab, in, out, H, W, D, pad, ph, s);   // right and left concurrently
	} else {
		if (pass_mask & 1)
			rc = zero_out ? launch_pass<K, VEC, 0, true>(tab, in, out, H, W, D, pad, ph, s)
				      : launch_pass<K, VEC, 0, false>(tab, in, out, H, W, D, pad, ph, s);
		if (rc) return rc;
		if ((pass_mask & 2) && (rc = launch_pass<K, VEC, 1, false>(tab, in, out, H, W, D, pad, ph, s))) return rc;
	}
	if (rc) return rc;
	if ((pass_mask & 4) && (rc = launch_pass<K, VEC, 2, false>(tab, in, out, H, W, D, pad, pv, s))) return rc;
	if (pass_mask & 8) rc = launch_pass<K, VEC, 3, false>(tab, in, out, H, W, D, pad, pv, s);
	return rc;
}

}  // namespace

// lanes carry 32*K disparity slots (K from D); the class tables are padded by that many columns so
// that the padding slots d >= D also index inside the row
static int sgm_slots(int D) { return D <= 32 ? 32 : (D <= 64 ? 64 : (D <= 128 ? 128 : (D <= 256 ? 256 : 512))); }

// four byte-class planes + the selector words of the vertical scans (128 bytes per pixel)
size_t adc_sgm_table_bytes(int H, int W, int D) { return sgm_sel_offset(H, W + 2 * sgm_slots(D)) + (size_t)128 * H * W; }

static int adc_sgm_classes(const float *x0, const float *x1, uint8_t *tab, int Ht, int Wt, int D, float tau_so, cudaStream_t s)
{
	const int pad = sgm_slots(D);
	const long plane = (long)Ht * (Wt + 2 * pad);
	sgm_class_kernel<<<adc_div_up(plane, 256), 256, 0, s>>>(x0, x1, tab, Ht, Wt, pad, tau_so);
	ADC_CHECK_LAUNCH();
	return 0;
}

// The selected passes over a volume (H,W,D) that is the band [yoff, yoff+H) x [xoff, xoff+W) of the
// Ht x Wt image whose class tables are in `tab` (adc_sgm_classes).  zero_out: `output` is known
// to be all zeros (main.lua:1014) -> the first (rightward) pass skips reading it.
// selector words of the vertical scans for the W columns at image offset xoff (all Ht table rows) and one `direction`
static int adc_sgm_selectors(uint8_t *tab, int W, int D, int Ht, int Wt, int xoff, int direction, cudaStream_t s)
{
	const int pad = sgm_slots(D);
	unsigned *sel = reinterpret_cast<unsigned *>(tab + sgm_sel_offset(Ht, Wt + 2 * pad));
	if (Ht > 65535) return ADCENSUS_ELIMIT;            // gridDim.y
	const dim3 grid(adc_div_up(W, 8), Ht), block(32, 8);
	switch (pad / 32) {
	case 1: sgm_sel_kernel<1><<<grid, block, 0, s>>>(tab, sel, Ht, W, Wt + 2 * pad, pad, xoff, direction); break;
	case 2: sgm_sel_kernel<2><<<grid, block, 0, s>>>(tab, sel, Ht, W, Wt + 2 * pad, pad, xoff, direction); break;
	case 4: sgm_sel_kernel<4><<<grid, block, 0, s>>>(tab, sel, Ht, W, Wt + 2 * pad, pad, xoff, direction); break;
	case 8: sgm_sel_kernel<8><<<grid, block, 0, s>>>(tab, sel, Ht, W, Wt + 2 * pad, pad, xoff, direction); break;
	default: sgm_sel_kernel<16><<<grid, block, 0, s>>>(tab, sel, Ht, W, Wt + 2 * pad, pad, xoff, direction); break;
	}
	ADC_CHECK_LAUNCH();
	return 0;
}

// the selected passes with tables (and, for vertical passes, selectors) already built; vertical passes may cover the
// columns [xa, xb) only and carry the line state across row bands (state_in / state_out, [W][32K] floats, NULL = border)
static int adc_sgm2_passes(const float *in, float *out, const uint8_t *tab, int H, int W, int D, int Ht, int Wt, int yoff, int xoff,
			   float pi1, float pi2, float tau_so, float alpha1, float q1, float q2, int direction,
			   bool zero_out, int pass_mask, int xa, int xb, const float *state_in, float *state_out, cudaStream_t s)
{
	SgmParams prm{pi1, pi2, tau_so, alpha1, q1, q2, direction, Ht, Wt, yoff, xoff, state_in, state_out, xa, xb};
	const int pad = sgm_slots(D);
	const bool vec = (D % 4 == 0) && (((uintptr_t)in | (uintptr_t)out) % 16 == 0);
	if (D <= 32) return launch_all<1, false>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s);
	if (D <= 64) return launch_all<2, false>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s);
	if (D <= 128) return vec ? launch_all<4, true>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s)
				 : launch_all<4, false>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s);
	if (D <= 256) return vec ? launch_all<8, true>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s)
				 : launch_all<8, false>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s);
	return vec ? launch_all<16, true>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s)
		   : launch_all<16, false>(tab, in, out, H, W, D, pad, prm, zero_out, pass_mask, s);
}

static int adc_sgm2_band(const float *in, float *out, const uint8_t *tab, int H, int W, int D, int Ht, int Wt, int yoff, int xoff,
			 float pi1, float pi2, float tau_so, float alpha1, float q1, float q2, int direction,
			 bool zero_out, int pass_mask, cudaStream_t s)
{
	if (pass_mask & 12) {                              // vertical scans: band = whole columns (H == Ht)
		int rc = adc_sgm_selectors(const_cast<uint8_t *>(tab), W, D, Ht, Wt, xoff, direction, s);
		if (rc) return rc;
	}
	return adc_sgm2_passes(in, out, tab, H, W, D, Ht, Wt, yoff, xoff, pi1, pi2, tau_so, alpha1, q1, q2, direction, zero_out, pass_mask,
			       0, 0, nullptr, nullptr, s);
}


// whole image, all four directions (what adcensus.sgm2 does).  tab: scratch of adc_sgm_table_bytes(H, W, D) bytes.
int adc_sgm2(const float *x0, const float *x1, const float *in, float *out, uint8_t *tab, int H, int W, int D,
	     float pi1, float pi2, float tau_so, float alpha1, float q1, float q2, int direction,
	     bool zero_out, cudaStream_t s)
{
	int rc = adc_sgm_classes(x0, x1, tab, H, W, D, tau_so, s);
	if (rc) return rc;
	return adc_sgm2_band(in, out, tab, H, W, D, H, W, 0, 0, pi1, pi2, tau_so, alpha1, q1, q2, direction, zero_out, 15, s);
}

// ---- band-wise entry point for the row-band / column-band multi-GPU split (rowband.py) ----------
// x0, x1: the FULL Ht x Wt images (replicated on every GPU); input/output: this GPU's band volume
// (H,W,D) at image offset (yoff, xoff); pass_mask selects scan directions (bit 0 right, 1 left,
// 2 down, 3 up).  A band must contain whole scanlines of every selected pass: row bands
// (W == Wt, xoff == 0) for the horizontal passes, column bands (H == Ht, yoff == 0) for the vertical.
extern "C" int mccnn_sgm2_band(const float *x0, const float *x1, const float *input, float *output,
			       int H, int W, int D, int Ht, int Wt, int yoff, int xoff,
			       float pi1, float pi2, float tau_so, float alpha1, float sgm_q1, float sgm_q2,
			       int direction, int pass_mask, int zero_out, adcensus_stream_t stream)
{
	if (!x0 || !x1 || !input || !output || input == output) return ADCENSUS_EINVAL;
	if (H < 1 || W < 1 || D < 1 || Ht < H || Wt < W || yoff < 0 || xoff < 0 || yoff + H > Ht || xoff + W > Wt) return ADCENSUS_EINVAL;
	if ((direction != 1 && direction != -1) || (pass_mask & ~15)) return ADCENSUS_EINVAL;
	if ((pass_mask & 3) && (W != Wt || xoff != 0)) return ADCENSUS_EINVAL;   // horizontal scanlines must be whole
	if ((pass_mask & 12) && (H != Ht || yoff != 0)) return ADCENSUS_EINVAL;  // vertical scanlines must be whole
	if (D > ADCENSUS_MAX_DISP) return ADCENSUS_ELIMIT;
	cudaStream_t s = adc_stream(stream);
	uint8_t *tab = nullptr;
	int rc = adc_scratch_alloc((void **)&tab, adc_sgm_table_bytes(Ht, Wt, D), s);
	if (rc) return rc;
	rc = adc_sgm_classes(x0, x1, tab, Ht, Wt, D, tau_so, s);
	if (!rc) rc = adc_sgm2_band(input, output, tab, H, W, D, Ht, Wt, yoff, xoff, pi1, pi2, tau_so, alpha1, sgm_q1, sgm_q2,
				    direction, zero_out != 0, pass_mask, s);
	int rc2 = adc_scratch_free(tab, s);
	return rc ? rc : rc2;
}

extern "C" int adcensus_sgm2(const float *x0, const float *x1, const float *input, float *output, float *tmp,
			     int H, int W, int D, float pi1, float pi2, float tau_so, float alpha1,
			     float sgm_q1, float sgm_q2, int direction, adcensus_stream_t stream)
{
	(void)tmp;  // the reference's global line-state scratch; state lives in registers here
	if (!x0 || !x1 || !input || !output || input == output) return ADCENSUS_EINVAL;
	if (H < 1 || W < 1 || D < 1 || (direction != 1 && direction != -1)) return ADCENSUS_EINVAL;
	if (D > ADCENSUS_MAX_DISP) return ADCENSUS_ELIMIT;
	cudaStream_t s = adc_stream(stream);
	uint8_t *tab = nullptr;
	int rc = adc_scratch_alloc((void **)&tab, adc_sgm_table_bytes(H, W, D), s);
	if (rc) return rc;
	rc = adc_sgm2(x0, x1, input, output, tab, H, W, D, pi1, pi2, tau_so, alpha1, sgm_q1, sgm_q2, direction, false, s);
	int rc2 = adc_scratch_free(tab, s);
	return rc ? rc : rc2;
}

// ---- wavefront split of the vertical scans over ROW bands (rowband.py) ------------------------------------------
// The class tables of an image pair are built once (mccnn_sgm_tables_build: classes + the selector words of one
// `direction`), then the passes run band by band: horizontal passes are band-local; a vertical pass over the rows
// [yoff, yoff + H) of the columns [xa, xb) takes the line state of the row before the band from state_in (NULL: the band
// touches the image border where the scan starts) and leaves the state of its last row in state_out ([W][sgm_state_pitch]
// floats), so that consecutive bands -- on different GPUs -- chain column chunk by column chunk.
extern "C" size_t mccnn_sgm_tables_bytes(int Ht, int Wt, int D) { return adc_sgm_table_bytes(Ht, Wt, D); }
extern "C" int mccnn_sgm_state_pitch(int D) { return sgm_slots(D); }

extern "C" int mccnn_sgm_tables_build(const float *x0, const float *x1, void *tab, int Ht, int Wt, int D, float tau_so,
				      int direction, adcensus_stream_t stream)
{
	if (!x0 || !x1 || !tab || Ht < 1 || Wt < 1 || D < 1 || (direction != 1 && direction != -1)) return ADCENSUS_EINVAL;
	if (D > ADCENSUS_MAX_DISP) return ADCENSUS_ELIMIT;
	int rc = adc_sgm_classes(x0, x1, (uint8_t *)tab, Ht, Wt, D, tau_so, adc_stream(stream));
	if (!rc) rc = adc_sgm_selectors((uint8_t *)tab, Wt, D, Ht, Wt, 0, direction, adc_stream(stream));
	return rc;
}

extern "C" int mccnn_sgm2_rows(const void *tab, const float *input, float *output, int H, int W, int D, int Ht, int yoff,
			       float pi1, float pi2, float tau_so, float alpha1, float sgm_q1, float sgm_q2,
			       int direction, int pass_mask, int zero_out, int xa, int xb,
			       const float *state_in, float *state_out, adcensus_stream_t stream)
{
	if (!tab || !input || !output || input == output) return ADCENSUS_EINVAL;
	if (H < 1 || W < 1 || D < 1 || Ht < H || yoff < 0 || yoff + H > Ht) return ADCENSUS_EINVAL;
	if ((direction != 1 && direction != -1) || (pass_mask & ~15) || !pass_mask) return ADCENSUS_EINVAL;
	if ((pass_mask & 12) && (xa < 0 || xb > W || xa >= xb)) return ADCENSUS_EINVAL;
	if ((pass_mask & 12) == 12 && (state_in || state_out)) return ADCENSUS_EINVAL;   // one vertical direction per call when chained
	if ((pass_mask & 4) && !state_in && yoff != 0) return ADCENSUS_EINVAL;           // a band below the top needs the state above it
	if ((pass_mask & 8) && !state_in && yoff + H != Ht) return ADCENSUS_EINVAL;
	if (D > ADCENSUS_MAX_DISP) return ADCENSUS_ELIMIT;
	return adc_sgm2_passes(input, output, (const uint8_t *)tab, H, W, D, Ht, W, yoff, 0, pi1, pi2, tau_so, alpha1, sgm_q1, sgm_q2,
			       direction, zero_out != 0, pass_mask, xa, xb, state_in, state_out, adc_stream(stream));
}
