// icgn2d.cu -- inverse-compositional Gauss-Newton subset registration, 2D, first-order (6
// parameters) and second-order (12 parameters) shape functions, for sm_100a.
//
// Replaces ICGN2D1::compute(POI2D*) (reference src/oc_icgn.cpp:144-341) and
// ICGN2D2::compute(POI2D*) (src/oc_icgn.cpp:685-898), including what ICGN2D*::prepare() feeds
// them (Gradient2D4, src/oc_gradient.cpp:37-79; BicubicBspline, src/oc_cubic_bspline.cpp:84-181).
//
// Round-2 structure in one paragraph: the setup pass and the sampling loop take TWO subset rows per lane and step in packed
// f32x2 arithmetic (ICGN2D_PAIRS), and in the Tensor-Memory variant (template flag TM: wide-enough subsets, queues that fill the
// GPU) a lane's per-sample constants live in its own TMEM lane instead of shared memory, which lifts the resident warps per SM
// from 11 to 16 at r = 16.  The reference's `any sample < 0` rejection is re-decided in the reference's own arithmetic when the
// smallest sample is borderline (icgn2d_exact_negative).  What follows describes the common skeleton.
//
// Mapping: ONE WARP PER POI, persistent warps pulling POIs from an atomic counter, no CTA barrier.
// Lanes run along x: lane c owns column c of the subset for every row (columns >= 32 are a short
// tail), so x-dependent factors are per-lane constants and y-dependent ones are warp-uniform.
//   stage   : the reference tile (subset + 2-pixel gradient halo) is staged in the warp's smem slab.
//   setup   : one pass computes R' = R - c0 (c0 = centre pixel, a pilot value that keeps every sum
//             well conditioned), the 4th-order gradients gx, gy (recomputed from the image, nothing
//             precomputed in HBM) and stores them to smem; the Hessian is accumulated as FACTORED
//             sums  sum g_a g_b y^Q  (x^P applied once per lane afterwards), so a sample costs 15
//             (6-parameter) / 30 (12-parameter) flops instead of 21 / 78 FMAs.  Mean and norm of the
//             reference subset come from the same pass.  Cholesky factorisation in registers.
//   iterate : the target tile (subset + bicubic support + slack), minus c0, replaces the reference
//             tile in the slab.  Each iteration evaluates the bicubic interpolant from the 4x4 pixel
//             block with explicit fp32 weights (the reference's 64 B/pixel LUT is never built) and
//             accumulates ONE pass of sums with d = t - R:  sum d, sum d^2, sum R'd, sum g_a d y^Q;
//             mean/norm of the warped target, ZNSSD and the Gauss-Newton right-hand side follow
//             algebraically (DESIGN.md "single-pass IC-GN sums").
//   update  : solve with the Cholesky factors, compose W <- W * W(dp)^-1 in registers.
// Samples whose 4x4 support leaves the staged tile (large deformation gradients) are read from
// global memory instead, so results never depend on the tile size.
#include <stdlib.h>
#include <string.h>

#include "ocb_kernels.h"
#include "ocb_tma.cuh"
#include "ocb_f32x2.cuh"
#include "ocb_tile2d.cuh"
#include "ocb_tmem.cuh"

namespace ocb {

#ifndef ICGN2D_PAIRS
// 1: the fast sampling loop takes TWO subset rows per lane and step and does their arithmetic in packed f32x2 pairs
// (FFMA2 / FMUL2 / FADD2, ocb_f32x2.cuh) -- position, bicubic weights, taps and all sums of rows r and r + 1 go through ONE
// instruction per pair, and the two 4x4 pixel blocks, which overlap in three rows, are fetched as one 4x5 block (20 LDS
// instead of 32).  The two rows are independent, so unlike packing WITHIN one sample (tried in round 1: 10 % slower)
// no dependency chain gets longer.  0: one row per step, scalar arithmetic (the round-1 loop), kept for A/B runs.
#define ICGN2D_PAIRS 1
#endif
#ifndef ICGN2D_PAIR_UNROLL
#define ICGN2D_PAIR_UNROLL 2 // row pairs in flight per lane
#endif
#ifndef ICGN2D_MINB
#define ICGN2D_MINB 16 // resident one-warp CTAs the 6-parameter kernels' register budget is sized for (16 -> 128 registers; measured best of 11/16/20)
#endif
#ifndef ICGN2D_UNROLL
#define ICGN2D_UNROLL 3
#endif
constexpr int ICGN2D_ROW_UNROLL = ICGN2D_UNROLL; // rows of the fast sampling loop in flight per lane
constexpr int ICGN2D_PAIR_UNROLL_N = ICGN2D_PAIR_UNROLL;
#ifndef ICGN2D_SETUP_UNROLL
#define ICGN2D_SETUP_UNROLL 3 // row pairs of the setup pass in flight per lane (1 / 2 / 3: 0.651 / 0.647 / 0.641 ms on config B)
#endif
constexpr int ICGN2D_SETUP_UNROLL_N = ICGN2D_SETUP_UNROLL;
constexpr int ICGN2D_TILE_MARGIN = 1; // slack (pixels) around subset+support in the target tile
// TMA tile loads need the innermost coordinate 16-byte aligned (x multiple of 4 floats; measured: an
// unaligned x raises 'illegal instruction'), so tile origins are rounded down to a multiple of 4 and
// the boxes are 3 columns wider.

__host__ __device__ inline int icgn2d_ref_w(int rx) { return round_up4(2 * rx + 1 + 4 + 3); }
__host__ __device__ inline int icgn2d_ref_h(int ry) { return 2 * ry + 1 + 4; }
__host__ __device__ inline int icgn2d_tar_w(int rx) { return round_up4(2 * rx + 1 + 3 + 2 * ICGN2D_TILE_MARGIN + 3); }
__host__ __device__ inline int icgn2d_tar_h(int ry) { return 2 * ry + 1 + 3 + 2 * ICGN2D_TILE_MARGIN; }
// per-warp slab (floats): [0,32) mbarrier + pad | tile T (TMA destination, 128-B aligned) | R', gx, gy
__host__ __device__ inline int icgn2d_tile_floats(int rx, int ry) {
	const int a = icgn2d_ref_w(rx) * icgn2d_ref_h(ry), b = icgn2d_tar_w(rx) * icgn2d_tar_h(ry);
	return round_up32(a > b ? a : b);
}
// lm: the Levenberg-Marquardt variant keeps the undamped Hessian (<= 78 floats) behind the constants;
// wpp > 1 (warps per POI): a reduction area follows -- wpp x 96 floats of setup partials, 2 x wpp x 32 floats of
// per-iteration partials (double-buffered by iteration parity)
constexpr int ICGN2D_RED_SETUP = 96, ICGN2D_RED_ITER = 32;
// TM variant (below): four independent warps per CTA; the {R, gx, gy} constants of the 32 row-mapped columns live in Tensor Memory
// (3 columns per subset row in the warp's quarter of the 128 TMEM lanes), only the tile and the tail columns' constants in smem
constexpr int ICGN2D_TM_WARPS = 4, ICGN2D_TM_COLS = 128;
__host__ __device__ inline int icgn2d_tm_slab_floats(int rx, int ry) {
	const int rem = (2 * rx + 1) - 32;
	return 32 + icgn2d_tile_floats(rx, ry) + round_up32(3 * (rem > 0 ? rem : 0) * (2 * ry + 1));
}
__host__ inline bool icgn2d_tm_supported(int rx, int ry) { return 2 * rx + 1 >= 32 && 3 * (2 * ry + 1) <= ICGN2D_TM_COLS; }
__host__ __device__ inline int icgn2d_slab_floats(int rx, int ry, bool lm, int wpp) {
	const int n = (2 * rx + 1) * (2 * ry + 1);
	return 32 + icgn2d_tile_floats(rx, ry) + round_up32(3 * n) + (lm ? 96 : 0) + (wpp > 1 ? wpp * (ICGN2D_RED_SETUP + 2 * ICGN2D_RED_ITER) : 0);
}

// Shape functions: sd = g_a * phi_i, phi = [1, x, y, x^2/2, xy, y^2/2] (first 3 for NP == 6);
// phi_i = c_i x^p_i y^q_i  (reference src/oc_icgn.cpp:191-196, :725-745)
__host__ __device__ constexpr int phi_p(int i) { return i == 1 ? 1 : (i == 3 ? 2 : (i == 4 ? 1 : 0)); }
__host__ __device__ constexpr int phi_q(int i) { return i == 2 ? 1 : (i == 4 ? 1 : (i == 5 ? 2 : 0)); }
__host__ __device__ constexpr float phi_c(int i) { return (i == 3 || i == 5) ? 0.5f : 1.f; }
// index of monomial x^P y^Q among all monomials ordered by total degree then Q
__host__ __device__ constexpr int mono(int P, int Q) { return (P + Q) * (P + Q + 1) / 2 + Q; }
__host__ __device__ constexpr int pair_idx(int a, int b) { return a + b; } // (x,x)=0 (x,y)=1 (y,y)=2

__device__ __forceinline__ float ipow(float x, int p) {
	float r = 1.f;
#pragma unroll
	for (int i = 0; i < 4; i++)
		if (i < p) r *= x;
	return r;
}

// W(p) of the second-order shape function (reference src/oc_deformation.cpp:301-350)
__device__ __forceinline__ void warp2d2_matrix(const float* p, float* W) {
	const float u = p[0], ux = p[1], uy = p[2], uxx = p[3], uxy = p[4], uyy = p[5];
	const float v = p[6], vx = p[7], vy = p[8], vxx = p[9], vxy = p[10], vyy = p[11];
	W[0] = 1.f + 2.f * ux + ux * ux + u * uxx;
	W[1] = 2.f * u * uxy + 2.f * (1.f + ux) * uy;
	W[2] = uy * uy + u * uyy;
	W[3] = 2.f * u * (1.f + ux);
	W[4] = 2.f * u * uy;
	W[5] = u * u;
	W[6] = 0.5f * (v * uxx + 2.f * (1.f + ux) * vx + u * vxx);
	W[7] = 1.f + uy * vx + ux * vy + v * uxy + u * vxy + vy + ux;
	W[8] = 0.5f * (v * uyy + 2.f * uy * (1.f + vy) + u * vyy);
	W[9] = v + v * ux + u * vx;
	W[10] = u + v * uy + u * vy;
	W[11] = u * v;
	W[12] = vx * vx + v * vxx;
	W[13] = 2.f * v * vxy + 2.f * vx * (1.f + vy);
	W[14] = 1.f + 2.f * vy + vy * vy + v * vyy;
	W[15] = 2.f * v * vx;
	W[16] = 2.f * v * (1.f + vy);
	W[17] = v * v;
	W[18] = 0.5f * uxx; W[19] = uxy; W[20] = 0.5f * uyy; W[21] = 1.f + ux; W[22] = uy; W[23] = u;
	W[24] = 0.5f * vxx; W[25] = vxy; W[26] = 0.5f * vyy; W[27] = vx; W[28] = 1.f + vy; W[29] = v;
	// row 5 = [0 0 0 0 0 1] is implicit
}

// rows <- rows * M^-1 for the 2x6 block `rows` (rows 3,4 of the running warp) and the 6x6 warp
// increment M whose last row is [0 0 0 0 0 1] (given as its first 5 rows, 30 floats).
// Gaussian elimination without pivoting: M = W(dp) is a perturbation of the identity.
// X M = R: reduce M = L U (unit lower L), Y U = R by forward substitution over columns, X = Y L^-1.
__device__ __forceinline__ void right_divide_2x6(float* rows, float* M) {
	float Lm[5][5];
#pragma unroll
	for (int k = 0; k < 5; k++) {
		float inv = 1.0f / M[k * 6 + k];
#pragma unroll
		for (int i = k + 1; i < 5; i++) {
			float l = M[i * 6 + k] * inv;
			Lm[i][k] = l;
#pragma unroll
			for (int j = k + 1; j < 6; j++) M[i * 6 + j] -= l * M[k * 6 + j];
		}
	}
#pragma unroll
	for (int r = 0; r < 2; r++) {
		float y[6];
#pragma unroll
		for (int j = 0; j < 6; j++) {
			float v = rows[r * 6 + j];
#pragma unroll
			for (int i = 0; i < j; i++) {
				if (i < 5) v -= y[i] * M[i * 6 + j];
			}
			y[j] = (j < 5) ? v / M[j * 6 + j] : v;
		}
#pragma unroll
		for (int k = 4; k >= 0; k--) {
			float v = y[k];
#pragma unroll
			for (int i = k + 1; i < 5; i++) v -= y[i] * Lm[i][k];
			y[k] = v;
		}
#pragma unroll
		for (int j = 0; j < 6; j++) rows[r * 6 + j] = y[j];
	}
}

// ---- the reference's `any interpolated sample < 0 -> zncc = -3` rule (src/oc_icgn.cpp:251-255, :792-796) --------------
// The sampling loops below evaluate the interpolant with explicit weights and fused multiply-adds; the reference goes
// through its 16-coefficient LUT and a 16-term polynomial (src/oc_cubic_bspline.cpp:98-129,159-177), and forms the warped
// position with separately rounded products (Deformation2D1::warp, src/oc_deformation.cpp:94-105).  Next to truly black
// pixels the B-spline overshoots by tiny amounts, so the sign of the smallest sample can hinge on those roundings.
// The loops therefore only track min(t); the decision is immediate when it is decisively negative (< -TRIGGER) or
// positive (>= TRIGGER), and otherwise re-made here sample by sample in the reference's own arithmetic: same operation
// order, every operation rounded separately (no FMA), the LUT cell rebuilt from the 4x4 pixel block.
constexpr float ICGN_NEG_TRIGGER = 0.125f; // covers one-ulp differences of the position (ulp 4.9e-4 px at x < 8192) times the steepest 8-bit edge
constexpr float ICGN_NEG_BAND = 4e-3f;     // fused vs separately rounded evaluation at the SAME position differ by < 3e-4 on 8-bit data
__constant__ float c_bc_matrix[4][4] = { // BC = B*C, src/oc_cubic_bspline.h:52-58
	{ -144.0f / 336.0f, 384.0f / 336.0f, -384.0f / 336.0f, 144.0f / 336.0f },
	{ 342.0f / 336.0f, -702.0f / 336.0f, 450.0f / 336.0f, -90.0f / 336.0f },
	{ -198.0f / 336.0f, -18.0f / 336.0f, 270.0f / 336.0f, -54.0f / 336.0f },
	{ 0.0f, 1.0f, 0.0f, 0.0f } };

// BicubicBspline::prepare for ONE cell + BicubicBspline::compute, reference operation order, no contraction.
// q: the 4x4 pixel block (row pitch `pitch`) whose element [1][1] is the pixel at (floor Y, floor X).
__device__ __noinline__ float bicubic_reference_order(const float* __restrict__ q, int pitch, float xd, float yd) {
	float coef[4][4]; // coefficient[k][l] = mat_p[3-k][3-l]
#pragma unroll 1
	for (int k = 0; k < 4; k++)
#pragma unroll 1
		for (int l = 0; l < 4; l++) {
			float acc = 0.f;
#pragma unroll
			for (int m = 0; m < 4; m++)
#pragma unroll
				for (int n = 0; n < 4; n++)
					acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(c_bc_matrix[l][m], c_bc_matrix[k][n]), q[n * pitch + m]));
			coef[3 - k][3 - l] = acc;
		}
	const float x2 = __fmul_rn(xd, xd), y2 = __fmul_rn(yd, yd), x3 = __fmul_rn(x2, xd), y3 = __fmul_rn(y2, yd);
	const float yp[4] = { 1.f, yd, y2, y3 }, xp[4] = { 1.f, xd, x2, x3 };
	float value = coef[0][0];
#pragma unroll
	for (int a = 0; a < 4; a++)
#pragma unroll
		for (int b = 0; b < 4; b++) {
			if (a == 0 && b == 0) continue;
			float term = coef[a][b];
			if (a > 0) term = __fmul_rn(term, yp[a]);
			if (b > 0) term = __fmul_rn(term, xp[b]);
			value = __fadd_rn(value, term);
		}
	return value;
}

// Does any of the samples idx = idx_begin, idx_begin + 32, ... < idx_end (row-major over the subset) of the warp Aw come
// out negative in the reference's arithmetic?  Aw: the running warp as the kernels keep it (NP == 6: W00 W01 W02 W10 W11
// W12; NP == 12: rows 3 and 4 of the 6x6 warp).  Reads the target image directly (rare path).
template <int NP>
__device__ __noinline__ bool icgn2d_exact_negative(const float* Aw, float pcx, float pcy, float ox, float oy, int rx, int ry,
	const float* __restrict__ tar, int w, int h, int idx_begin, int idx_end) {
	const int sw = 2 * rx + 1;
	bool negative = false;
	float A[12];
#pragma unroll
	for (int k = 0; k < (NP == 6 ? 6 : 12); k++) A[k] = Aw[k];
	for (int idx = idx_begin; idx < idx_end; idx += 32) {
		const int r = idx / sw, c = idx - r * sw;
		const float xl = (float)(c - rx) - ox, yl = (float)(r - ry) - oy;
		float wx, wy;
		if constexpr (NP == 6) { // warp_matrix * (x, y, 1): products summed left to right
			wx = __fadd_rn(__fadd_rn(__fmul_rn(A[0], xl), __fmul_rn(A[1], yl)), A[2]);
			wy = __fadd_rn(__fadd_rn(__fmul_rn(A[3], xl), __fmul_rn(A[4], yl)), A[5]);
		} else { // rows 3, 4 of warp_matrix * (x^2, xy, y^2, x, y, 1), src/oc_deformation.cpp:268-282
			const float v0 = __fmul_rn(xl, xl), v1 = __fmul_rn(xl, yl), v2 = __fmul_rn(yl, yl);
			wx = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A[0], v0), __fmul_rn(A[1], v1)), __fmul_rn(A[2], v2)), __fmul_rn(A[3], xl)),
						__fmul_rn(A[4], yl)), A[5]);
			wy = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A[6], v0), __fmul_rn(A[7], v1)), __fmul_rn(A[8], v2)), __fmul_rn(A[9], xl)),
						__fmul_rn(A[10], yl)), A[11]);
		}
		const float X = __fadd_rn(pcx, wx), Y = __fadd_rn(pcy, wy); // center + warped, src/oc_icgn.cpp:238-239
		if (!((X >= 1.f) && (Y >= 1.f) && (X < (float)(w - 2)) && (Y < (float)(h - 2)))) { // BicubicBspline::compute returns -1 (NaN too)
			negative = true;
			continue;
		}
		const float xf = floorf(X), yf = floorf(Y);
		const float* q = tar + (size_t)((int)yf - 1) * w + ((int)xf - 1);
		float blk[16], top = 0.f;
#pragma unroll
		for (int n = 0; n < 4; n++)
#pragma unroll
			for (int m = 0; m < 4; m++) {
				blk[n * 4 + m] = __ldg(q + (size_t)n * w + m);
				top = fmaxf(top, fabsf(blk[n * 4 + m]));
			}
		if (top == 0.f) continue; // an all-zero block gives exactly 0 in any arithmetic
		const float xd = __fsub_rn(X, xf), yd = __fsub_rn(Y, yf);
		float wxx[4], wyy[4];
		bicubic_weights(xd, wxx);
		bicubic_weights(yd, wyy);
		float t = 0.f;
#pragma unroll
		for (int n = 0; n < 4; n++) {
			const float row = fmaf(blk[n * 4 + 3], wxx[3], fmaf(blk[n * 4 + 2], wxx[2], fmaf(blk[n * 4 + 1], wxx[1], blk[n * 4] * wxx[0])));
			t = fmaf(row, wyy[n], t);
		}
		if (t >= ICGN_NEG_BAND) continue;
		if (t <= -ICGN_NEG_BAND || bicubic_reference_order(blk, 4, xd, yd) < 0.f) negative = true;
	}
	return negative;
}

// RC > 0: subset radius known at compile time (rx == ry == RC), so tile pitches and trip counts fold
// into immediates; RC == 0: any radii at run time.
// LM: inverse-compositional Levenberg-Marquardt siblings ICLM2D1 / ICLM2D2 (reference src/oc_iclm.cpp:150-358,
// :502-730): the Hessian is damped with lambda*I and re-factorised every iteration, a step is accepted only
// when ZNSSD decreased, and out-of-range samples are NOT rejected (the interpolant's -1 is used as a value).
// WPP: warps per POI.  One CTA = WPP warps = one POI at a time; the subset rows are split between the warps, which
// share the POI's slab and meet at a CTA barrier once per pass (partial sums through the slab).  Everything after the
// sums (statistics, solve, warp update) is computed redundantly by every warp from the same totals, so the warps
// never diverge in control flow.  With the slab unchanged this doubles the resident warps per SM (r=16: 22 instead
// of 11), which is what the latency-bound row loops need.
// (the second launch bound keeps the register file from limiting residency below what the slab allows: 16 one-warp CTAs for the
//  6-parameter kernels of any radius, 12 for the r = 16 specialisation, whose 20 KB slab admits 11)
// TM: Tensor-Memory variant (WPP == 1, not LM, subset at least 32 columns wide, at most 42 rows).  A CTA is four warps, each
// registering its own POIs exactly like a one-warp CTA; what changes is where a lane keeps the constants of its subset column:
// in its own TMEM lane (tcgen05.st in the setup pass, tcgen05.ld in every iteration) instead of 13 of the 20 KB of shared
// memory per warp.  Shared memory then holds 16 warps per SM instead of 11, and the constants of a row pair come back as the
// register pairs the packed loop wants.  TMEM: 128 columns per CTA, 4 CTAs per SM = all 512 columns.
template <int NP, int RC, bool LM, int WPP, bool TM = false>
__global__ void __launch_bounds__(TM ? 32 * ICGN2D_TM_WARPS : 32 * WPP, TM ? (NP == 6 ? 4 : 1) : (NP == 6 ? (RC == 16 ? 12 : ICGN2D_MINB) / WPP : 7)) icgn2d_kernel(Image2D img, float* __restrict__ pois, int n_poi, int rx_arg, int ry_arg,
	float conv_criterion, float stop_condition, int* __restrict__ work_counter, const __grid_constant__ CUtensorMap tm_ref,
	const __grid_constant__ CUtensorMap tm_tar, int use_tma, const float* __restrict__ center_offsets, float lm_lambda, float lm_alpha,
	float lm_beta) {
	extern __shared__ __align__(128) float smem[];
	constexpr int NH = NP * (NP + 1) / 2;
	constexpr int NPHI = NP / 2;           // 3 or 6 shape monomials per displacement component
	constexpr int DEG = (NP == 6) ? 1 : 2; // degree of the shape function
	constexpr int D2 = 2 * DEG;
	constexpr int NM = (D2 + 1) * (D2 + 2) / 2; // monomials x^P y^Q with P+Q <= 2*DEG: 6 or 15
	const int rx = RC ? RC : rx_arg, ry = RC ? RC : ry_arg;
	const int lane = threadIdx.x & 31;
	static_assert(!TM || (WPP == 1 && !LM), "the Tensor-Memory variant is one warp per POI, plain IC-GN");
	const int sub = WPP > 1 ? (int)(threadIdx.x >> 5) : 0; // this warp's share of the POI
	const int warp_in_cta = (int)(threadIdx.x >> 5);
	const bool poi_leader = TM ? lane == 0 : threadIdx.x == 0; // the thread that speaks for the POI (TMA issue, single stores)
	const int sw = 2 * rx + 1, sh = 2 * ry + 1, N = sw * sh;
	const int rows_per = (sh + WPP - 1) / WPP;
	const int r_lo = sub * rows_per, r_hi = (r_lo + rows_per) < sh ? (r_lo + rows_per) : sh; // rows [r_lo, r_hi) belong to this warp
	const int ncol = sw < 32 ? sw : 32;        // columns handled by the row-mapped main loops
	const int rem = sw - ncol;                  // columns 32.. handled by the tail loops
	const int ntail = rem * sh;
	const int RW = icgn2d_ref_w(rx), RH = icgn2d_ref_h(ry);
	const int TW = icgn2d_tar_w(rx), TH = icgn2d_tar_h(ry);
	float* slab = TM ? smem + warp_in_cta * icgn2d_tm_slab_floats(rx, ry) : smem;
	uint64_t* bar = (uint64_t*)slab;
	int* s_poi = (int*)(slab + 8);              // WPP > 1: the POI index fetched by thread 0
	float* T = slab + 32;
	float* sC = T + icgn2d_tile_floats(rx, ry); // per-sample constants, interleaved {R, gx, gy} (12-byte lane stride: conflict-free); TM: tail columns only
	float* sH = sC + round_up32(3 * N);         // LM only: the undamped Hessian, packed lower triangle
	float* sRedS = sH + (LM ? 96 : 0);          // WPP > 1: setup partials [WPP][ICGN2D_RED_SETUP]
	float* sRedI = sRedS + WPP * ICGN2D_RED_SETUP; // WPP > 1: iteration partials [2][WPP][ICGN2D_RED_ITER]
	uint32_t bar_phase = 0;
	auto gsync = [&]() { // all warps of this POI
		if constexpr (WPP > 1) __syncthreads();
		else __syncwarp();
	};
	if (use_tma) {
		if (poi_leader) mbar_init(bar, 1);
		gsync();
	}
	// TM: the CTA's Tensor-Memory columns; a lane's constants of subset rows (2p, 2p+1) sit in columns 6p .. 6p+5 of its TMEM lane
	// as {R_a, R_b, gx_a, gx_b, gy_a, gy_b}, those of a last single row in 6p .. 6p+2
	uint32_t tm_base = 0, s_tmem_base_value = 0;
	if constexpr (TM) {
		__shared__ uint32_t s_tmem_base;
		if (warp_in_cta == 0) tmem_alloc<ICGN2D_TM_COLS>(&s_tmem_base);
		tmem_fence_before_sync();
		__syncthreads();
		tmem_fence_after_sync();
		s_tmem_base_value = s_tmem_base;
		tm_base = tmem_warp_base(s_tmem_base_value, warp_in_cta);
	}
	// the constants of tail column c >= 32 at row r (smem in both variants)
	auto tail_consts = [&](int r, int c) -> float* { return TM ? sC + 3 * (r * rem + (c - 32)) : sC + 3 * (r * sw + c); };
	// TM: single-row access to a lane's constants (column of R; gx and gy follow at +stride, +2 stride)
	auto tm_row = [&](int r, int& stride) -> uint32_t {
		const bool single = (sh & 1) && r == sh - 1;
		stride = single ? 1 : 2;
		return tm_base + (single ? 3 * r : 6 * (r >> 1) + (r & 1));
	};
	const float* __restrict__ ref = img.ref;
	const float* __restrict__ tar = img.tar;
	const int w = img.w, h = img.h;
	const float inv_n = 1.0f / (float)N;
	const bool lane_on = lane < ncol;
	const int lane_c = lane_on ? lane : ncol - 1; // idle lanes (subsets narrower than 32) shadow the last column

	// WPP == 1: the work counter is drawn and the record requested one POI AHEAD (the queue may be read in place from page-locked
	// host memory; the round trip then hides behind the current POI)
	int poi_next = 0;
	float rec_next = 0.f;
	if constexpr (WPP == 1) {
		if (lane == 0) poi_next = atomicAdd(work_counter, 1);
		poi_next = __shfl_sync(0xffffffffu, poi_next, 0);
		if (poi_next < n_poi && lane < P2_N) rec_next = pois[(size_t)poi_next * P2_N + lane];
	}
	while (true) {
		int poi = 0;
		float rec;
		if constexpr (WPP > 1) {
			gsync(); // every warp is done with the previous POI (slab, s_poi)
			if (threadIdx.x == 0) *s_poi = atomicAdd(work_counter, 1);
			gsync();
			poi = *s_poi;
			if (poi >= n_poi) break;
			rec = lane < P2_N ? pois[(size_t)poi * P2_N + lane] : 0.f;
		} else {
			poi = poi_next;
			if (poi >= n_poi) break;
			rec = rec_next;
			if (lane == 0) poi_next = atomicAdd(work_counter, 1);
			poi_next = __shfl_sync(0xffffffffu, poi_next, 0);
			if (poi_next < n_poi && lane < P2_N) rec_next = pois[(size_t)poi_next * P2_N + lane];
		}
		float* P = pois + (size_t)poi * P2_N;
		const float px = __shfl_sync(0xffffffffu, rec, P2_X);
		const float py = __shfl_sync(0xffffffffu, rec, P2_Y);
		const float u_in = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_U);
		const float v_in = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_V);
		const float zncc_in = __shfl_sync(0xffffffffu, rec, P2_ZNCC);
		// guard, reference src/oc_icgn.cpp:160-167 / :701-708 (NaN coordinates are rejected too)
		if (py - ry < 0 || px - rx < 0 || py + ry > h - 1 || px + rx > w - 1 || fabsf(u_in) >= w || fabsf(v_in) >= h
			|| zncc_in < 0 || is_nan_f(u_in) || is_nan_f(v_in) || is_nan_f(px) || is_nan_f(py)) {
			if (poi_leader) P[P2_ZNCC] = zncc_in >= 0 ? -3.f : zncc_in;
			continue;
		}
		gsync(); // every warp has read the record before thread 0 may write results / TMA may overwrite the slab
		// compute(POI2D*, Point2D& center_offset), src/oc_icgn.cpp:353-547 / :910-1126: local coordinates are
		// (integer - offset) and the target subset is centred at poi + offset; (0, 0) for the plain overload
		float ox = 0.f, oy = 0.f;
		if (center_offsets != nullptr) {
			ox = __ldg(center_offsets + 2 * (size_t)poi);
			oy = __ldg(center_offsets + 2 * (size_t)poi + 1);
		}
		const float xl_lane = (float)(lane - rx) - ox;
		const float pcx = px + ox, pcy = py + oy;

		// ---------------- stage the reference tile ----------------
		const int x0 = (int)px - rx, y0 = (int)py - ry; // Subset2D::fill upper-left, src/oc_subset.cpp:41-42
		const int rox = floor4(x0 - 2), ex = (x0 - 2) - rox; // 16-byte aligned tile origin, column offset 0..3
		if (use_tma) {
			if (poi_leader) {
				fence_proxy_async(); // earlier generic-proxy accesses to T are ordered before the async-proxy write
				mbar_expect_tx(bar, (uint32_t)(RW * RH * sizeof(float)));
				tma_load_2d(T, &tm_ref, rox, y0 - 2, bar);
			}
			mbar_wait(bar, bar_phase);
			bar_phase ^= 1;
		} else {
			if (sub == 0) stage_tile(T, ref, w, h, rox, y0 - 2, RW, RH, 0.f, lane);
			gsync();
		}
		const float c0 = T[(ry + 2) * RW + rx + 2 + ex]; // pilot value: the centre pixel

		// ---------------- setup: R', gradients, factored Hessian sums ----------------
		float r1 = 0.f, r2 = 0.f;
		float accH[3][D2 + 1];   // sum g_a g_b y^Q over this lane's column
		float accS[2][DEG + 1];  // sum g_a y^Q
		float accR[2][DEG + 1];  // sum g_a R' y^Q
#pragma unroll
		for (int a = 0; a < 3; a++)
#pragma unroll
			for (int q = 0; q <= D2; q++) accH[a][q] = 0.f;
#pragma unroll
		for (int a = 0; a < 2; a++)
#pragma unroll
			for (int q = 0; q <= DEG; q++) { accS[a][q] = 0.f; accR[a][q] = 0.f; }
		{
			const int xg = x0 + lane;
			const bool gx_ok = lane_on && xg >= 2 && xg < w - 2; // gradient maps are zero on a 2-pixel border (src/oc_gradient.cpp:42,46)
			int r_first = r_lo;
#if ICGN2D_PAIRS
			if (lane_on) {
				// rows (r, r + 1) in lanes {.x, .y} of packed pairs: the same operations as the one-row loop below (the gradients keep
				// the reference's separately rounded products and sums), and the six pixels of this lane's column that the two y
				// gradients need are fetched once
				float2 r1p = make_float2(0.f, 0.f), r2p = r1p;
				float2 accH2[3][D2 + 1], accS2[2][DEG + 1], accR2[2][DEG + 1];
#pragma unroll
				for (int a = 0; a < 3; a++)
#pragma unroll
					for (int qq = 0; qq <= D2; qq++) accH2[a][qq] = r1p;
#pragma unroll
				for (int a = 0; a < 2; a++)
#pragma unroll
					for (int qq = 0; qq <= DEG; qq++) { accS2[a][qq] = r1p; accR2[a][qq] = r1p; }
				const float2 f1 = bcast2(1.f / 12.f), f2 = bcast2(2.f / 3.f);
				const int npair = (r_hi - r_lo) >> 1;
#pragma unroll ICGN2D_SETUP_UNROLL_N
				for (int pr = 0; pr < npair; pr++) {
					const int r = r_lo + 2 * pr;
					const int yg = y0 + r;
					const float* q = T + (r + 2) * RW + lane + 2 + ex;
					const float v0 = q[-2 * RW], v1 = q[-RW], v2 = q[0], v3 = q[RW], v4 = q[2 * RW], v5 = q[3 * RW];
					const float2 yl2 = make_float2((float)(r - ry) - oy, (float)(r + 1 - ry) - oy);
					const float2 Rraw = make_float2(v2, v3);
					const float2 R2 = fsub2(Rraw, bcast2(c0));
					// grad4: ((0 - f(+2)/12) + f(+1)*2/3) - f(-1)*2/3 + f(-2)/12, every operation rounded separately (src/oc_gradient.cpp:49-54)
					float2 gx2 = fsub2(bcast2(0.f), fmul2(make_float2(q[2], q[RW + 2]), f1));
					gx2 = fadd2(gx2, fmul2(make_float2(q[1], q[RW + 1]), f2));
					gx2 = fsub2(gx2, fmul2(make_float2(q[-1], q[RW - 1]), f2));
					gx2 = fadd2(gx2, fmul2(make_float2(q[-2], q[RW - 2]), f1));
					float2 gy2 = fsub2(bcast2(0.f), fmul2(make_float2(v4, v5), f1));
					gy2 = fadd2(gy2, fmul2(make_float2(v3, v4), f2));
					gy2 = fsub2(gy2, fmul2(make_float2(v1, v2), f2));
					gy2 = fadd2(gy2, fmul2(make_float2(v0, v1), f1));
					if (!gx_ok) gx2 = make_float2(0.f, 0.f);
					if (!(yg >= 2 && yg < h - 2)) gy2.x = 0.f;
					if (!(yg + 1 >= 2 && yg + 1 < h - 2)) gy2.y = 0.f;
					if constexpr (TM) {
						tmem_st4(tm_base + 3 * r, v2, v3, gx2.x, gx2.y);
						tmem_st2(tm_base + 3 * r + 4, gy2.x, gy2.y);
					} else {
						float* pc = sC + 3 * (r * sw + lane);
						pc[0] = v2; pc[1] = gx2.x; pc[2] = gy2.x;
						pc[3 * sw] = v3; pc[3 * sw + 1] = gx2.y; pc[3 * sw + 2] = gy2.y;
					}
					r1p = fadd2(r1p, R2);
					r2p = ffma2(R2, R2, r2p);
					float2 g[3] = { fmul2(gx2, gx2), fmul2(gx2, gy2), fmul2(gy2, gy2) };
#pragma unroll
					for (int a = 0; a < 3; a++) {
						float2 t = g[a];
#pragma unroll
						for (int qq = 0; qq <= D2; qq++) {
							accH2[a][qq] = fadd2(accH2[a][qq], t);
							if (qq < D2) t = fmul2(t, yl2);
						}
					}
					float2 g1[2] = { gx2, gy2 };
#pragma unroll
					for (int a = 0; a < 2; a++) {
						float2 t = g1[a], tr = fmul2(g1[a], R2);
#pragma unroll
						for (int qq = 0; qq <= DEG; qq++) {
							accS2[a][qq] = fadd2(accS2[a][qq], t);
							accR2[a][qq] = fadd2(accR2[a][qq], tr);
							if (qq < DEG) { t = fmul2(t, yl2); tr = fmul2(tr, yl2); }
						}
					}
				}
				r1 = r1p.x + r1p.y;
				r2 = r2p.x + r2p.y;
#pragma unroll
				for (int a = 0; a < 3; a++)
#pragma unroll
					for (int qq = 0; qq <= D2; qq++) accH[a][qq] = accH2[a][qq].x + accH2[a][qq].y;
#pragma unroll
				for (int a = 0; a < 2; a++)
#pragma unroll
					for (int qq = 0; qq <= DEG; qq++) { accS[a][qq] = accS2[a][qq].x + accS2[a][qq].y; accR[a][qq] = accR2[a][qq].x + accR2[a][qq].y; }
				r_first = r_lo + 2 * npair;
			}
#endif
			for (int r = r_first; r < r_hi; r++) {
				const int yg = y0 + r;
				const bool gy_ok = yg >= 2 && yg < h - 2;
				const float yl = (float)(r - ry) - oy;
				if (lane_on) {
					const float* q = T + (r + 2) * RW + lane + 2 + ex;
					const float R = q[0] - c0;
					float gx = 0.f, gy = 0.f;
					if (gx_ok) gx = grad4(q[-2], q[-1], q[1], q[2]);
					if (gy_ok) gy = grad4(q[-2 * RW], q[-RW], q[RW], q[2 * RW]);
					if constexpr (TM) { // (every lane is on in this variant: the stores are warp-convergent)
						int st;
						const uint32_t ta = tm_row(r, st);
						tmem_st1(ta, q[0]);
						tmem_st1(ta + st, gx);
						tmem_st1(ta + 2 * st, gy);
					} else {
						float* pc = sC + 3 * (r * sw + lane);
						pc[0] = q[0]; // raw R
						pc[1] = gx;
						pc[2] = gy;
					}
					r1 += R;
					r2 = fmaf(R, R, r2);
					float g[3] = { gx * gx, gx * gy, gy * gy };
#pragma unroll
					for (int a = 0; a < 3; a++) {
						float t = g[a];
#pragma unroll
						for (int qq = 0; qq <= D2; qq++) {
							accH[a][qq] += t;
							if (qq < D2) t *= yl;
						}
					}
					float g1[2] = { gx, gy };
#pragma unroll
					for (int a = 0; a < 2; a++) {
						float t = g1[a], tr = g1[a] * R;
#pragma unroll
						for (int qq = 0; qq <= DEG; qq++) {
							accS[a][qq] += t;
							accR[a][qq] += tr;
							if (qq < DEG) { t *= yl; tr *= yl; }
						}
					}
				}
			}
		}
		// expand with this lane's x powers: M[pair][mono(P,Q)] = x^P * accH[pair][Q]
		float M[3][NM], Sg[2][NPHI], SRg[2][NPHI];
		{
			float xp[D2 + 1];
			xp[0] = 1.f;
#pragma unroll
			for (int p = 1; p <= D2; p++) xp[p] = xp[p - 1] * xl_lane;
#pragma unroll
			for (int Pp = 0; Pp <= D2; Pp++)
#pragma unroll
				for (int Q = 0; Q <= D2; Q++)
					if (Pp + Q <= D2) {
#pragma unroll
						for (int a = 0; a < 3; a++) M[a][mono(Pp, Q)] = xp[Pp] * accH[a][Q];
					}
#pragma unroll
			for (int i = 0; i < NPHI; i++)
#pragma unroll
				for (int a = 0; a < 2; a++) {
					Sg[a][i] = xp[phi_p(i)] * accS[a][phi_q(i)];
					SRg[a][i] = xp[phi_p(i)] * accR[a][phi_q(i)];
				}
		}
		// tail columns (>= 32): lanes run over (row, column) pairs, general x and y
		for (int idx = sub * 32 + lane; idx < ntail; idx += 32 * WPP) {
			const int r = idx / rem, c = 32 + (idx - r * rem);
			const int xg = x0 + c, yg = y0 + r;
			const float xl = (float)(c - rx) - ox, yl = (float)(r - ry) - oy;
			const float* q = T + (r + 2) * RW + c + 2 + ex;
			const float R = q[0] - c0;
			float gx = 0.f, gy = 0.f;
			if (xg >= 2 && xg < w - 2) gx = grad4(q[-2], q[-1], q[1], q[2]);
			if (yg >= 2 && yg < h - 2) gy = grad4(q[-2 * RW], q[-RW], q[RW], q[2 * RW]);
			float* pc = tail_consts(r, c);
			pc[0] = q[0];
			pc[1] = gx;
			pc[2] = gy;
			r1 += R;
			r2 = fmaf(R, R, r2);
			float g[3] = { gx * gx, gx * gy, gy * gy };
			float g1[2] = { gx, gy };
#pragma unroll
			for (int Pp = 0; Pp <= D2; Pp++)
#pragma unroll
				for (int Q = 0; Q <= D2; Q++)
					if (Pp + Q <= D2) {
						const float mm = ipow(xl, Pp) * ipow(yl, Q);
#pragma unroll
						for (int a = 0; a < 3; a++) M[a][mono(Pp, Q)] = fmaf(g[a], mm, M[a][mono(Pp, Q)]);
					}
#pragma unroll
			for (int ii = 0; ii < NPHI; ii++) {
				const float mm = ipow(xl, phi_p(ii)) * ipow(yl, phi_q(ii));
#pragma unroll
				for (int a = 0; a < 2; a++) {
					Sg[a][ii] = fmaf(g1[a], mm, Sg[a][ii]);
					SRg[a][ii] = fmaf(g1[a] * R, mm, SRg[a][ii]);
				}
			}
		}
		r1 = warp_sum(r1);
		r2 = warp_sum(r2);
#pragma unroll
		for (int a = 0; a < 3; a++)
#pragma unroll
			for (int m = 0; m < NM; m++) M[a][m] = warp_sum(M[a][m]);
#pragma unroll
		for (int a = 0; a < 2; a++)
#pragma unroll
			for (int i = 0; i < NPHI; i++) { Sg[a][i] = warp_sum(Sg[a][i]); SRg[a][i] = warp_sum(SRg[a][i]); }
		if constexpr (WPP > 1) {
			// partial sums of the warps meet here; every warp then adds them in the same order
			static_assert(2 + 3 * NM + 4 * NPHI <= ICGN2D_RED_SETUP, "setup partials do not fit");
			if (lane == 0) {
				float* o = sRedS + sub * ICGN2D_RED_SETUP;
				o[0] = r1;
				o[1] = r2;
#pragma unroll
				for (int a = 0; a < 3; a++)
#pragma unroll
					for (int m = 0; m < NM; m++) o[2 + a * NM + m] = M[a][m];
#pragma unroll
				for (int a = 0; a < 2; a++)
#pragma unroll
					for (int i = 0; i < NPHI; i++) { o[2 + 3 * NM + a * NPHI + i] = Sg[a][i]; o[2 + 3 * NM + 2 * NPHI + a * NPHI + i] = SRg[a][i]; }
			}
			gsync(); // also: every warp is done with the reference tile
			r1 = 0.f;
			r2 = 0.f;
#pragma unroll
			for (int a = 0; a < 3; a++)
#pragma unroll
				for (int m = 0; m < NM; m++) M[a][m] = 0.f;
#pragma unroll
			for (int a = 0; a < 2; a++)
#pragma unroll
				for (int i = 0; i < NPHI; i++) { Sg[a][i] = 0.f; SRg[a][i] = 0.f; }
#pragma unroll
			for (int ww = 0; ww < WPP; ww++) {
				const float* o = sRedS + ww * ICGN2D_RED_SETUP;
				r1 += o[0];
				r2 += o[1];
#pragma unroll
				for (int a = 0; a < 3; a++)
#pragma unroll
					for (int m = 0; m < NM; m++) M[a][m] += o[2 + a * NM + m];
#pragma unroll
				for (int a = 0; a < 2; a++)
#pragma unroll
					for (int i = 0; i < NPHI; i++) { Sg[a][i] += o[2 + 3 * NM + a * NPHI + i]; SRg[a][i] += o[2 + 3 * NM + 2 * NPHI + a * NPHI + i]; }
			}
		}
		// reference subset statistics (Subset2D::zeroMeanNorm, src/oc_subset.cpp:46-53), relative to c0
		const float rbar = r1 * inv_n;              // mean(R) - c0
		const float f2 = r2 - r1 * rbar;            // sum f^2, f = R - mean(R)
		const float ref_norm = sqrtf(f2);
		// S_k = sum sd_k, SF_k = sum sd_k f = sum sd_k R' - rbar * S_k ; H = sum sd sd^T (src/oc_icgn.cpp:198-205)
		float H[NH], S[NP], SF[NP];
#pragma unroll
		for (int a = 0; a < 2; a++)
#pragma unroll
			for (int i = 0; i < NPHI; i++) {
				const int k = a * NPHI + i;
				S[k] = phi_c(i) * Sg[a][i];
				SF[k] = phi_c(i) * (SRg[a][i] - rbar * Sg[a][i]);
#pragma unroll
				for (int b = 0; b < 2; b++)
#pragma unroll
					for (int j = 0; j < NPHI; j++) {
						const int l = b * NPHI + j;
						if (l <= k) H[k * (k + 1) / 2 + l] = phi_c(i) * phi_c(j) * M[pair_idx(a, b)][mono(phi_p(i) + phi_p(j), phi_q(i) + phi_q(j))];
					}
			}
		if constexpr (LM) {
			if (threadIdx.x == 0) {
#pragma unroll
				for (int k = 0; k < NH; k++) sH[k] = H[k];
			}
			gsync();
		} else {
			cholesky_packed<NP>(H);
		}
		float lm_cur = 0.f, znssd0 = 4.f; // src/oc_iclm.cpp:234-235

		if constexpr (TM) tmem_wait_st(); // the setup pass's constants are in Tensor Memory before the first iteration reads them
		// ---------------- stage the target tile over the reference tile ----------------
		// (WPP > 1: the barrier of the setup reduction already ordered every warp's last read of the reference tile)
		if constexpr (WPP == 1) __syncwarp();
		const int tx0 = floor4((int)floorf(pcx + u_in) - rx - 1 - ICGN2D_TILE_MARGIN);
		const int ty0 = (int)floorf(pcy + v_in) - ry - 1 - ICGN2D_TILE_MARGIN;
		if (use_tma) {
			if (poi_leader) {
				fence_proxy_async();
				mbar_expect_tx(bar, (uint32_t)(TW * TH * sizeof(float)));
				tma_load_2d(T, &tm_tar, tx0, ty0, bar);
			}
			mbar_wait(bar, bar_phase);
			bar_phase ^= 1;
		} else {
			if (sub == 0) stage_tile(T, tar, w, h, tx0, ty0, TW, TH, 0.f, lane);
			gsync();
		}
		// a sample is "fast" when it is valid (src/oc_cubic_bspline.cpp:137-142) AND its support is in the tile
		const float xlo = fmaxf(1.f, (float)(tx0 + 1)), xhi = fminf((float)(w - 2), (float)(tx0 + TW - 2));
		const float ylo = fmaxf(1.f, (float)(ty0 + 1)), yhi = fminf((float)(h - 2), (float)(ty0 + TH - 2));
		const float xmax = (float)(w - 2), ymax = (float)(h - 2);

		// ---------------- IC-GN iterations ----------------
		// running warp: NP==6 -> A = {W00,W01,W02,W10,W11,W12}; NP==12 -> rows 3,4 of the 6x6 warp
		float A[12];
		{
			const float ux = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_UX), uy = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_UY);
			const float vx = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_VX), vy = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_VY);
			if constexpr (NP == 6) {
				A[0] = 1.f + ux; A[1] = uy; A[2] = u_in; A[3] = vx; A[4] = 1.f + vy; A[5] = v_in;
			} else { // second-order terms of the incoming guess are dropped (src/oc_icgn.cpp:765-770)
				A[0] = 0.f; A[1] = 0.f; A[2] = 0.f; A[3] = 1.f + ux; A[4] = uy; A[5] = u_in;
				A[6] = 0.f; A[7] = 0.f; A[8] = 0.f; A[9] = vx; A[10] = 1.f + vy; A[11] = v_in;
			}
		}
		int iteration = 0;
		float dp_norm = 0.f, zncc = 0.f;
		bool left_image = false;
		float dp[NP];
		do {
			iteration++;
			float d1 = 0.f, d2 = 0.f, rd = 0.f;
			float G[2][DEG + 1]; // sum g_a d y^Q over this lane's column
#pragma unroll
			for (int a = 0; a < 2; a++)
#pragma unroll
				for (int q = 0; q <= DEG; q++) G[a][q] = 0.f;
			bool invalid = false;
			float tmin = 3.0e38f; // smallest interpolated sample of this pass (see icgn2d_exact_negative)
			// per-lane x part of the warp (Deformation2D1::warp src/oc_deformation.cpp:94-105,
			// Deformation2D2::warp rows 3,4 :268-282): X = px + (ax2*y^2 + ax1*y + ax0)
			float ax0, ax1, ax2, ay0, ay1, ay2;
			if constexpr (NP == 6) {
				ax0 = fmaf(A[0], xl_lane, A[2]); ax1 = A[1]; ax2 = 0.f;
				ay0 = fmaf(A[3], xl_lane, A[5]); ay1 = A[4]; ay2 = 0.f;
			} else {
				ax0 = fmaf(A[0] * xl_lane + A[3], xl_lane, A[5]); ax1 = fmaf(A[1], xl_lane, A[4]); ax2 = A[2];
				ay0 = fmaf(A[6] * xl_lane + A[9], xl_lane, A[11]); ay1 = fmaf(A[7], xl_lane, A[10]); ay2 = A[8];
			}
			// Can every row-mapped sample take the fast path (valid + support inside the tile)?  The
			// affine part of the warp maps the subset to a parallelogram, so its 4 corners decide;
			// the second-order part is bounded by qx/qy and shrinks the window.
			bool iter_fast;
			{
				float qx = 0.f, qy = 0.f;
				const float fx = (float)rx + fabsf(ox), fy = (float)ry + fabsf(oy);
				float a0, a1, a2, b0, b1, b2; // X = px + a0 x + a1 y + a2 (+ quadratic), same for Y
				if constexpr (NP == 6) {
					a0 = A[0]; a1 = A[1]; a2 = A[2]; b0 = A[3]; b1 = A[4]; b2 = A[5];
				} else {
					a0 = A[3]; a1 = A[4]; a2 = A[5]; b0 = A[9]; b1 = A[10]; b2 = A[11];
					qx = fabsf(A[0]) * fx * fx + fabsf(A[1]) * fx * fy + fabsf(A[2]) * fy * fy;
					qy = fabsf(A[6]) * fx * fx + fabsf(A[7]) * fx * fy + fabsf(A[8]) * fy * fy;
				}
				const float cx = pcx + a2, cy = pcy + b2;
				const float ex_ = fabsf(a0) * fx + fabsf(a1) * fy + qx, ey_ = fabsf(b0) * fx + fabsf(b1) * fy + qy;
				iter_fast = (cx - ex_ >= xlo) && (cx + ex_ < xhi) && (cy - ey_ >= ylo) && (cy + ey_ < yhi); // false for NaN
			}
			if (iter_fast) {
				// branch-free row loop: no per-sample validity tests (min(t) is tested after the loop)
				float yl = (float)(r_lo - ry) - oy;
				const float* pc = sC + 3 * (r_lo * sw + lane_c);
				float xs0, xs1, xs2, ys0, ys1, ys2;
				{
					const float xl = (float)(lane_c - rx) - ox;
					// the warped offset is formed first and the POI centre added last, with ONE rounding at
					// the large magnitude, like the reference's `center + warped` (src/oc_icgn.cpp:238-239):
					// at x ~ 4096 a float ulp is 4.9e-4 px, so the association order is visible in the result
					if constexpr (NP == 6) {
						xs0 = fmaf(A[0], xl, A[2]); xs1 = A[1]; xs2 = 0.f;
						ys0 = fmaf(A[3], xl, A[5]); ys1 = A[4]; ys2 = 0.f;
					} else {
						xs0 = fmaf(A[0] * xl + A[3], xl, A[5]); xs1 = fmaf(A[1], xl, A[4]); xs2 = A[2];
						ys0 = fmaf(A[6] * xl + A[9], xl, A[11]); ys1 = fmaf(A[7], xl, A[10]); ys2 = A[8];
					}
				}
				const float* tbase = T - (ty0 + 1) * TW - (tx0 + 1);
				int r_first = r_lo; // first row of the one-row-per-step loop below
#if ICGN2D_PAIRS
				{
					// rows (r, r + 1) as lanes {.x, .y} of packed pairs; the same operations, in the same order, as the one-row loop
					float2 d1p = make_float2(0.f, 0.f), d2p = d1p, rdp = d1p;
					float2 Gp[2][DEG + 1];
#pragma unroll
					for (int a = 0; a < 2; a++)
#pragma unroll
						for (int qq = 0; qq <= DEG; qq++) Gp[a][qq] = d1p;
					const float2 pcx2 = bcast2(pcx), pcy2 = bcast2(pcy);
					const float2 xs0p = bcast2(xs0), xs1p = bcast2(xs1), xs2p = bcast2(xs2), ys0p = bcast2(ys0), ys1p = bcast2(ys1), ys2p = bcast2(ys2);
					constexpr float s336 = 1.0f / 336.0f;
					// w_j(t) = ((a_j t + b_j) t + c_j) t + e_j, the reference's BC matrix by columns (ocb_common.cuh bicubic_weights)
					constexpr float BA[4] = { -144.0f * s336, 384.0f * s336, -384.0f * s336, 144.0f * s336 };
					constexpr float BB[4] = { 342.0f * s336, -702.0f * s336, 450.0f * s336, -90.0f * s336 };
					constexpr float BC_[4] = { -198.0f * s336, -18.0f * s336, 270.0f * s336, -54.0f * s336 };
					constexpr float BE[4] = { 0.f, 1.f, 0.f, 0.f };
					float2 yl2 = make_float2(yl, yl + 1.f);
					const int npair = (r_hi - r_lo) >> 1;
#pragma unroll (TM ? 1 : ICGN2D_PAIR_UNROLL_N) // (16 resident warps need less unrolling than 11: measured 0.647 vs 0.653 ms on config B)
					for (int pr = 0; pr < npair; pr++) {
						float2 R2c, gx2c, gy2c; // the two rows' constants
						if constexpr (TM) { // requested now, needed after the taps
							const uint32_t ta = tm_base + 3 * (r_lo + 2 * pr);
							tmem_ld4(ta, R2c.x, R2c.y, gx2c.x, gx2c.y);
							tmem_ld2(ta + 4, gy2c.x, gy2c.y);
						}
						float2 X2, Y2;
						if constexpr (NP == 6) {
							X2 = fadd2(pcx2, ffma2(xs1p, yl2, xs0p));
							Y2 = fadd2(pcy2, ffma2(ys1p, yl2, ys0p));
						} else {
							X2 = fadd2(pcx2, ffma2(ffma2(xs2p, yl2, xs1p), yl2, xs0p));
							Y2 = fadd2(pcy2, ffma2(ffma2(ys2p, yl2, ys1p), yl2, ys0p));
						}
						const float xfa = floorf(X2.x), xfb = floorf(X2.y), yfa = floorf(Y2.x), yfb = floorf(Y2.y);
						const float2 tx = fsub2(X2, make_float2(xfa, xfb)), ty = fsub2(Y2, make_float2(yfa, yfb));
						// weights of both rows: WX[j] = {w_j(tx.x), w_j(tx.y)}, WYu[j] likewise in y.  The rows of the shared 4x5 block
						// are j = 0..4 and row r + 1 starts one block row lower: block rows 1..3 serve both samples (packed, y weights
						// {w_j(ty.x), w_{j-1}(ty.y)}), row 0 only the first and row 4 only the second (scalar on that half of the pair)
						float2 WX[4], WYu[4], WY[3];
#pragma unroll
						for (int j = 0; j < 4; j++) {
							WX[j] = ffma2(ffma2(ffma2(bcast2(BA[j]), tx, bcast2(BB[j])), tx, bcast2(BC_[j])), tx, bcast2(BE[j]));
							WYu[j] = ffma2(ffma2(ffma2(bcast2(BA[j]), ty, bcast2(BB[j])), ty, bcast2(BC_[j])), ty, bcast2(BE[j]));
						}
#pragma unroll
						for (int j = 1; j < 4; j++) WY[j - 1] = make_float2(WYu[j].x, WYu[j - 1].y);
						const float* q = tbase + (int)yfa * TW + (int)xfa;
						float2 t2;
						{
							const float row = fmaf(q[3], WX[3].x, fmaf(q[2], WX[2].x, fmaf(q[1], WX[1].x, q[0] * WX[0].x)));
							t2 = make_float2(fmaf(row, WYu[0].x, 0.f), 0.f);
						}
#pragma unroll
						for (int j = 1; j < 4; j++) {
							const float2 row = ffma2(bcast2(q[j * TW + 3]), WX[3], ffma2(bcast2(q[j * TW + 2]), WX[2], ffma2(bcast2(q[j * TW + 1]), WX[1], fmul2(bcast2(q[j * TW]), WX[0]))));
							t2 = ffma2(row, WY[j - 1], t2);
						}
						{
							const float row = fmaf(q[4 * TW + 3], WX[3].y, fmaf(q[4 * TW + 2], WX[2].y, fmaf(q[4 * TW + 1], WX[1].y, q[4 * TW] * WX[0].y)));
							t2.y = fmaf(row, WYu[3].y, t2.y);
						}
						// row r + 1 normally sits one block row below row r in the same columns; where the warp's shear or stretch
						// breaks that (a few lanes per POI), its sample is evaluated on its own
						if (xfb != xfa || yfb != yfa + 1.f) t2.y = bicubic_sample(T, TW, tx0, ty0, tar, w, X2.y, Y2.y, true);
						tmin = fminf(tmin, fminf(t2.x, t2.y));
						if constexpr (TM) tmem_wait_ld();
						else { R2c = make_float2(pc[0], pc[3 * sw]); gx2c = make_float2(pc[1], pc[3 * sw + 1]); gy2c = make_float2(pc[2], pc[3 * sw + 2]); }
						const float2 R2 = R2c;
						float2 dd = fsub2(t2, R2);
						if (!lane_on) dd = make_float2(0.f, 0.f);
						d1p = fadd2(d1p, dd);
						d2p = ffma2(dd, dd, d2p);
						rdp = ffma2(R2, dd, rdp);
						float2 gd[2] = { fmul2(gx2c, dd), fmul2(gy2c, dd) };
#pragma unroll
						for (int a = 0; a < 2; a++) {
							float2 tt = gd[a];
#pragma unroll
							for (int qq = 0; qq <= DEG; qq++) {
								Gp[a][qq] = fadd2(Gp[a][qq], tt);
								if (qq < DEG) tt = fmul2(tt, yl2);
							}
						}
						pc += 6 * sw;
						yl2 = fadd2(yl2, bcast2(2.f));
					}
					d1 = d1p.x + d1p.y;
					d2 = d2p.x + d2p.y;
					rd = rdp.x + rdp.y;
#pragma unroll
					for (int a = 0; a < 2; a++)
#pragma unroll
						for (int qq = 0; qq <= DEG; qq++) G[a][qq] = Gp[a][qq].x + Gp[a][qq].y;
					r_first = r_lo + 2 * npair;
					yl += (float)(2 * npair);
				}
#endif
#pragma unroll ICGN2D_ROW_UNROLL
				for (int r = r_first; r < r_hi; r++) {
					float X, Y;
					if constexpr (NP == 6) {
						X = pcx + fmaf(xs1, yl, xs0);
						Y = pcy + fmaf(ys1, yl, ys0);
					} else {
						X = pcx + fmaf(fmaf(xs2, yl, xs1), yl, xs0);
						Y = pcy + fmaf(fmaf(ys2, yl, ys1), yl, ys0);
					}
					const float xf = floorf(X), yf = floorf(Y);
					float wx[4], wy[4];
					bicubic_weights(X - xf, wx);
					bicubic_weights(Y - yf, wy);
					const float* q = tbase + (int)yf * TW + (int)xf;
					float t = 0.f;
#pragma unroll
					for (int nn = 0; nn < 4; nn++) {
						float row = fmaf(q[nn * TW + 3], wx[3], fmaf(q[nn * TW + 2], wx[2], fmaf(q[nn * TW + 1], wx[1], q[nn * TW] * wx[0])));
						t = fmaf(row, wy[nn], t);
					}
					tmin = fminf(tmin, t);
					float R, gxc, gyc;
					if constexpr (TM) {
						int st;
						const uint32_t ta = tm_row(r, st);
						R = tmem_ld1(ta);
						gxc = tmem_ld1(ta + st);
						gyc = tmem_ld1(ta + 2 * st);
						tmem_wait_ld();
					} else {
						R = pc[0]; gxc = pc[1]; gyc = pc[2];
					}
					const float d = lane_on ? t - R : 0.f;
					d1 += d;
					d2 = fmaf(d, d, d2);
					rd = fmaf(R, d, rd);
					float gd[2] = { gxc * d, gyc * d };
#pragma unroll
					for (int a = 0; a < 2; a++) {
						float tt = gd[a];
#pragma unroll
						for (int qq = 0; qq <= DEG; qq++) {
							G[a][qq] += tt;
							if (qq < DEG) tt *= yl;
						}
					}
					pc += 3 * sw;
					yl += 1.f;
				}
			} else {
				for (int r = r_lo; r < r_hi; r++) {
					const float yl = (float)(r - ry) - oy;
					float X, Y;
					if constexpr (NP == 6) {
						X = pcx + fmaf(ax1, yl, ax0);
						Y = pcy + fmaf(ay1, yl, ay0);
					} else {
						X = pcx + fmaf(fmaf(ax2, yl, ax1), yl, ax0);
						Y = pcy + fmaf(fmaf(ay2, yl, ay1), yl, ay0);
					}
					float Rt = 0.f, gxt = 0.f, gyt = 0.f;
					if constexpr (TM) { // warp-convergent: before the per-lane branches
						int st;
						const uint32_t ta = tm_row(r, st);
						Rt = tmem_ld1(ta);
						gxt = tmem_ld1(ta + st);
						gyt = tmem_ld1(ta + 2 * st);
						tmem_wait_ld();
					}
					if (lane_on) {
						const bool fast = (X >= xlo) && (X < xhi) && (Y >= ylo) && (Y < yhi);
						const bool ok = fast || ((X >= 1.f) && (Y >= 1.f) && (X < xmax) && (Y < ymax)); // NaN fails
						if (!ok && !LM) {
							invalid = true;
						} else {
							const float t = ok ? bicubic_sample(T, TW, tx0, ty0, tar, w, X, Y, fast) : -1.f; // BicubicBspline::compute returns -1 outside
							tmin = fminf(tmin, t);
							if constexpr (!TM) {
								const float* pc = sC + 3 * (r * sw + lane);
								Rt = pc[0]; gxt = pc[1]; gyt = pc[2];
							}
							const float R = Rt;
							const float d = t - R;
							d1 += d;
							d2 = fmaf(d, d, d2);
							rd = fmaf(R, d, rd);
							float gd[2] = { gxt * d, gyt * d };
#pragma unroll
							for (int a = 0; a < 2; a++) {
								float tt = gd[a];
#pragma unroll
								for (int qq = 0; qq <= DEG; qq++) {
									G[a][qq] += tt;
									if (qq < DEG) tt *= yl;
								}
							}
						}
					}
				}
			}
			float SD[NP];
			{
				float xp[DEG + 1];
				xp[0] = 1.f;
#pragma unroll
				for (int p = 1; p <= DEG; p++) xp[p] = xp[p - 1] * xl_lane;
#pragma unroll
				for (int a = 0; a < 2; a++)
#pragma unroll
					for (int i = 0; i < NPHI; i++) SD[a * NPHI + i] = phi_c(i) * xp[phi_p(i)] * G[a][phi_q(i)];
			}
			for (int idx = sub * 32 + lane; idx < ntail; idx += 32 * WPP) {
				const int r = idx / rem, c = 32 + (idx - r * rem);
				const float xl = (float)(c - rx) - ox, yl = (float)(r - ry) - oy;
				float X, Y;
				if constexpr (NP == 6) {
					X = pcx + fmaf(A[0], xl, fmaf(A[1], yl, A[2]));
					Y = pcy + fmaf(A[3], xl, fmaf(A[4], yl, A[5]));
				} else {
					const float m0 = xl * xl, m1 = xl * yl, m2 = yl * yl;
					X = pcx + fmaf(A[0], m0, fmaf(A[1], m1, fmaf(A[2], m2, fmaf(A[3], xl, fmaf(A[4], yl, A[5])))));
					Y = pcy + fmaf(A[6], m0, fmaf(A[7], m1, fmaf(A[8], m2, fmaf(A[9], xl, fmaf(A[10], yl, A[11])))));
				}
				const bool fast = (X >= xlo) && (X < xhi) && (Y >= ylo) && (Y < yhi);
				const bool ok = fast || ((X >= 1.f) && (Y >= 1.f) && (X < xmax) && (Y < ymax));
				if (!ok && !LM) {
					invalid = true;
				} else {
					const float t = ok ? bicubic_sample(T, TW, tx0, ty0, tar, w, X, Y, fast) : -1.f;
					tmin = fminf(tmin, t);
					const float* pc = tail_consts(r, c);
					const float R = pc[0];
					const float d = t - R;
					d1 += d;
					d2 = fmaf(d, d, d2);
					rd = fmaf(R, d, rd);
					float gd[2] = { pc[1] * d, pc[2] * d };
#pragma unroll
					for (int ii = 0; ii < NPHI; ii++) {
						const float mm = phi_c(ii) * ipow(xl, phi_p(ii)) * ipow(yl, phi_q(ii));
#pragma unroll
						for (int a = 0; a < 2; a++) SD[a * NPHI + ii] = fmaf(gd[a], mm, SD[a * NPHI + ii]);
					}
				}
			}
			if constexpr (!LM) { // src/oc_icgn.cpp:251-255: any sample < 0 rejects the POI (the ICLM siblings have no such test)
				if (tmin < -ICGN_NEG_TRIGGER) invalid = true;
				const bool borderline = !(tmin >= ICGN_NEG_TRIGGER);
				if (__any_sync(0xffffffffu, borderline) && !__any_sync(0xffffffffu, invalid)) {
					float* sA = slab + 16; // the running warp, handed over through the slab header
					if (lane == 0) {
#pragma unroll
						for (int k = 0; k < (NP == 6 ? 6 : 12); k++) sA[k] = A[k];
					}
					__syncwarp();
					if (icgn2d_exact_negative<NP>(sA, pcx, pcy, ox, oy, rx, ry, tar, w, h, lane, N)) invalid = true;
				}
			}
			bool any_invalid = __any_sync(0xffffffffu, invalid);
			d1 = warp_sum(d1);
			d2 = warp_sum(d2);
			rd = warp_sum(rd);
#pragma unroll
			for (int k = 0; k < NP; k++) SD[k] = warp_sum(SD[k]);
			if constexpr (WPP > 1) {
				static_assert(4 + NP <= ICGN2D_RED_ITER, "iteration partials do not fit");
				float* o = sRedI + ((iteration & 1) * WPP + sub) * ICGN2D_RED_ITER; // double-buffered: one barrier per iteration
				if (lane == 0) {
					o[0] = d1;
					o[1] = d2;
					o[2] = rd;
					o[3] = any_invalid ? 1.f : 0.f;
#pragma unroll
					for (int k = 0; k < NP; k++) o[4 + k] = SD[k];
				}
				gsync();
				d1 = 0.f;
				d2 = 0.f;
				rd = 0.f;
				float inv_flag = 0.f;
#pragma unroll
				for (int k = 0; k < NP; k++) SD[k] = 0.f;
#pragma unroll
				for (int ww = 0; ww < WPP; ww++) {
					const float* q = sRedI + ((iteration & 1) * WPP + ww) * ICGN2D_RED_ITER;
					d1 += q[0];
					d2 += q[1];
					rd += q[2];
					inv_flag += q[3];
#pragma unroll
					for (int k = 0; k < NP; k++) SD[k] += q[4 + k];
				}
				any_invalid = inv_flag > 0.f;
			}
			if (any_invalid) { // src/oc_icgn.cpp:251-255
				left_image = true;
				break;
			}
			// warped-target statistics: g = t - mean(t) = f + (d - dbar); sum f d = sum R'd - rbar * sum d
			const float dbar = d1 * inv_n;
			const float fd = (rd - c0 * d1) - rbar * d1; // rd holds sum R d with the raw R
			const float g2 = f2 + 2.f * fd + (d2 - d1 * dbar);
			const float tar_norm = sqrtf(g2);
			const float factor = ref_norm / tar_norm; // src/oc_icgn.cpp:260
			zncc = (f2 + fd) / (ref_norm * tar_norm); // == 0.5*(2 - znssd), src/oc_icgn.cpp:263,320
			float b[NP];
#pragma unroll
			for (int k = 0; k < NP; k++) b[k] = factor * (SF[k] + SD[k] - dbar * S[k]) - SF[k];
			bool accept = true;
			if constexpr (LM) {
				const float znssd = 2.f - 2.f * zncc;
				if (iteration == 1) lm_cur = powf(lm_lambda, znssd / znssd0) - 1.f; // src/oc_iclm.cpp:258-263
#pragma unroll
				for (int k = 0; k < NH; k++) H[k] = sH[k];
#pragma unroll
				for (int k = 0; k < NP; k++) H[k * (k + 1) / 2 + k] += lm_cur; // hessian + lambda * I, :266
				cholesky_packed<NP>(H);
				accept = znssd < znssd0; // :292-310
				if (accept) { lm_cur *= lm_alpha; znssd0 = znssd; }
				else lm_cur *= lm_beta;
			}
			cholesky_solve<NP>(H, b, dp);
			if constexpr (NP == 6) {
				// W <- W * W(dp)^-1, 3x3 affine (src/oc_icgn.cpp:290)
				const float a = dp[1], bb = dp[2], cc = dp[0], d = dp[4], e = dp[5], ff = dp[3];
				const float det = (1.f + a) * (1.f + e) - bb * d;
				const float id = 1.0f / det;
				const float i00 = (1.f + e) * id, i01 = -bb * id, i02 = (bb * ff - cc * (1.f + e)) * id;
				const float i10 = -d * id, i11 = (1.f + a) * id, i12 = (cc * d - (1.f + a) * ff) * id;
				const float n00 = A[0] * i00 + A[1] * i10, n01 = A[0] * i01 + A[1] * i11, n02 = A[0] * i02 + A[1] * i12 + A[2];
				const float n10 = A[3] * i00 + A[4] * i10, n11 = A[3] * i01 + A[4] * i11, n12 = A[3] * i02 + A[4] * i12 + A[5];
				if (accept) { A[0] = n00; A[1] = n01; A[2] = n02; A[3] = n10; A[4] = n11; A[5] = n12; }
				const float rx2 = (float)(rx * rx), ry2 = (float)(ry * ry);
				dp_norm = dp[0] * dp[0] + dp[1] * dp[1] * rx2 + dp[2] * dp[2] * ry2
					+ dp[3] * dp[3] + dp[4] * dp[4] * rx2 + dp[5] * dp[5] * ry2; // src/oc_icgn.cpp:296-306
			} else {
				if (accept) {
					float Mw[30];
					warp2d2_matrix(dp, Mw);
					right_divide_2x6(A, Mw); // rows 3,4 of W * W(dp)^-1 (src/oc_icgn.cpp:831)
				}
				const int rx2 = rx * rx, ry2 = ry * ry;
				const float rxy2 = (float)(rx2 * ry2);
				const float rx4 = (float)(int)((float)(rx2 * rx2) * 0.25f); // float->int truncation, src/oc_icgn.cpp:840-841
				const float ry4 = (float)(int)((float)(ry2 * ry2) * 0.25f);
				dp_norm = dp[0] * dp[0] + dp[1] * dp[1] * (float)rx2 + dp[2] * dp[2] * (float)ry2
					+ dp[3] * dp[3] * rx4 + dp[5] * dp[5] * ry4 + dp[4] * dp[4] * rxy2
					+ dp[6] * dp[6] + dp[7] * dp[7] * (float)rx2 + dp[8] * dp[8] * (float)ry2
					+ dp[9] * dp[9] * rx4 + dp[11] * dp[11] * ry4 + dp[10] * dp[10] * rxy2;
			}
			dp_norm = sqrtf(dp_norm);
		} while ((float)iteration < stop_condition && dp_norm >= conv_criterion);

		if (left_image) {
			if (poi_leader) P[P2_ZNCC] = -3.f;
			__syncwarp();
			continue;
		}
		// ---------------- results, src/oc_icgn.cpp:310-340 / :859-897 ----------------
		// Every lane holds the same final state; the record goes out as ONE coalesced store, lane k writing float k (fields the
		// reference leaves alone keep the value read at the start) -- the queue may live in page-locked host memory, where
		// separate 4-byte stores would each cross PCIe on their own.
		if (TM || threadIdx.x < 32) {
			float u, v;
			float out = rec;
			auto put = [&](int field, float value) { if (lane == field) out = value; };
			if constexpr (NP == 6) {
				u = A[2]; v = A[5];
				put(P2_DEF + D2_U, u); put(P2_DEF + D2_UX, A[0] - 1.f); put(P2_DEF + D2_UY, A[1]);
				put(P2_DEF + D2_V, v); put(P2_DEF + D2_VX, A[3]); put(P2_DEF + D2_VY, A[4] - 1.f);
			} else { // Deformation2D2::setDeformation(), src/oc_deformation.cpp:284-299
				u = A[5]; v = A[11];
				put(P2_DEF + D2_U, u); put(P2_DEF + D2_UX, A[3] - 1.f); put(P2_DEF + D2_UY, A[4]);
				put(P2_DEF + D2_UXX, A[0] * 2.f); put(P2_DEF + D2_UXY, A[1]); put(P2_DEF + D2_UYY, A[2] * 2.f);
				put(P2_DEF + D2_V, v); put(P2_DEF + D2_VX, A[9]); put(P2_DEF + D2_VY, A[10] - 1.f);
				put(P2_DEF + D2_VXX, A[6] * 2.f); put(P2_DEF + D2_VXY, A[7]); put(P2_DEF + D2_VYY, A[8] * 2.f);
			}
			put(P2_U0, u_in);
			put(P2_V0, v_in);
			float zout = zncc;
			put(P2_ITER, (float)iteration);
			put(P2_CONV, dp_norm);
			put(P2_RX, (float)rx);
			put(P2_RY, (float)ry);
			if (dp_norm >= conv_criterion && (float)iteration >= stop_condition) zout = -4.f;
			if (is_nan_f(zout) || is_nan_f(u) || is_nan_f(v)) {
				put(P2_DEF + D2_U, u_in);
				put(P2_DEF + D2_V, v_in);
				zout = -5.f;
			}
			put(P2_ZNCC, zout);
			if (lane < P2_N) P[lane] = out;
		}
		__syncwarp();
	}
	if constexpr (WPP == 1) {
		// The queue head resets itself: the last worker to leave zeroes it (and the departure count 8 ints further on), so a
		// launch needs no memset in front of it (2-3 us of an otherwise empty stream per launch).  The host zeroes both once.
		if (lane == 0) {
			const int workers = (int)gridDim.x * (TM ? ICGN2D_TM_WARPS : 1);
			__threadfence();
			if (atomicAdd(work_counter + 8, 1) == workers - 1) {
				work_counter[0] = 0;
				work_counter[8] = 0;
			}
		}
	}
	if constexpr (TM) { // every warp has drained the queue: release the CTA's Tensor-Memory columns
		tmem_fence_before_sync();
		__syncthreads();
		if (warp_in_cta == 0) tmem_dealloc<ICGN2D_TM_COLS>(s_tmem_base_value);
	}
}

// host-side launch ---------------------------------------------------------------------------
// Returns 0, -1 when one warp's slab does not fit in shared memory, -2 on a CUDA error.
// d_counter: a work-queue head owned by the context (64 ints; see ocb_create: [k] is zeroed per launch, [32 + k] and [40 + k] are
// the self-resetting head and departure count of the one-warp-per-POI kernels).
typedef void (*Icgn2dKernel)(Image2D, float*, int, int, int, float, float, int*, const CUtensorMap, const CUtensorMap, int, const float*, float, float, float);

// *rc: the compile-time subset radius of the instantiation picked (0: any radius)
template <int WPP>
static Icgn2dKernel icgn2d_pick(int np, int rx, int ry, bool lm, int* rc) {
	*rc = 0;
	if (lm) return (np == 6) ? icgn2d_kernel<6, 0, true, WPP> : icgn2d_kernel<12, 0, true, WPP>;
	if (np == 6) {
		if (rx == 16 && ry == 16) { *rc = 16; return icgn2d_kernel<6, 16, false, WPP>; }
		return icgn2d_kernel<6, 0, false, WPP>;
	}
	if (rx == 20 && ry == 20) { *rc = 20; return icgn2d_kernel<12, 20, false, WPP>; }
	return icgn2d_kernel<12, 0, false, WPP>;
}

size_t icgn2d_slab_bytes(int rx, int ry) { return (size_t)icgn2d_slab_floats(rx, ry, false, 1) * sizeof(float); }

int icgn2d_launch(int np, const Image2D& img, float* d_pois, size_t n, int rx, int ry, float conv, float stop, int sm_count,
	size_t smem_optin, int* d_counter, const float* d_center_offsets, const float* lm_damping, cudaStream_t stream, cudaError_t* err,
	LaunchInfo* info) {
	const bool lm = lm_damping != nullptr;
	// Warps per POI.  Measured on B200 (tools/ab_icgn2d.sh): with the GPU full, one warp per POI wins (config B 0.853 vs
	// 0.906 ms, C 2.22 vs 2.43 ms, E 8.38 vs 8.87 ms) -- the second warp doubles the resident warps but also the per-POI
	// fixed work and adds a barrier per pass; with fewer POIs than resident slots, two warps per POI shorten the tail
	// (config A, 200 POIs: 24.6 vs 32.5 us).  So: 2 only when the queue cannot fill the machine.
	auto slots = [&](int wpp_) {
		const size_t b = (size_t)icgn2d_slab_floats(rx, ry, lm, wpp_) * sizeof(float);
		if (b > smem_optin) return 0;
		int k = (int)((228 * 1024) / (b + 1024));
		return k > 32 ? 32 : k;
	};
	int wpp = ((long long)n < (long long)sm_count * slots(1) && (2 * ry + 1) >= 8 && slots(2) > 0) ? 2 : 1;
	if (const char* e = getenv("OCB_ICGN2D_WPP")) { // tuning knob
		const int v = atoi(e);
		if (v == 1 || (v == 2 && slots(2) > 0)) wpp = v;
	}
	size_t smem = (size_t)icgn2d_slab_floats(rx, ry, lm, wpp) * sizeof(float);
	if (smem > smem_optin) return -1;
	// Tensor-Memory variant: when the queue fills the machine, the subset is >= 32 columns wide and <= 42 rows high (3 TMEM columns
	// per row, 128 per CTA).  OCB_ICGN2D_TMEM=0 switches it off (A/B runs).
	const char* tm_env = getenv("OCB_ICGN2D_TMEM");
	// (and four such CTAs must fit the SM's shared memory, or the point of the variant -- 16 resident warps -- is lost)
	const size_t tm_cta_smem = (size_t)ICGN2D_TM_WARPS * icgn2d_tm_slab_floats(rx, ry) * sizeof(float);
	const bool use_tm = !lm && np == 6 && wpp == 1 && icgn2d_tm_supported(rx, ry) && !(tm_env && atoi(tm_env) == 0)
		&& (long long)n >= (long long)sm_count * ICGN2D_TM_WARPS * 4 && ICGN2D_PAIRS && tm_cta_smem <= smem_optin
		&& 4 * (tm_cta_smem + 1024) <= (size_t)(228 * 1024);
	int blocks_per_sm = slots(wpp);
	if (blocks_per_sm < 1) blocks_per_sm = 1;
	if (const char* cap = getenv("OCB_ICGN2D_MAX_WARPS")) { // tuning knob: cap the resident warps per SM
		const int c = atoi(cap) / wpp;
		if (c >= 1 && c < blocks_per_sm) blocks_per_sm = c;
	}
	CUtensorMap tm_ref, tm_tar;
	memset(&tm_ref, 0, sizeof(tm_ref));
	memset(&tm_tar, 0, sizeof(tm_tar));
	const int dims[2] = { img.w, img.h };
	const int box_ref[2] = { icgn2d_ref_w(rx), icgn2d_ref_h(ry) }, box_tar[2] = { icgn2d_tar_w(rx), icgn2d_tar_h(ry) };
	const int use_tma = !getenv("OCB_NO_TMA") && tma_make_map(&tm_ref, img.ref, 2, dims, box_ref) && tma_make_map(&tm_tar, img.tar, 2, dims, box_tar);
	int rc = 0;
	Icgn2dKernel kern = wpp == 2 ? icgn2d_pick<2>(np, rx, ry, lm, &rc) : icgn2d_pick<1>(np, rx, ry, lm, &rc);
	int threads = wpp * 32;
	if (use_tm) {
		// (6-parameter kernels only: the 12-parameter ones need ~250 registers, which already limits them to 8 warps per SM)
		rc = (rx == 16 && ry == 16) ? 16 : 0;
		kern = rc == 16 ? icgn2d_kernel<6, 16, false, 1, true> : icgn2d_kernel<6, 0, false, 1, true>;
		smem = tm_cta_smem;
		threads = ICGN2D_TM_WARPS * 32;
		blocks_per_sm = 512 / ICGN2D_TM_COLS; // Tensor Memory: 512 columns per SM
	}
	*err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (*err != cudaSuccess) return -2;
	if (wpp != 1) {
		*err = cudaMemsetAsync(d_counter, 0, sizeof(int), stream);
		if (*err != cudaSuccess) return -2;
	} else {
		d_counter += 32; // the one-warp-per-POI kernels reset their queue head themselves: a set of heads nobody else touches
	}
	long long resident = (long long)sm_count * blocks_per_sm;
	if (use_tm && (long long)n < resident * ICGN2D_TM_WARPS) resident = ((long long)n + ICGN2D_TM_WARPS - 1) / ICGN2D_TM_WARPS;
	int grid = (int)((long long)n < resident ? (long long)n : resident); // persistent: one wave, one POI per CTA (TM: per warp) at a time
	if (grid < 1) grid = 1;
	if (info) {
		info->op = "icgn2d";
		info->np = np; info->rc = rc; info->lm = lm; info->wpp = wpp; info->tm = use_tm; info->tma = use_tma;
		info->grid = grid; info->threads = threads;
	}
	kern<<<grid, threads, smem, stream>>>(img, d_pois, (int)n, rx, ry, conv, stop, d_counter, tm_ref, tm_tar, use_tma, d_center_offsets,
		lm ? lm_damping[0] : 0.f, lm ? lm_damping[1] : 0.f, lm ? lm_damping[2] : 0.f);
	*err = cudaGetLastError();
	return *err == cudaSuccess ? 0 : -2;
}

} // namespace ocb
