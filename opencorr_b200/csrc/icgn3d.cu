// icgn3d.cu -- DVC: ICGN3D1 (first-order shape function, 12 parameters) and the device-side
// ICGN3D1::prepare() products, for sm_100a.
//
// Replaces ICGN3D1::compute(POI3D*) (reference src/oc_icgn.cpp:1270-1490), Gradient3D4
// (src/oc_gradient.cpp:143-231) and TricubicBspline::prepare/compute
// (src/oc_cubic_bspline.cpp:214-405).
//
// Round-2 structure in one paragraph: the setup pass runs with lanes along x and accumulates FACTORED Hessian sums
// (ICGN3D_FACTORED_SETUP); when a whole z-slab of samples lies inside the staged tile (one warp-uniform corner test) every lane
// takes TWO y-adjacent samples per step, their 4x4x4 blocks fetched as one 4x5x4 block and evaluated in packed f32x2
// arithmetic (ICGN3D_PAIRS); the `any sample < 0` rejection is re-decided in the reference's own arithmetic when the smallest
// sample is borderline (icgn3d_exact_negative).  What follows describes the common skeleton.
//
// Mapping: ONE CTA (256 threads) PER POI, persistent CTAs pulling POIs from an atomic counter; the
// (2r+1)^3 samples are strided over the CTA with x fastest, so the reference-volume reads (value + 3
// gradient volumes) are coalesced.  The 64-tap tricubic evaluation reads a B-spline coefficient TILE
// staged in shared memory by TMA.  A (2r+8)^3 tile does not fit next to a second CTA, so the subset
// is processed in z-SLABS: per iteration and slab, one 3D TMA box (x origin 16-byte aligned, centred
// on the CURRENT warp) lands in smem, all samples of the slab are evaluated from it, the next slab
// replaces it; two CTAs per SM overlap one CTA's load with the other's math.  Samples whose support
// leaves the tile (large deformation gradients) read the coefficient volume through L1/L2 instead.
// Per-iteration single-pass sums as in icgn2d.cu; the 12x12 Cholesky factor and the running 3x4
// warp live in shared memory and are updated by one thread between two barriers.
#include <stdlib.h>
#include <string.h>

#include "ocb_kernels.h"
#include "ocb_f32x2.cuh"
#include "ocb_tma.cuh"

namespace ocb {

constexpr int ICGN3D_MAX_WARPS = 16; // CTAs run 8 warps (two CTAs per SM) or, when only one slab-carrying CTA fits, 16

// ---- ICGN3D1::prepareRef: Gradient3D4::getGradientX/Y/Z, src/oc_gradient.cpp:143-231 ----------
// Output is packed {ref, gx, gy, gz} per voxel so that IC-GN fetches a sample's constants with one 16-byte load.
__global__ void gradient3d_kernel(const float* __restrict__ f, float4* __restrict__ rg, int dx, int dy, int dz) {
	const size_t total = (size_t)dx * dy * dz;
	const size_t sy = (size_t)dx, sz = (size_t)dx * dy;
	for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
		const int k = (int)(i % dx), j = (int)((i / dx) % dy), ii = (int)(i / sz);
		float vx = 0.f, vy = 0.f, vz = 0.f; // borders stay zero (calloc in new3D, src/oc_array.h:60)
		if (k >= 2 && k < dx - 2) vx = grad4(f[i - 2], f[i - 1], f[i + 1], f[i + 2]);
		if (j >= 2 && j < dy - 2) vy = grad4(f[i - 2 * sy], f[i - sy], f[i + sy], f[i + 2 * sy]);
		if (ii >= 2 && ii < dz - 2) vz = grad4(f[i - 2 * sz], f[i - sz], f[i + sz], f[i + 2 * sz]);
		rg[i] = make_float4(f[i], vx, vy, vz);
	}
}

// ---- ICGN3D1::prepareTar: one 15-tap FIR pass of TricubicBspline::prepare -----------------------
// (src/oc_cubic_bspline.cpp:224-348; taps src/oc_cubic_bspline.h:80-90).  The reference's interior
// and edge branches are the same expression with the indices clamped to [0, dim-1]; the operation
// order b0*x + b1*(..) + b2*(..) ... is kept and evaluated without FMA so the coefficient volume
// is bit-identical to the CPU result.
__constant__ float c_prefilter[8] = { 1.732176555412860f, -0.464135309171000f, 0.124364681271139f, -0.033323415913556f,
	0.008928982383084f, -0.002392513618779f, 0.000641072092032f, -0.000171774749350f };

__global__ void prefilter3d_kernel(const float* __restrict__ in, float* __restrict__ out, int dx, int dy, int dz, int axis) {
	const size_t total = (size_t)dx * dy * dz;
	const size_t sy = (size_t)dx, sz = (size_t)dx * dy;
	const size_t stride = axis == 0 ? 1 : (axis == 1 ? sy : sz);
	const int dim = axis == 0 ? dx : (axis == 1 ? dy : dz);
	for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
		const int k = (int)(i % dx), j = (int)((i / dx) % dy), ii = (int)(i / sz);
		const int pos = axis == 0 ? k : (axis == 1 ? j : ii);
		const float* line = in + (i - (size_t)pos * stride);
		float v = __fmul_rn(c_prefilter[0], line[(size_t)pos * stride]);
#pragma unroll
		for (int t = 1; t <= 7; t++) {
			const int lo = pos - t < 0 ? 0 : pos - t;
			const int hi = pos + t > dim - 1 ? dim - 1 : pos + t;
			v = __fadd_rn(v, __fmul_rn(c_prefilter[t], __fadd_rn(line[(size_t)lo * stride], line[(size_t)hi * stride])));
		}
		out[i] = v;
	}
}

void gradient3d_launch(const float* ref, float4* rg, int dx, int dy, int dz, int sm_count, cudaStream_t s) {
	gradient3d_kernel<<<sm_count * 8, 256, 0, s>>>(ref, rg, dx, dy, dz);
}
void prefilter3d_launch(const float* in, float* out, int dx, int dy, int dz, int axis, int sm_count, cudaStream_t s) {
	prefilter3d_kernel<<<sm_count * 8, 256, 0, s>>>(in, out, dx, dy, dz, axis);
}

// ---- ICGN3D1::compute ---------------------------------------------------------------------------
constexpr int NP3 = 12;
constexpr int NH3 = NP3 * (NP3 + 1) / 2; // 78
constexpr int NSETUP = NH3 + 2 * NP3 + 2; // Hessian + S + SR + r1 + r2 = 104
constexpr int NITER = 3 + NP3;            // d1, d2, rd, SD[12]
constexpr int ICGN3D_TILE_MARGIN = 1;

struct Icgn3dShared {
	float part[ICGN3D_MAX_WARPS][NSETUP]; // per-warp partial sums
	float tot[NSETUP];
	float L[NH3];   // packed Cholesky factor (diag = 1/L_ii)
	float S[NP3], SF[NP3];
	float A[12];    // running warp rows: [1+ux uy uz u | vx 1+vy vz v | wx wy 1+wz w]
	float f2, rbar, c0;
	float dp_norm, zncc;
	int keep_going;
	int poi;
};

// floor(x / d) for 0 <= x < 2^21, d >= 1 (inv = 1.0f / d); see fftcc.cu
__device__ __forceinline__ int fdiv3(int x, float inv) { return __float2int_rz(((float)x + 0.5f) * inv); }

// Cubic B-spline basis (src/oc_cubic_bspline.cpp:35-53), 12 operations: b0 = (1-t)^3/6, b3 = t^3/6,
// b1 = 2/3 - t^2 (1 - t/2), b2 = 1 - b0 - b1 - b3 (partition of unity)
__device__ __forceinline__ void bspline_basis_fast(float t, float* b) {
	const float om = 1.f - t, t2 = t * t;
	b[0] = om * om * om * (1.f / 6.f);
	b[3] = t2 * t * (1.f / 6.f);
	b[1] = fmaf(t2, fmaf(0.5f, t, -1.f), 2.f / 3.f);
	b[2] = ((1.f - b[0]) - b[1]) - b[3];
}

// 64-tap evaluation (src/oc_cubic_bspline.cpp:390-401) from a dense array with pitches (py_, pz_) floats
template <bool GLOBAL>
__device__ __forceinline__ float tricubic_taps(const float* __restrict__ base, int py_, int pz_, const float* bx, const float* by, const float* bz) {
	float value = 0.f;
#pragma unroll
	for (int i = 0; i < 4; i++) {
		float sy_acc = 0.f;
#pragma unroll
		for (int j = 0; j < 4; j++) {
			const float* row = base + i * pz_ + j * py_;
			float sx_acc;
			if (GLOBAL) {
				sx_acc = __ldg(row) * bx[0];
				sx_acc = fmaf(__ldg(row + 1), bx[1], sx_acc);
				sx_acc = fmaf(__ldg(row + 2), bx[2], sx_acc);
				sx_acc = fmaf(__ldg(row + 3), bx[3], sx_acc);
			} else {
				sx_acc = row[0] * bx[0];
				sx_acc = fmaf(row[1], bx[1], sx_acc);
				sx_acc = fmaf(row[2], bx[2], sx_acc);
				sx_acc = fmaf(row[3], bx[3], sx_acc);
			}
			sy_acc = fmaf(sx_acc, by[j], sy_acc);
		}
		value = fmaf(sy_acc, bz[i], value);
	}
	return value;
}

// ---- the reference's `any interpolated sample < 0 -> zncc = -3` rule (src/oc_icgn.cpp:1378-1390) ------------------------
// Same scheme as icgn2d.cu: the sampling loop tracks min(t); a decisively negative (< -TRIGGER) or positive (>= TRIGGER)
// minimum decides at once, anything in between is re-decided here in the reference's own arithmetic -- Deformation3D1::warp
// with separately rounded products (src/oc_deformation.cpp:518-530), TricubicBspline::compute with its basis polynomials
// and its sum order (src/oc_cubic_bspline.cpp:35-53,353-405), no FMA anywhere.
constexpr float ICGN3D_NEG_TRIGGER = 0.125f;
constexpr float ICGN3D_NEG_BAND = 4e-3f;

__device__ __forceinline__ void bspline_basis_reference_order(float t, float* b) {
	const float s = 1.f / 6.f;
	b[0] = __fmul_rn(s, __fadd_rn(__fmul_rn(t, __fsub_rn(__fmul_rn(t, __fadd_rn(-t, 3.f)), 3.f)), 1.f));
	b[1] = __fmul_rn(s, __fadd_rn(__fmul_rn(__fmul_rn(t, t), __fsub_rn(__fmul_rn(3.f, t), 6.f)), 4.f));
	b[2] = __fmul_rn(s, __fadd_rn(__fmul_rn(t, __fadd_rn(__fmul_rn(t, __fadd_rn(__fmul_rn(-3.f, t), 3.f)), 3.f)), 1.f));
	b[3] = __fmul_rn(s, __fmul_rn(__fmul_rn(t, t), t));
}

// Does any of the samples i = first, first + stride, ... < N of the warp A (rows [1+ux uy uz u | vx 1+vy vz v | wx wy 1+wz w])
// come out negative in the reference's arithmetic?  Reads the coefficient volume directly (rare path).
__device__ __noinline__ bool icgn3d_exact_negative(const float* A, float px, float py, float pz, int rx, int ry, int rz,
	const float* __restrict__ coef, int dx, int dy, int dz, int first, int stride) {
	const int sx = 2 * rx + 1, sy = 2 * ry + 1, sz = 2 * rz + 1, slice = sx * sy, N = slice * sz;
	bool negative = false;
	for (int i = first; i < N; i += stride) {
		const int ii = i / slice, r2 = i - ii * slice, j = r2 / sx, k = r2 - j * sx;
		const float xl = (float)(k - rx), yl = (float)(j - ry), zl = (float)(ii - rz);
		const float wx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A[0], xl), __fmul_rn(A[1], yl)), __fmul_rn(A[2], zl)), A[3]);
		const float wy = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A[4], xl), __fmul_rn(A[5], yl)), __fmul_rn(A[6], zl)), A[7]);
		const float wz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(A[8], xl), __fmul_rn(A[9], yl)), __fmul_rn(A[10], zl)), A[11]);
		const float X = __fadd_rn(px, wx), Y = __fadd_rn(py, wy), Z = __fadd_rn(pz, wz); // center + warped, src/oc_icgn.cpp:1376
		if (!((X >= 1.f) && (Y >= 1.f) && (Z >= 1.f) && (X < (float)(dx - 2)) && (Y < (float)(dy - 2)) && (Z < (float)(dz - 2)))) {
			negative = true; // TricubicBspline::compute returns -1
			continue;
		}
		const float xf = floorf(X), yf = floorf(Y), zf = floorf(Z);
		const float xd = __fsub_rn(X, xf), yd = __fsub_rn(Y, yf), zd = __fsub_rn(Z, zf);
		const float* base = coef + ((size_t)((int)zf - 1) * dy + ((int)yf - 1)) * dx + ((int)xf - 1);
		float bx[4], by[4], bz[4];
		bspline_basis_fast(xd, bx);
		bspline_basis_fast(yd, by);
		bspline_basis_fast(zd, bz);
		const float t = tricubic_taps<true>(base, dx, dx * dy, bx, by, bz);
		if (t >= ICGN3D_NEG_BAND) continue;
		if (t <= -ICGN3D_NEG_BAND) {
			negative = true;
			continue;
		}
		bspline_basis_reference_order(xd, bx);
		bspline_basis_reference_order(yd, by);
		bspline_basis_reference_order(zd, bz);
		float sum_y[4];
#pragma unroll 1
		for (int a = 0; a < 4; a++) {
			float sum_x[4];
#pragma unroll
			for (int b = 0; b < 4; b++) {
				const float* row = base + (size_t)a * dx * dy + (size_t)b * dx;
				sum_x[b] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(bx[0], __ldg(row)), __fmul_rn(bx[1], __ldg(row + 1))), __fmul_rn(bx[2], __ldg(row + 2))),
					__fmul_rn(bx[3], __ldg(row + 3)));
			}
			sum_y[a] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(by[0], sum_x[0]), __fmul_rn(by[1], sum_x[1])), __fmul_rn(by[2], sum_x[2])), __fmul_rn(by[3], sum_x[3]));
		}
		const float value = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(bz[0], sum_y[0]), __fmul_rn(bz[1], sum_y[1])), __fmul_rn(bz[2], sum_y[2])), __fmul_rn(bz[3], sum_y[3]));
		if (value < 0.f) negative = true;
	}
	return negative;
}

#ifndef ICGN3D_FACTORED_SETUP
#define ICGN3D_FACTORED_SETUP 1 // setup pass with lanes along x and factored Hessian sums (0: the round-1 loop, for A/B runs)
#endif
#ifndef ICGN3D_PAIRS
// 1: when a whole z-slab of samples has its support inside the staged tile (the normal case: one warp-uniform corner test
// per slab replaces the per-sample range tests), every lane takes TWO y-adjacent samples per step.  Their 4x4x4 blocks
// overlap in three of four block rows, so the pair is evaluated from ONE 4x5x4 block (80 LDS instead of 128 -- the kernel
// was bound by the shared-memory pipe at 64 LDS per sample), and the arithmetic of the two samples runs in packed f32x2
// pairs (FFMA2), rows (j, j+1) in lanes {.x, .y}: 104 instead of 168 issue slots for the taps, the same operations in the
// same order as the one-sample path (the results are bit-identical).  0: one sample per step (round-1 loop), for A/B runs.
#define ICGN3D_PAIRS 1
#endif

// packed cubic B-spline basis: bspline_basis_fast on two arguments at once
__device__ __forceinline__ void bspline_basis_fast2(float2 t, float2* b) {
	const float2 om = fsub2(bcast2(1.f), t), t2 = fmul2(t, t);
	b[0] = fmul2(fmul2(fmul2(om, om), om), bcast2(1.f / 6.f));
	b[3] = fmul2(fmul2(t2, t), bcast2(1.f / 6.f));
	b[1] = ffma2(t2, ffma2(bcast2(0.5f), t, bcast2(-1.f)), bcast2(2.f / 3.f));
	b[2] = fsub2(fsub2(fsub2(bcast2(1.f), b[0]), b[1]), b[3]);
}

__host__ __device__ inline int icgn3d_tile_x(int rx) { return round_up4(2 * rx + 1 + 3 + 2 * ICGN3D_TILE_MARGIN + 3); }
__host__ __device__ inline int icgn3d_tile_y(int ry) { return 2 * ry + 1 + 3 + 2 * ICGN3D_TILE_MARGIN; }
__host__ __device__ inline int icgn3d_tile_z(int slab_k) { return slab_k + 3 + 2 * ICGN3D_TILE_MARGIN; }

// RC > 0: radius known at compile time (rx == ry == rz == RC): tile pitches become immediates.
// THREADS: 256 (two CTAs per SM) or 512 (large radii: the slab leaves room for one CTA only, which then brings 16 warps)
template <int RC, int THREADS>
__global__ void __launch_bounds__(THREADS, 512 / THREADS) icgn3d1_kernel(Image3D img, float* __restrict__ pois, int n_poi, int rx_arg, int ry_arg, int rz_arg,
	float conv_criterion, float stop_condition, int slab_k, int* __restrict__ work_counter, const __grid_constant__ CUtensorMap tm_coef, int use_tma) {
	constexpr int ICGN3D_THREADS = THREADS, ICGN3D_WARPS = THREADS / 32;
	extern __shared__ __align__(128) float dsmem[];
	__shared__ Icgn3dShared sh;
	uint64_t* bar = (uint64_t*)dsmem;
	float* T = dsmem + 32;
	const int rx = RC ? RC : rx_arg, ry = RC ? RC : ry_arg, rz = RC ? RC : rz_arg;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int sx = 2 * rx + 1, sy = 2 * ry + 1, sz = 2 * rz + 1;
	const int slice = sx * sy, N = slice * sz;
	const int dx = img.dx, dy = img.dy, dz = img.dz;
	const int TX = icgn3d_tile_x(rx), TY = icgn3d_tile_y(ry), TZ = icgn3d_tile_z(slab_k);
	const int TXY = TX * TY;
	const float inv_n = 1.0f / (float)N, inv_slice = 1.0f / (float)slice, inv_sx = 1.0f / (float)sx, inv_sy = 1.0f / (float)sy;
	const int ncol = sx < 32 ? sx : 32, rem = sx - ncol;
	const float inv_rem = rem > 0 ? 1.0f / (float)rem : 1.f;
	const float* __restrict__ coef = img.coef;
	uint32_t bar_phase = 0;
	if (tid == 0 && use_tma) mbar_init(bar, 1);
	__syncthreads();

	while (true) {
		if (tid == 0) sh.poi = atomicAdd(work_counter, 1);
		__syncthreads();
		const int poi = sh.poi;
		if (poi >= n_poi) break;
		float* P = pois + (size_t)poi * P3_N;
		const float px = P[P3_X], py = P[P3_Y], pz = P[P3_Z];
		const float u_in = P[P3_DEF + 0], v_in = P[P3_DEF + 4], w_in = P[P3_DEF + 8];
		const float zncc_in = P[P3_ZNCC];
		__syncthreads(); // everyone has read the record (and sh.poi) before thread 0 may overwrite them
		// guard, src/oc_icgn.cpp:1279-1286
		if ((px - rx) < 0 || (py - ry) < 0 || (pz - rz) < 0 || (px + rx) > (dx - 1) || (py + ry) > (dy - 1) || (pz + rz) > (dz - 1)
			|| fabsf(u_in) >= dx || fabsf(v_in) >= dy || fabsf(w_in) >= dz || zncc_in < 0
			|| is_nan_f(u_in) || is_nan_f(v_in) || is_nan_f(w_in) || is_nan_f(px) || is_nan_f(py) || is_nan_f(pz)) {
			if (tid == 0) P[P3_ZNCC] = zncc_in >= 0 ? -3.f : zncc_in;
			continue;
		}
		const int x0 = (int)px - rx, y0 = (int)py - ry, z0 = (int)pz - rz;
		const size_t goff = ((size_t)z0 * dy + y0) * dx + x0;
		const float c0 = __ldg(img.ref + ((size_t)(int)pz * dy + (int)py) * dx + (int)px); // pilot value: centre voxel

		// ---- reference subset statistics + steepest-descent images + Hessian (src/oc_icgn.cpp:1291-1337)
		{
			float acc[NSETUP];
#pragma unroll
			for (int k = 0; k < NSETUP; k++) acc[k] = 0.f;
			// One sample's contribution, everything spelled out: 12 steepest-descent values, 78 Hessian products (tail column, and
			// the whole subset when ICGN3D_FACTORED_SETUP is 0)
			auto setup_sample = [&](const float4& c4, float xl, float yl, float zl) {
				const float R = c4.x - c0;
				const float gx = c4.y, gy = c4.z, gz = c4.w;
				float sd[NP3];
				sd[0] = gx; sd[1] = gx * xl; sd[2] = gx * yl; sd[3] = gx * zl;
				sd[4] = gy; sd[5] = gy * xl; sd[6] = gy * yl; sd[7] = gy * zl;
				sd[8] = gz; sd[9] = gz * xl; sd[10] = gz * yl; sd[11] = gz * zl;
#pragma unroll
				for (int a = 0; a < NP3; a++) {
					acc[NH3 + a] += sd[a];
					acc[NH3 + NP3 + a] = fmaf(sd[a], R, acc[NH3 + NP3 + a]);
#pragma unroll
					for (int b = 0; b <= a; b++) acc[a * (a + 1) / 2 + b] = fmaf(sd[a], sd[b], acc[a * (a + 1) / 2 + b]);
				}
				acc[NSETUP - 2] += R;
				acc[NSETUP - 1] = fmaf(R, R, acc[NSETUP - 1]);
			};
#if ICGN3D_FACTORED_SETUP
			// Lanes along x (lane = subset column, like the sampling loops), warps over the (y, z) rows: x is a per-lane constant, y and z
			// are warp-uniform, so a lane accumulates the FACTORED sums  sum g_a g_b {1, y, z, y^2, yz, z^2}  (36 instead of 78 Hessian
			// products per sample),  sum g_a {1, y, z}  and  sum g_a R {1, y, z},  and applies its powers of x once at the end.  The row's
			// constants (one coalesced 512-byte request per warp) are requested one row ahead: nothing of this is in L1.
			{
				float aH[6][6], aS[3][3], aR[3][3], r1 = 0.f, r2 = 0.f;
#pragma unroll
				for (int a = 0; a < 6; a++)
#pragma unroll
					for (int q = 0; q < 6; q++) aH[a][q] = 0.f;
#pragma unroll
				for (int a = 0; a < 3; a++)
#pragma unroll
					for (int q = 0; q < 3; q++) { aS[a][q] = 0.f; aR[a][q] = 0.f; }
				const int nrows_all = sy * sz;
				const bool col_on = lane < ncol;
				auto row_offset = [&](int row) {
					const int ii = fdiv3(row, inv_sy), j = row - ii * sy;
					return goff + ((size_t)ii * dy + j) * dx + lane;
				};
				float4 c_next = make_float4(0.f, 0.f, 0.f, 0.f);
				if (warp < nrows_all && col_on) c_next = __ldg(img.rg + row_offset(warp));
				for (int row = warp; row < nrows_all; row += ICGN3D_WARPS) {
					const int ii = fdiv3(row, inv_sy), j = row - ii * sy;
					const float4 c4 = c_next;
					if (row + ICGN3D_WARPS < nrows_all && col_on) c_next = __ldg(img.rg + row_offset(row + ICGN3D_WARPS));
					if (col_on) {
						const float yl = (float)(j - ry), zl = (float)(ii - rz);
						const float m[6] = { 1.f, yl, zl, yl * yl, yl * zl, zl * zl };
						const float R = c4.x - c0;
						const float g[3] = { c4.y, c4.z, c4.w };
						const float p[6] = { g[0] * g[0], g[0] * g[1], g[0] * g[2], g[1] * g[1], g[1] * g[2], g[2] * g[2] };
#pragma unroll
						for (int a = 0; a < 6; a++) {
							aH[a][0] += p[a];
#pragma unroll
							for (int q = 1; q < 6; q++) aH[a][q] = fmaf(p[a], m[q], aH[a][q]);
						}
#pragma unroll
						for (int a = 0; a < 3; a++) {
							const float gr = g[a] * R;
							aS[a][0] += g[a];
							aS[a][1] = fmaf(g[a], yl, aS[a][1]);
							aS[a][2] = fmaf(g[a], zl, aS[a][2]);
							aR[a][0] += gr;
							aR[a][1] = fmaf(gr, yl, aR[a][1]);
							aR[a][2] = fmaf(gr, zl, aR[a][2]);
						}
						r1 += R;
						r2 = fmaf(R, R, r2);
					}
				}
				// expand with this lane's powers of x: sd index 4a + i, phi = [1, x, y, z]; phi_i phi_j = x^px * (a monomial of y, z)
				const float xl = (float)(lane - rx), xp[3] = { 1.f, xl, xl * xl };
#pragma unroll
				for (int a = 0; a < 3; a++)
#pragma unroll
					for (int i = 0; i < 4; i++) {
						const int k = 4 * a + i;
						const int pxi = i == 1 ? 1 : 0, qi = i == 2 ? 1 : (i == 3 ? 2 : 0); // x power and {1,y,z} index of phi_i
						acc[NH3 + k] = xp[pxi] * aS[a][qi];
						acc[NH3 + NP3 + k] = xp[pxi] * aR[a][qi];
#pragma unroll
						for (int b = 0; b < 3; b++)
#pragma unroll
							for (int jj = 0; jj < 4; jj++) {
								const int l = 4 * b + jj;
								if (l > k) continue;
								const int pxj = jj == 1 ? 1 : 0, qj = jj == 2 ? 1 : (jj == 3 ? 2 : 0);
								// monomial of (y, z) in phi_i phi_j: index into {1, y, z, yy, yz, zz}
								const int ny = (qi == 1) + (qj == 1), nz_ = (qi == 2) + (qj == 2);
								const int mq = ny == 0 ? (nz_ == 0 ? 0 : (nz_ == 1 ? 2 : 5)) : (ny == 1 ? (nz_ == 0 ? 1 : 4) : 3);
								const int pa = a <= b ? a : b, pb = a <= b ? b : a;                 // symmetric gradient pair (pa <= pb)
								const int pidx = pa == 0 ? pb : (pa == 1 ? 2 + pb : 5);             // xx xy xz yy yz zz
								acc[k * (k + 1) / 2 + l] = xp[pxi + pxj] * aH[pidx][mq];
							}
					}
				acc[NSETUP - 2] = r1;
				acc[NSETUP - 1] = r2;
				if (!col_on) {
#pragma unroll
					for (int k = 0; k < NSETUP; k++) acc[k] = 0.f;
				}
				// columns >= 32: a short tail, spelled-out sums
				for (int i = tid; i < nrows_all * rem; i += ICGN3D_THREADS) {
					const int row = fdiv3(i, inv_rem), k = 32 + (i - row * rem);
					const int ii = fdiv3(row, inv_sy), j = row - ii * sy;
					setup_sample(__ldg(img.rg + (goff + ((size_t)ii * dy + j) * dx + k)), (float)(k - rx), (float)(j - ry), (float)(ii - rz));
				}
			}
#else
			auto sample_offset = [&](int i) {
				const int ii = fdiv3(i, inv_slice), rem = i - ii * slice, j = fdiv3(rem, inv_sx), k = rem - j * sx;
				return goff + ((size_t)ii * dy + j) * dx + k;
			};
			float4 c_next = make_float4(0.f, 0.f, 0.f, 0.f);
			if (tid < N) c_next = __ldg(img.rg + sample_offset(tid));
			for (int i = tid; i < N; i += ICGN3D_THREADS) {
				const int ii = fdiv3(i, inv_slice), rem = i - ii * slice, j = fdiv3(rem, inv_sx), k = rem - j * sx;
				const float4 c4 = c_next;
				if (i + ICGN3D_THREADS < N) c_next = __ldg(img.rg + sample_offset(i + ICGN3D_THREADS));
				setup_sample(c4, (float)(k - rx), (float)(j - ry), (float)(ii - rz));
			}
#endif
#pragma unroll
			for (int k = 0; k < NSETUP; k++) {
				float v = warp_sum(acc[k]);
				if (lane == 0) sh.part[warp][k] = v;
			}
		}
		__syncthreads();
		if (tid < NSETUP) {
			float t = 0.f;
			for (int i = 0; i < ICGN3D_WARPS; i++) t += sh.part[i][tid];
			sh.tot[tid] = t;
		}
		__syncthreads();
		if (tid == 0) {
			float Hh[NH3];
#pragma unroll
			for (int k = 0; k < NH3; k++) Hh[k] = sh.tot[k];
			cholesky_packed<NP3>(Hh);
#pragma unroll
			for (int k = 0; k < NH3; k++) sh.L[k] = Hh[k];
			const float r1 = sh.tot[NSETUP - 2], r2 = sh.tot[NSETUP - 1];
			const float rbar = r1 * inv_n; // mean(R) - c0  (Subset3D::zeroMeanNorm, src/oc_subset.cpp:104-132)
			sh.rbar = rbar;
			sh.f2 = r2 - r1 * rbar;
			sh.c0 = c0;
			for (int k = 0; k < NP3; k++) {
				sh.S[k] = sh.tot[NH3 + k];
				sh.SF[k] = sh.tot[NH3 + NP3 + k] - rbar * sh.tot[NH3 + k]; // sum sd_k f = sum sd_k R' - rbar sum sd_k
			}
			// initial warp (Deformation3D1::setWarp, src/oc_deformation.cpp:495-516)
			sh.A[0] = 1.f + P[P3_DEF + 1]; sh.A[1] = P[P3_DEF + 2]; sh.A[2] = P[P3_DEF + 3]; sh.A[3] = u_in;
			sh.A[4] = P[P3_DEF + 5]; sh.A[5] = 1.f + P[P3_DEF + 6]; sh.A[6] = P[P3_DEF + 7]; sh.A[7] = v_in;
			sh.A[8] = P[P3_DEF + 9]; sh.A[9] = P[P3_DEF + 10]; sh.A[10] = 1.f + P[P3_DEF + 11]; sh.A[11] = w_in;
		}
		__syncthreads();

		// ---- IC-GN iterations (src/oc_icgn.cpp:1355-1447)
		const float xmax = (float)(dx - 2), ymax = (float)(dy - 2), zmax = (float)(dz - 2);
		int iteration = 0;
		bool left_image = false;
		while (true) {
			iteration++;
			float A[12];
#pragma unroll
			for (int k = 0; k < 12; k++) A[k] = sh.A[k];
			float acc[NITER];
#pragma unroll
			for (int k = 0; k < NITER; k++) acc[k] = 0.f;
			int invalid = 0;
			float tmin = 3.0e38f; // smallest interpolated sample of this pass (see icgn3d_exact_negative)
			// tile origin in x, y follows the CURRENT translation; x is 16-byte aligned for TMA
			const int tx0 = floor4((int)floorf(px + A[3]) - rx - 1 - ICGN3D_TILE_MARGIN);
			const int ty0 = (int)floorf(py + A[7]) - ry - 1 - ICGN3D_TILE_MARGIN;
			const float xlo = fmaxf(1.f, (float)(tx0 + 1)), xhi = fminf(xmax, (float)(tx0 + TX - 2));
			const float ylo = fmaxf(1.f, (float)(ty0 + 1)), yhi = fminf(ymax, (float)(ty0 + TY - 2));
			for (int zs = 0; zs < sz; zs += slab_k) {
				const int nz = (sz - zs) < slab_k ? (sz - zs) : slab_k;
				// slab centre line in z: Z = pz + w + (1 + wz) zl (+ shear); origin from its first layer
				const float zl0 = (float)(zs - rz);
				const float zc_lo = pz + A[11] + fminf(A[10] * zl0, A[10] * (zl0 + (float)(nz - 1)));
				const int tz0 = (int)floorf(zc_lo) - 1 - ICGN3D_TILE_MARGIN;
				const float zlo = fmaxf(1.f, (float)(tz0 + 1)), zhi = fminf(zmax, (float)(tz0 + TZ - 2));
				__syncthreads(); // previous slab's readers are done with T
				if (use_tma) {
					if (tid == 0) {
						fence_proxy_async();
						mbar_expect_tx(bar, (uint32_t)(TXY * TZ * sizeof(float)));
						tma_load_3d(T, &tm_coef, tx0, ty0, tz0, bar);
					}
					mbar_wait(bar, bar_phase);
					bar_phase ^= 1;
				} else {
					const float inv_txy = 1.0f / (float)TXY, inv_tx = 1.0f / (float)TX;
					for (int i = tid; i < TXY * TZ; i += ICGN3D_THREADS) {
						const int tz = fdiv3(i, inv_txy), rem = i - tz * TXY, ty = fdiv3(rem, inv_tx), tx = rem - ty * TX;
						const int gx_ = tx0 + tx, gy_ = ty0 + ty, gz_ = tz0 + tz;
						float v = 0.f;
						if (gx_ >= 0 && gx_ < dx && gy_ >= 0 && gy_ < dy && gz_ >= 0 && gz_ < dz) v = __ldg(coef + ((size_t)gz_ * dy + gy_) * dx + gx_);
						T[i] = v;
					}
					__syncthreads();
				}
				const float* tbase = T - ((tz0 + 1) * TXY + (ty0 + 1) * TX + (tx0 + 1));
				// single-pass sums of one sample (DESIGN.md "single-pass IC-GN sums"); c4 = {R, gx, gy, gz}
				auto accumulate = [&](float t, const float4& c4, float xl, float yl, float zl) {
					tmin = fminf(tmin, t);
					const float R = c4.x;
					const float d = t - R;
					acc[0] += d;
					acc[1] = fmaf(d, d, acc[1]);
					acc[2] = fmaf(R, d, acc[2]);
					const float gxd = c4.y * d, gyd = c4.z * d, gzd = c4.w * d;
					acc[3] += gxd; acc[4] = fmaf(gxd, xl, acc[4]); acc[5] = fmaf(gxd, yl, acc[5]); acc[6] = fmaf(gxd, zl, acc[6]);
					acc[7] += gyd; acc[8] = fmaf(gyd, xl, acc[8]); acc[9] = fmaf(gyd, yl, acc[9]); acc[10] = fmaf(gyd, zl, acc[10]);
					acc[11] += gzd; acc[12] = fmaf(gzd, xl, acc[12]); acc[13] = fmaf(gzd, yl, acc[13]); acc[14] = fmaf(gzd, zl, acc[14]);
				};
				// One sample: warp, 64-tap B-spline evaluation, single-pass sums.  CHECKED: per-sample range tests (tile / volume).
				auto sample = [&](int ii, int j, int k, bool checked) {
					const float4 c4 = __ldg(img.rg + (goff + ((size_t)ii * dy + j) * dx + k)); // issued first: its latency hides under the taps
					const float xl = (float)(k - rx), yl = (float)(j - ry), zl = (float)(ii - rz);
					// Deformation3D1::warp, src/oc_deformation.cpp:518-530; centre + warped (:1376)
					const float X = px + fmaf(A[0], xl, fmaf(A[1], yl, fmaf(A[2], zl, A[3])));
					const float Y = py + fmaf(A[4], xl, fmaf(A[5], yl, fmaf(A[6], zl, A[7])));
					const float Z = pz + fmaf(A[8], xl, fmaf(A[9], yl, fmaf(A[10], zl, A[11])));
					bool fast = true;
					if (checked) {
						fast = (X >= xlo) && (X < xhi) && (Y >= ylo) && (Y < yhi) && (Z >= zlo) && (Z < zhi);
						if (!fast) {
							// TricubicBspline::compute validity, src/oc_cubic_bspline.cpp:356-361 (NaN fails too)
							const bool ok = (X >= 1.f) && (Y >= 1.f) && (Z >= 1.f) && (X < xmax) && (Y < ymax) && (Z < zmax);
							if (!ok) {
								invalid = 1;
								return;
							}
						}
					}
					const float xf = floorf(X), yf = floorf(Y), zf = floorf(Z);
					float bx[4], by[4], bz[4];
					bspline_basis_fast(X - xf, bx);
					bspline_basis_fast(Y - yf, by);
					bspline_basis_fast(Z - zf, bz);
					float t;
					if (fast) t = tricubic_taps<false>(tbase + ((int)zf * TXY + (int)yf * TX + (int)xf), TX, TXY, bx, by, bz);
					else t = tricubic_taps<true>(coef + ((size_t)((int)zf - 1) * dy + ((int)yf - 1)) * dx + ((int)xf - 1), dx, dx * dy, bx, by, bz);
					accumulate(t, c4, xl, yl, zl);
				};
#if ICGN3D_PAIRS
				// Two y-adjacent samples (ii, j, k) and (ii, j + 1, k), support known to be inside the tile: packed pairs, lanes {.x, .y}
				auto sample_pair = [&](int ii, int j, int k) {
					const size_t o = goff + ((size_t)ii * dy + j) * dx + k;
					const float4 ca = __ldg(img.rg + o), cb = __ldg(img.rg + o + dx);
					const float xl = (float)(k - rx), yl = (float)(j - ry), zl = (float)(ii - rz);
					const float2 yl2 = make_float2(yl, yl + 1.f), xl2 = bcast2(xl);
					const float2 X2 = fadd2(bcast2(px), ffma2(bcast2(A[0]), xl2, ffma2(bcast2(A[1]), yl2, bcast2(fmaf(A[2], zl, A[3])))));
					const float2 Y2 = fadd2(bcast2(py), ffma2(bcast2(A[4]), xl2, ffma2(bcast2(A[5]), yl2, bcast2(fmaf(A[6], zl, A[7])))));
					const float2 Z2 = fadd2(bcast2(pz), ffma2(bcast2(A[8]), xl2, ffma2(bcast2(A[9]), yl2, bcast2(fmaf(A[10], zl, A[11])))));
					const float2 xf = make_float2(floorf(X2.x), floorf(X2.y)), yf = make_float2(floorf(Y2.x), floorf(Y2.y)), zf = make_float2(floorf(Z2.x), floorf(Z2.y));
					float2 BX[4], BY[4], BZ[4];
					bspline_basis_fast2(fsub2(X2, xf), BX);
					bspline_basis_fast2(fsub2(Y2, yf), BY);
					bspline_basis_fast2(fsub2(Z2, zf), BZ);
					// block rows jj = 0..4 of the shared 4x5x4 block: the second sample starts one row lower.  Rows 1..3 serve both
					// samples (packed, y weights {by_a[jj], by_b[jj-1]}); row 0 serves only the first and row 4 only the second
					// (scalar on that half of the pair): no multiply is spent on a padded zero weight, and each sample still sees
					// its four rows in the order of the one-sample path
					float2 BYs[3];
#pragma unroll
					for (int jj = 1; jj < 4; jj++) BYs[jj - 1] = make_float2(BY[jj].x, BY[jj - 1].y);
					const float* base = tbase + ((int)zf.x * TXY + (int)yf.x * TX + (int)xf.x);
					float2 val = make_float2(0.f, 0.f);
#pragma unroll
					for (int i = 0; i < 4; i++) {
						float2 ys;
						{
							const float* row = base + i * TXY;
							float rs = row[0] * BX[0].x;
							rs = fmaf(row[1], BX[1].x, rs);
							rs = fmaf(row[2], BX[2].x, rs);
							rs = fmaf(row[3], BX[3].x, rs);
							ys = make_float2(fmaf(rs, BY[0].x, 0.f), 0.f);
						}
#pragma unroll
						for (int jj = 1; jj < 4; jj++) {
							const float* row = base + i * TXY + jj * TX;
							float2 rs = fmul2(bcast2(row[0]), BX[0]);
							rs = ffma2(bcast2(row[1]), BX[1], rs);
							rs = ffma2(bcast2(row[2]), BX[2], rs);
							rs = ffma2(bcast2(row[3]), BX[3], rs);
							ys = ffma2(rs, BYs[jj - 1], ys);
						}
						{
							const float* row = base + i * TXY + 4 * TX;
							float rs = row[0] * BX[0].y;
							rs = fmaf(row[1], BX[1].y, rs);
							rs = fmaf(row[2], BX[2].y, rs);
							rs = fmaf(row[3], BX[3].y, rs);
							ys.y = fmaf(rs, BY[3].y, ys.y);
						}
						val = ffma2(ys, BZ[i], val);
					}
					// the second sample normally sits one block row below the first in the same columns and planes; where the
					// warp's shear or stretch breaks that (a few lanes per POI) it is evaluated on its own
					if (xf.y != xf.x || zf.y != zf.x || yf.y != yf.x + 1.f) {
						const float bx1[4] = { BX[0].y, BX[1].y, BX[2].y, BX[3].y }, by1[4] = { BY[0].y, BY[1].y, BY[2].y, BY[3].y };
						const float bz1[4] = { BZ[0].y, BZ[1].y, BZ[2].y, BZ[3].y };
						val.y = tricubic_taps<false>(tbase + ((int)zf.y * TXY + (int)yf.y * TX + (int)xf.y), TX, TXY, bx1, by1, bz1);
					}
					accumulate(val.x, ca, xl, yl, zl);
					accumulate(val.y, cb, xl, yl + 1.f, zl);
				};
				// Can every sample of this slab take the unchecked path (valid, support inside the tile)?  The affine warp maps
				// the slab's box of local coordinates to a parallelepiped: centre +- half extents per axis.
				bool slab_fast;
				{
					const float zh = 0.5f * (float)(nz - 1), zc = zl0 + zh, fx = (float)rx, fy = (float)ry, eps = 2e-3f;
					const float cx = px + fmaf(A[2], zc, A[3]), ex = fabsf(A[0]) * fx + fabsf(A[1]) * fy + fabsf(A[2]) * zh + eps;
					const float cy = py + fmaf(A[6], zc, A[7]), ey = fabsf(A[4]) * fx + fabsf(A[5]) * fy + fabsf(A[6]) * zh + eps;
					const float cz = pz + fmaf(A[10], zc, A[11]), ez = fabsf(A[8]) * fx + fabsf(A[9]) * fy + fabsf(A[10]) * zh + eps;
					slab_fast = (cx - ex >= xlo) && (cx + ex < xhi) && (cy - ey >= ylo) && (cy + ey < yhi) && (cz - ez >= zlo) && (cz + ez < zhi); // false for NaN
				}
#else
				const bool slab_fast = false;
#endif
				// Lanes run along x within ONE row (y, z) per warp: consecutive tile addresses, no bank
				// conflicts (a linear index over 33-wide rows straddles two rows and conflicts 2-way);
				// columns >= 32 form a short tail with lanes over rows.
				const int nrows = nz * sy;
#if ICGN3D_PAIRS
				if (slab_fast) {
					const int npy = (sy + 1) >> 1; // row pairs per layer; the last one is a single row when sy is odd
					const float inv_npy = 1.0f / (float)npy;
					for (int u = warp; u < nz * npy; u += ICGN3D_WARPS) {
						const int il = fdiv3(u, inv_npy), j = 2 * (u - il * npy);
						if (lane < ncol) {
							if (j + 1 < sy) sample_pair(zs + il, j, lane);
							else sample(zs + il, j, lane, false);
						}
					}
				} else
#endif
				{
					for (int row = warp; row < nrows; row += ICGN3D_WARPS) {
						const int il = fdiv3(row, inv_sy), j = row - il * sy;
						if (lane < ncol) sample(zs + il, j, lane, true);
					}
				}
				for (int i = tid; i < nrows * rem; i += ICGN3D_THREADS) {
					const int row = fdiv3(i, inv_rem), k = 32 + (i - row * rem);
					const int il = fdiv3(row, inv_sy), j = row - il * sy;
					sample(zs + il, j, k, true);
				}
			}
			// the reference rejects the POI when any interpolated value is < 0 (src/oc_icgn.cpp:1378-1390)
			if (tmin < -ICGN3D_NEG_TRIGGER) invalid = 1;
			const int borderline = !(tmin >= ICGN3D_NEG_TRIGGER) ? 2 : 0;
#pragma unroll
			for (int k = 0; k < NITER; k++) {
				float v = warp_sum(acc[k]);
				if (lane == 0) sh.part[warp][k] = v;
			}
			int verdict = __syncthreads_or(invalid | borderline); // bit 0: some sample is decisively out / negative; bit 1: some minimum is borderline
			if (verdict == 2) // sh.A still holds this iteration's warp (thread 0 updates it after the next barrier)
				verdict = __syncthreads_or(icgn3d_exact_negative(sh.A, px, py, pz, rx, ry, rz, coef, dx, dy, dz, tid, ICGN3D_THREADS) ? 1 : 0);
			if (verdict & 1) {
				left_image = true;
				break;
			}
			if (tid == 0) {
				float tot[NITER];
#pragma unroll
				for (int k = 0; k < NITER; k++) {
					float t = 0.f;
					for (int i = 0; i < ICGN3D_WARPS; i++) t += sh.part[i][k];
					tot[k] = t;
				}
				const float f2 = sh.f2, rbar = sh.rbar;
				const float d1 = tot[0], d2 = tot[1];
				const float fd = (tot[2] - sh.c0 * d1) - rbar * d1; // sum f d, from sum R d with the raw R
				const float dbar = d1 * inv_n;
				const float g2 = f2 + 2.f * fd + (d2 - d1 * dbar);
				const float ref_norm = sqrtf(f2), tar_norm = sqrtf(g2);
				const float factor = ref_norm / tar_norm;
				sh.zncc = (f2 + fd) / (ref_norm * tar_norm);
				float b[NP3], dp[NP3], Lr[NH3];
#pragma unroll
				for (int k = 0; k < NP3; k++) b[k] = factor * (sh.SF[k] + tot[3 + k] - dbar * sh.S[k]) - sh.SF[k];
#pragma unroll
				for (int k = 0; k < NH3; k++) Lr[k] = sh.L[k];
				cholesky_solve<NP3>(Lr, b, dp);
				// W <- W * W(dp)^-1 (src/oc_icgn.cpp:1439): affine 4x4, inverse = [B^-1 | -B^-1 t]
				const float m00 = 1.f + dp[1], m01 = dp[2], m02 = dp[3], t0 = dp[0];
				const float m10 = dp[5], m11 = 1.f + dp[6], m12 = dp[7], t1 = dp[4];
				const float m20 = dp[9], m21 = dp[10], m22 = 1.f + dp[11], t2 = dp[8];
				const float c00 = m11 * m22 - m12 * m21, c01 = m12 * m20 - m10 * m22, c02 = m10 * m21 - m11 * m20;
				const float det = m00 * c00 + m01 * c01 + m02 * c02;
				const float id = 1.0f / det;
				float I[9];
				I[0] = c00 * id; I[1] = (m02 * m21 - m01 * m22) * id; I[2] = (m01 * m12 - m02 * m11) * id;
				I[3] = c01 * id; I[4] = (m00 * m22 - m02 * m20) * id; I[5] = (m02 * m10 - m00 * m12) * id;
				I[6] = c02 * id; I[7] = (m01 * m20 - m00 * m21) * id; I[8] = (m00 * m11 - m01 * m10) * id;
				const float it0 = -(I[0] * t0 + I[1] * t1 + I[2] * t2);
				const float it1 = -(I[3] * t0 + I[4] * t1 + I[5] * t2);
				const float it2 = -(I[6] * t0 + I[7] * t1 + I[8] * t2);
#pragma unroll
				for (int r = 0; r < 3; r++) {
					const float a0 = sh.A[r * 4 + 0], a1 = sh.A[r * 4 + 1], a2 = sh.A[r * 4 + 2], a3 = sh.A[r * 4 + 3];
					sh.A[r * 4 + 0] = a0 * I[0] + a1 * I[3] + a2 * I[6];
					sh.A[r * 4 + 1] = a0 * I[1] + a1 * I[4] + a2 * I[7];
					sh.A[r * 4 + 2] = a0 * I[2] + a1 * I[5] + a2 * I[8];
					sh.A[r * 4 + 3] = a0 * it0 + a1 * it1 + a2 * it2 + a3;
				}
				const float dn = sqrtf(dp[0] * dp[0] + dp[4] * dp[4] + dp[8] * dp[8]); // translation only, :1445
				sh.dp_norm = dn;
				sh.keep_going = ((float)iteration < stop_condition && dn >= conv_criterion) ? 1 : 0;
			}
			__syncthreads();
			if (!sh.keep_going) break;
		}
		if (left_image) {
			if (tid == 0) P[P3_ZNCC] = -3.f;
			__syncthreads();
			continue;
		}
		// ---- results, src/oc_icgn.cpp:1450-1489
		if (tid == 0) {
			const float u = sh.A[3], v = sh.A[7], wv = sh.A[11];
			P[P3_DEF + 0] = u; P[P3_DEF + 1] = sh.A[0] - 1.f; P[P3_DEF + 2] = sh.A[1]; P[P3_DEF + 3] = sh.A[2];
			P[P3_DEF + 4] = v; P[P3_DEF + 5] = sh.A[4]; P[P3_DEF + 6] = sh.A[5] - 1.f; P[P3_DEF + 7] = sh.A[6];
			P[P3_DEF + 8] = wv; P[P3_DEF + 9] = sh.A[8]; P[P3_DEF + 10] = sh.A[9]; P[P3_DEF + 11] = sh.A[10] - 1.f;
			P[P3_U0] = u_in; P[P3_V0] = v_in; P[P3_W0] = w_in;
			float zout = sh.zncc;
			const float dn = sh.dp_norm;
			P[P3_ITER] = (float)iteration;
			P[P3_CONV] = dn;
			P[P3_RX] = (float)rx; P[P3_RY] = (float)ry; P[P3_RZ] = (float)rz;
			if (dn >= conv_criterion && (float)iteration >= stop_condition) zout = -4.f;
			if (is_nan_f(zout) || is_nan_f(u) || is_nan_f(v) || is_nan_f(wv)) {
				P[P3_DEF + 0] = u_in; P[P3_DEF + 4] = v_in; P[P3_DEF + 8] = w_in;
				zout = -5.f;
			}
			P[P3_ZNCC] = zout;
		}
		__syncthreads();
	}
}

// Returns 0, -1 when even a one-layer slab does not fit in shared memory, -2 on a CUDA error.
int icgn3d1_launch(const Image3D& img, float* d_pois, size_t n, int rx, int ry, int rz, float conv, float stop, int sm_count, size_t smem_optin,
	int* d_counter, cudaStream_t stream, cudaError_t* err, LaunchInfo* info) {
	const int sz = 2 * rz + 1;
	const size_t layer = (size_t)icgn3d_tile_x(rx) * icgn3d_tile_y(ry) * sizeof(float);
	const size_t fixed = 128 + sizeof(Icgn3dShared) + 1024; // barrier pad + static smem + per-CTA reservation
	const int halo = 3 + 2 * ICGN3D_TILE_MARGIN;
	// prefer two CTAs per SM (one loads while the other computes) when that leaves slabs of >= 6 layers
	int ctas = 2;
	long long k = (long long)(((228 * 1024) / 2 - fixed) / layer) - halo;
	if (k < 6 && k < sz) {
		ctas = 1;
		size_t budget = smem_optin < (size_t)(227 * 1024) ? smem_optin : (size_t)(227 * 1024);
		k = (long long)((budget - 128 - sizeof(Icgn3dShared)) / layer) - halo;
	}
	if (k < 1) return -1;
	if (k > sz) k = sz;
	const int nslab = (int)((sz + k - 1) / k);
	const int slab_k = (sz + nslab - 1) / nslab; // even out the slabs
	const size_t smem = 128 + layer * icgn3d_tile_z(slab_k);
	CUtensorMap tm;
	memset(&tm, 0, sizeof(tm));
	const int dims[3] = { img.dx, img.dy, img.dz };
	const int box[3] = { icgn3d_tile_x(rx), icgn3d_tile_y(ry), icgn3d_tile_z(slab_k) };
	const int use_tma = !getenv("OCB_NO_TMA") && tma_make_map(&tm, img.coef, 3, dims, box);
	void (*kern)(Image3D, float*, int, int, int, int, float, float, int, int*, const CUtensorMap, int);
	const int threads = ctas == 1 ? 512 : 256;
	int rc = 0;
	if (ctas == 1) { // 61^3: the reference's own DVC example
		if (rx == 30 && ry == 30 && rz == 30) rc = 30;
		kern = rc == 30 ? icgn3d1_kernel<30, 512> : icgn3d1_kernel<0, 512>;
	} else {
		if (rx == 16 && ry == 16 && rz == 16) rc = 16;
		kern = rc == 16 ? icgn3d1_kernel<16, 256> : icgn3d1_kernel<0, 256>;
	}
	*err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (*err != cudaSuccess) return -2;
	*err = cudaMemsetAsync(d_counter, 0, sizeof(int), stream);
	if (*err != cudaSuccess) return -2;
	long long grid = (long long)sm_count * ctas;
	if (grid > (long long)n) grid = (long long)n;
	if (grid < 1) grid = 1;
	if (info) {
		info->op = "icgn3d";
		info->rc = rc; info->threads = threads; info->slab_k = slab_k; info->nslab = nslab; info->tma = use_tma; info->grid = (int)grid;
	}
	kern<<<(int)grid, threads, smem, stream>>>(img, d_pois, (int)n, rx, ry, rz, conv, stop, slab_k, d_counter, tm, use_tma);
	*err = cudaGetLastError();
	return *err == cudaSuccess ? 0 : -2;
}

} // namespace ocb
