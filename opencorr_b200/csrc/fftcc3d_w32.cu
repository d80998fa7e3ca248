// fftcc3d_w32.cu -- FFT-CC for the 32x32x32 window (subvolume radius 16, BASELINE config D):
// one CTA (8 warps) per POI, every 32-point transform lives in registers (fft32.cuh).
//
// Same algorithm as fftcc3d_kernel (reference src/oc_fftcc.cpp:327-427), slab-decomposed:
//   pass 0 : means of both windows (coalesced rows, block reduction).
//   phase A: warp per z-slice.  lane = x column: gather, zero-mean, norms; DIF FFT along y in registers,
//            transpose through a padded smem tile, DIF FFT along x; the slice spectrum goes to the CTA's
//            scratch volume as S[z][kx][ky] (lanes = ky: coalesced 256-byte rows).
//   phase B: warp per kx column block.  lane = ky, registers over z (coalesced loads from S); DIF FFT
//            along z; the Hermitian partner Z(-kz,-ky,-kx) belongs to the warp handling -kx, so (kx,-kx)
//            pairs are scheduled on neighbouring warps and exchanged through smem; cross spectrum
//            C = conj(A) B; DIT inverse FFT along kz; back to S.
//   phase C: warp per z-slice: DIT inverse along kx, transpose, DIT inverse along ky, running
//            first-maximum argmax (linear index (z*32 + y)*32 + x).
// The scratch volume (256 KB per CTA, 2 CTAs per SM -> 76 MB) stays L2-resident.
// Phase A's slice loads go through TMA when the POI and its guess sit on whole voxels and the volume pitch allows it: one
// cp.async.bulk.tensor.3d box of 36 x 32 x 1 floats per window and slice (x origin rounded down to 16 bytes), straight into the
// warp's two transpose tiles, completion on a per-warp mbarrier; otherwise the lanes gather their columns (the reference's
// float-coordinate truncation per voxel).  Same values either way.
#include <stdlib.h>
#include <string.h>

#include "fft32.cuh"
#include "ocb_kernels.h"
#include "ocb_tma.cuh"

namespace ocb {

constexpr int F3_WARPS = 8;
constexpr int F3_PITCH = 33;
constexpr int F3_BOX_W = 36;              // TMA box: 32 columns + up to 3 of alignment slack
constexpr int F3_TILE = 32 * F3_BOX_W;    // floats per tile: a TMA box (36 x 32) or a padded transpose tile (32 x 33)

__device__ __forceinline__ void argmax_merge3(float& bv, int& bi, float v, int i) {
	if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
}

__global__ void __launch_bounds__(F3_WARPS * 32, 2) fftcc3d_w32_kernel(Image3D img, float* __restrict__ pois, int n_poi, float2* __restrict__ scratch,
	const __grid_constant__ CUtensorMap tm_ref, const __grid_constant__ CUtensorMap tm_tar, int use_tma) {
	extern __shared__ __align__(128) float f3_smem[]; // 2 x 8 tiles of F3_TILE floats (73.7 KB: above the static limit)
	__shared__ __align__(8) uint64_t s_bar[F3_WARPS];
	float* s_re_all = f3_smem;
	float* s_im_all = f3_smem + F3_WARPS * F3_TILE;
	__shared__ float red[4 * 32];
	constexpr int R = 16, NW = 32;
	constexpr int M = NW * NW * NW;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	float* sre = s_re_all + warp * F3_TILE;
	float* sim = s_im_all + warp * F3_TILE;
	uint64_t* bar = &s_bar[warp];
	uint32_t bar_phase = 0;
	if (use_tma) {
		if (lane == 0) mbar_init(bar, 1);
		__syncwarp();
	}
	const int dx = img.dx, dy = img.dy, dz = img.dz;
	float2* S = scratch + (size_t)blockIdx.x * M; // S[z][kx][ky]

	for (int poi = blockIdx.x; poi < n_poi; poi += gridDim.x) {
		float* P = pois + (size_t)poi * P3_N;
		const float px = P[P3_X], py = P[P3_Y], pz = P[P3_Z];
		const float u0 = P[P3_DEF + 0], v0 = P[P3_DEF + 4], w0 = P[P3_DEF + 8];
		// The reference has no border test here and would read out of bounds; such a POI is left untouched.
		{
			const int x0 = (int)(px - R), y0 = (int)(py - R), z0 = (int)(pz - R);
			const int x1 = (int)(px + (NW - 1) - R), y1 = (int)(py + (NW - 1) - R), z1 = (int)(pz + (NW - 1) - R);
			const int tx0 = (int)(px - R + u0), ty0 = (int)(py - R + v0), tz0 = (int)(pz - R + w0);
			const int tx1 = (int)(px + (NW - 1) - R + u0), ty1 = (int)(py + (NW - 1) - R + v0), tz1 = (int)(pz + (NW - 1) - R + w0);
			if (x0 < 0 || y0 < 0 || z0 < 0 || x1 >= dx || y1 >= dy || z1 >= dz || tx0 < 0 || ty0 < 0 || tz0 < 0 || tx1 >= dx || ty1 >= dy || tz1 >= dz
				|| px - R < 0 || py - R < 0 || pz - R < 0 || px - R + u0 < 0 || py - R + v0 < 0 || pz - R + w0 < 0
				|| is_nan_f(px) || is_nan_f(py) || is_nan_f(pz) || is_nan_f(u0) || is_nan_f(v0) || is_nan_f(w0))
				continue;
		}
		__syncthreads(); // the previous POI is completely finished (record read, smem free)
		// float coordinate arithmetic then (int) truncation, as the reference (src/oc_fftcc.cpp:353-360)
		const float rpx = px + lane - R;
		const int ax = (int)rpx, bx = (int)(rpx + u0);

		// ---- pass 0: means
		float sa = 0.f, sb = 0.f;
		for (int z = warp; z < NW; z += F3_WARPS) {
			const float rpz = pz + z - R;
			const float* pa = img.ref + (size_t)(int)rpz * dy * dx + ax;
			const float* pb = img.tar + (size_t)(int)(rpz + w0) * dy * dx + bx;
#pragma unroll 8
			for (int r = 0; r < NW; r++) {
				const float rpy = py + r - R;
				sa += __ldg(pa + (size_t)(int)rpy * dx);
				sb += __ldg(pb + (size_t)(int)(rpy + v0) * dx);
			}
		}
		sa = warp_sum(sa);
		sb = warp_sum(sb);
		if (lane == 0) { red[warp] = sa; red[32 + warp] = sb; }
		__syncthreads();
		float ref_mean = 0.f, tar_mean = 0.f;
#pragma unroll
		for (int i = 0; i < F3_WARPS; i++) { ref_mean += red[i]; tar_mean += red[32 + i]; }
		ref_mean /= (float)M;
		tar_mean /= (float)M;

		// ---- phase A: per z-slice forward 2D transform
		float na = 0.f, nb = 0.f;
		// whole-voxel POI and guess (CTA-uniform): every truncation is the identity, a slice of a window is one box
		const bool boxes = use_tma && px == floorf(px) && py == floorf(py) && pz == floorf(pz) && u0 == floorf(u0) && v0 == floorf(v0) && w0 == floorf(w0);
		for (int z = warp; z < NW; z += F3_WARPS) {
			float re[32], im[32];
			const float rpz = pz + z - R;
			if (boxes) {
				const int x0r = (int)px - R, y0r = (int)py - R, x0t = (int)(px + u0) - R, y0t = (int)(py + v0) - R;
				const int axr = floor4(x0r), axt = floor4(x0t);
				if (lane == 0) {
					fence_proxy_async(); // the previous slice's generic-proxy accesses to the tiles come first
					mbar_expect_tx(bar, (uint32_t)(2 * F3_TILE * sizeof(float)));
					tma_load_3d(sre, &tm_ref, axr, y0r, (int)rpz, bar);
					tma_load_3d(sim, &tm_tar, axt, y0t, (int)(rpz + w0), bar);
				}
				mbar_wait(bar, bar_phase);
				bar_phase ^= 1;
				const float* cr = sre + (x0r - axr) + lane;
				const float* ci = sim + (x0t - axt) + lane;
#pragma unroll
				for (int r = 0; r < 32; r++) {
					re[r] = cr[r * F3_BOX_W] - ref_mean;
					im[r] = ci[r * F3_BOX_W] - tar_mean;
					na = fmaf(re[r], re[r], na);
					nb = fmaf(im[r], im[r], nb);
				}
			} else {
				const float* pa = img.ref + (size_t)(int)rpz * dy * dx + ax;
				const float* pb = img.tar + (size_t)(int)(rpz + w0) * dy * dx + bx;
#pragma unroll
				for (int r = 0; r < 32; r++) {
					const float rpy = py + r - R;
					re[r] = __ldg(pa + (size_t)(int)rpy * dx) - ref_mean;
					im[r] = __ldg(pb + (size_t)(int)(rpy + v0) * dx) - tar_mean;
					na = fmaf(re[r], re[r], na);
					nb = fmaf(im[r], im[r], nb);
				}
			}
			fft32_dif<false>(re, im); // along y: register i holds ky = brev5(i), lane = x
			__syncwarp();
#pragma unroll
			for (int i = 0; i < 32; i++) {
				sre[brev5(i) * F3_PITCH + lane] = re[i];
				sim[brev5(i) * F3_PITCH + lane] = im[i];
			}
			__syncwarp();
#pragma unroll
			for (int i = 0; i < 32; i++) { // lane = ky, register i = x
				re[i] = sre[lane * F3_PITCH + i];
				im[i] = sim[lane * F3_PITCH + i];
			}
			fft32_dif<false>(re, im); // along x: register i holds kx = brev5(i), lane = ky
			float2* dst = S + (size_t)z * (NW * NW) + lane;
#pragma unroll
			for (int i = 0; i < 32; i++) dst[brev5(i) * NW] = make_float2(re[i], im[i]);
		}
		na = warp_sum(na);
		nb = warp_sum(nb);
		if (lane == 0) { red[64 + warp] = na; red[96 + warp] = nb; }
		__syncthreads(); // S complete (same-CTA global writes are visible after the barrier), norms published

		// ---- phase B: z transform, cross spectrum, inverse z transform.  17 (kx, -kx) pairs, 4 per round:
		// pair 0 = (0,0), pair 1 = (16,16), pair p>=2 = (p-1, 33-p); warps (2s, 2s+1) take one pair.
		for (int rnd = 0; rnd < 5; rnd++) {
			const int pr = rnd * 4 + (warp >> 1);
			const bool active = pr < 17;
			int kxa = 0, kxb = 0;
			if (active) {
				if (pr == 0) { kxa = 0; kxb = 0; }
				else if (pr == 1) { kxa = 16; kxb = 16; }
				else { kxa = pr - 1; kxb = 33 - pr; }
			}
			const int kx = (warp & 1) ? kxb : kxa;
			const bool work = active && !((warp & 1) && kxa == kxb); // self-paired columns need one warp only
			float re[32], im[32];
			if (work) {
				const float2* src = S + (size_t)kx * NW + lane; // S[z][kx][ky = lane]
#pragma unroll
				for (int z = 0; z < 32; z++) {
					const float2 v = __ldcg(src + (size_t)z * (NW * NW));
					re[z] = v.x;
					im[z] = v.y;
				}
				fft32_dif<false>(re, im); // along z: register i holds kz = brev5(i), lane = ky
#pragma unroll
				for (int i = 0; i < 32; i++) { // publish Z[kz][ky] for the partner warp
					sre[brev5(i) * F3_PITCH + lane] = re[i];
					sim[brev5(i) * F3_PITCH + lane] = im[i];
				}
			}
			__syncthreads();
			if (work) {
				const int pw = (kxa == kxb) ? warp : (warp ^ 1); // tile that holds column -kx
				const float* pre = s_re_all + pw * F3_TILE;
				const float* pim = s_im_all + pw * F3_TILE;
				const int plane = (32 - lane) & 31;
#pragma unroll
				for (int i = 0; i < 32; i++) {
					const int nkz = (32 - brev5(i)) & 31;
					const float nr = pre[nkz * F3_PITCH + plane], ni = pim[nkz * F3_PITCH + plane];
					float cr, ci;
					cross32(re[i], im[i], nr, ni, cr, ci);
					re[i] = cr;
					im[i] = ci;
				}
				fft32_dit<true>(re, im); // inverse along kz: register i = z
				float2* dst = S + (size_t)kx * NW + lane;
#pragma unroll
				for (int z = 0; z < 32; z++) dst[(size_t)z * (NW * NW)] = make_float2(re[z], im[z]);
			}
			__syncthreads(); // tiles free for the next round; S rows written
		}

		// ---- phase C: per z-slice inverse 2D transform + running argmax
		float bv = -2.f;
		int bi = 0;
		for (int z = warp; z < NW; z += F3_WARPS) {
			float re[32], im[32];
			const float2* src = S + (size_t)z * (NW * NW) + lane; // [kx][ky = lane]
#pragma unroll
			for (int i = 0; i < 32; i++) { // register i holds kx = brev5(i)
				const float2 v = __ldcg(src + brev5(i) * NW);
				re[i] = v.x;
				im[i] = v.y;
			}
			fft32_dit<true>(re, im); // inverse along kx: register i = x, lane = ky
			__syncwarp();
#pragma unroll
			for (int i = 0; i < 32; i++) {
				sre[lane * F3_PITCH + i] = re[i];
				sim[lane * F3_PITCH + i] = im[i];
			}
			__syncwarp();
#pragma unroll
			for (int i = 0; i < 32; i++) { // lane = x, register i holds ky = brev5(i)
				re[i] = sre[brev5(i) * F3_PITCH + lane];
				im[i] = sim[brev5(i) * F3_PITCH + lane];
			}
			fft32_dit<true>(re, im); // inverse along ky: register i = y, lane = x
#pragma unroll
			for (int y = 0; y < 32; y++) argmax_merge3(bv, bi, re[y], (z * 32 + y) * 32 + lane);
		}
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) {
			const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
			const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
			argmax_merge3(bv, bi, ov, oi);
		}
		if (lane == 0) { red[warp] = bv; ((int*)red)[32 + warp] = bi; }
		__syncthreads();
		if (tid == 0) {
			float fv = red[0];
			int fi = ((int*)red)[32];
			for (int i = 1; i < F3_WARPS; i++) argmax_merge3(fv, fi, red[i], ((int*)red)[32 + i]);
			float tna = 0.f, tnb = 0.f;
			for (int i = 0; i < F3_WARPS; i++) { tna += red[64 + i]; tnb += red[96 + i]; }
			int du = fi & 31, dv = (fi >> 5) & 31, dw = fi >> 10;
			if (du > R) du -= NW;
			if (dv > R) dv -= NW;
			if (dw > R) dw -= NW;
			P[P3_DEF + 0] = (float)du + u0;
			P[P3_DEF + 4] = (float)dv + v0;
			P[P3_DEF + 8] = (float)dw + w0;
			P[P3_U0] = u0;
			P[P3_V0] = v0;
			P[P3_W0] = w0;
			P[P3_ZNCC] = fv / (sqrtf(tna * tnb) * (float)M); // src/oc_fftcc.cpp:426
		}
	}
}

int fftcc3d_w32_grid(int sm_count) { return sm_count * 2; }

int fftcc3d_w32_launch(const Image3D& img, float* d_pois, size_t n, float2* scratch, int grid, cudaStream_t stream, cudaError_t* err,
	int* use_tma_out) {
	if ((long long)grid > (long long)n) grid = (int)n;
	if (grid < 1) grid = 1;
	const size_t smem = (size_t)2 * F3_WARPS * F3_TILE * sizeof(float);
	CUtensorMap tm_ref, tm_tar;
	memset(&tm_ref, 0, sizeof(tm_ref));
	memset(&tm_tar, 0, sizeof(tm_tar));
	const int dims[3] = { img.dx, img.dy, img.dz }, box[3] = { F3_BOX_W, 32, 1 };
	const int use_tma = !getenv("OCB_NO_TMA") && tma_make_map(&tm_ref, img.ref, 3, dims, box) && tma_make_map(&tm_tar, img.tar, 3, dims, box);
	*err = cudaFuncSetAttribute(fftcc3d_w32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (*err != cudaSuccess) return -2;
	if (use_tma_out) *use_tma_out = use_tma;
	fftcc3d_w32_kernel<<<grid, F3_WARPS * 32, smem, stream>>>(img, d_pois, (int)n, scratch, tm_ref, tm_tar, use_tma);
	*err = cudaGetLastError();
	return *err == cudaSuccess ? 0 : -2;
}

} // namespace ocb
