// fftcc2d_w32.cu -- FFT-CC for the 32x32 window (subset radius 16, the headline configuration):
// ONE WARP PER POI, the 32-point transforms live entirely in registers.
//
// Same algorithm as fftcc2d_kernel (reference src/oc_fftcc.cpp:177-275), specialised:
//   lane = window column: each lane gathers its column of both windows (coalesced rows), the packed
//     z = ref + i*tar column is transformed along y with a fully unrolled radix-2 DIF FFT
//     (compile-time twiddles, natural order in -> bit-reversed order out, tracked statically);
//   transpose through a padded 32x33 shared tile; lane = ky: DIF FFT along x;
//   cross spectrum C = conj(A) B from Z(k) and Z(-k): the partner bin sits in lane (32-ky)%32 at a
//     statically known register, fetched with warp shuffles;
//   inverse: DIT FFT along kx (bit-reversed in -> natural out), transpose back, DIT along ky;
//   first-maximum argmax over registers + warp shuffle reduction.
// No CTA barrier, no integer division, ~2.6k warp instructions per POI (the generic kernel: ~23k).
//
// Window loads: when the POI and its guess sit on whole pixels (the normal FFT-CC case: grid POIs, integer guess) and the
// image pitch allows it, the two 32x32 windows arrive by TMA -- one cp.async.bulk.tensor.2d box of 36 x 32 floats each
// (x origin rounded down to 16 bytes), straight into the shared tiles the transposes use afterwards, completion on a
// per-warp mbarrier -- and every lane then picks its column out of shared memory.  Otherwise the lanes gather their
// columns with coalesced global loads (the reference's float-coordinate truncation, src/oc_fftcc.cpp:204-219, evaluated
// per pixel).  Both paths deliver the same 2 x 1024 values.
#include <stdlib.h>
#include <string.h>

#include "fft32.cuh"
#include "ocb_kernels.h"
#include "ocb_tma.cuh"

namespace ocb {

constexpr int FFTW32_WARPS = 4;
constexpr int FFTW32_PITCH = 33;
constexpr int FFTW32_BOX_W = 36;                 // TMA box: 32 columns + up to 3 of alignment slack
constexpr int FFTW32_TILE = 32 * FFTW32_BOX_W;   // floats per tile: holds a TMA box (36 x 32) or a transpose tile (32 x 33)

__global__ void __launch_bounds__(FFTW32_WARPS * 32) fftcc2d_w32_kernel(Image2D img, float* __restrict__ pois, int n_poi,
	const __grid_constant__ CUtensorMap tm_ref, const __grid_constant__ CUtensorMap tm_tar, int use_tma) {
	__shared__ __align__(128) float s_re[FFTW32_WARPS][FFTW32_TILE];
	__shared__ __align__(128) float s_im[FFTW32_WARPS][FFTW32_TILE];
	__shared__ __align__(8) uint64_t s_bar[FFTW32_WARPS];
	constexpr int R = 16, NW = 32, M = NW * NW;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	float* sre = s_re[warp];
	float* sim = s_im[warp];
	uint64_t* bar = &s_bar[warp];
	uint32_t bar_phase = 0;
	if (use_tma) {
		if (lane == 0) mbar_init(bar, 1);
		__syncwarp();
	}
	const int w = img.w, h = img.h;
	const int plane = (32 - lane) & 31;

	// the record of the NEXT POI of this warp is requested one POI ahead: the queue may be read in place from page-locked host
	// memory, a few microseconds away
	const int poi_stride = gridDim.x * FFTW32_WARPS;
	int poi = blockIdx.x * FFTW32_WARPS + warp;
	float rec_next = (poi < n_poi && lane < P2_N) ? pois[(size_t)poi * P2_N + lane] : 0.f;
	for (; poi < n_poi; poi += poi_stride) {
		float* P = pois + (size_t)poi * P2_N;
		const float rec = rec_next;
		if (poi + poi_stride < n_poi && lane < P2_N) rec_next = pois[(size_t)(poi + poi_stride) * P2_N + lane];
		const float px = __shfl_sync(0xffffffffu, rec, P2_X), py = __shfl_sync(0xffffffffu, rec, P2_Y);
		const float u0 = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_U), v0 = __shfl_sync(0xffffffffu, rec, P2_DEF + D2_V);
		// border guard: the POI is left untouched (src/oc_fftcc.cpp:190-196)
		if ((int)px < R || (int)px >= w - R || (int)py < R || (int)py >= h - R || (int)(px + u0) < R || (int)(px + u0) >= w - R
			|| (int)(py + v0) < R || (int)(py + v0) >= h - R || is_nan_f(px) || is_nan_f(py) || is_nan_f(u0) || is_nan_f(v0))
			continue;
		// gather: lane = column; float coordinate arithmetic then (int) truncation (src/oc_fftcc.cpp:204-219)
		float re[32], im[32];
		{
			float sa = 0.f, sb = 0.f;
			// whole-pixel POI and guess (warp-uniform): every truncation below is the identity, the windows are two boxes
			if (use_tma && px == floorf(px) && py == floorf(py) && u0 == floorf(u0) && v0 == floorf(v0)) {
				const int x0r = (int)px - R, y0r = (int)py - R, x0t = (int)(px + u0) - R, y0t = (int)(py + v0) - R;
				const int axr = floor4(x0r), axt = floor4(x0t);
				if (lane == 0) {
					fence_proxy_async(); // the previous POI's generic-proxy accesses to the tiles come first
					mbar_expect_tx(bar, (uint32_t)(2 * FFTW32_TILE * sizeof(float)));
					tma_load_2d(sre, &tm_ref, axr, y0r, bar);
					tma_load_2d(sim, &tm_tar, axt, y0t, bar);
				}
				mbar_wait(bar, bar_phase);
				bar_phase ^= 1;
				const float* cr = sre + (x0r - axr) + lane;
				const float* ci = sim + (x0t - axt) + lane;
#pragma unroll
				for (int r = 0; r < 32; r++) {
					re[r] = cr[r * FFTW32_BOX_W];
					im[r] = ci[r * FFTW32_BOX_W];
					sa += re[r];
					sb += im[r];
				}
			} else {
				const float rpx = px + lane - R;
				const int ax = (int)rpx, bx = (int)(rpx + u0);
#pragma unroll
				for (int r = 0; r < 32; r++) {
					const float rpy = py + r - R;
					re[r] = __ldg(img.ref + (size_t)(int)rpy * w + ax);
					im[r] = __ldg(img.tar + (size_t)(int)(rpy + v0) * w + bx);
					sa += re[r];
					sb += im[r];
				}
			}
			sa = warp_sum(sa) / (float)M;
			sb = warp_sum(sb) / (float)M;
#pragma unroll
			for (int r = 0; r < 32; r++) {
				re[r] -= sa;
				im[r] -= sb;
			}
		}
		float na = 0.f, nb = 0.f;
#pragma unroll
		for (int r = 0; r < 32; r++) {
			na = fmaf(re[r], re[r], na);
			nb = fmaf(im[r], im[r], nb);
		}
		na = warp_sum(na);
		nb = warp_sum(nb);

		fft32_dif<false>(re, im); // along y: register i holds ky = brev5(i)
		__syncwarp();
#pragma unroll
		for (int i = 0; i < 32; i++) {
			sre[brev5(i) * FFTW32_PITCH + lane] = re[i];
			sim[brev5(i) * FFTW32_PITCH + lane] = im[i];
		}
		__syncwarp();
#pragma unroll
		for (int i = 0; i < 32; i++) { // lane = ky, register i = x
			re[i] = sre[lane * FFTW32_PITCH + i];
			im[i] = sim[lane * FFTW32_PITCH + i];
		}
		fft32_dif<false>(re, im); // along x: register i holds kx = brev5(i)

		// cross spectrum; partner of (ky, kx) is (-ky, -kx): lane `plane`, register brev5((32 - kx) % 32)
#pragma unroll
		for (int i = 0; i < 32; i++) {
			const int ip = brev5((32 - brev5(i)) & 31);
			if (ip < i) continue;
			const float pr_i = __shfl_sync(0xffffffffu, re[i], plane), pi_i = __shfl_sync(0xffffffffu, im[i], plane);
			if (ip == i) {
				float cr, ci;
				cross32(re[i], im[i], pr_i, pi_i, cr, ci);
				re[i] = cr;
				im[i] = ci;
			} else {
				const float pr_p = __shfl_sync(0xffffffffu, re[ip], plane), pi_p = __shfl_sync(0xffffffffu, im[ip], plane);
				float c0r, c0i, c1r, c1i;
				cross32(re[i], im[i], pr_p, pi_p, c0r, c0i);
				cross32(re[ip], im[ip], pr_i, pi_i, c1r, c1i);
				re[i] = c0r; im[i] = c0i;
				re[ip] = c1r; im[ip] = c1i;
			}
		}

		fft32_dit<true>(re, im); // inverse along kx: register i = x
		__syncwarp();
#pragma unroll
		for (int i = 0; i < 32; i++) {
			sre[lane * FFTW32_PITCH + i] = re[i];
			sim[lane * FFTW32_PITCH + i] = im[i];
		}
		__syncwarp();
#pragma unroll
		for (int i = 0; i < 32; i++) { // lane = x, register i holds ky = brev5(i)
			re[i] = sre[brev5(i) * FFTW32_PITCH + lane];
			im[i] = sim[brev5(i) * FFTW32_PITCH + lane];
		}
		fft32_dit<true>(re, im); // inverse along ky: register i = y, lane = x

		// first maximum in linear order y*32 + x (src/oc_fftcc.cpp:246-255)
		float bv = -2.f;
		int bi = 0;
#pragma unroll
		for (int y = 0; y < 32; y++) {
			if (re[y] > bv) { bv = re[y]; bi = y * 32 + lane; }
		}
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) {
			const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
			const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
			if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
		}
		{ // one store instruction for the five result fields (the queue may sit in page-locked host memory)
			int du = bi & 31, dv = bi >> 5;
			if (du > R) du -= NW;
			if (dv > R) dv -= NW;
			float out = 0.f;
			if (lane == P2_DEF + D2_U) out = (float)du + u0;
			if (lane == P2_DEF + D2_V) out = (float)dv + v0;
			if (lane == P2_U0) out = u0;
			if (lane == P2_V0) out = v0;
			if (lane == P2_ZNCC) out = bv / (sqrtf(na * nb) * (float)M); // src/oc_fftcc.cpp:274
			if (lane == P2_DEF + D2_U || lane == P2_DEF + D2_V || lane == P2_U0 || lane == P2_V0 || lane == P2_ZNCC) P[lane] = out;
		}
		__syncwarp();
	}
}

int fftcc2d_w32_launch(const Image2D& img, float* d_pois, size_t n, int sm_count, cudaStream_t stream, cudaError_t* err, int* use_tma_out) {
	long long blocks_needed = ((long long)n + FFTW32_WARPS - 1) / FFTW32_WARPS;
	long long grid = (long long)sm_count * 16;
	if (grid > blocks_needed) grid = blocks_needed;
	if (grid < 1) grid = 1;
	CUtensorMap tm_ref, tm_tar;
	memset(&tm_ref, 0, sizeof(tm_ref));
	memset(&tm_tar, 0, sizeof(tm_tar));
	const int dims[2] = { img.w, img.h }, box[2] = { FFTW32_BOX_W, 32 };
	const int use_tma = !getenv("OCB_NO_TMA") && tma_make_map(&tm_ref, img.ref, 2, dims, box) && tma_make_map(&tm_tar, img.tar, 2, dims, box);
	if (use_tma_out) *use_tma_out = use_tma;
	fftcc2d_w32_kernel<<<(int)grid, FFTW32_WARPS * 32, 0, stream>>>(img, d_pois, (int)n, tm_ref, tm_tar, use_tma);
	*err = cudaGetLastError();
	return *err == cudaSuccess ? 0 : -2;
}

} // namespace ocb
