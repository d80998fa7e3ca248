// ocb_kernels.h -- host-visible launch interfaces of the sm_100a kernels (internal to the library).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "ocb_common.cuh"

namespace ocb {

// Factorisation of one FFT axis into Stockham stages (radix 4/2/3/5, generic odd radix <= 31).
struct FftAxis {
	int n;
	int nstage;
	int radix[16];
};

inline bool fft_plan_axis(int n, FftAxis* ax) {
	ax->n = n;
	ax->nstage = 0;
	int m = n;
	while (m % 4 == 0) { ax->radix[ax->nstage++] = 4; m /= 4; }
	while (m % 2 == 0) { ax->radix[ax->nstage++] = 2; m /= 2; }
	while (m % 3 == 0) { ax->radix[ax->nstage++] = 3; m /= 3; }
	while (m % 5 == 0) { ax->radix[ax->nstage++] = 5; m /= 5; }
	for (int p = 7; m > 1; p += 2) {
		while (m % p == 0) {
			if (p > 31 || ax->nstage >= 15) return false;
			ax->radix[ax->nstage++] = p;
			m /= p;
		}
	}
	return true;
}

// Which kernel instantiation a launcher picked, and how it launched it (ocb_last_launch formats it).  Fields a launcher
// does not own stay at their defaults.
struct LaunchInfo {
	const char* op = "";     // "icgn2d", "icgn3d", "fftcc2d", "fftcc3d"
	const char* kernel = ""; // FFT-CC: "w32", "reg" or "generic"
	int np = 0;              // IC-GN 2D: 6 (first order) or 12 (second order)
	int rc = 0;              // compile-time subset radius of the instantiation (0: generic)
	int lm = 0, wpp = 0, tm = 0;
	int tma = 0;             // tile loads by TMA (0: staged loads)
	int grid = 0, threads = 0;
	int slab_k = 0, nslab = 0; // IC-GN 3D: layers per z-slab, slabs per subvolume
	int n = 0;               // FFT-CC register kernels: window points per axis
};

// icgn2d.cu
int icgn2d_launch(int np, const Image2D& img, float* d_pois, size_t n, int rx, int ry, float conv, float stop, int sm_count,
	size_t smem_optin, int* d_counter, const float* d_center_offsets, const float* lm_damping, cudaStream_t stream, cudaError_t* err,
	LaunchInfo* info);
size_t icgn2d_slab_bytes(int rx, int ry); // shared memory one POI needs (plain IC-GN, one warp per POI)
// nr2d.cu
int nr2d1_launch(const Image2D& img, float* d_pois, size_t n, int rx, int ry, float conv, float stop, int sm_count, size_t smem_optin,
	int* d_counter, cudaStream_t stream, cudaError_t* err);
// epipolar.cu
int epipolar_slots(int search_radius, int search_step);
void epipolar_candidates_launch(const float* d_pois, size_t poi0, size_t n_poi, const float* fundamental, const float* parallax_x,
	const float* parallax_y, int search_radius, int search_step, int rx, int ry, int w, int h, int slots, float* d_cand, int sm_count,
	cudaStream_t stream);
void epipolar_select_launch(float* d_pois, size_t poi0, size_t n_poi, int slots, const float* d_cand, int sm_count, cudaStream_t stream);
// strain.cu
size_t strain_workspace_bytes(size_t n);
int strain_launch(int dim, float* d_pois, size_t n, float radius, int k_min, float zncc_threshold, int approximation, long long only, void* workspace,
	int sm_count, cudaStream_t stream, cudaError_t* err, long long* launches);
// fftcc.cu
size_t fftcc2d_smem_bytes(int rx, int ry);
int fftcc2d_launch(const Image2D& img, float* d_pois, size_t n, int rx, int ry, const FftAxis& ax, const FftAxis& ay,
	const float2* tw_x, const float2* tw_y, int sm_count, cudaStream_t stream, cudaError_t* err);
// fftcc2d_w32.cu (32x32 window, one warp per POI, register FFT)
int fftcc2d_w32_launch(const Image2D& img, float* d_pois, size_t n, int sm_count, cudaStream_t stream, cudaError_t* err, int* use_tma_out);
// fftcc2d_reg.cu (square windows of 2^a 3^b 5^c <= 64 points, one thread per row, register FFT codelets)
bool fftcc2d_reg_supported(int r);
int fftcc2d_reg_launch(const Image2D& img, float* d_pois, size_t n, int r, int sm_count, cudaStream_t stream, cudaError_t* err);
// fftcc3d_reg.cu (cubic windows of 2^a 3^b 5^c <= 64 points, one thread per 1D transform, register FFT codelets)
bool fftcc3d_reg_supported(int r);
int fftcc3d_reg_grid(int r, int sm_count);
int fftcc3d_reg_launch(const Image3D& img, float* d_pois, size_t n_poi, int r, float2* scratch, int grid, cudaStream_t stream, cudaError_t* err);
size_t fftcc3d_smem_bytes(int rx, int ry, int rz);
int fftcc3d_grid(int rx, int ry, int rz, int sm_count);
int fftcc3d_launch(const Image3D& img, float* d_pois, size_t n, int rx, int ry, int rz, const FftAxis& ax, const FftAxis& ay,
	const FftAxis& az, const float2* tw_x, const float2* tw_y, const float2* tw_z, float2* scratch, int grid, cudaStream_t stream,
	cudaError_t* err);
// fftcc3d_w32.cu (32^3 window, register FFTs)
int fftcc3d_w32_grid(int sm_count);
int fftcc3d_w32_launch(const Image3D& img, float* d_pois, size_t n, float2* scratch, int grid, cudaStream_t stream, cudaError_t* err,
	int* use_tma_out);
// icgn3d.cu
void gradient3d_launch(const float* ref, float4* rg, int dx, int dy, int dz, int sm_count, cudaStream_t s);
void prefilter3d_launch(const float* in, float* out, int dx, int dy, int dz, int axis, int sm_count, cudaStream_t s);
int icgn3d1_launch(const Image3D& img, float* d_pois, size_t n, int rx, int ry, int rz, float conv, float stop, int sm_count, size_t smem_optin,
	int* d_counter, cudaStream_t stream, cudaError_t* err, LaunchInfo* info);

} // namespace ocb
