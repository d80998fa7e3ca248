// ocb_api.cu -- host side of the C ABI declared in include/opencorr_b200.h.
// Owns the per-GPU context (device images, DVC tables, FFT twiddles/scratch, POI staging buffer)
// and forwards to the sm_100a kernels.  No CPU compute path exists here by design.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/opencorr_b200.h"
#include "ocb_kernels.h"

namespace ocb {
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int w, int h) {
	// in: column-major [w][h] (element (r,c) at c*h + r)  ->  out: row-major [h][w]
	__shared__ float t[32][33];
	const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
	for (int j = threadIdx.y; j < 32; j += blockDim.y) {
		const int c = c0 + j, r = r0 + threadIdx.x;
		if (c < w && r < h) t[j][threadIdx.x] = in[(size_t)c * h + r];
	}
	__syncthreads();
	for (int j = threadIdx.y; j < 32; j += blockDim.y) {
		const int r = r0 + j, c = c0 + threadIdx.x;
		if (c < w && r < h) out[(size_t)r * w + c] = t[threadIdx.x][j];
	}
}
__global__ void widen_u8_kernel(const unsigned char* __restrict__ in, float* __restrict__ out, size_t n) {
	// 4 pixels per thread: one 32-bit load, one 128-bit store (n4 = n / 4 handled vectorised, tail scalar)
	const size_t n4 = n / 4;
	for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
		const uchar4 v = reinterpret_cast<const uchar4*>(in)[i];
		reinterpret_cast<float4*>(out)[i] = make_float4((float)v.x, (float)v.y, (float)v.z, (float)v.w);
	}
	for (size_t i = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) out[i] = (float)in[i];
}
} // namespace ocb

static thread_local std::string g_last_error = "";

// One persistent host thread per extra member of a GROUP context (ocb_create(-1) / ocb_create_multi): the members' copies
// and launches are issued concurrently, each device moving its share over its own PCIe link.
struct ocb_worker {
	std::thread th;
	std::mutex mu;
	std::condition_variable cv;
	std::function<int()> job;
	int result = 0;
	std::atomic<int> state{ 0 }; // 0 idle, 1 job posted, 2 job done
	bool stop = false;
	// A call on a group context is a handful of sub-millisecond phases, so both sides first spin on `state` (a condition-variable
	// round trip costs tens of microseconds per phase and member) and only then go to sleep.
	static bool spin_until(const std::atomic<int>& st, int want) {
		for (int i = 0; i < 20000; i++) {
			if (st.load(std::memory_order_acquire) == want) return true;
#if defined(__x86_64__)
			__builtin_ia32_pause();
#endif
		}
		return false;
	}
	void loop() {
		for (;;) {
			if (!spin_until(state, 1)) {
				std::unique_lock<std::mutex> lk(mu);
				cv.wait(lk, [&] { return state.load(std::memory_order_acquire) == 1 || stop; });
			}
			if (stop && state.load(std::memory_order_acquire) != 1) return;
			result = job();
			{
				std::lock_guard<std::mutex> lk(mu);
				state.store(2, std::memory_order_release);
			}
			cv.notify_all();
		}
	}
	void post(std::function<int()> f) {
		job = std::move(f);
		{
			std::lock_guard<std::mutex> lk(mu);
			state.store(1, std::memory_order_release);
		}
		cv.notify_all();
	}
	int wait() {
		if (!spin_until(state, 2)) {
			std::unique_lock<std::mutex> lk(mu);
			cv.wait(lk, [&] { return state.load(std::memory_order_acquire) == 2; });
		}
		state.store(0, std::memory_order_release);
		return result;
	}
};

struct ocb_ctx {
	// GROUP context: non-empty `members` (single-device contexts owned by the group); none of the per-device fields below
	// is used.  Host-buffer entry points shard their POI queue over the members; *_dev entry points are refused.
	std::vector<ocb_ctx*> members;
	std::vector<ocb_worker*> workers; // workers[i] serves members[i + 1]; member 0 runs on the calling thread
	bool peer_ok = false;             // group: every member can address every other member's memory (NVLink / NVSwitch)
	cudaEvent_t ev_idle = nullptr, ev_pushed = nullptr; // member of a group: see group_distribute_pair
	ocb_ctx* group = nullptr;          // member: the group it belongs to
	bool need_peer_wait = false;       // member: its stream has not yet been ordered after the peers' image pushes
	int device = 0;
	int sm_count = 0;
	size_t smem_optin = 0;
	cudaStream_t own_stream = nullptr;
	cudaStream_t stream = nullptr;
	std::string last_error;
	long long launches = 0;
	std::string last_launch; // ocb_last_launch

	// 2D images
	float* own_ref2 = nullptr;
	float* own_tar2 = nullptr;
	size_t own2_elems = 0;
	ocb::Image2D img2{ nullptr, nullptr, 0, 0 };
	bool prepared2 = false;
	bool prepared_nr2 = false;

	// 3D images + tables
	float* own_ref3 = nullptr;
	float* own_tar3 = nullptr;
	size_t own3_elems = 0;
	float4* rg3 = nullptr;   // packed {ref, gx, gy, gz}
	float* coef3 = nullptr;  // tricubic B-spline coefficients
	float* tmp3 = nullptr;
	size_t tab3_elems = 0;
	ocb::Image3D img3{ nullptr, nullptr, nullptr, nullptr, 0, 0, 0 };
	bool prepared3 = false;

	// FFT
	std::map<int, float2*> twiddles;
	float2* fft_scratch = nullptr;
	size_t fft_scratch_elems = 0;

	int* d_counter = nullptr; // work-queue heads of the persistent kernels

	// POI staging
	float* d_poi = nullptr;
	size_t d_poi_bytes = 0;
	unsigned char* d_u8 = nullptr; // staging for 8-bit image uploads
	size_t d_u8_bytes = 0;
	float* d_off = nullptr; // centre offsets (2 floats per POI)
	size_t d_off_bytes = 0;
	// host-queue calls on large 2D queues are split into chunks whose H2D copy, kernel and D2H copy run on separate
	// streams, so the PCIe transfers of one chunk overlap the kernel of another
	cudaStream_t pipe[4] = { nullptr, nullptr, nullptr, nullptr };
	cudaEvent_t pipe_ready = nullptr;
	// ocb_set_images_2d uploads the pair in OCB_BANDS row bands (ref band, tar band, event) so that the FFT-CC call that follows
	// can start on the POIs of the first rows while the rest of the pair is still crossing PCIe
	cudaEvent_t band_done[4] = { nullptr, nullptr, nullptr, nullptr };
	int band_end[4] = { 0, 0, 0, 0 }; // first row NOT covered once band_done[b] has fired
	bool bands_fresh = false;         // nothing has been enqueued on `stream` since the banded upload
	float* d_cand = nullptr; // EpipolarSearch candidate queue
	size_t d_cand_bytes = 0;
	void* d_strain_ws = nullptr; // Strain: sort keys / compact neighbour arrays / cub scratch
	size_t d_strain_ws_bytes = 0;
};

static int set_error(ocb_ctx* ctx, int code, const char* fmt, ...) {
	char buf[512];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof(buf), fmt, ap);
	va_end(ap);
	g_last_error = buf;
	if (ctx) ctx->last_error = buf;
	return code;
}

// Keep a key=value description of the kernel launch that just went out (ocb_last_launch).
static void record_launch(ocb_ctx* ctx, const ocb::LaunchInfo& li) {
	char buf[192];
	const std::string op = li.op;
	if (op == "icgn2d")
		snprintf(buf, sizeof(buf), "op=icgn2d np=%d rc=%d lm=%d wpp=%d tm=%d tma=%d grid=%d threads=%d", li.np, li.rc, li.lm, li.wpp, li.tm,
			li.tma, li.grid, li.threads);
	else if (op == "icgn3d")
		snprintf(buf, sizeof(buf), "op=icgn3d rc=%d threads=%d slab_k=%d nslab=%d tma=%d grid=%d", li.rc, li.threads, li.slab_k, li.nslab,
			li.tma, li.grid);
	else
		snprintf(buf, sizeof(buf), "op=%s kernel=%s n=%d tma=%d", li.op, li.kernel, li.n, li.tma);
	ctx->last_launch = buf;
}

static ocb::LaunchInfo fftcc_info(const char* op, const char* kernel, int n, int tma) {
	ocb::LaunchInfo li;
	li.op = op;
	li.kernel = kernel;
	li.n = n;
	li.tma = tma;
	return li;
}

#define OCB_CUDA(ctx, call)                                                                                   \
	do {                                                                                                      \
		cudaError_t e_ = (call);                                                                              \
		if (e_ != cudaSuccess) return set_error(ctx, OCB_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
	} while (0)

static int ensure_device(ocb_ctx* ctx) {
	OCB_CUDA(ctx, cudaSetDevice(ctx->device));
	return OCB_OK;
}

static int get_twiddles(ocb_ctx* ctx, int n, const float2** out) {
	auto it = ctx->twiddles.find(n);
	if (it != ctx->twiddles.end()) {
		*out = it->second;
		return OCB_OK;
	}
	std::vector<float2> h(n);
	for (int k = 0; k < n; k++) {
		double a = -2.0 * M_PI * (double)k / (double)n;
		h[k] = make_float2((float)cos(a), (float)sin(a));
	}
	float2* d = nullptr;
	OCB_CUDA(ctx, cudaMalloc(&d, sizeof(float2) * n));
	OCB_CUDA(ctx, cudaMemcpy(d, h.data(), sizeof(float2) * n, cudaMemcpyHostToDevice));
	ctx->twiddles[n] = d;
	*out = d;
	return OCB_OK;
}

static int stage_pois(ocb_ctx* ctx, const void* host, size_t bytes) {
	if (bytes > ctx->d_poi_bytes) {
		if (ctx->d_poi) cudaFree(ctx->d_poi);
		ctx->d_poi = nullptr;
		ctx->d_poi_bytes = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->d_poi, bytes));
		ctx->d_poi_bytes = bytes;
	}
	OCB_CUDA(ctx, cudaMemcpyAsync(ctx->d_poi, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
	return OCB_OK;
}

static int unstage_pois(ocb_ctx* ctx, void* host, size_t bytes) {
	OCB_CUDA(ctx, cudaMemcpyAsync(host, ctx->d_poi, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return OCB_OK;
}

// Host-queue driver for the per-POI independent 2D operators: stage -> dev_call(d_queue, n, first) -> unstage.
// Queues of >= OCB_PIPE_MIN records are processed in 4 chunks on 4 internal streams (each chunk: H2D, kernel, D2H), which
// hides most of the POI traffic behind the kernels; results do not depend on the split (the POIs are independent).
// dev_call launches on ctx->stream with ctx->d_counter, both of which are redirected per chunk.
static const size_t OCB_PIPE_MIN = 16384;
// Device-visible address of a host queue that is page-locked (cudaHostAlloc / cudaHostRegister / ocb_host_alloc), else NULL.
static float* mapped_queue(const void* host) {
	if (getenv("OCB_NO_ZEROCOPY")) return nullptr;
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, host) != cudaSuccess) {
		cudaGetLastError();
		return nullptr;
	}
	return (a.type == cudaMemoryTypeHost && a.devicePointer) ? (float*)a.devicePointer : nullptr;
}

static const int OCB_BANDS = 4;
// fftcc_radius_y > 0: the call is FFT-CC right after a banded image upload -- a chunk only waits for the bands its windows touch
template <class F>
static int run_host_queue_2d(ocb_ctx* ctx, void* host, size_t n, F dev_call, bool allow_mapped = false, int fftcc_radius_y = 0) {
	const size_t rec = OCB_POI2D_FLOATS * sizeof(float);
	int rc;
	const bool banded = fftcc_radius_y > 0 && ctx->bands_fresh && ctx->stream == ctx->own_stream;
	ctx->bands_fresh = false;
	// A page-locked queue is not copied at all: the kernels read each 100-byte record and write its results straight through
	// PCIe (one coalesced load, one coalesced store per POI), which also keeps the copy engines free for the image upload.
	float* const mapped = allow_mapped ? mapped_queue(host) : nullptr; // (only kernels that store a record with one coalesced write)
	if (mapped && !(banded && n >= OCB_PIPE_MIN)) {
		if ((rc = dev_call(mapped, n, (size_t)0))) return rc;
		OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		return OCB_OK;
	}
	if (n < OCB_PIPE_MIN || getenv("OCB_NO_PIPELINE")) {
		if ((rc = stage_pois(ctx, host, n * rec))) return rc;
		if ((rc = dev_call((float*)ctx->d_poi, n, (size_t)0))) return rc;
		return unstage_pois(ctx, host, n * rec);
	}
	if (!mapped && n * rec > ctx->d_poi_bytes) {
		if (ctx->d_poi) cudaFree(ctx->d_poi);
		ctx->d_poi = nullptr;
		ctx->d_poi_bytes = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->d_poi, n * rec));
		ctx->d_poi_bytes = n * rec;
	}
	const int K = 4;
	if (!ctx->pipe_ready) {
		OCB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->pipe_ready, cudaEventDisableTiming));
		for (int i = 0; i < K; i++) OCB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->pipe[i], cudaStreamNonBlocking));
	}
	// everything enqueued so far on the caller-visible stream (image uploads, prepare, offsets) comes first
	OCB_CUDA(ctx, cudaEventRecord(ctx->pipe_ready, ctx->stream));
	cudaStream_t saved_stream = ctx->stream;
	int* saved_counter = ctx->d_counter;
	rc = OCB_OK;
	for (int c = 0; c < K && rc == OCB_OK; c++) {
		const size_t a = n * (size_t)c / K, b = n * (size_t)(c + 1) / K;
		if (b == a) continue;
		char* h = (char*)host + a * rec;
		float* d = mapped ? mapped + a * OCB_POI2D_FLOATS : ctx->d_poi + a * OCB_POI2D_FLOATS;
		cudaEvent_t gate = ctx->pipe_ready;
		if (banded) { // last image row this chunk's windows read: max over its POIs of max(y, y + v0) + r (src/oc_fftcc.cpp:204-219)
			float ymax = -1e30f;
			bool finite = true;
			const float* q = (const float*)h;
			for (size_t i = 0; i < b - a; i++) {
				const float y = q[i * OCB_POI2D_FLOATS + 1], v0 = q[i * OCB_POI2D_FLOATS + 2 + 6];
				const float top = y > y + v0 ? y : y + v0;
				if (!(top == top) || top > 1e9f) finite = false;
				ymax = top > ymax ? top : ymax;
			}
			if (finite) {
				const int need = (int)ymax + fftcc_radius_y + 1;
				for (int k = 0; k < OCB_BANDS; k++)
					if (ctx->band_end[k] >= need || k == OCB_BANDS - 1) { gate = ctx->band_done[k]; break; }
			}
		}
		cudaError_t e = cudaStreamWaitEvent(ctx->pipe[c], gate, 0);
		if (e == cudaSuccess && !mapped) e = cudaMemcpyAsync(d, h, (b - a) * rec, cudaMemcpyHostToDevice, ctx->pipe[c]);
		if (e != cudaSuccess) { rc = set_error(ctx, OCB_ERR_CUDA, "pipelined upload failed: %s", cudaGetErrorString(e)); break; }
		ctx->stream = ctx->pipe[c];
		ctx->d_counter = saved_counter + c;
		rc = dev_call(d, b - a, a);
		ctx->stream = saved_stream;
		ctx->d_counter = saved_counter;
		if (rc != OCB_OK) break;
		if (!mapped) {
			e = cudaMemcpyAsync(h, d, (b - a) * rec, cudaMemcpyDeviceToHost, ctx->pipe[c]);
			if (e != cudaSuccess) rc = set_error(ctx, OCB_ERR_CUDA, "pipelined download failed: %s", cudaGetErrorString(e));
		}
	}
	for (int c = 0; c < K; c++) {
		cudaError_t e = cudaStreamSynchronize(ctx->pipe[c]);
		if (e != cudaSuccess && rc == OCB_OK) rc = set_error(ctx, OCB_ERR_CUDA, "pipelined queue failed: %s", cudaGetErrorString(e));
	}
	return rc;
}


// ---- GROUP contexts: one process, several devices -------------------------------------------------------------------
static inline bool is_group(const ocb_ctx* ctx) { return ctx && !ctx->members.empty(); }

// Run f(member, index) on the first `used` members concurrently (member 0 on the calling thread); first failure wins.
// (member, on its own thread) order the member's stream after every peer's image pushes, once per upload
static int member_settle(ocb_ctx* m) {
	if (!m->need_peer_wait) return OCB_OK;
	m->need_peer_wait = false;
	if (cudaSetDevice(m->device) != cudaSuccess) return set_error(m, OCB_ERR_CUDA, "cudaSetDevice failed");
	for (ocb_ctx* other : m->group->members)
		if (other != m && cudaStreamWaitEvent(m->stream, other->ev_pushed, 0) != cudaSuccess) return set_error(m, OCB_ERR_CUDA, "cudaStreamWaitEvent failed");
	return OCB_OK;
}

template <class F>
static int group_run(ocb_ctx* g, int used, F f) {
	if (used > (int)g->members.size()) used = (int)g->members.size();
	auto job = [f](ocb_ctx* m, int i) {
		const int rc = member_settle(m);
		return rc ? rc : f(m, i);
	};
	for (int i = 1; i < used; i++) {
		ocb_ctx* m = g->members[i];
		g->workers[i - 1]->post([job, m, i]() { return job(m, i); });
	}
	int rc = job(g->members[0], 0), bad = 0;
	for (int i = 1; i < used; i++) {
		const int r = g->workers[i - 1]->wait();
		if (rc == OCB_OK && r != OCB_OK) { rc = r; bad = i; }
	}
	if (rc != OCB_OK) {
		g->last_error = "device " + std::to_string(g->members[bad]->device) + ": " + g->members[bad]->last_error;
		g_last_error = g->last_error;
	}
	return rc;
}
template <class F>
static int group_each(ocb_ctx* g, F f) {
	return group_run(g, (int)g->members.size(), [f](ocb_ctx* m, int) { return f(m); });
}
// Contiguous block split of a host queue of n records of rec_bytes: member i gets records [n i / G, n (i+1) / G) and
// copies them in and out of the caller's array itself (its own PCIe link, straight into the caller's slice).  Queues
// too short to fill every device use fewer of them (min_per_device records each).  f(member, slice, count, first).
template <class F>
static int group_shard(ocb_ctx* g, void* queue, size_t n, size_t rec_bytes, size_t min_per_device, F f) {
	if (n == 0) return OCB_OK;
	size_t used = n / min_per_device;
	if (used < 1) used = 1;
	if (used > g->members.size()) used = g->members.size();
	const int G = (int)used;
	char* base = (char*)queue;
	return group_run(g, G, [=](ocb_ctx* m, int i) {
		const size_t a = n * (size_t)i / (size_t)G, b = n * (size_t)(i + 1) / (size_t)G;
		if (b == a) return (int)OCB_OK;
		return f(m, (void*)(base + a * rec_bytes), b - a, a);
	});
}
// Smallest shard worth a device.  2D: a launch that cannot fill the GPU lets two warps share a POI (icgn2d_launch), which splits
// its sums differently and changes the last bits of the result; shards of >= 8192 POIs take the same one-warp-per-POI path as
// the undivided queue on one device, so sharded results stay bit-identical.
static const size_t OCB_GROUP_MIN_2D = 8192, OCB_GROUP_MIN_3D = 64;
#define OCB_NO_GROUP(ctx, what) \
	if (is_group(ctx)) return set_error(ctx, OCB_ERR_ARG, what ": device-pointer / stream entry points need a single-device context (ocb_member)")

static ocb_ctx* create_group(const int* devices, int n) {
	ocb_ctx* g = new ocb_ctx;
	g->device = -1;
	for (int i = 0; i < n; i++) {
		ocb_ctx* m = ocb_create(devices[i]);
		if (!m) {
			for (ocb_ctx* p : g->members) ocb_destroy(p);
			delete g;
			return nullptr; // ocb_create left the message in the process-wide slot
		}
		m->group = g;
		g->members.push_back(m);
	}
	for (int i = 1; i < n; i++) {
		ocb_worker* w = new ocb_worker;
		w->th = std::thread([w]() { w->loop(); });
		g->workers.push_back(w);
	}
	// peer access between all members (NVLink through NVSwitch on an HGX board): images are then uploaded once, in slices, and
	// exchanged between the devices instead of crossing PCIe once per device
	g->peer_ok = n > 1 && !getenv("OCB_NO_PEER");
	for (int i = 0; i < n && g->peer_ok; i++) {
		cudaSetDevice(devices[i]);
		for (int j = 0; j < n && g->peer_ok; j++) {
			if (i == j) continue;
			int can = 0;
			if (cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) != cudaSuccess || !can) { g->peer_ok = false; break; }
			const cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
			if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) g->peer_ok = false;
			cudaGetLastError();
		}
	}
	for (ocb_ctx* m : g->members) {
		cudaSetDevice(m->device);
		if (cudaEventCreateWithFlags(&m->ev_idle, cudaEventDisableTiming) != cudaSuccess
			|| cudaEventCreateWithFlags(&m->ev_pushed, cudaEventDisableTiming) != cudaSuccess)
			g->peer_ok = false;
	}
	cudaGetLastError();
	return g;
}

// Image buffers of a single-device context (grow-only)
static int ensure_buffers_2d(ocb_ctx* ctx, size_t elems) {
	if (elems > ctx->own2_elems) {
		cudaFree(ctx->own_ref2);
		cudaFree(ctx->own_tar2);
		ctx->own_ref2 = ctx->own_tar2 = nullptr;
		ctx->own2_elems = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_ref2, elems * sizeof(float)));
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_tar2, elems * sizeof(float)));
		ctx->own2_elems = elems;
	}
	return OCB_OK;
}
static int ensure_buffers_3d(ocb_ctx* ctx, size_t elems) {
	if (elems > ctx->own3_elems) {
		cudaFree(ctx->own_ref3);
		cudaFree(ctx->own_tar3);
		ctx->own_ref3 = ctx->own_tar3 = nullptr;
		ctx->own3_elems = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_ref3, elems * sizeof(float)));
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_tar3, elems * sizeof(float)));
		ctx->own3_elems = elems;
	}
	return OCB_OK;
}

// GROUP upload of an image pair (elems floats each) into every member's buffers: member m copies ONLY slice m of both images
// from the host (its own PCIe link, all members concurrently), then pushes the slice to every other member over NVLink
// (cudaMemcpyPeerAsync); each member's stream finally waits for everybody's pushes.  Per device the PCIe traffic drops from the
// whole pair to 1/G of it; the exchange runs at NVLink rate through the switch.  dim: 2 or 3 (which buffers).
static int group_distribute_pair(ocb_ctx* g, const float* ref, const float* tar, size_t elems, int dim) {
	const int G = (int)g->members.size();
	int rc = OCB_OK;
	for (ocb_ctx* m : g->members) { // buffers first: a peer may push into them as soon as the exchange starts
		if (ensure_device(m)) return OCB_ERR_CUDA;
		rc = dim == 2 ? ensure_buffers_2d(m, elems) : ensure_buffers_3d(m, elems);
		if (rc == OCB_OK && cudaEventRecord(m->ev_idle, m->stream) != cudaSuccess) rc = set_error(m, OCB_ERR_CUDA, "cudaEventRecord failed");
		if (rc) {
			g->last_error = m->last_error;
			return rc;
		}
	}
	const size_t gran = 64; // floats: slices start on 256-byte boundaries
	rc = group_run(g, G, [=](ocb_ctx* m, int i) {
		if (ensure_device(m)) return (int)OCB_ERR_CUDA;
		const size_t a = (elems * (size_t)i / (size_t)G) / gran * gran, b = i + 1 == G ? elems : (elems * (size_t)(i + 1) / (size_t)G) / gran * gran;
		const size_t len = (b - a) * sizeof(float);
		float* mine[2] = { dim == 2 ? m->own_ref2 : m->own_ref3, dim == 2 ? m->own_tar2 : m->own_tar3 };
		const float* src[2] = { ref, tar };
		if (len) {
			for (int k = 0; k < 2; k++) OCB_CUDA(m, cudaMemcpyAsync(mine[k] + a, src[k] + a, len, cudaMemcpyHostToDevice, m->stream));
			for (int jj = 1; jj < G; jj++) { // start with the next neighbour so that the pushes of all members spread over the peers
				ocb_ctx* peer = g->members[(i + jj) % G];
				OCB_CUDA(m, cudaStreamWaitEvent(m->stream, peer->ev_idle, 0)); // the peer is done with its old images
				float* theirs[2] = { dim == 2 ? peer->own_ref2 : peer->own_ref3, dim == 2 ? peer->own_tar2 : peer->own_tar3 };
				for (int k = 0; k < 2; k++) OCB_CUDA(m, cudaMemcpyPeerAsync(theirs[k] + a, peer->device, mine[k] + a, m->device, len, m->stream));
			}
		}
		OCB_CUDA(m, cudaEventRecord(m->ev_pushed, m->stream));
		return (int)OCB_OK;
	});
	if (rc) return rc;
	// nobody uses the pair before every slice has arrived: each member orders its stream after the peers' pushes at the start of
	// its next job, on its own thread (member_settle)
	for (ocb_ctx* m : g->members) m->need_peer_wait = true;
	return OCB_OK;
}

extern "C" {

int ocb_device_count(void) {
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess) return set_error(nullptr, OCB_ERR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
	return n;
}

ocb_ctx* ocb_create(int device) {
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0) {
		set_error(nullptr, OCB_ERR_CUDA, "no usable CUDA device (%s); this engine has no CPU fallback",
			e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
		return nullptr;
	}
	if (device == -1) { // every visible device: a GROUP context
		std::vector<int> all(n);
		for (int i = 0; i < n; i++) all[i] = i;
		return n == 1 ? ocb_create(0) : create_group(all.data(), n);
	}
	if (device < 0 || device >= n) {
		set_error(nullptr, OCB_ERR_ARG, "device %d out of range [0,%d)", device, n);
		return nullptr;
	}
	ocb_ctx* ctx = new ocb_ctx;
	ctx->device = device;
	cudaDeviceProp prop;
	if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess
		|| (e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
		set_error(nullptr, OCB_ERR_CUDA, "context creation on device %d failed: %s", device, cudaGetErrorString(e));
		delete ctx;
		return nullptr;
	}
	if (prop.major < 10) {
		set_error(nullptr, OCB_ERR_CUDA, "device %d is sm_%d%d; this library ships sm_100a code only", device, prop.major, prop.minor);
		cudaStreamDestroy(ctx->own_stream);
		delete ctx;
		return nullptr;
	}
	ctx->stream = ctx->own_stream;
	ctx->sm_count = prop.multiProcessorCount;
	ctx->smem_optin = prop.sharedMemPerBlockOptin;
	// work-queue heads: [0, 16) are zeroed by a memset in front of every launch that uses one; [32, 48) belong to the kernels that
	// reset their head themselves (icgn2d, one warp per POI) and are zeroed once, here
	if ((e = cudaMalloc(&ctx->d_counter, 64 * sizeof(int))) != cudaSuccess || (e = cudaMemset(ctx->d_counter, 0, 64 * sizeof(int))) != cudaSuccess) {
		set_error(nullptr, OCB_ERR_CUDA, "context creation on device %d failed: %s", device, cudaGetErrorString(e));
		cudaStreamDestroy(ctx->own_stream);
		delete ctx;
		return nullptr;
	}
	return ctx;
}

ocb_ctx* ocb_create_multi(const int* devices, int n_devices) {
	if (!devices || n_devices < 1) {
		set_error(nullptr, OCB_ERR_ARG, "create_multi: need at least one device");
		return nullptr;
	}
	for (int i = 0; i < n_devices; i++)
		for (int j = 0; j < i; j++)
			if (devices[i] == devices[j]) {
				set_error(nullptr, OCB_ERR_ARG, "create_multi: device %d listed twice", devices[i]);
				return nullptr;
			}
	return create_group(devices, n_devices);
}

int ocb_member_count(const ocb_ctx* ctx) { return !ctx ? 0 : (is_group(ctx) ? (int)ctx->members.size() : 1); }

ocb_ctx* ocb_member(ocb_ctx* ctx, int index) {
	if (!ctx) return nullptr;
	if (!is_group(ctx)) return index == 0 ? ctx : nullptr;
	if (index < 0 || index >= (int)ctx->members.size()) return nullptr;
	member_settle(ctx->members[index]); // the caller may go on with device-pointer calls on this member: its images must be complete
	return ctx->members[index];
}

void* ocb_host_alloc_on(ocb_ctx* ctx, size_t bytes) {
	if (ctx) {
		const ocb_ctx* c = is_group(ctx) ? ctx->members[0] : ctx;
		if (cudaSetDevice(c->device) != cudaSuccess) {
			cudaGetLastError();
			return nullptr;
		}
	}
	return ocb_host_alloc(bytes);
}

void* ocb_host_alloc(size_t bytes) {
	if (!bytes) return nullptr;
	void* p = nullptr;
	cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
	if (e != cudaSuccess) {
		cudaGetLastError();
		set_error(nullptr, OCB_ERR_CUDA, "cudaHostAlloc failed: %s", cudaGetErrorString(e));
		return nullptr;
	}
	return p;
}

void ocb_host_free(void* host) {
	if (host) cudaFreeHost(host);
}

int ocb_host_register(void* host, size_t bytes) {
	if (!host || !bytes) return set_error(nullptr, OCB_ERR_ARG, "host_register: bad arguments");
	cudaError_t e = cudaHostRegister(host, bytes, cudaHostRegisterPortable);
	if (e != cudaSuccess) {
		cudaGetLastError();
		return set_error(nullptr, OCB_ERR_CUDA, "cudaHostRegister failed: %s", cudaGetErrorString(e));
	}
	return OCB_OK;
}

int ocb_host_unregister(void* host) {
	if (!host) return set_error(nullptr, OCB_ERR_ARG, "host_unregister: bad arguments");
	cudaError_t e = cudaHostUnregister(host);
	if (e != cudaSuccess) {
		cudaGetLastError();
		return set_error(nullptr, OCB_ERR_CUDA, "cudaHostUnregister failed: %s", cudaGetErrorString(e));
	}
	return OCB_OK;
}

void ocb_destroy(ocb_ctx* ctx) {
	if (!ctx) return;
	if (is_group(ctx)) {
		for (ocb_worker* w : ctx->workers) {
			{
				std::lock_guard<std::mutex> lk(w->mu);
				w->stop = true;
			}
			w->cv.notify_all();
			w->th.join();
			delete w;
		}
		for (ocb_ctx* m : ctx->members) {
			cudaSetDevice(m->device);
			if (m->ev_idle) cudaEventDestroy(m->ev_idle);
			if (m->ev_pushed) cudaEventDestroy(m->ev_pushed);
			ocb_destroy(m);
		}
		delete ctx;
		return;
	}
	cudaSetDevice(ctx->device);
	cudaDeviceSynchronize();
	cudaFree(ctx->own_ref2);
	cudaFree(ctx->own_tar2);
	cudaFree(ctx->own_ref3);
	cudaFree(ctx->own_tar3);
	cudaFree(ctx->rg3);
	cudaFree(ctx->coef3);
	cudaFree(ctx->tmp3);
	for (auto& kv : ctx->twiddles) cudaFree(kv.second);
	cudaFree(ctx->fft_scratch);
	cudaFree(ctx->d_poi);
	cudaFree(ctx->d_off);
	cudaFree(ctx->d_strain_ws);
	cudaFree(ctx->d_cand);
	for (int i = 0; i < 4; i++)
		if (ctx->pipe[i]) cudaStreamDestroy(ctx->pipe[i]);
	if (ctx->pipe_ready) cudaEventDestroy(ctx->pipe_ready);
	for (int i = 0; i < 4; i++)
		if (ctx->band_done[i]) cudaEventDestroy(ctx->band_done[i]);
	cudaFree(ctx->d_u8);
	cudaFree(ctx->d_counter);
	cudaStreamDestroy(ctx->own_stream);
	delete ctx;
}

const char* ocb_last_error(const ocb_ctx* ctx) { return ctx ? ctx->last_error.c_str() : g_last_error.c_str(); }

const char* ocb_last_launch(const ocb_ctx* ctx) { return ctx ? ctx->last_launch.c_str() : ""; }

int ocb_set_stream(ocb_ctx* ctx, void* cuda_stream) {
	if (!ctx) return set_error(nullptr, OCB_ERR_ARG, "null context");
	OCB_NO_GROUP(ctx, "set_stream");
	ctx->stream = (cudaStream_t)cuda_stream;
	return OCB_OK;
}

int ocb_use_own_stream(ocb_ctx* ctx) {
	if (!ctx) return set_error(nullptr, OCB_ERR_ARG, "null context");
	if (is_group(ctx)) return OCB_OK;
	ctx->stream = ctx->own_stream;
	return OCB_OK;
}

int ocb_sync(ocb_ctx* ctx) {
	if (!ctx) return set_error(nullptr, OCB_ERR_ARG, "null context");
	if (is_group(ctx)) return group_each(ctx, [](ocb_ctx* m) { return ocb_sync(m); });
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return OCB_OK;
}

long long ocb_launch_count(const ocb_ctx* ctx) {
	if (!ctx) return 0;
	long long total = ctx->launches;
	for (const ocb_ctx* m : ctx->members) total += m->launches;
	return total;
}

// ---- images ----------------------------------------------------------------------------------
int ocb_set_images_2d_dev(ocb_ctx* ctx, const float* d_ref, const float* d_tar, int width, int height) {
	OCB_NO_GROUP(ctx, "set_images_2d_dev");
	if (!ctx || !d_ref || !d_tar || width < 5 || height < 5) return set_error(ctx, OCB_ERR_ARG, "set_images_2d: bad arguments");
	ctx->img2 = ocb::Image2D{ d_ref, d_tar, width, height };
	ctx->bands_fresh = false;
	ctx->prepared2 = false;
	ctx->prepared_nr2 = false;
	return OCB_OK;
}

int ocb_set_images_2d(ocb_ctx* ctx, const float* ref, const float* tar, int width, int height, int col_major) {
	if (is_group(ctx)) {
		if (ctx->peer_ok && !col_major && ref && tar && width >= 5 && height >= 5) {
			int rc = group_distribute_pair(ctx, ref, tar, (size_t)width * height, 2);
			if (rc) return rc;
			for (ocb_ctx* m : ctx->members)
				if ((rc = ocb_set_images_2d_dev(m, m->own_ref2, m->own_tar2, width, height))) return rc;
			return OCB_OK;
		}
		return group_each(ctx, [=](ocb_ctx* m) { return ocb_set_images_2d(m, ref, tar, width, height, col_major); });
	}
	if (!ctx || !ref || !tar || width < 5 || height < 5) return set_error(ctx, OCB_ERR_ARG, "set_images_2d: bad arguments");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const size_t elems = (size_t)width * height;
	{
		const int rcb = ensure_buffers_2d(ctx, elems);
		if (rcb) return rcb;
	}
	bool banded = false;
	if (!col_major) {
		if (ctx->stream == ctx->own_stream && elems >= ((size_t)1 << 20) && !getenv("OCB_NO_PIPELINE")) {
			for (int b = 0; b < OCB_BANDS; b++) {
				if (!ctx->band_done[b]) OCB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->band_done[b], cudaEventDisableTiming));
				const size_t r0 = (size_t)height * b / OCB_BANDS, r1 = (size_t)height * (b + 1) / OCB_BANDS;
				const size_t off = r0 * (size_t)width, len = (r1 - r0) * (size_t)width * sizeof(float);
				OCB_CUDA(ctx, cudaMemcpyAsync(ctx->own_ref2 + off, ref + off, len, cudaMemcpyHostToDevice, ctx->stream));
				OCB_CUDA(ctx, cudaMemcpyAsync(ctx->own_tar2 + off, tar + off, len, cudaMemcpyHostToDevice, ctx->stream));
				OCB_CUDA(ctx, cudaEventRecord(ctx->band_done[b], ctx->stream));
				ctx->band_end[b] = (int)r1;
			}
			banded = true;
		} else {
			OCB_CUDA(ctx, cudaMemcpyAsync(ctx->own_ref2, ref, elems * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
			OCB_CUDA(ctx, cudaMemcpyAsync(ctx->own_tar2, tar, elems * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
		}
	} else {
		float* tmp = nullptr;
		OCB_CUDA(ctx, cudaMalloc(&tmp, elems * sizeof(float)));
		dim3 grid((width + 31) / 32, (height + 31) / 32), block(32, 8);
		const float* src[2] = { ref, tar };
		float* dst[2] = { ctx->own_ref2, ctx->own_tar2 };
		for (int i = 0; i < 2; i++) {
			OCB_CUDA(ctx, cudaMemcpyAsync(tmp, src[i], elems * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
			ocb::transpose_kernel<<<grid, block, 0, ctx->stream>>>(tmp, dst[i], width, height);
			ctx->launches++;
		}
		OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		cudaFree(tmp);
	}
	const int rc_dev = ocb_set_images_2d_dev(ctx, ctx->own_ref2, ctx->own_tar2, width, height);
	ctx->bands_fresh = banded && rc_dev == OCB_OK;
	return rc_dev;
}

// upload `elems` bytes twice (ref, tar) and widen into the context-owned float buffers dst_ref/dst_tar
static int upload_u8_pair(ocb_ctx* ctx, const unsigned char* ref, const unsigned char* tar, size_t elems, float* dst_ref, float* dst_tar) {
	// the widening kernel reads uchar4: the second image starts at a 16-byte aligned offset whatever the pixel count
	const size_t tar_off = (elems + 15) & ~(size_t)15;
	if (tar_off + elems > ctx->d_u8_bytes) {
		cudaFree(ctx->d_u8);
		ctx->d_u8 = nullptr;
		ctx->d_u8_bytes = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->d_u8, tar_off + elems));
		ctx->d_u8_bytes = tar_off + elems;
	}
	OCB_CUDA(ctx, cudaMemcpyAsync(ctx->d_u8, ref, elems, cudaMemcpyHostToDevice, ctx->stream));
	OCB_CUDA(ctx, cudaMemcpyAsync(ctx->d_u8 + tar_off, tar, elems, cudaMemcpyHostToDevice, ctx->stream));
	const int grid = ctx->sm_count * 8;
	ocb::widen_u8_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->d_u8, dst_ref, elems);
	ocb::widen_u8_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->d_u8 + tar_off, dst_tar, elems);
	ctx->launches += 2;
	OCB_CUDA(ctx, cudaGetLastError());
	return OCB_OK;
}

int ocb_set_images_2d_u8(ocb_ctx* ctx, const unsigned char* ref, const unsigned char* tar, int width, int height) {
	if (is_group(ctx)) return group_each(ctx, [=](ocb_ctx* m) { return ocb_set_images_2d_u8(m, ref, tar, width, height); });
	if (!ctx || !ref || !tar || width < 5 || height < 5) return set_error(ctx, OCB_ERR_ARG, "set_images_2d_u8: bad arguments");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const size_t elems = (size_t)width * height;
	if (elems > ctx->own2_elems) {
		cudaFree(ctx->own_ref2);
		cudaFree(ctx->own_tar2);
		ctx->own_ref2 = ctx->own_tar2 = nullptr;
		ctx->own2_elems = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_ref2, elems * sizeof(float)));
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_tar2, elems * sizeof(float)));
		ctx->own2_elems = elems;
	}
	int rc = upload_u8_pair(ctx, ref, tar, elems, ctx->own_ref2, ctx->own_tar2);
	if (rc) return rc;
	return ocb_set_images_2d_dev(ctx, ctx->own_ref2, ctx->own_tar2, width, height);
}

int ocb_set_images_3d_u8(ocb_ctx* ctx, const unsigned char* ref, const unsigned char* tar, int dim_x, int dim_y, int dim_z) {
	if (is_group(ctx)) return group_each(ctx, [=](ocb_ctx* m) { return ocb_set_images_3d_u8(m, ref, tar, dim_x, dim_y, dim_z); });
	if (!ctx || !ref || !tar || dim_x < 15 || dim_y < 15 || dim_z < 15)
		return set_error(ctx, OCB_ERR_ARG, "set_images_3d_u8: bad arguments (each dimension must be >= 15)");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const size_t elems = (size_t)dim_x * dim_y * dim_z;
	if (elems > ctx->own3_elems) {
		cudaFree(ctx->own_ref3);
		cudaFree(ctx->own_tar3);
		ctx->own_ref3 = ctx->own_tar3 = nullptr;
		ctx->own3_elems = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_ref3, elems * sizeof(float)));
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_tar3, elems * sizeof(float)));
		ctx->own3_elems = elems;
	}
	int rc = upload_u8_pair(ctx, ref, tar, elems, ctx->own_ref3, ctx->own_tar3);
	if (rc) return rc;
	return ocb_set_images_3d_dev(ctx, ctx->own_ref3, ctx->own_tar3, dim_x, dim_y, dim_z);
}

int ocb_set_images_3d_dev(ocb_ctx* ctx, const float* d_ref, const float* d_tar, int dim_x, int dim_y, int dim_z) {
	OCB_NO_GROUP(ctx, "set_images_3d_dev");
	if (!ctx || !d_ref || !d_tar || dim_x < 15 || dim_y < 15 || dim_z < 15) // TricubicBspline needs >= 15 (src/oc_cubic_bspline.cpp:201)
		return set_error(ctx, OCB_ERR_ARG, "set_images_3d: bad arguments (each dimension must be >= 15)");
	ctx->img3 = ocb::Image3D{ d_ref, d_tar, nullptr, nullptr, dim_x, dim_y, dim_z };
	ctx->prepared3 = false;
	return OCB_OK;
}

int ocb_set_images_3d(ocb_ctx* ctx, const float* ref, const float* tar, int dim_x, int dim_y, int dim_z) {
	if (is_group(ctx)) {
		if (ctx->peer_ok && ref && tar && dim_x >= 15 && dim_y >= 15 && dim_z >= 15) {
			int rc = group_distribute_pair(ctx, ref, tar, (size_t)dim_x * dim_y * dim_z, 3);
			if (rc) return rc;
			for (ocb_ctx* m : ctx->members)
				if ((rc = ocb_set_images_3d_dev(m, m->own_ref3, m->own_tar3, dim_x, dim_y, dim_z))) return rc;
			return OCB_OK;
		}
		return group_each(ctx, [=](ocb_ctx* m) { return ocb_set_images_3d(m, ref, tar, dim_x, dim_y, dim_z); });
	}
	if (!ctx || !ref || !tar || dim_x < 15 || dim_y < 15 || dim_z < 15)
		return set_error(ctx, OCB_ERR_ARG, "set_images_3d: bad arguments (each dimension must be >= 15)");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const size_t elems = (size_t)dim_x * dim_y * dim_z;
	if (elems > ctx->own3_elems) {
		cudaFree(ctx->own_ref3);
		cudaFree(ctx->own_tar3);
		ctx->own_ref3 = ctx->own_tar3 = nullptr;
		ctx->own3_elems = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_ref3, elems * sizeof(float)));
		OCB_CUDA(ctx, cudaMalloc(&ctx->own_tar3, elems * sizeof(float)));
		ctx->own3_elems = elems;
	}
	OCB_CUDA(ctx, cudaMemcpyAsync(ctx->own_ref3, ref, elems * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
	OCB_CUDA(ctx, cudaMemcpyAsync(ctx->own_tar3, tar, elems * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
	return ocb_set_images_3d_dev(ctx, ctx->own_ref3, ctx->own_tar3, dim_x, dim_y, dim_z);
}

// ---- FFT-CC ----------------------------------------------------------------------------------
int ocb_fftcc2d_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, int rx, int ry) {
	OCB_NO_GROUP(ctx, "fftcc2d_dev");
	if (!ctx || (!d_poi2d && n) || rx < 1 || ry < 1) return set_error(ctx, OCB_ERR_ARG, "fftcc2d: bad arguments");
	if (!ctx->img2.ref) return set_error(ctx, OCB_ERR_STATE, "fftcc2d: images not set");
	if (n == 0) return OCB_OK;
	if (n > 0x7fffffffull) return set_error(ctx, OCB_ERR_ARG, "fftcc2d: too many POIs in one call");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	if (rx == 16 && ry == 16 && !getenv("OCB_FFTCC2D_GENERIC")) { // specialised register-FFT kernel for the 32x32 window
		cudaError_t err32;
		int tma = 0;
		if (ocb::fftcc2d_w32_launch(ctx->img2, (float*)d_poi2d, n, ctx->sm_count, ctx->stream, &err32, &tma))
			return set_error(ctx, OCB_ERR_CUDA, "fftcc2d launch failed: %s", cudaGetErrorString(err32));
		ctx->launches++;
		record_launch(ctx, fftcc_info("fftcc2d", "w32", 32, tma));
		return OCB_OK;
	}
	if (rx == ry && ocb::fftcc2d_reg_supported(rx) && !getenv("OCB_FFTCC2D_GENERIC")) { // thread-per-row register FFTs, N = 2^a 3^b 5^c <= 64
		cudaError_t errr;
		if (ocb::fftcc2d_reg_launch(ctx->img2, (float*)d_poi2d, n, rx, ctx->sm_count, ctx->stream, &errr))
			return set_error(ctx, OCB_ERR_CUDA, "fftcc2d launch failed: %s", cudaGetErrorString(errr));
		ctx->launches++;
		record_launch(ctx, fftcc_info("fftcc2d", "reg", 2 * rx, 0));
		return OCB_OK;
	}
	ocb::FftAxis ax, ay;
	if (!ocb::fft_plan_axis(2 * rx, &ax) || !ocb::fft_plan_axis(2 * ry, &ay))
		return set_error(ctx, OCB_ERR_UNSUPPORTED, "fftcc2d: window size %dx%d has a prime factor > 31", 2 * rx, 2 * ry);
	if (ocb::fftcc2d_smem_bytes(rx, ry) > ctx->smem_optin)
		return set_error(ctx, OCB_ERR_UNSUPPORTED, "fftcc2d: %dx%d window needs %zu B of shared memory (> %zu)", 2 * rx, 2 * ry,
			ocb::fftcc2d_smem_bytes(rx, ry), ctx->smem_optin);
	const float2 *twx, *twy;
	int rc;
	if ((rc = get_twiddles(ctx, 2 * rx, &twx)) || (rc = get_twiddles(ctx, 2 * ry, &twy))) return rc;
	cudaError_t err;
	if (ocb::fftcc2d_launch(ctx->img2, (float*)d_poi2d, n, rx, ry, ax, ay, twx, twy, ctx->sm_count, ctx->stream, &err))
		return set_error(ctx, OCB_ERR_CUDA, "fftcc2d launch failed: %s", cudaGetErrorString(err));
	ctx->launches++;
	record_launch(ctx, fftcc_info("fftcc2d", "generic", 2 * rx, 0));
	return OCB_OK;
}

int ocb_fftcc2d(ocb_ctx* ctx, void* poi2d, size_t n, int rx, int ry) {
	if (is_group(ctx) && poi2d) return group_shard(ctx, poi2d, n, OCB_POI2D_FLOATS * sizeof(float), OCB_GROUP_MIN_2D, [=](ocb_ctx* m, void* q, size_t c, size_t) { return ocb_fftcc2d(m, q, c, rx, ry); });
	if (!ctx || (!poi2d && n)) return set_error(ctx, OCB_ERR_ARG, "fftcc2d: bad arguments");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	return run_host_queue_2d(ctx, poi2d, n, [&](float* d, size_t m, size_t) { return ocb_fftcc2d_dev(ctx, d, m, rx, ry); },
		rx == 16 && ry == 16 && !getenv("OCB_FFTCC2D_GENERIC"), ry > 0 ? ry : 0);
}

int ocb_fftcc3d_dev(ocb_ctx* ctx, void* d_poi3d, size_t n, int rx, int ry, int rz) {
	OCB_NO_GROUP(ctx, "fftcc3d_dev");
	if (!ctx || (!d_poi3d && n) || rx < 1 || ry < 1 || rz < 1) return set_error(ctx, OCB_ERR_ARG, "fftcc3d: bad arguments");
	if (!ctx->img3.ref) return set_error(ctx, OCB_ERR_STATE, "fftcc3d: images not set");
	if (n == 0) return OCB_OK;
	if (n > 0x7fffffffull) return set_error(ctx, OCB_ERR_ARG, "fftcc3d: too many POIs in one call");
	if ((size_t)8 * rx * ry * rz > 0x7fffffffull) return set_error(ctx, OCB_ERR_UNSUPPORTED, "fftcc3d: window too large");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	if (rx == 16 && ry == 16 && rz == 16 && !getenv("OCB_FFTCC3D_GENERIC")) { // specialised register-FFT kernel for the 32^3 window
		int grid32 = ocb::fftcc3d_w32_grid(ctx->sm_count);
		if ((size_t)grid32 > n) grid32 = (int)n;
		const size_t need32 = (size_t)grid32 * 32768;
		if (need32 > ctx->fft_scratch_elems) {
			OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
			cudaFree(ctx->fft_scratch);
			ctx->fft_scratch = nullptr;
			ctx->fft_scratch_elems = 0;
			OCB_CUDA(ctx, cudaMalloc(&ctx->fft_scratch, need32 * sizeof(float2)));
			ctx->fft_scratch_elems = need32;
		}
		cudaError_t err32;
		int tma = 0;
		if (ocb::fftcc3d_w32_launch(ctx->img3, (float*)d_poi3d, n, ctx->fft_scratch, grid32, ctx->stream, &err32, &tma))
			return set_error(ctx, OCB_ERR_CUDA, "fftcc3d launch failed: %s", cudaGetErrorString(err32));
		ctx->launches++;
		record_launch(ctx, fftcc_info("fftcc3d", "w32", 32, tma));
		return OCB_OK;
	}
	if (rx == ry && ry == rz && ocb::fftcc3d_reg_supported(rx) && !getenv("OCB_FFTCC3D_GENERIC")) { // register FFT codelets, N = 2^a 3^b 5^c <= 64
		int gridr = ocb::fftcc3d_reg_grid(rx, ctx->sm_count);
		if ((size_t)gridr > n) gridr = (int)n;
		const size_t needr = (size_t)gridr * 2 * 8 * rx * ry * rz; // two scratch volumes of (2r)^3 complex per CTA
		if (needr > ctx->fft_scratch_elems) {
			OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
			cudaFree(ctx->fft_scratch);
			ctx->fft_scratch = nullptr;
			ctx->fft_scratch_elems = 0;
			OCB_CUDA(ctx, cudaMalloc(&ctx->fft_scratch, needr * sizeof(float2)));
			ctx->fft_scratch_elems = needr;
		}
		cudaError_t errr;
		if (ocb::fftcc3d_reg_launch(ctx->img3, (float*)d_poi3d, n, rx, ctx->fft_scratch, gridr, ctx->stream, &errr))
			return set_error(ctx, OCB_ERR_CUDA, "fftcc3d launch failed: %s", cudaGetErrorString(errr));
		ctx->launches++;
		record_launch(ctx, fftcc_info("fftcc3d", "reg", 2 * rx, 0));
		return OCB_OK;
	}
	ocb::FftAxis ax, ay, az;
	if (!ocb::fft_plan_axis(2 * rx, &ax) || !ocb::fft_plan_axis(2 * ry, &ay) || !ocb::fft_plan_axis(2 * rz, &az))
		return set_error(ctx, OCB_ERR_UNSUPPORTED, "fftcc3d: window size has a prime factor > 31");
	if (ocb::fftcc3d_smem_bytes(rx, ry, rz) > ctx->smem_optin)
		return set_error(ctx, OCB_ERR_UNSUPPORTED, "fftcc3d: window needs %zu B of shared memory (> %zu)", ocb::fftcc3d_smem_bytes(rx, ry, rz),
			ctx->smem_optin);
	const float2 *twx, *twy, *twz;
	int rc;
	if ((rc = get_twiddles(ctx, 2 * rx, &twx)) || (rc = get_twiddles(ctx, 2 * ry, &twy)) || (rc = get_twiddles(ctx, 2 * rz, &twz))) return rc;
	int grid = ocb::fftcc3d_grid(rx, ry, rz, ctx->sm_count);
	if ((size_t)grid > n) grid = (int)n;
	const size_t need = (size_t)grid * 8 * rx * ry * rz;
	if (need > ctx->fft_scratch_elems) {
		OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		cudaFree(ctx->fft_scratch);
		ctx->fft_scratch = nullptr;
		ctx->fft_scratch_elems = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->fft_scratch, need * sizeof(float2)));
		ctx->fft_scratch_elems = need;
	}
	cudaError_t err;
	if (ocb::fftcc3d_launch(ctx->img3, (float*)d_poi3d, n, rx, ry, rz, ax, ay, az, twx, twy, twz, ctx->fft_scratch, grid, ctx->stream, &err))
		return set_error(ctx, OCB_ERR_CUDA, "fftcc3d launch failed: %s", cudaGetErrorString(err));
	ctx->launches++;
	record_launch(ctx, fftcc_info("fftcc3d", "generic", 2 * rx, 0));
	return OCB_OK;
}

int ocb_fftcc3d(ocb_ctx* ctx, void* poi3d, size_t n, int rx, int ry, int rz) {
	if (is_group(ctx) && poi3d) return group_shard(ctx, poi3d, n, OCB_POI3D_FLOATS * sizeof(float), OCB_GROUP_MIN_3D, [=](ocb_ctx* m, void* q, size_t c, size_t) { return ocb_fftcc3d(m, q, c, rx, ry, rz); });
	if (!ctx || (!poi3d && n)) return set_error(ctx, OCB_ERR_ARG, "fftcc3d: bad arguments");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	int rc;
	const size_t bytes = n * OCB_POI3D_FLOATS * sizeof(float);
	if ((rc = stage_pois(ctx, poi3d, bytes))) return rc;
	if ((rc = ocb_fftcc3d_dev(ctx, ctx->d_poi, n, rx, ry, rz))) return rc;
	return unstage_pois(ctx, poi3d, bytes);
}

// ---- IC-GN -----------------------------------------------------------------------------------
int ocb_icgn2d_prepare(ocb_ctx* ctx) {
	if (is_group(ctx)) { // flag only: no need to wake the members' threads
		for (ocb_ctx* m : ctx->members) {
			const int rc = ocb_icgn2d_prepare(m);
			if (rc) { ctx->last_error = m->last_error; return rc; }
		}
		return OCB_OK;
	}
	if (!ctx) return set_error(nullptr, OCB_ERR_ARG, "null context");
	if (!ctx->img2.ref) return set_error(ctx, OCB_ERR_STATE, "icgn2d_prepare: images not set");
	ctx->prepared2 = true; // gradients and bicubic weights are recomputed on chip per POI
	return OCB_OK;
}

static int icgn2d_dev(ocb_ctx* ctx, int np, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop, const float* d_offsets = nullptr,
	const float* lm_damping = nullptr) {
	OCB_NO_GROUP(ctx, "icgn2d_dev");
	if (!ctx || (!d_poi2d && n) || rx < 1 || ry < 1) return set_error(ctx, OCB_ERR_ARG, "icgn2d: bad arguments");
	if (!ctx->img2.ref) return set_error(ctx, OCB_ERR_STATE, "icgn2d: images not set");
	if (!ctx->prepared2) return set_error(ctx, OCB_ERR_STATE, "icgn2d: prepare() has not been called since setImages()");
	if (n == 0) return OCB_OK;
	if (n > 0x7fffffffull) return set_error(ctx, OCB_ERR_ARG, "icgn2d: too many POIs in one call");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	cudaError_t err = cudaSuccess;
	ocb::LaunchInfo li;
	int rc = ocb::icgn2d_launch(np, ctx->img2, (float*)d_poi2d, n, rx, ry, conv, stop, ctx->sm_count, ctx->smem_optin, ctx->d_counter, d_offsets, lm_damping,
		ctx->stream, &err, &li);
	if (rc == -1) return set_error(ctx, OCB_ERR_UNSUPPORTED, "icgn2d: subset radius (%d,%d) exceeds the shared-memory design limit", rx, ry);
	if (rc) return set_error(ctx, OCB_ERR_CUDA, "icgn2d launch failed: %s", cudaGetErrorString(err));
	ctx->launches++;
	record_launch(ctx, li);
	return OCB_OK;
}

int ocb_icgn2d1_dev(ocb_ctx* ctx, void* d, size_t n, int rx, int ry, float conv, float stop) { return icgn2d_dev(ctx, 6, d, n, rx, ry, conv, stop); }
int ocb_icgn2d2_dev(ocb_ctx* ctx, void* d, size_t n, int rx, int ry, float conv, float stop) { return icgn2d_dev(ctx, 12, d, n, rx, ry, conv, stop); }

static int icgn2d_host(ocb_ctx* ctx, int np, void* poi2d, size_t n, int rx, int ry, float conv, float stop) {
	if (is_group(ctx) && poi2d) return group_shard(ctx, poi2d, n, OCB_POI2D_FLOATS * sizeof(float), OCB_GROUP_MIN_2D, [=](ocb_ctx* m, void* q, size_t c, size_t) { return icgn2d_host(m, np, q, c, rx, ry, conv, stop); });
	if (!ctx || (!poi2d && n)) return set_error(ctx, OCB_ERR_ARG, "icgn2d: bad arguments");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	return run_host_queue_2d(ctx, poi2d, n, [&](float* d, size_t m, size_t) { return icgn2d_dev(ctx, np, d, m, rx, ry, conv, stop); }, true);
}
int ocb_icgn2d1(ocb_ctx* ctx, void* p, size_t n, int rx, int ry, float conv, float stop) { return icgn2d_host(ctx, 6, p, n, rx, ry, conv, stop); }
int ocb_icgn2d2(ocb_ctx* ctx, void* p, size_t n, int rx, int ry, float conv, float stop) { return icgn2d_host(ctx, 12, p, n, rx, ry, conv, stop); }

int ocb_icgn2d_ex_dev(ocb_ctx* ctx, int order, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop, const float* d_center_offsets) {
	if (order != 1 && order != 2) return set_error(ctx, OCB_ERR_ARG, "icgn2d_ex: order must be 1 or 2");
	return icgn2d_dev(ctx, order == 1 ? 6 : 12, d_poi2d, n, rx, ry, conv, stop, d_center_offsets);
}

// one launch over a host queue (all POIs share the radius), optional host offsets
static int icgn2d_host_group(ocb_ctx* ctx, int np, float* poi2d, size_t n, int rx, int ry, float conv, float stop, const float* offsets) {
	const float* d_off = nullptr;
	if (offsets) {
		const size_t ob = n * 2 * sizeof(float);
		if (ob > ctx->d_off_bytes) {
			cudaFree(ctx->d_off);
			ctx->d_off = nullptr;
			ctx->d_off_bytes = 0;
			OCB_CUDA(ctx, cudaMalloc(&ctx->d_off, ob));
			ctx->d_off_bytes = ob;
		}
		OCB_CUDA(ctx, cudaMemcpyAsync(ctx->d_off, offsets, ob, cudaMemcpyHostToDevice, ctx->stream));
		d_off = ctx->d_off;
	}
	return run_host_queue_2d(ctx, poi2d, n,
		[&](float* d, size_t m, size_t first) { return icgn2d_dev(ctx, np, d, m, rx, ry, conv, stop, d_off ? d_off + 2 * first : nullptr); }, true);
}

int ocb_icgn2d_ex(ocb_ctx* ctx, int order, void* poi2d, size_t n, int rx, int ry, float conv, float stop, const float* center_offsets,
	int self_adaptive) {
	if (is_group(ctx) && poi2d)
		return group_shard(ctx, poi2d, n, OCB_POI2D_FLOATS * sizeof(float), OCB_GROUP_MIN_2D, [=](ocb_ctx* m, void* q, size_t c, size_t first) {
			return ocb_icgn2d_ex(m, order, q, c, rx, ry, conv, stop, center_offsets ? center_offsets + 2 * first : nullptr, self_adaptive);
		});
	if (!ctx || (!poi2d && n)) return set_error(ctx, OCB_ERR_ARG, "icgn2d_ex: bad arguments");
	if (order != 1 && order != 2) return set_error(ctx, OCB_ERR_ARG, "icgn2d_ex: order must be 1 or 2");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const int np = order == 1 ? 6 : 12;
	float* q = (float*)poi2d;
	if (!self_adaptive) return icgn2d_host_group(ctx, np, q, n, rx, ry, conv, stop, center_offsets);
	// self-adaptive: group the POIs by their own (subset_radius.x, subset_radius.y); one launch per group
	std::map<std::pair<int, int>, std::vector<size_t>> groups;
	for (size_t i = 0; i < n; i++) {
		const float* p = q + i * OCB_POI2D_FLOATS;
		groups[std::make_pair((int)p[23], (int)p[24])].push_back(i);
	}
	for (auto& kv : groups) // refuse before anything is launched: no partial results
		if (kv.first.first >= 1 && kv.first.second >= 1
			&& (size_t)ocb::icgn2d_slab_bytes(kv.first.first, kv.first.second) > ctx->smem_optin)
			return set_error(ctx, OCB_ERR_UNSUPPORTED, "icgn2d_ex: subset radius (%d,%d) of a self-adaptive POI exceeds the shared-memory design limit",
				kv.first.first, kv.first.second);
	std::vector<float> gq, goff;
	for (auto& kv : groups) {
		const int grx = kv.first.first, gry = kv.first.second;
		const std::vector<size_t>& idx = kv.second;
		if (grx < 1 || gry < 1) { // the reference would size its scratch from a radius < 1 (undefined); reject like a failed guard
			for (size_t i : idx)
				if (q[i * OCB_POI2D_FLOATS + 16] >= 0) q[i * OCB_POI2D_FLOATS + 16] = -3.f;
			continue;
		}
		gq.resize(idx.size() * OCB_POI2D_FLOATS);
		for (size_t k = 0; k < idx.size(); k++) memcpy(&gq[k * OCB_POI2D_FLOATS], q + idx[k] * OCB_POI2D_FLOATS, OCB_POI2D_FLOATS * sizeof(float));
		const float* off = nullptr;
		if (center_offsets) {
			goff.resize(idx.size() * 2);
			for (size_t k = 0; k < idx.size(); k++) { goff[2 * k] = center_offsets[2 * idx[k]]; goff[2 * k + 1] = center_offsets[2 * idx[k] + 1]; }
			off = goff.data();
		}
		int rc = icgn2d_host_group(ctx, np, gq.data(), idx.size(), grx, gry, conv, stop, off);
		if (rc) return rc;
		for (size_t k = 0; k < idx.size(); k++) memcpy(q + idx[k] * OCB_POI2D_FLOATS, &gq[k * OCB_POI2D_FLOATS], OCB_POI2D_FLOATS * sizeof(float));
	}
	return OCB_OK;
}

// ---- ICLM (SURVEY.md section 8(f) N2) ----------------------------------------------------------------
int ocb_iclm2d_dev(ocb_ctx* ctx, int order, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop, float lambda, float alpha, float beta) {
	if (order != 1 && order != 2) return set_error(ctx, OCB_ERR_ARG, "iclm2d: order must be 1 or 2");
	const float damping[3] = { lambda, alpha, beta };
	return icgn2d_dev(ctx, order == 1 ? 6 : 12, d_poi2d, n, rx, ry, conv, stop, nullptr, damping);
}

int ocb_iclm2d(ocb_ctx* ctx, int order, void* poi2d, size_t n, int rx, int ry, float conv, float stop, float lambda, float alpha, float beta) {
	if (is_group(ctx) && poi2d)
		return group_shard(ctx, poi2d, n, OCB_POI2D_FLOATS * sizeof(float), OCB_GROUP_MIN_2D,
			[=](ocb_ctx* m, void* q, size_t c, size_t) { return ocb_iclm2d(m, order, q, c, rx, ry, conv, stop, lambda, alpha, beta); });
	if (!ctx || (!poi2d && n)) return set_error(ctx, OCB_ERR_ARG, "iclm2d: bad arguments");
	if (order != 1 && order != 2) return set_error(ctx, OCB_ERR_ARG, "iclm2d: order must be 1 or 2");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	return run_host_queue_2d(ctx, poi2d, n,
		[&](float* d, size_t m, size_t) { return ocb_iclm2d_dev(ctx, order, d, m, rx, ry, conv, stop, lambda, alpha, beta); }, true);
}

// ---- NR2D1 (SURVEY.md section 8(f) N2) ---------------------------------------------------------------
int ocb_nr2d_prepare(ocb_ctx* ctx) {
	if (is_group(ctx)) {
		for (ocb_ctx* m : ctx->members) {
			const int rc = ocb_nr2d_prepare(m);
			if (rc) { ctx->last_error = m->last_error; return rc; }
		}
		return OCB_OK;
	}
	if (!ctx) return set_error(nullptr, OCB_ERR_ARG, "null context");
	if (!ctx->img2.ref) return set_error(ctx, OCB_ERR_STATE, "nr2d_prepare: images not set");
	ctx->prepared_nr2 = true; // target gradients and the three interpolants are evaluated on chip per POI
	return OCB_OK;
}

int ocb_nr2d1_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop) {
	OCB_NO_GROUP(ctx, "nr2d1_dev");
	if (!ctx || (!d_poi2d && n) || rx < 1 || ry < 1) return set_error(ctx, OCB_ERR_ARG, "nr2d1: bad arguments");
	if (!ctx->img2.ref) return set_error(ctx, OCB_ERR_STATE, "nr2d1: images not set");
	if (!ctx->prepared_nr2) return set_error(ctx, OCB_ERR_STATE, "nr2d1: prepare() has not been called since setImages()");
	if (n == 0) return OCB_OK;
	if (n > 0x7fffffffull) return set_error(ctx, OCB_ERR_ARG, "nr2d1: too many POIs in one call");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	cudaError_t err = cudaSuccess;
	int rc = ocb::nr2d1_launch(ctx->img2, (float*)d_poi2d, n, rx, ry, conv, stop, ctx->sm_count, ctx->smem_optin, ctx->d_counter, ctx->stream, &err);
	if (rc == -1) return set_error(ctx, OCB_ERR_UNSUPPORTED, "nr2d1: subset radius (%d,%d) exceeds the shared-memory design limit", rx, ry);
	if (rc) return set_error(ctx, OCB_ERR_CUDA, "nr2d1 launch failed: %s", cudaGetErrorString(err));
	ctx->launches++;
	return OCB_OK;
}

int ocb_nr2d1(ocb_ctx* ctx, void* poi2d, size_t n, int rx, int ry, float conv, float stop) {
	if (is_group(ctx) && poi2d) return group_shard(ctx, poi2d, n, OCB_POI2D_FLOATS * sizeof(float), OCB_GROUP_MIN_2D, [=](ocb_ctx* m, void* q, size_t c, size_t) { return ocb_nr2d1(m, q, c, rx, ry, conv, stop); });
	if (!ctx || (!poi2d && n)) return set_error(ctx, OCB_ERR_ARG, "nr2d1: bad arguments");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	return run_host_queue_2d(ctx, poi2d, n, [&](float* d, size_t m, size_t) { return ocb_nr2d1_dev(ctx, d, m, rx, ry, conv, stop); });
}

// ---- EpipolarSearch candidate sweep (SURVEY.md section 8(f) N4) ----------------------------------------
int ocb_epipolar_search2d_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, const float* fundamental, const float* parallax_x, const float* parallax_y,
	int search_radius, int search_step, int rx, int ry, float conv, float stop) {
	OCB_NO_GROUP(ctx, "epipolar_search2d_dev");
	if (!ctx || (!d_poi2d && n) || !fundamental || !parallax_x || !parallax_y || rx < 1 || ry < 1)
		return set_error(ctx, OCB_ERR_ARG, "epipolar_search2d: bad arguments");
	if (search_step < 1 || search_radius < search_step)
		return set_error(ctx, OCB_ERR_ARG, "epipolar_search2d: search radius is less than search step"); // EpipolarSearch::setSearch, src/oc_epipolar_search.cpp:44-53
	if (!ctx->img2.ref) return set_error(ctx, OCB_ERR_STATE, "epipolar_search2d: images not set");
	if (!ctx->prepared2) return set_error(ctx, OCB_ERR_STATE, "epipolar_search2d: prepare() has not been called since setImages()");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const int slots = ocb::epipolar_slots(search_radius, search_step);
	// candidates of a block of POIs at a time: at most ~2^22 records (420 MB) in flight
	size_t block = ((size_t)1 << 22) / (size_t)slots;
	if (block < 1) block = 1;
	if (block > n) block = n;
	const size_t need = block * (size_t)slots * OCB_POI2D_FLOATS * sizeof(float);
	if (need > ctx->d_cand_bytes) {
		if (ctx->d_cand) cudaFree(ctx->d_cand);
		ctx->d_cand = nullptr;
		ctx->d_cand_bytes = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->d_cand, need));
		ctx->d_cand_bytes = need;
	}
	for (size_t p0 = 0; p0 < n; p0 += block) {
		const size_t nb = n - p0 < block ? n - p0 : block;
		ocb::epipolar_candidates_launch((const float*)d_poi2d, p0, nb, fundamental, parallax_x, parallax_y, search_radius, search_step, rx, ry, ctx->img2.w,
			ctx->img2.h, slots, ctx->d_cand, ctx->sm_count, ctx->stream);
		OCB_CUDA(ctx, cudaGetLastError());
		ctx->launches++;
		int rc = icgn2d_dev(ctx, 6, ctx->d_cand, nb * (size_t)slots, rx, ry, conv, stop);
		if (rc) return rc;
		ocb::epipolar_select_launch((float*)d_poi2d, p0, nb, slots, ctx->d_cand, ctx->sm_count, ctx->stream);
		OCB_CUDA(ctx, cudaGetLastError());
		ctx->launches++;
	}
	return OCB_OK;
}

int ocb_epipolar_search2d(ocb_ctx* ctx, void* poi2d, size_t n, const float* fundamental, const float* parallax_x, const float* parallax_y,
	int search_radius, int search_step, int rx, int ry, float conv, float stop) {
	if (is_group(ctx) && poi2d)
		return group_shard(ctx, poi2d, n, OCB_POI2D_FLOATS * sizeof(float), 256, [=](ocb_ctx* m, void* q, size_t c, size_t) {
			return ocb_epipolar_search2d(m, q, c, fundamental, parallax_x, parallax_y, search_radius, search_step, rx, ry, conv, stop);
		});
	if (!ctx || (!poi2d && n)) return set_error(ctx, OCB_ERR_ARG, "epipolar_search2d: bad arguments");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	int rc;
	const size_t bytes = n * OCB_POI2D_FLOATS * sizeof(float);
	if ((rc = stage_pois(ctx, poi2d, bytes))) return rc;
	if ((rc = ocb_epipolar_search2d_dev(ctx, ctx->d_poi, n, fundamental, parallax_x, parallax_y, search_radius, search_step, rx, ry, conv, stop))) return rc;
	return unstage_pois(ctx, poi2d, bytes);
}

// ---- Strain (SURVEY.md section 8(f) N4) ---------------------------------------------------------------
static int strain_dev(ocb_ctx* ctx, int dim, void* d_poi, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation,
	long long only = -1) {
	OCB_NO_GROUP(ctx, "strain_dev");
	if (!ctx || (!d_poi && n) || only >= (long long)n) return set_error(ctx, OCB_ERR_ARG, "strain: bad arguments");
	if (n == 0) return OCB_OK;
	if (n > 0x7fffffffull) return set_error(ctx, OCB_ERR_ARG, "strain: too many POIs in one call");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const size_t need = ocb::strain_workspace_bytes(n);
	if (need > ctx->d_strain_ws_bytes) {
		if (ctx->d_strain_ws) cudaFree(ctx->d_strain_ws);
		ctx->d_strain_ws = nullptr;
		ctx->d_strain_ws_bytes = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->d_strain_ws, need));
		ctx->d_strain_ws_bytes = need;
	}
	cudaError_t err = cudaSuccess;
	int rc = ocb::strain_launch(dim, (float*)d_poi, n, radius, min_neighbors, zncc_threshold, approximation, only, ctx->d_strain_ws, ctx->sm_count, ctx->stream,
		&err, &ctx->launches);
	if (rc) return set_error(ctx, OCB_ERR_CUDA, "strain launch failed: %s", cudaGetErrorString(err));
	return OCB_OK;
}

static int strain_host(ocb_ctx* ctx, int dim, void* poi, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation,
	long long only = -1) {
	if (is_group(ctx)) { // every POI needs its neighbours wherever they are in the queue: not sharded, the first member runs it
		const int rc = strain_host(ctx->members[0], dim, poi, n, radius, min_neighbors, zncc_threshold, approximation, only);
		if (rc) ctx->last_error = ctx->members[0]->last_error;
		return rc;
	}
	if (!ctx || (!poi && n)) return set_error(ctx, OCB_ERR_ARG, "strain: bad arguments");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	int rc;
	const size_t bytes = n * (dim == 2 ? OCB_POI2D_FLOATS : (dim == 3 ? OCB_POI3D_FLOATS : OCB_POI2DS_FLOATS)) * sizeof(float);
	if ((rc = stage_pois(ctx, poi, bytes))) return rc;
	if ((rc = strain_dev(ctx, dim, ctx->d_poi, n, radius, min_neighbors, zncc_threshold, approximation, only))) return rc;
	return unstage_pois(ctx, poi, bytes);
}

int ocb_strain2d(ocb_ctx* ctx, void* poi2d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_host(ctx, 2, poi2d, n, radius, min_neighbors, zncc_threshold, approximation);
}
int ocb_strain3d(ocb_ctx* ctx, void* poi3d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_host(ctx, 3, poi3d, n, radius, min_neighbors, zncc_threshold, approximation);
}
int ocb_strain2ds(ocb_ctx* ctx, void* poi2ds, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_host(ctx, 23, poi2ds, n, radius, min_neighbors, zncc_threshold, approximation);
}
int ocb_strain2ds_dev(ocb_ctx* ctx, void* d_poi2ds, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_dev(ctx, 23, d_poi2ds, n, radius, min_neighbors, zncc_threshold, approximation);
}
int ocb_strain2d_single(ocb_ctx* ctx, void* poi2d, size_t n, size_t index, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_host(ctx, 2, poi2d, n, radius, min_neighbors, zncc_threshold, approximation, (long long)index);
}
int ocb_strain3d_single(ocb_ctx* ctx, void* poi3d, size_t n, size_t index, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_host(ctx, 3, poi3d, n, radius, min_neighbors, zncc_threshold, approximation, (long long)index);
}
int ocb_strain2d_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_dev(ctx, 2, d_poi2d, n, radius, min_neighbors, zncc_threshold, approximation);
}
int ocb_strain3d_dev(ocb_ctx* ctx, void* d_poi3d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation) {
	return strain_dev(ctx, 3, d_poi3d, n, radius, min_neighbors, zncc_threshold, approximation);
}

int ocb_icgn3d_prepare(ocb_ctx* ctx) {
	if (is_group(ctx)) return group_each(ctx, [](ocb_ctx* m) { return ocb_icgn3d_prepare(m); });
	if (!ctx) return set_error(nullptr, OCB_ERR_ARG, "null context");
	if (!ctx->img3.ref) return set_error(ctx, OCB_ERR_STATE, "icgn3d_prepare: images not set");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const int dx = ctx->img3.dx, dy = ctx->img3.dy, dz = ctx->img3.dz;
	const size_t elems = (size_t)dx * dy * dz;
	if (elems > ctx->tab3_elems) {
		cudaFree(ctx->rg3);
		cudaFree(ctx->coef3);
		cudaFree(ctx->tmp3);
		ctx->rg3 = nullptr;
		ctx->coef3 = ctx->tmp3 = nullptr;
		ctx->tab3_elems = 0;
		OCB_CUDA(ctx, cudaMalloc(&ctx->rg3, elems * sizeof(float4)));
		OCB_CUDA(ctx, cudaMalloc(&ctx->coef3, elems * sizeof(float)));
		OCB_CUDA(ctx, cudaMalloc(&ctx->tmp3, elems * sizeof(float)));
		ctx->tab3_elems = elems;
	}
	ocb::gradient3d_launch(ctx->img3.ref, ctx->rg3, dx, dy, dz, ctx->sm_count, ctx->stream);
	// TricubicBspline::prepare: x -> coefficient, y -> conv_buffer, z -> coefficient
	ocb::prefilter3d_launch(ctx->img3.tar, ctx->coef3, dx, dy, dz, 0, ctx->sm_count, ctx->stream);
	ocb::prefilter3d_launch(ctx->coef3, ctx->tmp3, dx, dy, dz, 1, ctx->sm_count, ctx->stream);
	ocb::prefilter3d_launch(ctx->tmp3, ctx->coef3, dx, dy, dz, 2, ctx->sm_count, ctx->stream);
	ctx->launches += 4;
	OCB_CUDA(ctx, cudaGetLastError());
	ctx->img3.rg = ctx->rg3;
	ctx->img3.coef = ctx->coef3;
	ctx->prepared3 = true;
	return OCB_OK;
}

int ocb_icgn3d1_dev(ocb_ctx* ctx, void* d_poi3d, size_t n, int rx, int ry, int rz, float conv, float stop) {
	OCB_NO_GROUP(ctx, "icgn3d1_dev");
	if (!ctx || (!d_poi3d && n) || rx < 1 || ry < 1 || rz < 1) return set_error(ctx, OCB_ERR_ARG, "icgn3d1: bad arguments");
	if (!ctx->img3.ref) return set_error(ctx, OCB_ERR_STATE, "icgn3d1: images not set");
	if (!ctx->prepared3) return set_error(ctx, OCB_ERR_STATE, "icgn3d1: prepare() has not been called since setImages()");
	if (n == 0) return OCB_OK;
	if (n > 0x7fffffffull) return set_error(ctx, OCB_ERR_ARG, "icgn3d1: too many POIs in one call");
	if ((size_t)(2 * rx + 1) * (2 * ry + 1) * (2 * rz + 1) > 0x3fffffffull) return set_error(ctx, OCB_ERR_UNSUPPORTED, "icgn3d1: subset too large");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	cudaError_t err = cudaSuccess;
	ocb::LaunchInfo li;
	const int rc3 = ocb::icgn3d1_launch(ctx->img3, (float*)d_poi3d, n, rx, ry, rz, conv, stop, ctx->sm_count, ctx->smem_optin, ctx->d_counter + 1,
		ctx->stream, &err, &li);
	if (rc3 == -1) return set_error(ctx, OCB_ERR_UNSUPPORTED, "icgn3d1: subset radius (%d,%d,%d) exceeds the shared-memory design limit", rx, ry, rz);
	if (rc3) return set_error(ctx, OCB_ERR_CUDA, "icgn3d1 launch failed: %s", cudaGetErrorString(err));
	ctx->launches++;
	record_launch(ctx, li);
	return OCB_OK;
}

int ocb_icgn3d1(ocb_ctx* ctx, void* poi3d, size_t n, int rx, int ry, int rz, float conv, float stop) {
	if (is_group(ctx) && poi3d) return group_shard(ctx, poi3d, n, OCB_POI3D_FLOATS * sizeof(float), OCB_GROUP_MIN_3D, [=](ocb_ctx* m, void* q, size_t c, size_t) { return ocb_icgn3d1(m, q, c, rx, ry, rz, conv, stop); });
	if (!ctx || (!poi3d && n)) return set_error(ctx, OCB_ERR_ARG, "icgn3d1: bad arguments");
	if (n == 0) return OCB_OK;
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	int rc;
	const size_t bytes = n * OCB_POI3D_FLOATS * sizeof(float);
	if ((rc = stage_pois(ctx, poi3d, bytes))) return rc;
	if ((rc = ocb_icgn3d1_dev(ctx, ctx->d_poi, n, rx, ry, rz, conv, stop))) return rc;
	return unstage_pois(ctx, poi3d, bytes);
}

int ocb_get_tables_3d(ocb_ctx* ctx, float* gx, float* gy, float* gz, float* coefficient) {
	if (is_group(ctx)) return ocb_get_tables_3d(ctx->members[0], gx, gy, gz, coefficient);
	if (!ctx) return set_error(nullptr, OCB_ERR_ARG, "null context");
	if (!ctx->prepared3) return set_error(ctx, OCB_ERR_STATE, "get_tables_3d: prepare() has not been called");
	if (ensure_device(ctx)) return OCB_ERR_CUDA;
	const size_t elems = (size_t)ctx->img3.dx * ctx->img3.dy * ctx->img3.dz;
	float* dst[3] = { gx, gy, gz };
	for (int i = 0; i < 3; i++) // de-interleave component i+1 of the packed {ref, gx, gy, gz} volume (inspection path, not hot)
		if (dst[i])
			OCB_CUDA(ctx, cudaMemcpy2DAsync(dst[i], sizeof(float), (const float*)ctx->rg3 + (i + 1), sizeof(float4), sizeof(float), elems,
				cudaMemcpyDeviceToHost, ctx->stream));
	if (coefficient) OCB_CUDA(ctx, cudaMemcpyAsync(coefficient, ctx->coef3, elems * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
	OCB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return OCB_OK;
}

} // extern "C"
