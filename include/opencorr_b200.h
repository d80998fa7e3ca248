/*
 * opencorr_b200.h -- C ABI of the B200-native FFT-CC -> IC-GN correlation engine.
 *
 * This is the drop-in boundary for ONE hot path of vincentjzy/OpenCorr: the per-POI
 * FFT-CC integer-pixel initial guess followed by inverse-compositional Gauss-Newton
 * registration.  Every entry point names the reference interface it replaces
 * (paths relative to the reference repo root).  Plain pointers and sizes only; no
 * C++/torch types.  The C++ shim in include/opencorr/ (same class names as the
 * reference) and the Python mirror in opencorr_b200/ are thin layers over this file.
 *
 * Conventions
 *   - POI arrays are the reference's own records, passed verbatim:
 *       POI2D  (src/oc_poi.h:102-136) = 25 floats / 100 bytes
 *         { x, y | u ux uy uxx uxy uyy v vx vy vxx vxy vyy | u0 v0 zncc iteration
 *           convergence feature | exx eyy exy | subset_radius.x subset_radius.y }
 *       POI3D  (src/oc_poi.h:187-222) = 31 floats / 124 bytes
 *         { x, y, z | u ux uy uz v vx vy vz w wx wy wz | u0 v0 w0 zncc iteration
 *           convergence feature | e[6] | subset_radius.x .y .z }
 *     They are mutated in place exactly as the reference's compute(std::vector<POI>&) does,
 *     including the sentinel ZNCC codes of src/oc_dic.h:28-34 (-3 rejected / left the image,
 *     -4 not converged, -5 NaN; a POI arriving with zncc < 0 is skipped).
 *   - Images: float32.  2D row-major [height][width] (col_major=1 accepts the reference's
 *     Eigen::MatrixXf storage, src/oc_image.h:36); volumes [z][y][x] contiguous, the payload
 *     of the reference's float*** (src/oc_array.h:56-74).
 *   - Every function returns OCB_OK (0) or a negative OCB_ERR_* code; the message is
 *     available from ocb_last_error().  There is NO CPU fallback: without a usable CUDA
 *     device ocb_create() fails (returns NULL) and says why.
 *   - Functions taking host POI arrays copy host->device, run, copy back and synchronise
 *     (the reference's blocking compute()); a page-locked array (cudaHostAlloc, ocb_host_alloc,
 *     ocb_host_register) is not copied by the 2D FFT-CC (r = 16) / IC-GN / IC-LM calls: the kernels
 *     read and write the caller's records in place.  The *_dev variants take a device pointer,
 *     enqueue on the context's stream and return without synchronising.
 *   - ocb_set_images_* return once the copies are enqueued: the host images must stay valid and
 *     unchanged until the next call that synchronises (any host-queue call, or ocb_sync()).
 *   - A context (single-device or group) is not to be used from two host threads at the same time.
 */
#ifndef OPENCORR_B200_H_
#define OPENCORR_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCB_OK 0
#define OCB_ERR_CUDA (-1)        /* CUDA runtime / driver error (message has the CUDA string) */
#define OCB_ERR_ARG (-2)         /* bad argument (null pointer, radius < 1, size mismatch ...) */
#define OCB_ERR_STATE (-3)       /* call order: images not set / prepare() not called */
#define OCB_ERR_UNSUPPORTED (-4) /* subset too large for the on-chip design (see DESIGN.md) */

#define OCB_POI2D_FLOATS 25
#define OCB_POI3D_FLOATS 31
#define OCB_POI2DS_FLOATS 28 /* stereo-DIC record, src/oc_poi.h:140-186 */

typedef struct ocb_ctx ocb_ctx;

/* ---- context ------------------------------------------------------------------------------ */
/* Number of CUDA devices visible, or a negative OCB_ERR_CUDA. */
int ocb_device_count(void);
/* One context = one GPU + one stream + the device copies the reference keeps per DIC/DVC
 * object (images, gradient / B-spline tables, scratch).  Replaces the constructors
 * FFTCC2D/FFTCC3D (src/oc_fftcc.cpp:151-163,300-313) and ICGN2D1/ICGN2D2/ICGN3D1
 * (src/oc_icgn.cpp:71-88,612-629,1197-1215): no per-thread pools are needed on the GPU.
 * Returns NULL on failure (see ocb_last_error(NULL)). */
ocb_ctx* ocb_create(int device);
/* Several devices behind ONE context (SURVEY.md section 8(e): one process, G devices): ocb_create(-1) takes every visible
 * device, ocb_create_multi() the listed ones.  A GROUP context replaces what the reference does with its OpenMP loop over
 * the POI queue, FFTCC2D::compute(std::vector<POI2D>&) src/oc_fftcc.cpp:277-285, ICGN2D1::compute(std::vector<POI2D>&)
 * src/oc_icgn.cpp:343-351 (and the siblings): setImages() uploads the pair to every member, each over its own PCIe link;
 * prepare() runs on every member; every host-queue compute() call splits the caller's array into contiguous blocks
 * (member i gets records [n*i/G, n*(i+1)/G)), and each member copies ITS block in, registers it and copies it back
 * straight into the caller's array, concurrently (one host thread per member).  Results are bit-identical to a
 * single-device context (the POIs are independent).  Queues too short to fill G devices use fewer of them.  Strain needs
 * every POI's neighbours and runs on the first member.  The *_dev / stream entry points need a single-device context:
 * use ocb_member(). */
ocb_ctx* ocb_create_multi(const int* devices, int n_devices);
/* 1 for a single-device context, G for a group; ocb_member(ctx, i) = the i-th member's single-device context (owned by the
 * group), or ctx itself for i == 0 of a single-device context. */
int ocb_member_count(const ocb_ctx* ctx);
ocb_ctx* ocb_member(ocb_ctx* ctx, int index);
void ocb_destroy(ocb_ctx* ctx);
/* Page-lock / release a caller-owned host buffer (an Image2D's pixels, a std::vector<POI2D>'s storage) so that the copies of
 * the host-buffer entry points run as asynchronous DMA at full PCIe rate instead of being staged by the driver.  Optional:
 * every entry point accepts pageable memory.  The range must stay allocated until it is unregistered. */
int ocb_host_register(void* host, size_t bytes);
int ocb_host_unregister(void* host);
/* Page-locked host memory for buffers the caller allocates anew (the shim's Image2D / Image3D keep their pixels in it).
 * ocb_host_alloc returns NULL when there is no usable CUDA device (callers then use ordinary memory). */
void* ocb_host_alloc(size_t bytes);
void* ocb_host_alloc_on(ocb_ctx* ctx, size_t bytes); /* same, after making ctx's (first) device current: no stray context on device 0 */
void ocb_host_free(void* host);
/* Last error message of this context (or of the process when ctx == NULL). Never NULL. */
const char* ocb_last_error(const ocb_ctx* ctx);
/* Enqueue on an external cudaStream_t (e.g. PyTorch's current stream).  The handle is used as given:
 * NULL is CUDA's legacy default stream, NOT "no stream".  ocb_use_own_stream() goes back to the
 * context's private non-blocking stream (the state after ocb_create). */
int ocb_set_stream(ocb_ctx* ctx, void* cuda_stream);
int ocb_use_own_stream(ocb_ctx* ctx);
/* Block until everything enqueued on the context's stream has finished. */
int ocb_sync(ocb_ctx* ctx);
/* Number of kernels this context has launched since creation (bench.py "gpu_launches"). */
long long ocb_launch_count(const ocb_ctx* ctx);
/* Which kernel the most recent FFT-CC 2D/3D, IC-GN/IC-LM 2D or ICGN3D1 call of this context launched, as space-separated
 * key=value pairs, so that a caller can tell which specialisation served its queue:
 *   "op=icgn2d np=6 rc=0 lm=0 wpp=1 tm=1 tma=1 grid=... threads=128"   (rc: compile-time subset radius, 0 = generic;
 *                                                                      wpp: warps per POI; tm: Tensor-Memory variant)
 *   "op=icgn3d rc=0 threads=256 slab_k=... nslab=... tma=1 grid=..."    (slab_k: layers per z-slab, nslab: slabs)
 *   "op=fftcc2d kernel=w32|reg|generic n=32 tma=1"                     (n: window points along x)
 * A host-queue 2D call of 16384 POIs or more goes out in four pipelined chunks, each its own launch: the description is
 * then that of the last chunk.  Never NULL; empty before the first such launch, and on a group context (ocb_member()
 * gives the member contexts, which keep their own). */
const char* ocb_last_launch(const ocb_ctx* ctx);

/* ---- images: DIC::setImages / DVC::setImages (src/oc_dic.cpp:22-26,44-48) ----------------- */
/* Host buffers; copied to the device (H2D on the context's stream). */
int ocb_set_images_2d(ocb_ctx* ctx, const float* ref, const float* tar, int width, int height, int col_major);
int ocb_set_images_3d(ocb_ctx* ctx, const float* ref, const float* tar, int dim_x, int dim_y, int dim_z);
/* 8-bit host images (what cv::imread(..., IMREAD_GRAYSCALE) hands the reference before cv2eigen turns
 * them into floats, src/oc_image.cpp:39,56): uploaded as bytes (4x fewer PCIe bytes) and widened to
 * f32 on the device; results are identical to passing the float copy.  Row-major / [z][y][x]. */
int ocb_set_images_2d_u8(ocb_ctx* ctx, const unsigned char* ref, const unsigned char* tar, int width, int height);
int ocb_set_images_3d_u8(ocb_ctx* ctx, const unsigned char* ref, const unsigned char* tar, int dim_x, int dim_y, int dim_z);
/* Device buffers (row-major / [z][y][x]); BORROWED like the reference borrows Image2D*. */
int ocb_set_images_2d_dev(ocb_ctx* ctx, const float* d_ref, const float* d_tar, int width, int height);
int ocb_set_images_3d_dev(ocb_ctx* ctx, const float* d_ref, const float* d_tar, int dim_x, int dim_y, int dim_z);

/* ---- FFT-CC: FFTCC2D::compute(std::vector<POI2D>&) src/oc_fftcc.cpp:277-285 (per POI
 *      :177-275) and FFTCC3D::compute(std::vector<POI3D>&) :429-437 (per POI :327-427) ------- */
int ocb_fftcc2d(ocb_ctx* ctx, void* poi2d, size_t n, int rx, int ry);
int ocb_fftcc3d(ocb_ctx* ctx, void* poi3d, size_t n, int rx, int ry, int rz);
int ocb_fftcc2d_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, int rx, int ry);
int ocb_fftcc3d_dev(ocb_ctx* ctx, void* d_poi3d, size_t n, int rx, int ry, int rz);

/* ---- IC-GN prepare(): ICGN2D1::prepare src/oc_icgn.cpp:138-142, ICGN2D2::prepare :679-683,
 *      ICGN3D1::prepare :1264-1268.  2D: nothing is materialised (gradients and bicubic
 *      weights are recomputed on chip); 3D: gradient volumes + tricubic B-spline coefficient
 *      volume are built on the device (src/oc_gradient.cpp:143-231, oc_cubic_bspline.cpp:214-351). */
int ocb_icgn2d_prepare(ocb_ctx* ctx);
int ocb_icgn3d_prepare(ocb_ctx* ctx);

/* ---- IC-GN compute(): ICGN2D1::compute(std::vector<POI2D>&) src/oc_icgn.cpp:343-351 (per POI
 *      :144-341); ICGN2D2 :900-908 (:685-898); ICGN3D1 :1492-1500 (:1270-1490).
 *      conv = conv_criterion, stop = stop_condition (a float in the reference, oc_icgn.h:52). */
int ocb_icgn2d1(ocb_ctx* ctx, void* poi2d, size_t n, int rx, int ry, float conv, float stop);
int ocb_icgn2d2(ocb_ctx* ctx, void* poi2d, size_t n, int rx, int ry, float conv, float stop);
int ocb_icgn3d1(ocb_ctx* ctx, void* poi3d, size_t n, int rx, int ry, int rz, float conv, float stop);
int ocb_icgn2d1_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop);
int ocb_icgn2d2_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop);
int ocb_icgn3d1_dev(ocb_ctx* ctx, void* d_poi3d, size_t n, int rx, int ry, int rz, float conv, float stop);

/* ---- IC-GN, the remaining overloads of the reference's class API (SURVEY.md section 8(f) N1) ------
 * order = 1 (ICGN2D1) or 2 (ICGN2D2).
 * center_offsets: NULL, or n (x, y) pairs -- compute(std::vector<POI2D>&, std::vector<Point2D>&
 *   center_offset_queue), src/oc_icgn.cpp:549-557 (per POI :353-547) and :1128-1136 (:910-1126): local
 *   coordinates are taken relative to poi + offset and the target subset is centred there.
 * self_adaptive != 0: DIC::setSelfAdaptive(true) -- every POI uses its own subset_radius.x/.y fields
 *   (src/oc_icgn.cpp:152-158) and rx, ry are ignored; POIs are grouped by radius on the host and each
 *   group is one launch.  The _dev variant takes device pointers and one radius for all POIs. */
int ocb_icgn2d_ex(ocb_ctx* ctx, int order, void* poi2d, size_t n, int rx, int ry, float conv, float stop, const float* center_offsets,
	int self_adaptive);
int ocb_icgn2d_ex_dev(ocb_ctx* ctx, int order, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop, const float* d_center_offsets);

/* ---- IC-LM siblings (SURVEY.md section 8(f) N2): ICLM2D1::compute(std::vector<POI2D>&) src/oc_iclm.cpp:360-368
 *      (per POI :150-358) and ICLM2D2 :732-740 (:502-730).  Same prepare() as IC-GN (ocb_icgn2d_prepare).
 *      lambda, alpha, beta = DampingParameter (src/oc_iclm.h:32-37; defaults 100, 0.1, 10; setDamping()). */
int ocb_iclm2d(ocb_ctx* ctx, int order, void* poi2d, size_t n, int rx, int ry, float conv, float stop, float lambda, float alpha, float beta);
int ocb_iclm2d_dev(ocb_ctx* ctx, int order, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop, float lambda, float alpha, float beta);

/* ---- NR2D1, forward-additive Newton-Raphson (SURVEY.md section 8(f) N2): NR2D1::prepare src/oc_nr.cpp:119-156
 *      (nothing is precomputed here: the target gradients and the three bicubic interpolants are evaluated
 *      on chip), NR2D1::compute(std::vector<POI2D>&) :327-334 (per POI :160-325). */
int ocb_nr2d_prepare(ocb_ctx* ctx);
int ocb_nr2d1(ocb_ctx* ctx, void* poi2d, size_t n, int rx, int ry, float conv, float stop);
int ocb_nr2d1_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, int rx, int ry, float conv, float stop);

/* ---- EpipolarSearch (SURVEY.md section 8(f) N4): EpipolarSearch::compute(std::vector<POI2D>&) src/oc_epipolar_search.cpp:197-205
 *      (per POI :133-195) as one batch: every POI spawns its candidates along the epipolar line of the secondary view
 *      (centre + every search_step pixels in x below search_radius, both directions), ICGN2D1(rx, ry, conv, stop) registers
 *      all of them, the candidate with the highest ZNCC replaces the POI's deformation and result.
 *      fundamental: the 3x3 fundamental matrix, row-major (updateFundementalMatrix :110-126); parallax_x/_y: the three
 *      coefficients of setParallax(float[3], float[3]) (setParallax(Point2D p) = {0, 0, p.x}, {0, 0, p.y}) -- host pointers in
 *      both variants.  Images = primary / secondary view (setImages), after ocb_icgn2d_prepare (prepareICGN :63-67). */
int ocb_epipolar_search2d(ocb_ctx* ctx, void* poi2d, size_t n, const float* fundamental, const float* parallax_x, const float* parallax_y,
	int search_radius, int search_step, int rx, int ry, float conv, float stop);
int ocb_epipolar_search2d_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, const float* fundamental, const float* parallax_x, const float* parallax_y,
	int search_radius, int search_step, int rx, int ry, float conv, float stop);

/* ---- Strain post-processing of a POI queue (SURVEY.md section 8(f) N4): Strain::prepare + Strain::compute(queue),
 *      src/oc_strain.cpp:100-111,150-156,239-250 (POI2D; per POI :158-237) and :476-487 (POI3D; per POI :373-474).
 *      radius = subregion_radius, min_neighbors = neighbor_number_min (constructor :32-36), zncc_threshold = setZnccThreshold
 *      (default 0.9, :38), approximation = setApproximation: 1 Cauchy (default), 2 Green.  Writes strain.exx.. of every POI
 *      whose own ZNCC and enough neighbours' ZNCC pass the threshold; other records are left untouched.
 *      (The stereo variant, POI2DS records, is ocb_strain2ds below.) */
int ocb_strain2d(ocb_ctx* ctx, void* poi2d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation);
int ocb_strain3d(ocb_ctx* ctx, void* poi3d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation);
/* Strain::compute(POI2D* poi, queue) / (POI3D* poi, queue) for the queue member `index`: fitted whatever its own ZNCC. */
int ocb_strain2d_single(ocb_ctx* ctx, void* poi2d, size_t n, size_t index, float radius, int min_neighbors, float zncc_threshold, int approximation);
int ocb_strain3d_single(ocb_ctx* ctx, void* poi3d, size_t n, size_t index, float radius, int min_neighbors, float zncc_threshold, int approximation);
/* Stereo-DIC queues (POI2DS records, OCB_POI2DS_FLOATS floats: x y | u v w | r1r2 r1t1 r1t2 ZNCC r2_x r2_y t1_x t1_y t2_x t2_y |
 * ref_coor | tar_coor | e[6] | subset_radius, src/oc_poi.h:140-186): Strain::compute(std::vector<POI2DS>&) src/oc_strain.cpp:362-371
 * (per POI :252-360) -- neighbours searched in the image plane, plane fit over ref_coor and u, v, w, all three ZNCCs tested. */
int ocb_strain2ds(ocb_ctx* ctx, void* poi2ds, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation);
int ocb_strain2ds_dev(ocb_ctx* ctx, void* d_poi2ds, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation);
int ocb_strain2d_dev(ocb_ctx* ctx, void* d_poi2d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation);
int ocb_strain3d_dev(ocb_ctx* ctx, void* d_poi3d, size_t n, float radius, int min_neighbors, float zncc_threshold, int approximation);

/* ---- inspection (parity tests of the prepare() products) ----------------------------------- */
/* Copy the device tables built by ocb_icgn3d_prepare() to host buffers of dim_x*dim_y*dim_z
 * floats each; any pointer may be NULL. */
int ocb_get_tables_3d(ocb_ctx* ctx, float* gx, float* gy, float* gz, float* coefficient);

#ifdef __cplusplus
}
#endif
#endif /* OPENCORR_B200_H_ */
