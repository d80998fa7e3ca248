"""Host-side mirror of the reference's operator interface for the FFT-CC -> IC-GN path.

Class names, constructor arguments and method meaning follow the reference (C++):
  FFTCC2D(int rx, int ry, int threads)                        src/oc_fftcc.h:61
  FFTCC3D(int rx, int ry, int rz, int threads)                src/oc_fftcc.h:82
  ICGN2D1 / ICGN2D2(int rx, int ry, float conv, float stop, int threads)   src/oc_icgn.h:58,113
  ICGN3D1(int rx, int ry, int rz, float conv, float stop, int threads)     src/oc_icgn.h:168
  setImages / setSubset / prepare / compute / setIteration    src/oc_dic.h:56-84, oc_icgn.h:61-76
Python spellings (set_images, ...) are provided next to the reference's camelCase names.

POI queues are numpy float32 arrays [n, 25] (POI2D) or [n, 31] (POI3D) -- the reference's
records viewed as floats (src/oc_poi.h:102-136,187-222) -- mutated in place like
compute(std::vector<POI>&).  Everything runs through the C ABI (include/opencorr_b200.h); the
`thread_number` argument is accepted for signature compatibility and ignored (no CPU threads).
"""
import ctypes

import numpy as np

from . import _capi

# ---- POI record layout (reference src/oc_poi.h) ------------------------------------------------
POI2D_FLOATS = 25
POI3D_FLOATS = 31
P2 = dict(x=0, y=1, u=2, ux=3, uy=4, uxx=5, uxy=6, uyy=7, v=8, vx=9, vy=10, vxx=11, vxy=12, vyy=13,
          u0=14, v0=15, zncc=16, iteration=17, convergence=18, feature=19, exx=20, eyy=21, exy=22,
          subset_rx=23, subset_ry=24)
P3 = dict(x=0, y=1, z=2, u=3, ux=4, uy=5, uz=6, v=7, vx=8, vy=9, vz=10, w=11, wx=12, wy=13, wz=14,
          u0=15, v0=16, w0=17, zncc=18, iteration=19, convergence=20, feature=21,
          exx=22, eyy=23, ezz=24, exy=25, eyz=26, ezx=27, subset_rx=28, subset_ry=29, subset_rz=30)


def make_poi2d(xy):
    """POI2D(Point2D) for every row of xy: location set, everything else cleared (oc_poi.h:112-135)."""
    xy = np.asarray(xy, dtype=np.float32).reshape(-1, 2)
    q = np.zeros((xy.shape[0], POI2D_FLOATS), np.float32)
    q[:, 0:2] = xy
    return q


def make_poi3d(xyz):
    xyz = np.asarray(xyz, dtype=np.float32).reshape(-1, 3)
    q = np.zeros((xyz.shape[0], POI3D_FLOATS), np.float32)
    q[:, 0:3] = xyz
    return q


def _vp(a):
    return ctypes.c_void_p(a.ctypes.data)


def _check_queue(q, floats):
    if not isinstance(q, np.ndarray) or q.dtype != np.float32 or q.ndim != 2 or q.shape[1] != floats \
            or not q.flags.c_contiguous:
        raise ValueError("POI queue must be a C-contiguous float32 array of shape [n, %d]" % floats)


class Engine:
    """One GPU context (ocb_ctx), or a GROUP context over several devices: device = -1 / "all" (every visible device) or a
    list of device indices -- host-queue calls then shard the queue over the devices inside the C ABI (one process, G
    devices; include/opencorr_b200.h ocb_create_multi).  Raises OpenCorrB200Error when no B200-class GPU is usable."""

    def __init__(self, device=0):
        self._lib = _capi.load()
        if isinstance(device, str):
            if device != "all":
                raise ValueError("device must be an index, -1 / 'all', or a list of indices")
            device = -1
        if isinstance(device, (list, tuple)):
            devs = (ctypes.c_int * len(device))(*[int(d) for d in device])
            self._ctx = self._lib.ocb_create_multi(devs, len(device))
            self.device = tuple(int(d) for d in device)
        else:
            self._ctx = self._lib.ocb_create(int(device))
            self.device = int(device)
        if not self._ctx:
            raise _capi.OpenCorrB200Error(_capi.OCB_ERR_CUDA, _capi.last_error(None))
        self._keep = []  # host arrays referenced by the last upload
        self.image_token = 0  # bumped by every set_images_*: lets an operator see that another one replaced its images

    @property
    def member_count(self):
        """Devices behind this context (1 unless it is a group)."""
        return int(self._lib.ocb_member_count(self._ctx))

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.ocb_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        _capi.check(rc, self._ctx)

    # images ------------------------------------------------------------------------------------
    def set_images_2d(self, ref, tar):
        """float32 images, or uint8 images (as read from an 8-bit file): the latter are uploaded as
        bytes and widened on the device -- same results, a quarter of the PCIe traffic."""
        ref, tar = np.asarray(ref), np.asarray(tar)
        if ref.ndim != 2 or ref.shape != tar.shape:
            raise ValueError("ref/tar must be 2-D arrays of equal shape")
        h, w = ref.shape
        if ref.dtype == np.uint8 and tar.dtype == np.uint8:
            ref, tar = np.ascontiguousarray(ref), np.ascontiguousarray(tar)
            self._ck(self._lib.ocb_set_images_2d_u8(self._ctx, _vp(ref), _vp(tar), w, h))
        else:
            ref = np.ascontiguousarray(ref, dtype=np.float32)
            tar = np.ascontiguousarray(tar, dtype=np.float32)
            self._ck(self._lib.ocb_set_images_2d(self._ctx, _vp(ref), _vp(tar), w, h, 0))
        self._ck(self._lib.ocb_sync(self._ctx))
        self.image_token += 1

    def set_images_3d(self, ref, tar):
        ref, tar = np.asarray(ref), np.asarray(tar)
        if ref.ndim != 3 or ref.shape != tar.shape:
            raise ValueError("ref/tar must be 3-D arrays [z, y, x] of equal shape")
        dz, dy, dx = ref.shape
        if ref.dtype == np.uint8 and tar.dtype == np.uint8:
            ref, tar = np.ascontiguousarray(ref), np.ascontiguousarray(tar)
            self._ck(self._lib.ocb_set_images_3d_u8(self._ctx, _vp(ref), _vp(tar), dx, dy, dz))
        else:
            ref = np.ascontiguousarray(ref, dtype=np.float32)
            tar = np.ascontiguousarray(tar, dtype=np.float32)
            self._ck(self._lib.ocb_set_images_3d(self._ctx, _vp(ref), _vp(tar), dx, dy, dz))
        self._ck(self._lib.ocb_sync(self._ctx))
        self.image_token += 1

    def set_images_2d_dev(self, d_ref, d_tar, width, height):
        self._ck(self._lib.ocb_set_images_2d_dev(self._ctx, int(d_ref), int(d_tar), width, height))
        self.image_token += 1

    def set_images_3d_dev(self, d_ref, d_tar, dim_x, dim_y, dim_z):
        self._ck(self._lib.ocb_set_images_3d_dev(self._ctx, int(d_ref), int(d_tar), dim_x, dim_y, dim_z))
        self.image_token += 1

    def set_stream(self, cuda_stream):
        """Enqueue on this cudaStream_t handle (0/None = CUDA's legacy default stream)."""
        self._ck(self._lib.ocb_set_stream(self._ctx, int(cuda_stream) if cuda_stream else None))

    def use_own_stream(self):
        self._ck(self._lib.ocb_use_own_stream(self._ctx))

    def sync(self):
        self._ck(self._lib.ocb_sync(self._ctx))

    def launch_count(self):
        return int(self._lib.ocb_launch_count(self._ctx))

    def last_launch(self):
        """The kernel the most recent FFT-CC / IC-GN / IC-LM / ICGN3D1 call launched (include/opencorr_b200.h
        ocb_last_launch), e.g. {"op": "icgn2d", "rc": 0, "tm": 1, ...}; numbers come back as int.  {} before any launch."""
        text = self._lib.ocb_last_launch(self._ctx).decode("utf-8", "replace")
        out = {}
        for item in text.split():
            key, _, value = item.partition("=")
            out[key] = int(value) if value.lstrip("-").isdigit() else value
        return out

    # hot path, host POI queues -------------------------------------------------------------------
    def fftcc2d(self, q, rx, ry):
        _check_queue(q, POI2D_FLOATS)
        self._ck(self._lib.ocb_fftcc2d(self._ctx, _vp(q), q.shape[0], rx, ry))

    def fftcc3d(self, q, rx, ry, rz):
        _check_queue(q, POI3D_FLOATS)
        self._ck(self._lib.ocb_fftcc3d(self._ctx, _vp(q), q.shape[0], rx, ry, rz))

    def icgn2d_prepare(self):
        self._ck(self._lib.ocb_icgn2d_prepare(self._ctx))

    def icgn3d_prepare(self):
        self._ck(self._lib.ocb_icgn3d_prepare(self._ctx))

    def icgn2d1(self, q, rx, ry, conv, stop):
        _check_queue(q, POI2D_FLOATS)
        self._ck(self._lib.ocb_icgn2d1(self._ctx, _vp(q), q.shape[0], rx, ry, conv, stop))

    def icgn2d2(self, q, rx, ry, conv, stop):
        _check_queue(q, POI2D_FLOATS)
        self._ck(self._lib.ocb_icgn2d2(self._ctx, _vp(q), q.shape[0], rx, ry, conv, stop))

    def icgn2d_ex(self, order, q, rx, ry, conv, stop, center_offsets=None, self_adaptive=False):
        """Offset-centre and/or self-adaptive overloads (reference src/oc_icgn.cpp:353-557, :910-1136)."""
        _check_queue(q, POI2D_FLOATS)
        off = None
        if center_offsets is not None:
            off = np.ascontiguousarray(center_offsets, dtype=np.float32).reshape(-1, 2)
            if off.shape[0] != q.shape[0]:
                raise ValueError("center_offsets must hold one (x, y) pair per POI")
        self._ck(self._lib.ocb_icgn2d_ex(self._ctx, int(order), _vp(q), q.shape[0], rx, ry, conv, stop,
                                         _vp(off) if off is not None else None, int(bool(self_adaptive))))

    def iclm2d(self, order, q, rx, ry, conv, stop, damping=(100.0, 0.1, 10.0)):
        """ICLM2D1 / ICLM2D2 (reference src/oc_iclm.cpp); damping = (lambda, alpha, beta)."""
        _check_queue(q, POI2D_FLOATS)
        self._ck(self._lib.ocb_iclm2d(self._ctx, int(order), _vp(q), q.shape[0], rx, ry, conv, stop,
                                      float(damping[0]), float(damping[1]), float(damping[2])))

    def epipolar_search2d(self, q, fundamental, parallax_x, parallax_y, search_radius, search_step, rx, ry, conv, stop):
        """EpipolarSearch::compute(queue) (reference src/oc_epipolar_search.cpp:133-205) as one batch."""
        _check_queue(q, POI2D_FLOATS)
        f = np.ascontiguousarray(fundamental, dtype=np.float32).reshape(9)
        ax = np.ascontiguousarray(parallax_x, dtype=np.float32).reshape(3)
        ay = np.ascontiguousarray(parallax_y, dtype=np.float32).reshape(3)
        self._ck(self._lib.ocb_epipolar_search2d(self._ctx, _vp(q), q.shape[0], _vp(f), _vp(ax), _vp(ay), int(search_radius),
                                                 int(search_step), rx, ry, conv, stop))

    def strain(self, q, radius, min_neighbors, zncc_threshold=0.9, approximation=1):
        """Strain::prepare + compute(queue) (reference src/oc_strain.cpp) on a POI2D [n,25] or POI3D [n,31] queue."""
        if q.ndim == 2 and q.shape[1] == 28:  # POI2DS records (stereo DIC)
            _check_queue(q, 28)
            fn = self._lib.ocb_strain2ds
        elif q.ndim == 2 and q.shape[1] == POI3D_FLOATS:
            _check_queue(q, POI3D_FLOATS)
            fn = self._lib.ocb_strain3d
        else:
            _check_queue(q, POI2D_FLOATS)
            fn = self._lib.ocb_strain2d
        self._ck(fn(self._ctx, _vp(q), q.shape[0], float(radius), int(min_neighbors), float(zncc_threshold), int(approximation)))

    def nr2d_prepare(self):
        self._ck(self._lib.ocb_nr2d_prepare(self._ctx))

    def nr2d1(self, q, rx, ry, conv, stop):
        """NR2D1 (reference src/oc_nr.cpp:160-334)."""
        _check_queue(q, POI2D_FLOATS)
        self._ck(self._lib.ocb_nr2d1(self._ctx, _vp(q), q.shape[0], rx, ry, conv, stop))

    def icgn3d1(self, q, rx, ry, rz, conv, stop):
        _check_queue(q, POI3D_FLOATS)
        self._ck(self._lib.ocb_icgn3d1(self._ctx, _vp(q), q.shape[0], rx, ry, rz, conv, stop))

    # hot path, device-resident POI queues (pointers as ints, e.g. torch.Tensor.data_ptr()) --------
    def fftcc2d_dev(self, d_q, n, rx, ry):
        self._ck(self._lib.ocb_fftcc2d_dev(self._ctx, int(d_q), n, rx, ry))

    def fftcc3d_dev(self, d_q, n, rx, ry, rz):
        self._ck(self._lib.ocb_fftcc3d_dev(self._ctx, int(d_q), n, rx, ry, rz))

    def icgn2d1_dev(self, d_q, n, rx, ry, conv, stop):
        self._ck(self._lib.ocb_icgn2d1_dev(self._ctx, int(d_q), n, rx, ry, conv, stop))

    def icgn2d2_dev(self, d_q, n, rx, ry, conv, stop):
        self._ck(self._lib.ocb_icgn2d2_dev(self._ctx, int(d_q), n, rx, ry, conv, stop))

    def icgn3d1_dev(self, d_q, n, rx, ry, rz, conv, stop):
        self._ck(self._lib.ocb_icgn3d1_dev(self._ctx, int(d_q), n, rx, ry, rz, conv, stop))


_default_engines = {}


def default_engine(device=0):
    """Process-wide engine per device, shared by the operator objects below (the reference's
    objects all borrow the same Image2D/Image3D; here they share one device copy)."""
    key = tuple(device) if isinstance(device, (list, tuple)) else device
    eng = _default_engines.get(key)
    if eng is None or not eng._ctx:
        eng = Engine(device)
        _default_engines[key] = eng
    return eng


class _DIC:
    def __init__(self, rx, ry, thread_number=0, engine=None):
        self.subset_radius_x = int(rx)
        self.subset_radius_y = int(ry)
        self.thread_number = int(thread_number)
        self.self_adaptive = False
        self.engine = engine if engine is not None else default_engine()
        self.ref_img = None
        self.tar_img = None
        self._token = None      # engine.image_token of this object's own upload
        self._prepared = False  # prepare() has been called since set_images()

    def set_images(self, ref_img, tar_img):
        self.ref_img, self.tar_img = ref_img, tar_img
        self.engine.set_images_2d(ref_img, tar_img)
        self._token = self.engine.image_token
        self._prepared = False

    def _bind(self):
        """The operators of one engine share its device images (like the reference's objects share Image2D pointers), but
        each keeps ITS pair and prepared state (the reference keeps per-object tables): if another object has replaced the
        engine's images since, upload this object's pair again and redo its prepare()."""
        if self.ref_img is None or self._token == self.engine.image_token:
            return
        self.engine.set_images_2d(self.ref_img, self.tar_img)
        self._token = self.engine.image_token
        if self._prepared:
            self._prepare_engine()

    def _prepare_engine(self):
        pass

    def set_subset(self, radius_x, radius_y):
        self.subset_radius_x, self.subset_radius_y = int(radius_x), int(radius_y)

    setImages = set_images
    setSubset = set_subset


class _DVC:
    def __init__(self, rx, ry, rz, thread_number=0, engine=None):
        self.subset_radius_x = int(rx)
        self.subset_radius_y = int(ry)
        self.subset_radius_z = int(rz)
        self.thread_number = int(thread_number)
        self.engine = engine if engine is not None else default_engine()
        self.ref_img = None
        self.tar_img = None
        self._token = None
        self._prepared = False

    def set_images(self, ref_img, tar_img):
        self.ref_img, self.tar_img = ref_img, tar_img
        self.engine.set_images_3d(ref_img, tar_img)
        self._token = self.engine.image_token
        self._prepared = False

    def _bind(self):
        """See _DIC._bind."""
        if self.ref_img is None or self._token == self.engine.image_token:
            return
        self.engine.set_images_3d(self.ref_img, self.tar_img)
        self._token = self.engine.image_token
        if self._prepared:
            self._prepare_engine()

    def _prepare_engine(self):
        pass

    def set_subset(self, radius_x, radius_y, radius_z):
        self.subset_radius_x, self.subset_radius_y, self.subset_radius_z = int(radius_x), int(radius_y), int(radius_z)

    setImages = set_images
    setSubset = set_subset


class FFTCC2D(_DIC):
    def prepare(self):
        pass

    def compute(self, poi_queue):
        self._bind()
        self.engine.fftcc2d(poi_queue, self.subset_radius_x, self.subset_radius_y)
        return poi_queue


class FFTCC3D(_DVC):
    def prepare(self):
        pass

    def compute(self, poi_queue):
        self._bind()
        self.engine.fftcc3d(poi_queue, self.subset_radius_x, self.subset_radius_y, self.subset_radius_z)
        return poi_queue


class _ICGN2D(_DIC):
    _order = 1

    def __init__(self, rx, ry, conv_criterion, stop_condition, thread_number=0, engine=None):
        super().__init__(rx, ry, thread_number, engine)
        self.conv_criterion = float(conv_criterion)
        self.stop_condition = float(stop_condition)

    def set_iteration(self, conv_criterion, stop_condition):
        self.conv_criterion, self.stop_condition = float(conv_criterion), float(stop_condition)

    def _prepare_engine(self):
        self.engine.icgn2d_prepare()

    def prepare(self):
        self._bind()
        self._prepare_engine()
        self._prepared = True

    prepare_ref = prepare
    prepare_tar = prepare

    def compute(self, poi_queue, center_offset_queue=None):
        """compute(queue) and compute(queue, center_offset_queue); honours set_self_adaptive(True)."""
        self._bind()
        if center_offset_queue is None and not self.self_adaptive:
            fn = self.engine.icgn2d1 if self._order == 1 else self.engine.icgn2d2
            fn(poi_queue, self.subset_radius_x, self.subset_radius_y, self.conv_criterion, self.stop_condition)
        else:
            self.engine.icgn2d_ex(self._order, poi_queue, self.subset_radius_x, self.subset_radius_y, self.conv_criterion,
                                  self.stop_condition, center_offset_queue, self.self_adaptive)
        return poi_queue

    def set_self_adaptive(self, is_self_adaptive):
        self.self_adaptive = bool(is_self_adaptive)

    setSelfAdaptive = set_self_adaptive

    setIteration = set_iteration
    prepareRef = prepare_ref
    prepareTar = prepare_tar


class ICGN2D1(_ICGN2D):
    _order = 1


class ICGN2D2(_ICGN2D):
    _order = 2


class _ICLM2D(_ICGN2D):
    """ICLM2D1 / ICLM2D2(int rx, int ry, float conv, float stop, int threads), reference src/oc_iclm.h:56-75,110-130."""

    def __init__(self, rx, ry, conv_criterion, stop_condition, thread_number=0, engine=None):
        super().__init__(rx, ry, conv_criterion, stop_condition, thread_number, engine)
        self.damping = (100.0, 0.1, 10.0)

    def set_damping(self, lambda_, alpha, beta):
        self.damping = (float(lambda_), float(alpha), float(beta))

    def compute(self, poi_queue):
        self._bind()
        self.engine.iclm2d(self._order, poi_queue, self.subset_radius_x, self.subset_radius_y, self.conv_criterion,
                           self.stop_condition, self.damping)
        return poi_queue

    setDamping = set_damping


class ICLM2D1(_ICLM2D):
    _order = 1


class ICLM2D2(_ICLM2D):
    _order = 2


class NR2D1(_DIC):
    """NR2D1(int rx, int ry, float conv, float stop, int threads), reference src/oc_nr.h:46-71."""

    def __init__(self, rx, ry, conv_criterion, stop_condition, thread_number=0, engine=None):
        super().__init__(rx, ry, thread_number, engine)
        self.conv_criterion = float(conv_criterion)
        self.stop_condition = float(stop_condition)

    def set_iteration(self, conv_criterion, stop_condition):
        self.conv_criterion, self.stop_condition = float(conv_criterion), float(stop_condition)

    def _prepare_engine(self):
        self.engine.nr2d_prepare()

    def prepare(self):
        self._bind()
        self._prepare_engine()
        self._prepared = True

    def compute(self, poi_queue):
        self._bind()
        self.engine.nr2d1(poi_queue, self.subset_radius_x, self.subset_radius_y, self.conv_criterion, self.stop_condition)
        return poi_queue

    setIteration = set_iteration


class Calibration:
    """The part of the reference's Calibration (src/oc_calibration.h:25-98, .cpp:36-88) EpipolarSearch needs: the
    intrinsic matrix, the rotation matrix from the rotation vector (rx, ry, rz) and the translation vector, float32."""

    def __init__(self, fx, fy, fs, cx, cy, tx=0.0, ty=0.0, tz=0.0, rx=0.0, ry=0.0, rz=0.0):
        self.intrinsics = dict(fx=fx, fy=fy, fs=fs, cx=cx, cy=cy)
        self.extrinsics = dict(tx=tx, ty=ty, tz=tz, rx=rx, ry=ry, rz=rz)
        self.update_matrices()

    def update_matrices(self):
        f32 = np.float32
        i, e = self.intrinsics, self.extrinsics
        self.intrinsic_matrix = np.array([[i["fx"], i["fs"], i["cx"]], [0, i["fy"], i["cy"]], [0, 0, 1]], f32)
        v = np.array([e["rx"], e["ry"], e["rz"]], f32)
        th = f32(np.linalg.norm(v))
        if th == 0:
            self.rotation_matrix = np.eye(3, dtype=f32)
        else:  # Eigen::AngleAxisf::toRotationMatrix, src/oc_calibration.cpp:50-60
            x, y, z = v / th
            c, s = f32(np.cos(th)), f32(np.sin(th))
            t = f32(1) - c
            self.rotation_matrix = np.array([[t * x * x + c, t * x * y - s * z, t * x * z + s * y],
                                             [t * x * y + s * z, t * y * y + c, t * y * z - s * x],
                                             [t * x * z - s * y, t * y * z + s * x, t * z * z + c]], f32)
        self.translation_vector = np.array([e["tx"], e["ty"], e["tz"]], f32)

    updateMatrices = update_matrices


class EpipolarSearch(_DIC):
    """EpipolarSearch(Calibration& view1_cam, Calibration& view2_cam, int thread_number), reference
    src/oc_epipolar_search.h:30-63.  set_images(view1, view2); the candidate sweep of all POIs runs as one GPU batch."""

    def __init__(self, view1_cam, view2_cam, thread_number=0, engine=None):
        super().__init__(0, 0, thread_number, engine)
        self.view1_cam, self.view2_cam = view1_cam, view2_cam
        self.search_radius, self.search_step = 0, 1
        self.parallax_x = np.zeros(3, np.float32)
        self.parallax_y = np.zeros(3, np.float32)
        self.fundamental_matrix = None
        self._icgn = None

    def set_search(self, search_radius, search_step):
        if search_radius < search_step:
            raise ValueError("Search radius is less than search step")
        self.search_radius, self.search_step = int(search_radius), int(search_step)

    def create_icgn(self, subset_radius_x, subset_radius_y, conv_criterion, stop_condition):
        self._icgn = (int(subset_radius_x), int(subset_radius_y), float(conv_criterion), float(stop_condition))

    def set_parallax(self, *args):
        """set_parallax((px, py))  or  set_parallax(coefficient_x[3], coefficient_y[3])  (src/oc_epipolar_search.cpp:74-95)."""
        if len(args) == 1:
            self.parallax_x = np.array([0, 0, args[0][0]], np.float32)
            self.parallax_y = np.array([0, 0, args[0][1]], np.float32)
        else:
            self.parallax_x = np.asarray(args[0], np.float32).reshape(3)
            self.parallax_y = np.asarray(args[1], np.float32).reshape(3)

    def update_cameras(self, view1_cam, view2_cam):
        self.view1_cam, self.view2_cam = view1_cam, view2_cam

    def update_fundamental_matrix(self):
        """src/oc_epipolar_search.cpp:110-126, float32."""
        f32 = np.float32
        c1, c2 = self.view1_cam, self.view2_cam
        t = c2.translation_vector
        tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]], f32)
        e = (tx @ c2.rotation_matrix).astype(f32)
        k2_inv_t = np.linalg.inv(c2.intrinsic_matrix.astype(np.float64)).T.astype(f32)
        k1_inv = np.linalg.inv(c1.intrinsic_matrix.astype(np.float64)).astype(f32)
        self.fundamental_matrix = (k2_inv_t @ e @ k1_inv).astype(f32)

    def prepare(self):
        self.view1_cam.update_matrices()
        self.view2_cam.update_matrices()
        self.update_fundamental_matrix()
        self._bind()
        self._prepare_engine()
        self._prepared = True

    def _prepare_engine(self):
        self.engine.icgn2d_prepare()

    def compute(self, poi_queue):
        if self._icgn is None or self.fundamental_matrix is None:
            raise _capi.OpenCorrB200Error(_capi.OCB_ERR_STATE, "EpipolarSearch: create_icgn() and prepare() must be called before compute()")
        self._bind()
        rx, ry, conv, stop = self._icgn
        self.engine.epipolar_search2d(poi_queue, self.fundamental_matrix, self.parallax_x, self.parallax_y, self.search_radius,
                                      self.search_step, rx, ry, conv, stop)
        return poi_queue

    setSearch = set_search
    createICGN = create_icgn
    setParallax = set_parallax
    updateCameras = update_cameras
    updateFundementalMatrix = update_fundamental_matrix


class Strain:
    """Strain(float subregion_radius, int neighbor_number_min, int thread_number), reference src/oc_strain.h:33-70."""

    def __init__(self, subregion_radius, neighbor_number_min, thread_number=0, engine=None):
        self.engine = engine if engine is not None else default_engine()
        self.subregion_radius = float(subregion_radius)
        self.neighbor_number_min = int(neighbor_number_min)
        self.zncc_threshold = 0.9  # src/oc_strain.cpp:38-40
        self.description = 1
        self.approximation = 1
        self.thread_number = thread_number

    def set_subregion_radius(self, r):
        self.subregion_radius = float(r)

    def set_neighbor_min(self, k):
        self.neighbor_number_min = int(k)

    def set_zncc_threshold(self, t):
        self.zncc_threshold = float(t)

    def set_description(self, d):
        self.description = int(d)

    def set_approximation(self, a):
        self.approximation = int(a)

    def prepare(self, poi_queue):
        """The reference builds its kd-trees here; the grid binning happens inside compute()."""

    def compute(self, poi_queue):
        self.engine.strain(poi_queue, self.subregion_radius, self.neighbor_number_min, self.zncc_threshold, self.approximation)
        return poi_queue

    setSubregionRadius = set_subregion_radius
    setNeighborMin = set_neighbor_min
    setZnccThreshold = set_zncc_threshold
    setDescription = set_description
    setApproximation = set_approximation


class ICGN3D1(_DVC):
    def __init__(self, rx, ry, rz, conv_criterion, stop_condition, thread_number=0, engine=None):
        super().__init__(rx, ry, rz, thread_number, engine)
        self.conv_criterion = float(conv_criterion)
        self.stop_condition = float(stop_condition)

    def set_iteration(self, conv_criterion, stop_condition):
        self.conv_criterion, self.stop_condition = float(conv_criterion), float(stop_condition)

    def _prepare_engine(self):
        self.engine.icgn3d_prepare()

    def prepare(self):
        self._bind()
        self._prepare_engine()
        self._prepared = True

    prepare_ref = prepare_tar = prepare

    def compute(self, poi_queue):
        self._bind()
        self.engine.icgn3d1(poi_queue, self.subset_radius_x, self.subset_radius_y, self.subset_radius_z,
                            self.conv_criterion, self.stop_condition)
        return poi_queue

    def tables(self):
        """(gx, gy, gz, coefficient) volumes built by prepare() -- for parity tests."""
        dz, dy, dx = np.asarray(self.ref_img).shape
        out = [np.empty((dz, dy, dx), np.float32) for _ in range(4)]
        eng = self.engine
        eng._ck(eng._lib.ocb_get_tables_3d(eng._ctx, _vp(out[0]), _vp(out[1]), _vp(out[2]), _vp(out[3])))
        return out

    setIteration = set_iteration
    prepareRef = prepareTar = prepare
