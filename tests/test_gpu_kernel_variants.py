"""Every IC-GN kernel instantiation the launchers pick at run time, asserted through Engine.last_launch() and compared with
the oracle.  icgn2d_launch chooses among template instantiations from the queue length, the subset radius, the image
width and what fits in shared memory (the Tensor-Memory variant, for one, only when the queue holds >= 16 POIs per SM);
icgn3d1_launch splits the subvolume into z-slabs and picks a two- or one-CTA-per-SM kernel.  A test that only lands on
one side of such a threshold by accident stops covering the kernel it was written for when the threshold moves, so
each case here states the variant it expects and fails, naming the variant it saw, when another one ran.

Parity bar: 1e-4 px and 1e-5 ZNCC, identical sentinel codes and u0/v0, iteration counts equal or one apart
(util.compare_2d / util.compare_3d)."""
import numpy as np
import pytest

import opencorr_b200 as ob
from opencorr_b200 import synth
from oracle.oracle import Oracle2D, Oracle3D
import util

pytestmark = pytest.mark.gpu

# Queues of 16384 POIs or more go out in four pipelined chunks (include/opencorr_b200.h ocb_last_launch): the Tensor-Memory
# queues below stay under that, so one launch serves the whole queue.
PIPELINE_MIN = 16384


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tm_queue_len():
    """POIs enough for the Tensor-Memory variant (>= 16 per SM, icgn2d.cu icgn2d_launch), in one launch."""
    n = 17 * _sm_count()
    assert n < PIPELINE_MIN
    return n


def _expect(engine, label, **want):
    got = engine.last_launch()
    bad = {k: v for k, v in want.items() if got.get(k) != v}
    assert not bad, "%s: expected %s, ran %s" % (label, want, got)
    return got


def _pair_and_queue(n, width, height, margin=40):
    """Synthetic pair and a queue of n POIs on a grid inside `margin`, seeded with the rounded true displacement."""
    ref, tar = synth.speckle_pair_2d(width, height)
    nx = int(np.ceil(np.sqrt(n * (width - 2 * margin) / (height - 2 * margin))))
    ny = (n + nx - 1) // nx
    sx = (width - 2 * margin) / nx
    sy = (height - 2 * margin) / ny
    xs = np.floor(margin + sx * np.arange(nx))
    ys = np.floor(margin + sy * np.arange(ny))
    yy, xx = np.meshgrid(ys, xs, indexing="ij")
    xy = np.stack([xx.ravel(), yy.ravel()], 1)[:n].astype(np.float32)
    q = ob.make_poi2d(xy)
    u, v = synth.displacement_2d(xy[:, 0], xy[:, 1], width, height)
    q[:, 2], q[:, 8] = np.round(u), np.round(v)
    return ref, tar, q


def _icgn2d1(engine, ref, tar, q, rx, ry, conv=0.001, stop=10, offsets=None):
    engine.set_images_2d(ref, tar)
    engine.icgn2d_prepare()
    out = q.copy()
    if offsets is None:
        engine.icgn2d1(out, rx, ry, conv, stop)
    else:
        engine.icgn2d_ex(1, out, rx, ry, conv, stop, center_offsets=offsets)
    return out


# ---- Tensor-Memory (TM) ICGN2D1 -----------------------------------------------------------------------------------------

# (20, 20) and (18, 19): tail columns and odd row counts; (24, 12): 17 tail columns; (16, 20): 41 rows, the most the
# 128 TMEM columns of a CTA hold (3 per row); (32, 8): 33 tail columns, more than one lane pass
TM_GENERIC_RADII = [(20, 20), (24, 12), (16, 20), (32, 8), (18, 19)]


@pytest.fixture(scope="module")
def tm_pair():
    n = _tm_queue_len()
    ref, tar, q = _pair_and_queue(n, 520, 480)
    return ref, tar, q


@pytest.mark.parametrize("rx,ry", TM_GENERIC_RADII)
def test_tm_generic_radii(engine, tm_pair, rx, ry):
    """The generic (run-time radius) Tensor-Memory kernel icgn2d_kernel<6, 0, false, 1, true> at the subset shapes where
    its layout differs from r = 16's."""
    ref, tar, q = tm_pair
    q_gpu = _icgn2d1(engine, ref, tar, q, rx, ry)
    _expect(engine, "r=(%d,%d)" % (rx, ry), op="icgn2d", np=6, tm=1, rc=0, wpp=1, lm=0)
    q_cpu = q.copy()
    Oracle2D(ref, tar).icgn2d1(q_cpu, rx, ry, 0.001, 10)
    stats = util.compare_2d(q_gpu, q_cpu, "TM r=(%d,%d)" % (rx, ry))
    assert stats["n_compared"] >= 0.95 * len(q)


@pytest.mark.parametrize("rx,ry", [(16, 16)] + TM_GENERIC_RADII)
def test_tm_matches_shared_memory_constants(engine, tm_pair, monkeypatch, rx, ry):
    """The TM kernel keeps the per-sample constants {R, gx, gy} of the 32 row-mapped columns in Tensor Memory; with
    OCB_ICGN2D_TMEM=0 the same queue runs the one-warp-per-POI kernel, which keeps them in shared memory.  Nothing else
    differs, so the records must be bit-identical."""
    ref, tar, q = tm_pair
    a = _icgn2d1(engine, ref, tar, q, rx, ry)
    _expect(engine, "TMEM on, r=(%d,%d)" % (rx, ry), tm=1, wpp=1)
    monkeypatch.setenv("OCB_ICGN2D_TMEM", "0")
    b = _icgn2d1(engine, ref, tar, q, rx, ry)
    _expect(engine, "TMEM off, r=(%d,%d)" % (rx, ry), tm=0, wpp=1)
    diff = np.where((a != b).any(1))[0]
    assert len(diff) == 0, "r=(%d,%d): %d of %d records differ between the TM and shared-memory kernels, first %s: %s vs %s" % (
        rx, ry, len(diff), len(q), diff[:5], a[diff[:2]], b[diff[:2]])


@pytest.mark.parametrize("rx,ry", [(16, 16), (20, 20)])
@pytest.mark.parametrize("how", ["width_1001", "no_tma"])
def test_tm_staged_tile_loads(engine, monkeypatch, rx, ry, how):
    """TM kernel with the staged (non-TMA) tile loads: an image width that is not a multiple of 4 (TMA needs a 16-byte
    aligned row pitch), and OCB_NO_TMA=1 on a width of 1024."""
    n = _tm_queue_len()
    width = 1001 if how == "width_1001" else 1024
    ref, tar, q = _pair_and_queue(n, width, 300)
    if how == "no_tma":
        monkeypatch.setenv("OCB_NO_TMA", "1")
    q_gpu = _icgn2d1(engine, ref, tar, q, rx, ry)
    _expect(engine, "%s r=(%d,%d)" % (how, rx, ry), tm=1, tma=0, rc=16 if rx == 16 and ry == 16 else 0)
    q_cpu = q.copy()
    Oracle2D(ref, tar).icgn2d1(q_cpu, rx, ry, 0.001, 10)
    stats = util.compare_2d(q_gpu, q_cpu, "TM staged %s r=(%d,%d)" % (how, rx, ry))
    assert stats["n_compared"] >= 0.95 * len(q)


@pytest.mark.parametrize("rx,ry", [(16, 16), (20, 20)])
def test_tm_center_offsets(engine, tm_pair, rx, ry):
    """compute(queue, center_offset_queue) (src/oc_icgn.cpp:353-557) on a queue long enough for the TM kernel."""
    ref, tar, q = tm_pair
    off = np.random.default_rng(11).uniform(-4, 4, (len(q), 2)).astype(np.float32)
    q_gpu = _icgn2d1(engine, ref, tar, q, rx, ry, offsets=off)
    _expect(engine, "offsets r=(%d,%d)" % (rx, ry), tm=1, rc=16 if rx == 16 else 0)
    q_cpu = q.copy()
    Oracle2D(ref, tar).icgn2d_ex(1, q_cpu, rx, ry, 0.001, 10, center_offsets=off)
    stats = util.compare_2d(q_gpu, q_cpu, "TM offsets r=(%d,%d)" % (rx, ry))
    assert stats["n_compared"] >= 0.95 * len(q)
    assert np.abs(q_gpu[:, 2] - _icgn2d1(engine, ref, tar, q, rx, ry)[:, 2]).max() > 1e-3  # the offsets were applied


def test_tm_self_adaptive_groups(engine):
    """setSelfAdaptive(true) launches once per radius group: two long groups take the TM kernel -- (16, 16) its RC = 16
    specialisation, (20, 14) the generic one -- and a short (12, 12) group two warps per POI.  Only the last launch is
    recorded, so each group is also run on its own, where its variant is asserted; the self-adaptive records must be
    bit-identical to those."""
    m = _tm_queue_len()
    groups = [((12, 12), 150), ((16, 16), m), ((20, 14), m)]
    ref, tar, q = _pair_and_queue(sum(k for _, k in groups), 720, 720)
    rng = np.random.default_rng(3)
    radii = np.concatenate([np.tile(np.array(r, np.float32), (k, 1)) for r, k in groups])
    q[:, 23:25] = radii[rng.permutation(len(q))]
    engine.set_images_2d(ref, tar)
    engine.icgn2d_prepare()
    q_gpu = q.copy()
    engine.icgn2d_ex(1, q_gpu, 99, 99, 0.001, 10, self_adaptive=True)
    _expect(engine, "self-adaptive, last group (20,14)", tm=1, rc=0)  # groups run in (rx, ry) order
    q_cpu = q.copy()
    Oracle2D(ref, tar).icgn2d_ex(1, q_cpu, 99, 99, 0.001, 10, self_adaptive=True)
    stats = util.compare_2d(q_gpu, q_cpu, "TM self-adaptive")
    assert stats["n_compared"] >= 0.95 * len(q)
    assert np.array_equal(q_gpu[:, 23:25], q[:, 23:25])
    want = {(12, 12): dict(tm=0, wpp=2), (16, 16): dict(tm=1, rc=16), (20, 14): dict(tm=1, rc=0)}
    for (rx, ry), _ in groups:
        sel = (q[:, 23] == rx) & (q[:, 24] == ry)
        alone = q[sel].copy()
        engine.icgn2d1(alone, rx, ry, 0.001, 10)
        _expect(engine, "group (%d,%d) alone" % (rx, ry), **want[(rx, ry)])
        assert np.array_equal(alone, q_gpu[sel]), "group (%d,%d): self-adaptive records differ from the group run alone" % (rx, ry)


@pytest.mark.parametrize("rx,ry", [(16, 16), (20, 20)])
def test_tm_sentinels(engine, tm_pair, rx, ry):
    """The rejection rules on a TM-length queue (pattern: test_gpu_2d.py::test_icgn2d_sentinels): subsets leaving the
    reference image (-3), an incoming ZNCC < 0 (skipped, code kept), guesses that push the target subset out (-3), then
    stop = 1 (-4, parameters kept).  Rejected records must be bit-identical to the oracle's."""
    ref, tar, q = tm_pair
    q = q.copy()
    h, w = ref.shape
    k = len(q) // 13
    border = {k: [5, 200], 2 * k: [200, 5], 3 * k: [w - 6, 200], 4 * k: [200, h - 6]}
    for i, xy in border.items():
        q[i, 0:2] = xy
    skipped = {5 * k: -1.0, 6 * k: -2.0, 7 * k + 1: -1.0}
    for i, z in skipped.items():
        q[i, 16] = z
    pushed = [8 * k, 9 * k]
    q[pushed[0], 2] = w - q[pushed[0], 0] - 5.0  # target subset mostly right of the image
    q[pushed[1], 8] = float(h)                   # |v| >= height
    q_cpu = q.copy()
    o = Oracle2D(ref, tar)
    o.icgn2d1(q_cpu, rx, ry, 0.001, 10)
    q_gpu = _icgn2d1(engine, ref, tar, q, rx, ry)
    _expect(engine, "sentinels r=(%d,%d)" % (rx, ry), tm=1, rc=16 if rx == 16 else 0)
    expect_codes = [-3.0] * len(border) + list(skipped.values()) + [-3.0, -3.0]
    idx = list(border) + list(skipped) + pushed
    assert list(q_cpu[idx, 16]) == expect_codes
    util.compare_2d(q_gpu, q_cpu, "TM sentinels r=(%d,%d)" % (rx, ry))
    rejected = np.isin(q_cpu[:, 16], [-1.0, -2.0, -3.0])
    assert np.array_equal(q_gpu[rejected], q_cpu[rejected])
    # stop = 1: no POI converges to 1e-6 in one step -> -4 everywhere else, parameters kept
    q_cpu = q.copy()
    o.icgn2d1(q_cpu, rx, ry, 1e-6, 1)
    q_gpu = _icgn2d1(engine, ref, tar, q, rx, ry, conv=1e-6, stop=1)
    _expect(engine, "sentinels stop=1 r=(%d,%d)" % (rx, ry), tm=1)
    assert (q_cpu[~rejected, 16] == -4).all()
    assert np.array_equal(q_gpu[:, 16], q_cpu[:, 16])
    assert np.array_equal(q_gpu[rejected], q_cpu[rejected])
    assert np.abs(q_gpu[~rejected][:, 2:14] - q_cpu[~rejected][:, 2:14]).max() < 1e-4


# ---- ICGN3D1 generic kernels -------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def vol120():
    ref, tar = synth.speckle_pair_3d(120, 120, 120)
    c = np.array([[60, 60, 60], [57, 62, 59], [63, 58, 61], [59, 59, 63], [61, 63, 57], [62, 61, 62], [58, 57, 58],
                  [60, 61, 60]], np.float32)
    return ref, tar, c


def _icgn3d_case(engine, vol, r, label):
    ref, tar, xyz = vol
    q = ob.make_poi3d(xyz)
    u, v, w = synth.displacement_3d(xyz[:, 0], xyz[:, 1], xyz[:, 2], 120, 120, 120)
    q[:, 3], q[:, 7], q[:, 11] = u, v, w
    q[-1, 4] = 0.05   # 5 % stretch guesses in x and z: the first iterations sample outside the slab tiles
    q[-1, 14] = 0.05
    icgn = ob.ICGN3D1(*r, 0.001, 20, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    q_gpu = q.copy()
    icgn.compute(q_gpu)
    got = engine.last_launch()
    q_cpu = q.copy()
    Oracle3D(ref, tar).icgn3d1(q_cpu, *r, 0.001, 20, exact=True)
    stats = util.compare_3d(q_gpu, q_cpu, "%s r=%s (%s)" % (label, r, got), max_iter_mismatch_frac=0.25)
    assert stats["n_compared"] >= 0.6 * len(q)
    return got


@pytest.mark.parametrize("r", [(12, 12, 12), (16, 16, 12), (14, 9, 20), (20, 20, 20)])
def test_icgn3d1_generic_two_ctas_per_sm_several_slabs(engine, vol120, r):
    """icgn3d1_kernel<0, 256> (two CTAs per SM) on subvolumes that need several z-slabs; (16, 16, 12) splits its 25
    layers so that the last slab is shorter than the others."""
    got = _icgn3d_case(engine, vol120, r, "2 CTAs/SM")
    assert got.get("op") == "icgn3d" and got.get("rc") == 0 and got.get("threads") == 256 and got.get("nslab", 0) > 1, \
        "r=%s: expected rc=0 threads=256 nslab>1, ran %s" % (r, got)
    assert got["tma"] == 1, "r=%s: %s" % (r, got)
    if r == (16, 16, 12):
        assert got["nslab"] * got["slab_k"] != 2 * r[2] + 1, "r=%s: expected an uneven last slab, ran %s" % (r, got)


@pytest.mark.parametrize("r,no_tma", [((24, 24, 24), False), ((30, 30, 22), False), ((22, 22, 22), True)])
def test_icgn3d1_generic_one_cta_per_sm(engine, vol120, monkeypatch, r, no_tma):
    """icgn3d1_kernel<0, 512> (one CTA per SM, 16 warps): subvolumes too large for two slab-carrying CTAs per SM;
    (22, 22, 22) with the staged slab loads (OCB_NO_TMA=1)."""
    if no_tma:
        monkeypatch.setenv("OCB_NO_TMA", "1")
    got = _icgn3d_case(engine, vol120, r, "1 CTA/SM")
    assert got.get("op") == "icgn3d" and got.get("rc") == 0 and got.get("threads") == 512 and got.get("nslab", 0) > 1, \
        "r=%s: expected rc=0 threads=512 nslab>1, ran %s" % (r, got)
    assert got["tma"] == (0 if no_tma else 1), "r=%s: %s" % (r, got)
