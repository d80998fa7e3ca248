"""GPU parity, 2D: FFTCC2D, ICGN2D1, ICGN2D2 through the C ABI vs the CPU oracle and vs the
reference's golden table.  Tolerances are north_star's: 1e-4 px displacement, 1e-5 ZNCC; integer
outputs (u0, v0, FFT-CC displacement, iteration count, sentinel codes) must be identical, with the
documented exception of POIs whose ||dp|| lands within float noise of the convergence threshold."""
import numpy as np
import pytest

import opencorr_b200 as ob
from opencorr_b200 import synth
from oracle.oracle import Oracle2D
import util

pytestmark = pytest.mark.gpu


def _config_a():
    cfg = synth.CONFIGS["A"]
    ref, tar = synth.speckle_pair_2d(*cfg["size"])
    xy = synth.grid_2d(*cfg["grid"])
    return ref, tar, xy, cfg["r"]


@pytest.fixture(scope="module")
def cfg_a():
    return _config_a()


@pytest.mark.parametrize("r", [15, 16, 20, 6])
def test_fftcc2d_matches_oracle(engine, cfg_a, r):
    ref, tar, xy, _ = cfg_a
    q_gpu = ob.make_poi2d(xy)
    q_cpu = q_gpu.copy()
    f = ob.FFTCC2D(r, r, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    Oracle2D(ref, tar).fftcc2d(q_cpu, r, r)
    assert np.array_equal(q_gpu[:, [2, 8, 14, 15]], q_cpu[:, [2, 8, 14, 15]])  # integer displacements: bit-exact
    assert np.abs(q_gpu[:, 16] - q_cpu[:, 16]).max() < 1e-5
    untouched = np.delete(np.arange(25), [2, 8, 14, 15, 16])
    assert np.array_equal(q_gpu[:, untouched], q_cpu[:, untouched])


@pytest.mark.parametrize("r", [4, 5, 8, 9, 10, 12, 18, 24, 25, 27, 30, 32])
def test_fftcc2d_register_kernels_all_sizes(engine, r):
    """Every window size served by fftcc2d_reg.cu (thread-per-row register FFTs), with a POI count that does not fill
    the last CTA, border POIs (left untouched) and a non-zero incoming guess."""
    ref, tar = synth.speckle_pair_2d(400, 360)
    xy = synth.grid_2d(70, 70, 9, 7, 29, 31)[:59]
    xy = np.vstack([xy, [[2, 2], [399, 100], [200, 358]]]).astype(np.float32)
    q_gpu = ob.make_poi2d(xy)
    q_gpu[::4, 2] = 1.0
    q_gpu[::5, 8] = -1.6
    q_cpu = q_gpu.copy()
    f = ob.FFTCC2D(r, r, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    Oracle2D(ref, tar).fftcc2d(q_cpu, r, r)
    assert np.array_equal(q_gpu[:, [2, 8, 14, 15]], q_cpu[:, [2, 8, 14, 15]])
    assert np.abs(q_gpu[:, 16] - q_cpu[:, 16]).max() < 1e-5
    untouched = np.delete(np.arange(25), [2, 8, 14, 15, 16])
    assert np.array_equal(q_gpu[:, untouched], q_cpu[:, untouched])
    assert np.all(q_gpu[-3:, 16] == 0)


def test_fftcc2d_generic_kernel_still_matches(engine, cfg_a, monkeypatch):
    """The Stockham-over-shared-memory kernel stays the fallback (non-square windows, other prime factors)."""
    monkeypatch.setenv("OCB_FFTCC2D_GENERIC", "1")
    ref, tar, xy, _ = cfg_a
    for r in (16, 20, 7):
        q_gpu = ob.make_poi2d(xy)
        q_cpu = q_gpu.copy()
        f = ob.FFTCC2D(r, r, engine=engine)
        f.set_images(ref, tar)
        f.compute(q_gpu)
        Oracle2D(ref, tar).fftcc2d(q_cpu, r, r)
        assert np.array_equal(q_gpu[:, [2, 8, 14, 15]], q_cpu[:, [2, 8, 14, 15]])
        assert np.abs(q_gpu[:, 16] - q_cpu[:, 16]).max() < 1e-5


def test_fftcc2d_nonsquare_window_and_initial_guess(engine, cfg_a):
    ref, tar, xy, _ = cfg_a
    q_gpu = ob.make_poi2d(xy)
    q_gpu[:, 2] = 1.0   # incoming guess shifts the target window (src/oc_fftcc.cpp:187,215)
    q_gpu[:, 8] = -2.0
    q_gpu[::3, 2] = 0.6  # fractional guesses exercise the (int) truncation
    q_cpu = q_gpu.copy()
    f = ob.FFTCC2D(12, 10, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    Oracle2D(ref, tar).fftcc2d(q_cpu, 12, 10)
    assert np.array_equal(q_gpu[:, [2, 8, 14, 15]], q_cpu[:, [2, 8, 14, 15]])
    assert np.abs(q_gpu[:, 16] - q_cpu[:, 16]).max() < 1e-5


def test_fftcc2d_border_pois_are_left_untouched(engine, cfg_a):
    ref, tar, _, _ = cfg_a
    h, w = ref.shape
    xy = np.array([[5, 100], [100, 5], [w - 6, 100], [100, h - 6], [15, 15], [16, 16], [w - 16, h - 16], [w - 17, h - 17]], np.float32)
    q_gpu = ob.make_poi2d(xy)
    q_gpu[:, 16] = 0.123  # marker that must survive on skipped POIs
    q_cpu = q_gpu.copy()
    f = ob.FFTCC2D(16, 16, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    Oracle2D(ref, tar).fftcc2d(q_cpu, 16, 16)
    assert np.array_equal(q_gpu[:, [2, 8, 14, 15]], q_cpu[:, [2, 8, 14, 15]])
    skipped = q_cpu[:, 16] == np.float32(0.123)
    assert skipped.sum() == 6
    assert np.array_equal(q_gpu[skipped], q_cpu[skipped])
    assert np.abs(q_gpu[:, 16] - q_cpu[:, 16]).max() < 1e-5


@pytest.mark.parametrize("exact", [0, 1])
def test_icgn2d1_config_a(engine, cfg_a, exact):
    ref, tar, xy, r = cfg_a
    q = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(q, r, r)
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN2D1(r, r, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    o.icgn2d1(q_cpu, r, r, 0.001, 10, exact=exact)
    stats = util.compare_2d(q_gpu, q_cpu, "icgn2d1 A exact=%d" % exact)
    assert stats["n_compared"] >= 0.95 * len(q)
    ok = (q_gpu[:, 16] >= 0) & (q_gpu[:, 17] == q_cpu[:, 17])
    assert np.abs(q_gpu[ok][:, [3, 4, 9, 10]] - q_cpu[ok][:, [3, 4, 9, 10]]).max() < 2e-5  # ux uy vx vy
    assert np.abs(q_gpu[ok, 18] - q_cpu[ok, 18]).max() < 1e-4                              # convergence
    assert np.array_equal(q_gpu[ok][:, 23:25], q_cpu[ok][:, 23:25])
    # ground truth of the synthetic field, loose sanity bound
    u_true, v_true = synth.displacement_2d(xy[:, 0], xy[:, 1], ref.shape[1], ref.shape[0])
    assert np.abs(q_gpu[ok, 2] - u_true[ok]).max() < 0.05 and np.abs(q_gpu[ok, 8] - v_true[ok]).max() < 0.05


def test_icgn2d1_golden_table(engine):
    """FFTCC2D -> ICGN2D1 on the reference's example pair: all 30 000 POIs of examples/test_2d_dic_fftcc_icgn1.cpp:50-66 against
    the oracle (every sentinel code identical; the POIs inside the specimen's hole end with -4), and the
    committed rows of the shipped result table as known answers."""
    ref, tar = util.oht_cfrp_pair()
    g = util.oht_cfrp_golden()
    xy = synth.grid_2d(30, 30, 100, 300, 2, 2)
    assert len(xy) == 30000
    q = ob.make_poi2d(xy)
    f = ob.FFTCC2D(16, 16, engine=engine)
    f.set_images(ref, tar)
    f.compute(q)
    qc = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(qc, 16, 16)
    # FFT-CC: identical integer guess everywhere except, possibly, where two correlation bins tie exactly (the three POIs
    # enumerated in the fixture, tests/test_oracle_golden.py::test_2d_fftcc_ties): there the arg-max hangs on the last bit
    ties = set(int(r) for r in g["fftcc_tie_rows"])
    guess_differs = np.where((q[:, 14] != qc[:, 14]) | (q[:, 15] != qc[:, 15]))[0]
    assert set(int(i) for i in guess_differs) <= ties, guess_differs
    q[:, 2:17] = qc[:, 2:17]  # same seed for both IC-GN runs, ties included
    icgn = ob.ICGN2D1(16, 16, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q)
    o.icgn2d1(qc, 16, 16, 0.001, 10)
    assert (qc[:, 16] == -4).sum() > 100  # the POIs inside the specimen's hole do not converge
    stats = util.compare_2d(q, qc, "oht_cfrp, all 30 000 POIs", max_iter_mismatch_frac=0.02)  # asserts identical sentinel codes
    assert stats["n_compared"] > 0.9 * len(q)
    # known answers: the shipped table (it predates the -4 code: converged rows only)
    tab, rows = g["table"], g["rows"]
    qt = q[rows]
    assert np.array_equal(qt[:, 0:2], tab[:, 0:2].astype(np.float32))
    ok = (qt[:, 14] == tab[:, 4]) & (qt[:, 15] == tab[:, 5]) & (tab[:, 7] < 10) & (qt[:, 17] == tab[:, 7])
    assert ok.sum() > 0.93 * len(tab)
    assert np.abs(qt[ok][:, [2, 8]] - tab[ok][:, [2, 3]]).max() < 1e-4
    assert np.abs(qt[ok, 16] - tab[ok, 6]).max() < 1e-5


@pytest.mark.parametrize("r", [20, 12])
def test_icgn2d2_matches_oracle(engine, r):
    ref, tar = synth.speckle_pair_2d(512, 512, second_order=True)
    xy = synth.grid_2d(64, 64, 16, 12, 24, 31)
    q = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(q, r, r)
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN2D2(r, r, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    got = engine.last_launch()  # 192 POIs cannot fill the GPU: two warps per POI; r = 20 has its own instantiation
    assert got.get("np") == 12 and got.get("wpp") == 2 and got.get("rc") == (20 if r == 20 else 0), "r=%d: ran %s" % (r, got)
    o.icgn2d2(q_cpu, r, r, 0.001, 10)
    stats = util.compare_2d(q_gpu, q_cpu, "icgn2d2 r=%d" % r, max_iter_mismatch_frac=0.03)
    assert stats["n_compared"] >= 0.9 * len(q)
    ok = (q_gpu[:, 16] >= 0) & (q_gpu[:, 17] == q_cpu[:, 17])
    assert np.abs(q_gpu[ok][:, 2:14] - q_cpu[ok][:, 2:14]).max() < 1e-4


def test_icgn2d_sentinels(engine, cfg_a):
    """-3 at the border / skip on incoming zncc<0 / -3 when the warped subset leaves the target /
    -4 when stop is reached (src/oc_icgn.cpp:160-167,251-255,329-332)."""
    ref, tar, _, r = cfg_a
    h, w = ref.shape
    xy = np.array([[10, 200], [200, 10], [w - 11, 200], [200, h - 11],  # 0-3: subset leaves the reference image
                   [200, 200], [260, 240],                               # 4,5: fine
                   [r, r], [w - 1 - r, h - 1 - r],                       # 6,7: guard passes, warped samples leave the target -> -3
                   [300, 300], [320, 300], [340, 300]], np.float32)      # 8: zncc<0 in, 9: guess pushes out, 10: |u|>=w
    q = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(q, r, r)
    q[8, 16] = -2.0
    q[9, 2] = w - 330.0   # target subset partly outside -> -3 during iteration 1
    q[10, 2] = float(w)
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN2D1(r, r, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    o.icgn2d1(q_cpu, r, r, 0.001, 10)
    assert list(q_cpu[[0, 1, 2, 3, 6, 7, 8, 9, 10], 16]) == [-3, -3, -3, -3, -3, -3, -2, -3, -3]
    util.compare_2d(q_gpu, q_cpu, "sentinels", max_iter_mismatch_frac=0.0)
    rejected = [0, 1, 2, 3, 6, 7, 8, 9, 10]
    assert np.array_equal(q_gpu[rejected], q_cpu[rejected])  # rejected records: bit-identical (nothing else written)
    # stop_condition = 1 -> every POI that does not converge in one step gets -4, parameters kept
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn.set_iteration(1e-6, 1)
    icgn.compute(q_gpu)
    o.icgn2d1(q_cpu, r, r, 1e-6, 1)
    assert (q_cpu[[4, 5], 16] == -4).all()
    assert np.array_equal(q_gpu[:, 16], q_cpu[:, 16])
    assert np.abs(q_gpu[[4, 5]][:, 2:14] - q_cpu[[4, 5]][:, 2:14]).max() < 1e-4


def test_icgn2d_requires_prepare_and_images():
    eng = ob.Engine(0)
    q = ob.make_poi2d([[100, 100]])
    with pytest.raises(ob.OpenCorrB200Error):
        eng.icgn2d1(q, 16, 16, 0.001, 10)       # images not set
    ref, tar = synth.speckle_pair_2d(128, 128)
    eng.set_images_2d(ref, tar)
    with pytest.raises(ob.OpenCorrB200Error):
        eng.icgn2d1(q, 16, 16, 0.001, 10)       # prepare() missing
    eng.icgn2d_prepare()
    eng.icgn2d1(q[:0], 16, 16, 0.001, 10)      # empty queue is a no-op
    with pytest.raises(ob.OpenCorrB200Error):
        eng.icgn2d1(q, 0, 16, 0.001, 10)        # radius < 1
    eng.close()


def test_large_deformation_gradient_falls_back_to_global_reads(engine):
    """Samples leaving the staged target tile are read from global memory; result must not change."""
    ref, _ = synth.speckle_pair_2d(384, 384)
    # target = reference stretched by 12 % about the centre (far beyond the tile slack at r=16)
    yy, xx = np.mgrid[0:384, 0:384].astype(np.float32)
    o_ref = Oracle2D(ref, ref)
    o_ref.prepare()
    src = np.stack([(192 + (xx - 192) / 1.12).ravel(), (192 + (yy - 192) / 1.12).ravel()], 1)
    tar = np.clip(o_ref.bicubic(src), 0, 255).reshape(384, 384).astype(np.float32)
    xy = synth.grid_2d(150, 150, 5, 5, 20, 20)
    q = ob.make_poi2d(xy)
    q[:, 2] = (xy[:, 0] - 192) * 0.12
    q[:, 8] = (xy[:, 1] - 192) * 0.12
    q[:, 3] = 0.12
    q[:, 10] = 0.12
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN2D1(16, 16, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    Oracle2D(ref, tar).icgn2d1(q_cpu, 16, 16, 0.001, 10)
    assert (q_cpu[:, 16] > 0.9).all()
    util.compare_2d(q_gpu, q_cpu, "stretch", max_iter_mismatch_frac=0.05)


@pytest.mark.parametrize("width", [330, 331, 333])
def test_icgn2d1_image_width_not_multiple_of_four(engine, width):
    """TMA tile loads need a 16-byte aligned row pitch; other widths take the staged-load path.
    Both must give the same answer as the oracle (the reference's example pair is 280 px wide)."""
    ref, tar = synth.speckle_pair_2d(width, 300)
    xy = synth.grid_2d(40, 40, 10, 8, 25, 27)
    q = ob.make_poi2d(xy)
    f = ob.FFTCC2D(16, 16, engine=engine)
    f.set_images(ref, tar)
    f.compute(q)
    q_gpu, q_cpu = q.copy(), q.copy()
    o = Oracle2D(ref, tar)
    qo = ob.make_poi2d(xy)
    o.fftcc2d(qo, 16, 16)
    assert np.array_equal(q[:, [2, 8]], qo[:, [2, 8]])
    icgn = ob.ICGN2D1(16, 16, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    got = engine.last_launch()
    assert got.get("rc") == 16 and got.get("tma") == 0 and got.get("wpp") == 2, "width %d: ran %s" % (width, got)
    o.icgn2d1(q_cpu, 16, 16, 0.001, 10)
    stats = util.compare_2d(q_gpu, q_cpu, "width %d" % width, max_iter_mismatch_frac=0.03)
    assert stats["n_compared"] >= 0.9 * len(q)


@pytest.mark.parametrize("rx,ry", [(16, 10), (9, 21), (33, 33), (4, 4)])
def test_icgn2d1_other_radii(engine, rx, ry):
    """Non-square subsets, a subset wider than 64 px (tail columns, two lane passes) and a tiny one."""
    ref, tar = synth.speckle_pair_2d(400, 360)
    xy = synth.grid_2d(100, 90, 6, 5, 33, 37)
    q = ob.make_poi2d(xy)
    u, v = synth.displacement_2d(xy[:, 0], xy[:, 1], 400, 360)
    q[:, 2], q[:, 8] = np.round(u), np.round(v)
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN2D1(rx, ry, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    Oracle2D(ref, tar).icgn2d1(q_cpu, rx, ry, 0.001, 10)
    stats = util.compare_2d(q_gpu, q_cpu, "r=(%d,%d)" % (rx, ry), max_iter_mismatch_frac=0.1)
    assert stats["n_compared"] >= 0.8 * len(q)


def test_borrowed_device_images_and_device_queue(engine):
    """The *_dev entry points: images and the POI queue stay on the device (torch is only the allocator)."""
    torch = pytest.importorskip("torch")
    ref, tar = synth.speckle_pair_2d(320, 256)
    xy = synth.grid_2d(40, 40, 12, 9, 20, 19)
    d_ref, d_tar = torch.from_numpy(ref).cuda(), torch.from_numpy(tar).cuda()
    eng = ob.Engine(0)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.set_images_2d_dev(d_ref.data_ptr(), d_tar.data_ptr(), 320, 256)
    d_q = torch.from_numpy(ob.make_poi2d(xy)).cuda()
    eng.fftcc2d_dev(d_q.data_ptr(), len(xy), 16, 16)
    eng.icgn2d_prepare()
    eng.icgn2d1_dev(d_q.data_ptr(), len(xy), 16, 16, 0.001, 10)
    torch.cuda.synchronize()
    q_gpu = d_q.cpu().numpy()
    q_cpu = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(q_cpu, 16, 16)
    o.icgn2d1(q_cpu, 16, 16, 0.001, 10)
    util.compare_2d(q_gpu, q_cpu, "device-resident", max_iter_mismatch_frac=0.03)
    assert eng.launch_count() == 2
    eng.close()


@pytest.mark.parametrize("order", [1, 2])
def test_icgn2d_center_offset_overload(engine, order):
    """compute(queue, center_offset_queue), reference src/oc_icgn.cpp:353-557 / :910-1136."""
    ref, tar = synth.speckle_pair_2d(400, 360, second_order=(order == 2))
    xy = synth.grid_2d(90, 80, 8, 6, 27, 33)
    rng = np.random.default_rng(5)
    off = rng.uniform(-4, 4, (len(xy), 2)).astype(np.float32)
    off[0] = 0.0
    q = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(q, 16, 16)
    q_gpu, q_cpu = q.copy(), q.copy()
    cls = ob.ICGN2D1 if order == 1 else ob.ICGN2D2
    icgn = cls(16, 16, 0.001, 10, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu, off)
    o.icgn2d_ex(order, q_cpu, 16, 16, 0.001, 10, center_offsets=off)
    stats = util.compare_2d(q_gpu, q_cpu, "offset order %d" % order, max_iter_mismatch_frac=0.05)
    assert stats["n_compared"] >= 0.9 * len(q)
    # the offset moves the point whose displacement is reported: it must differ from the plain overload
    q_plain = q.copy()
    icgn.compute(q_plain)
    assert np.abs(q_plain[1:, 2] - q_gpu[1:, 2]).max() > 1e-3
    assert np.abs(q_plain[0, 2:14] - q_gpu[0, 2:14]).max() < 1e-6  # zero offset == plain overload


def test_icgn2d1_self_adaptive(engine):
    """setSelfAdaptive(true): every POI uses its own subset_radius (src/oc_icgn.cpp:152-158)."""
    ref, tar = synth.speckle_pair_2d(400, 360)
    xy = synth.grid_2d(90, 80, 9, 7, 25, 30)
    q = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(q, 16, 16)
    radii = np.array([[10, 10], [16, 16], [12, 20], [23, 9]], np.float32)
    q[:, 23:25] = radii[np.arange(len(q)) % 4]
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN2D1(99, 99, 0.001, 10, engine=engine)  # the constructor radius is ignored in this mode
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.set_self_adaptive(True)
    icgn.compute(q_gpu)
    o.icgn2d_ex(1, q_cpu, 99, 99, 0.001, 10, self_adaptive=True)
    stats = util.compare_2d(q_gpu, q_cpu, "self-adaptive", max_iter_mismatch_frac=0.05)
    assert stats["n_compared"] >= 0.9 * len(q)
    assert np.array_equal(q_gpu[:, 23:25], q[:, 23:25])


def test_u8_image_upload_gives_identical_results(engine):
    """8-bit images uploaded as bytes (ocb_set_images_2d_u8) == the same images passed as float32."""
    ref, tar = util.oht_cfrp_pair()
    xy = synth.grid_2d(40, 60, 20, 30, 10, 26)
    res = []
    for cast in (np.float32, np.uint8):
        q = ob.make_poi2d(xy)
        f = ob.FFTCC2D(16, 16, engine=engine)
        f.set_images(ref.astype(cast), tar.astype(cast))
        f.compute(q)
        icgn = ob.ICGN2D1(16, 16, 0.001, 10, engine=engine)
        icgn.set_images(ref.astype(cast), tar.astype(cast))
        icgn.prepare()
        icgn.compute(q)
        res.append(q)
    assert np.array_equal(res[0], res[1])


def _iclm_compare(q_gpu, q_cpu, label):
    """ICLM parity: sentinel codes, guesses and iteration counts as for IC-GN; displacements within 1e-4 px
    for >= 98 % of the POIs and within conv (1e-3 px) for all -- at convergence the accept/reject test of the
    last step (`znssd < znssd0`, src/oc_iclm.cpp:292) is decided by rounding (see test_oracle_golden)."""
    assert np.array_equal(q_gpu[:, 14:16], q_cpu[:, 14:16])
    neg = (q_gpu[:, 16] < 0) | (q_cpu[:, 16] < 0)
    it_same = q_gpu[:, 17] == q_cpu[:, 17]
    assert it_same.mean() > 0.95, label
    assert np.array_equal(q_gpu[neg & it_same, 16], q_cpu[neg & it_same, 16]), label
    ok = ~neg & it_same
    d = np.abs(q_gpu[ok][:, [2, 8]] - q_cpu[ok][:, [2, 8]]).max(1)
    assert (d < 1e-4).mean() >= 0.98, (label, float((d < 1e-4).mean()))
    assert d.max() < 1.5e-3, (label, float(d.max()))
    assert np.abs(q_gpu[ok, 16] - q_cpu[ok, 16]).max() < 1e-5, label


@pytest.mark.parametrize("order,second", [(1, False), (2, True)])
def test_iclm2d_matches_oracle(engine, order, second):
    ref, tar = synth.speckle_pair_2d(512, 512, second_order=second)
    xy = synth.grid_2d(64, 64, 16, 12, 24, 31)
    q = ob.make_poi2d(xy)
    o = Oracle2D(ref, tar)
    o.fftcc2d(q, 16, 16)
    q_gpu, q_cpu = q.copy(), q.copy()
    iclm = (ob.ICLM2D1 if order == 1 else ob.ICLM2D2)(16, 16, 0.001, 10, engine=engine)
    iclm.set_images(ref, tar)
    iclm.prepare()
    iclm.compute(q_gpu)
    o.iclm2d(order, q_cpu, 16, 16, 0.001, 10)
    _iclm_compare(q_gpu, q_cpu, "iclm order %d" % order)
    # non-default damping
    q_gpu, q_cpu = q.copy(), q.copy()
    iclm.set_damping(10.0, 0.5, 4.0)
    iclm.compute(q_gpu)
    o.iclm2d(order, q_cpu, 16, 16, 0.001, 10, damping=(10.0, 0.5, 4.0))
    _iclm_compare(q_gpu, q_cpu, "iclm order %d damping" % order)


def test_iclm2d1_golden_table(engine):
    """FFTCC2D -> ICLM2D1 vs the reference's shipped examples/2d_dic/oht_cfrp_4_fftcc_iclm1_r16.csv."""
    ref, tar = util.oht_cfrp_pair()
    tab = util.oht_cfrp_iclm_golden()["table"]
    q = ob.make_poi2d(tab[:, 0:2])
    f = ob.FFTCC2D(16, 16, engine=engine)
    f.set_images(ref, tar)
    f.compute(q)
    iclm = ob.ICLM2D1(16, 16, 0.001, 10, engine=engine)
    iclm.set_images(ref, tar)
    iclm.prepare()
    iclm.compute(q)
    same = (q[:, 14] == tab[:, 4]) & (q[:, 15] == tab[:, 5])
    assert same.mean() > 0.998
    ok = same & (tab[:, 6] >= 0) & (q[:, 17] == tab[:, 7])
    assert ok.sum() > 0.9 * len(tab)
    d = np.abs(q[ok][:, [2, 8]] - tab[ok][:, [2, 3]]).max(1)
    assert np.percentile(d, 98) < 1e-4 and d.max() < 1.5e-3
    assert np.abs(q[ok, 16] - tab[ok, 6]).max() < 1e-5


@pytest.mark.parametrize("wpp", ["1", "2"])
@pytest.mark.parametrize("order", [1, 2])
def test_icgn2d_warps_per_poi_variants(engine, cfg_a, monkeypatch, wpp, order):
    """The launch picks one or two warps per POI from the queue length (icgn2d.cu icgn2d_launch); both code paths must
    meet the same parity bar, also with sentinels, an odd row split and the LM variant of the same order (ICLM2D1,
    ICLM2D2: icgn2d_kernel<6 or 12, 0, true, WPP>)."""
    monkeypatch.setenv("OCB_ICGN2D_WPP", wpp)
    ref, tar, xy, _ = cfg_a
    o = Oracle2D(ref, tar)
    for rx, ry in ((15, 15), (16, 13)):
        q = ob.make_poi2d(np.vstack([xy, [[3, 3], [ref.shape[1] - 2, 50]]]).astype(np.float32))
        o.fftcc2d(q, rx, ry)
        a, b = q.copy(), q.copy()
        cls = ob.ICGN2D1 if order == 1 else ob.ICGN2D2
        ic = cls(rx, ry, 0.001, 10, engine=engine)
        ic.set_images(ref, tar)
        ic.prepare()
        ic.compute(a)
        (o.icgn2d1 if order == 1 else o.icgn2d2)(b, rx, ry, 0.001, 10)
        got = engine.last_launch()
        assert got.get("np") == 6 * order and got.get("wpp") == int(wpp) and got.get("lm") == 0 and got.get("tm") == 0, \
            "wpp=%s order=%d: ran %s" % (wpp, order, got)
        util.compare_2d(a, b, "wpp=%s order=%d r=(%d,%d)" % (wpp, order, rx, ry), order=order)
        assert a[-1, 16] == -3 and a[-2, 16] == -3
    lm = (ob.ICLM2D1 if order == 1 else ob.ICLM2D2)(16, 16, 0.001, 10, engine=engine)
    lm.set_images(ref, tar)
    lm.prepare()
    q = ob.make_poi2d(xy)
    o.fftcc2d(q, 16, 16)
    a, b = q.copy(), q.copy()
    lm.compute(a)
    got = engine.last_launch()
    assert got.get("np") == 6 * order and got.get("wpp") == int(wpp) and got.get("lm") == 1 and got.get("rc") == 0, \
        "ICLM wpp=%s order=%d: ran %s" % (wpp, order, got)
    o.iclm2d(order, b, 16, 16, 0.001, 10)
    same = a[:, 17] == b[:, 17]
    assert same.mean() > 0.97
    assert np.abs(a[same][:, [2, 8]] - b[same][:, [2, 8]]).max() < 1e-4


def test_icgn2d2_known_answers(engine):
    """ICGN2D2 seeded with the u0, v0 of the reference's shipped GPU table examples/2d_dic/oht_cfrp_4_sift_icgn2(gpu)_r16.csv
    (see tests/test_oracle_golden.py::test_icgn2d2_known_answers for why only the same-iteration rows are compared)."""
    ref, tar = util.oht_cfrp_pair()
    tab = util.oht_cfrp_icgn2_golden()["table"]
    q = ob.make_poi2d(tab[:, 0:2])
    q[:, 2], q[:, 8] = tab[:, 4], tab[:, 5]
    ic = ob.ICGN2D2(16, 16, 0.001, 10, engine=engine)
    ic.set_images(ref, tar)
    ic.prepare()
    ic.compute(q)
    ok = (q[:, 17] == tab[:, 7]) & (tab[:, 7] < 10) & (tab[:, 6] >= 0.9)
    assert ok.mean() > 0.6
    d = np.abs(q[ok][:, [2, 8]] - tab[ok][:, [2, 3]]).max(1)
    assert np.percentile(d, 99) < 1e-4 and np.median(d) < 2e-5
    assert np.abs(q[ok, 16] - tab[ok, 6]).max() < 1e-5


def test_self_adaptive_icgn2d1_known_answers(engine):
    """Per-POI subset radii through ocb_icgn2d_ex vs the reference's shipped examples/2d_dic/utn_30_self_adaptive.csv."""
    ref, tar, tab = util.utn_self_adaptive_fixture()
    q = util.utn_self_adaptive_queue(tab)
    ic = ob.ICGN2D1(30, 30, 0.001, 10, engine=engine)
    ic.set_images(ref, tar)
    ic.set_self_adaptive(True)
    ic.prepare()
    ic.compute(q)
    assert (q[:, 16] > 0.9).all()
    assert np.abs(q[:, [2, 8]] - tab[:, [2, 3]]).max() < 1.5e-4     # displacements of ~480 px: a float32 ulp is 3e-5 there
    assert np.abs(q[:, 16] - tab[:, 6]).max() < 1e-5
    assert np.array_equal(q[:, 23:25], tab[:, 13:15])


def test_u8_upload_of_odd_sized_images(engine):
    """Pixel counts that are not a multiple of 4 (501 x 333): the second image of the 8-bit staging buffer must still start
    on an aligned address (the widening kernel reads uchar4)."""
    ref, tar = synth.speckle_pair_2d(501, 333)
    xy = synth.grid_2d(40, 40, 14, 9, 30, 28)
    res = []
    for cast in (np.float32, np.uint8):
        q = ob.make_poi2d(xy)
        engine.set_images_2d(ref.astype(cast), tar.astype(cast))
        engine.fftcc2d(q, 16, 16)
        engine.icgn2d_prepare()
        engine.icgn2d1(q, 16, 16, 0.001, 10)
        res.append(q)
    assert np.array_equal(res[0], res[1])
    assert (res[0][:, 16] > 0.9).all()


def test_two_operators_with_different_pairs_interleaved(engine):
    """Each DIC object keeps ITS image pair and prepared state, like the reference's per-object tables: preparing B between
    A.prepare() and A.compute() must not change A's result (nor make it fail)."""
    ref_a, tar_a = synth.speckle_pair_2d(320, 300)
    ref_b, tar_b = synth.speckle_pair_2d(320, 300, seed=99)
    xy = synth.grid_2d(40, 40, 10, 9, 24, 24)
    seed_a, seed_b = ob.make_poi2d(xy), ob.make_poi2d(xy)
    Oracle2D(ref_a, tar_a).fftcc2d(seed_a, 16, 16)
    Oracle2D(ref_b, tar_b).fftcc2d(seed_b, 16, 16)

    def alone(ref, tar, seed):
        q = seed.copy()
        op = ob.ICGN2D1(16, 16, 0.001, 10, engine=engine)
        op.set_images(ref, tar)
        op.prepare()
        op.compute(q)
        return q

    want_a, want_b = alone(ref_a, tar_a, seed_a), alone(ref_b, tar_b, seed_b)
    assert not np.array_equal(want_a[:, 2], want_b[:, 2])
    a = ob.ICGN2D1(16, 16, 0.001, 10, engine=engine)
    b = ob.ICGN2D1(16, 16, 0.001, 10, engine=engine)
    a.set_images(ref_a, tar_a)
    a.prepare()
    b.set_images(ref_b, tar_b)
    b.prepare()
    qa, qb = seed_a.copy(), seed_b.copy()
    a.compute(qa)  # B's images are on the device at this point
    b.compute(qb)
    assert np.array_equal(qa, want_a) and np.array_equal(qb, want_b)
    f = ob.FFTCC2D(16, 16, engine=engine)
    f.set_images(ref_a, tar_a)
    qb = seed_b.copy()
    b.compute(qb)  # and again after a third object took the engine
    assert np.array_equal(qb, want_b)


def test_large_deformation_gradient_tensor_memory_variant(engine):
    """The 12 % stretch of test_large_deformation_gradient_falls_back_to_global_reads on a queue of 3 136 POIs: the
    Tensor-Memory variant of the kernel, whose row-by-row path fetches a lane's constants from TMEM one row at a time."""
    ref, _ = synth.speckle_pair_2d(704, 704)
    yy, xx = np.mgrid[0:704, 0:704].astype(np.float32)
    o_ref = Oracle2D(ref, ref)
    o_ref.prepare()
    src = np.stack([(352 + (xx - 352) / 1.12).ravel(), (352 + (yy - 352) / 1.12).ravel()], 1)
    tar = np.clip(o_ref.bicubic(src), 0, 255).reshape(704, 704).astype(np.float32)
    xy = synth.grid_2d(100, 100, 56, 56, 9, 9)
    q = ob.make_poi2d(xy)
    q[:, 2] = (xy[:, 0] - 352) * 0.12
    q[:, 8] = (xy[:, 1] - 352) * 0.12
    q[:, 3] = 0.12
    q[:, 10] = 0.12
    q_gpu, q_cpu = q.copy(), q.copy()
    engine.set_images_2d(ref, tar)
    engine.icgn2d_prepare()
    engine.icgn2d1(q_gpu, 16, 16, 0.001, 10)
    Oracle2D(ref, tar).icgn2d1(q_cpu, 16, 16, 0.001, 10)
    assert (q_cpu[:, 16] > 0.9).all()
    stats = util.compare_2d(q_gpu, q_cpu, "stretch, TM variant", max_iter_mismatch_frac=0.05)
    assert stats["n_compared"] > 0.9 * len(q)
