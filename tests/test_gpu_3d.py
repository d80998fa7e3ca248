"""GPU parity, DVC: ICGN3D1::prepare products (bit-exact), FFTCC3D, ICGN3D1 vs the CPU oracle and
vs the reference's golden tables (al_foam4 crop)."""
import numpy as np
import pytest

import opencorr_b200 as ob
from opencorr_b200 import synth
from oracle.oracle import Oracle3D
import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vol():
    ref, tar = synth.speckle_pair_3d(72, 64, 80)
    xyz = synth.grid_3d(24, 22, 26, 4, 3, 4, 7, 9, 8)
    return ref, tar, xyz


def test_prepare_tables_bit_exact(engine, vol):
    ref, tar, _ = vol
    icgn = ob.ICGN3D1(8, 8, 8, 0.001, 20, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    gx, gy, gz, coef = icgn.tables()
    o = Oracle3D(ref, tar)
    o.prepare()
    ogx, ogy, ogz = o.gradients()
    assert np.array_equal(gx, ogx) and np.array_equal(gy, ogy) and np.array_equal(gz, ogz)
    assert np.array_equal(coef, o.coefficients())


@pytest.mark.parametrize("r", [(8, 8, 8), (10, 6, 9), (15, 15, 15)])
def test_fftcc3d_matches_oracle(engine, vol, r):
    ref, tar, xyz = vol
    if max(r) > 10:
        xyz = np.array([[36, 32, 40], [34, 30, 38]], np.float32)
    q_gpu = ob.make_poi3d(xyz)
    q_cpu = q_gpu.copy()
    f = ob.FFTCC3D(*r, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    q_exact = q_cpu.copy()
    Oracle3D(ref, tar).fftcc3d(q_cpu, *r)
    Oracle3D(ref, tar).fftcc3d(q_exact, *r, exact=True)
    assert np.array_equal(q_gpu[:, [3, 7, 11, 15, 16, 17]], q_cpu[:, [3, 7, 11, 15, 16, 17]])
    # 1e-5 against exact arithmetic; the ref-faithful flavour sums up to 27 000 float32 values
    # sequentially (src/oc_fftcc.cpp:346-376) and carries ~1e-5 of its own rounding noise
    assert np.abs(q_gpu[:, 18] - q_exact[:, 18]).max() < 1e-5
    assert np.abs(q_gpu[:, 18] - q_cpu[:, 18]).max() < 5e-5
    assert (q_cpu[:, 18] > 0.3).all()


@pytest.mark.parametrize("r", [4, 5, 6, 9, 10, 12, 18, 20, 24, 25, 27, 32])
def test_fftcc3d_register_kernels(engine, r):
    """Every cubic window fftcc3d_reg.cu serves through the dispatch (one thread per 1D transform, register codelets,
    OCB_F3R_SIZES) apart from r = 15 and 30, which test_fftcc3d_matches_oracle and the golden DVC table cover: N = 2r
    from 8 to 64, with 2 * 5^2 and 2 * 3^3 among them.  r = 16 takes fftcc3d_w32 instead (test_fftcc3d_w32_specialised_kernel),
    so fftcc3d_reg_kernel<32> is never launched.  Includes a POI too close to the border (left untouched) and a non-zero
    incoming guess."""
    ref, tar = synth.speckle_pair_3d(96, 88, 80)
    c = np.array([[48, 44, 40], [50, 41, 38], [44, 46, 42], [3, 44, 40]], np.float32)
    if r > 12:
        c = c[[0, 3]]
    q_gpu = ob.make_poi3d(c)
    q_gpu[0, 3] = 1.0
    q_gpu[0, 11] = -1.4
    q_cpu = q_gpu.copy()
    f = ob.FFTCC3D(r, r, r, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    got = engine.last_launch()
    assert got.get("op") == "fftcc3d" and got.get("kernel") == "reg" and got.get("n") == 2 * r, \
        "r=%d: expected kernel=reg n=%d, ran %s" % (r, 2 * r, got)
    o = Oracle3D(ref, tar)
    o.fftcc3d(q_cpu, r, r, r, exact=True)
    assert q_cpu[0, 18] > 0.3  # the window (and the guess) fit the volume: a real correlation, not a skipped POI
    assert np.array_equal(q_gpu[:, [3, 7, 11, 15, 16, 17]], q_cpu[:, [3, 7, 11, 15, 16, 17]])
    assert np.abs(q_gpu[:, 18] - q_cpu[:, 18]).max() < 1e-5
    assert q_gpu[-1, 18] == 0 and np.all(q_gpu[-1, 3:15] == 0)


def test_fftcc3d_generic_kernel_still_matches(engine, vol, monkeypatch):
    """The Stockham kernel stays the fallback (non-cubic windows, other prime factors)."""
    monkeypatch.setenv("OCB_FFTCC3D_GENERIC", "1")
    ref, tar, xyz = vol
    for r in (8, 7):
        q_gpu = ob.make_poi3d(xyz)
        q_cpu = q_gpu.copy()
        f = ob.FFTCC3D(r, r, r, engine=engine)
        f.set_images(ref, tar)
        f.compute(q_gpu)
        Oracle3D(ref, tar).fftcc3d(q_cpu, r, r, r, exact=True)
        assert np.array_equal(q_gpu[:, [3, 7, 11, 15, 16, 17]], q_cpu[:, [3, 7, 11, 15, 16, 17]])
        assert np.abs(q_gpu[:, 18] - q_cpu[:, 18]).max() < 1e-5


def test_fftcc3d_out_of_volume_pois_are_left_untouched(engine, vol):
    ref, tar, _ = vol
    xyz = np.array([[5, 30, 30], [30, 5, 30], [30, 30, 5], [70, 30, 30], [36, 32, 40]], np.float32)
    q_gpu = ob.make_poi3d(xyz)
    q_gpu[:, 18] = 0.5
    q_cpu = q_gpu.copy()
    f = ob.FFTCC3D(8, 8, 8, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    Oracle3D(ref, tar).fftcc3d(q_cpu, 8, 8, 8)
    assert np.array_equal(q_gpu[:4], q_cpu[:4])
    assert (q_gpu[:4, 18] == 0.5).all() and q_gpu[4, 18] != 0.5


@pytest.mark.parametrize("exact", [0, 1])
def test_icgn3d1_matches_oracle(engine, vol, exact):
    ref, tar, xyz = vol
    r = 8
    q = ob.make_poi3d(xyz)
    o = Oracle3D(ref, tar)
    o.fftcc3d(q, r, r, r)
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN3D1(r, r, r, 0.001, 20, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    o.icgn3d1(q_cpu, r, r, r, 0.001, 20, exact=exact)
    stats = util.compare_3d(q_gpu, q_cpu, "icgn3d1 exact=%d" % exact, max_iter_mismatch_frac=0.05)
    assert stats["n_compared"] >= 0.9 * len(q)
    ok = (q_gpu[:, 18] >= 0) & (q_gpu[:, 19] == q_cpu[:, 19])
    assert np.abs(q_gpu[ok][:, 3:15] - q_cpu[ok][:, 3:15]).max() < 1e-4
    u, v, w = synth.displacement_3d(xyz[:, 0], xyz[:, 1], xyz[:, 2], 72, 64, 80)
    assert np.abs(q_gpu[ok, 3] - u[ok]).max() < 0.1 and np.abs(q_gpu[ok, 11] - w[ok]).max() < 0.1


def test_icgn3d1_sentinels(engine, vol):
    ref, tar, _ = vol
    xyz = np.array([[5, 30, 30], [36, 32, 40], [36, 32, 40], [36, 32, 40], [30, 30, 72]], np.float32)
    q = ob.make_poi3d(xyz)
    q[2, 18] = -1.0          # skipped, keeps its code
    q[3, 3] = 30.0           # guess pushes the subvolume out of the target -> -3
    q[1, 3], q[1, 7], q[1, 11] = 1.0, -1.0, 2.0
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN3D1(8, 8, 8, 0.001, 20, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    Oracle3D(ref, tar).icgn3d1(q_cpu, 8, 8, 8, 0.001, 20)
    assert list(q_cpu[[0, 2, 3, 4], 18]) == [-3, -1, -3, -3]
    assert np.array_equal(q_gpu[[0, 2, 3, 4]], q_cpu[[0, 2, 3, 4]])
    util.compare_3d(q_gpu, q_cpu, "3d sentinels", max_iter_mismatch_frac=0.0)


def test_dvc_golden_tables(engine):
    """FFTCC3D -> ICGN3D1 at r=30 on the al_foam4 crop vs the reference's CPU table, its GPU table
    and the oracle (the reference CPU path carries ~2e-5 of float32 summation noise at 61^3,
    BASELINE.md section 2, so the bound against its CPU table is looser than against its GPU table)."""
    ref, tar, z0, cpu, gpu = util.al_foam_crop()
    sel = np.arange(0, len(cpu), 5)
    xyz = cpu[sel, 0:3].copy()
    xyz[:, 2] -= z0
    q = ob.make_poi3d(xyz)
    f = ob.FFTCC3D(30, 30, 30, engine=engine)
    f.set_images(ref, tar)
    f.compute(q)
    assert np.array_equal(q[:, [3, 7, 11]], cpu[sel][:, 6:9])
    q10 = q.copy()
    icgn = ob.ICGN3D1(30, 30, 30, 0.001, 20, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q)
    same = q[:, 19] == cpu[sel, 10]
    assert same.mean() > 0.9
    assert np.abs(q[same][:, [3, 7, 11]] - cpu[sel][same][:, 3:6]).max() < 1e-4
    assert np.abs(q[same, 18] - cpu[sel][same, 9]).max() < 5e-5
    icgn.set_iteration(0.001, 10)  # the reference GPU table was made with stop=10 (test_dvc_gpu_icgn.cpp:46-50)
    icgn.compute(q10)
    same = (q10[:, 19] == gpu[sel, 10]) & (q10[:, 18] >= 0)
    assert same.mean() > 0.85
    assert np.abs(q10[same][:, [3, 7, 11]] - gpu[sel][same][:, 3:6]).max() < 1e-4
    assert np.abs(q10[same, 18] - gpu[sel][same, 9]).max() < 1e-5


def test_icgn3d1_volume_width_not_multiple_of_four(engine):
    """dim_x % 4 != 0 disables the TMA slab loads; the staged path must agree with the oracle too."""
    ref, tar = synth.speckle_pair_3d(70, 64, 66)
    xyz = synth.grid_3d(24, 22, 24, 3, 3, 2, 8, 9, 9)
    q = ob.make_poi3d(xyz)
    o = Oracle3D(ref, tar)
    o.fftcc3d(q, 8, 8, 8)
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN3D1(8, 8, 8, 0.001, 20, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    o.icgn3d1(q_cpu, 8, 8, 8, 0.001, 20)
    util.compare_3d(q_gpu, q_cpu, "dx=70", max_iter_mismatch_frac=0.1)


def test_icgn3d1_nonuniform_radii_and_large_gradient(engine, vol):
    """Non-cubic subvolume; a 6 % stretch guess drives samples out of the slab tile (global fallback)."""
    ref, tar, _ = vol
    xyz = np.array([[36, 32, 40], [33, 30, 37], [38, 34, 42]], np.float32)
    q = ob.make_poi3d(xyz)
    u, v, w = synth.displacement_3d(xyz[:, 0], xyz[:, 1], xyz[:, 2], 72, 64, 80)
    q[:, 3], q[:, 7], q[:, 11] = u, v, w
    q[2, 4] = 0.06  # ux guess far from the truth: first iterations sample outside the tile
    q_gpu, q_cpu = q.copy(), q.copy()
    icgn = ob.ICGN3D1(10, 7, 9, 0.001, 20, engine=engine)
    icgn.set_images(ref, tar)
    icgn.prepare()
    icgn.compute(q_gpu)
    Oracle3D(ref, tar).icgn3d1(q_cpu, 10, 7, 9, 0.001, 20)
    util.compare_3d(q_gpu, q_cpu, "radii (10,7,9)", max_iter_mismatch_frac=0.34)


def test_fftcc3d_w32_specialised_kernel(engine):
    """radius 16 takes the register-FFT 32^3 kernel; it must agree with the oracle and with the generic
    kernel (selected with OCB_FFTCC3D_GENERIC)."""
    import os
    ref, tar = synth.speckle_pair_3d(80, 76, 72)
    xyz = synth.grid_3d(30, 28, 27, 4, 3, 3, 6, 8, 7)
    q_gpu = ob.make_poi3d(xyz)
    q_gpu[::4, 3] = 1.0   # incoming guesses shift the target window
    q_gpu[::5, 11] = -1.0
    q_cpu, q_gen = q_gpu.copy(), q_gpu.copy()
    f = ob.FFTCC3D(16, 16, 16, engine=engine)
    f.set_images(ref, tar)
    f.compute(q_gpu)
    os.environ["OCB_FFTCC3D_GENERIC"] = "1"
    try:
        f.compute(q_gen)
    finally:
        del os.environ["OCB_FFTCC3D_GENERIC"]
    o = Oracle3D(ref, tar)
    q_exact = q_cpu.copy()
    o.fftcc3d(q_cpu, 16, 16, 16)
    o.fftcc3d(q_exact, 16, 16, 16, exact=True)
    for q in (q_gpu, q_gen):
        assert np.array_equal(q[:, [3, 7, 11, 15, 16, 17]], q_cpu[:, [3, 7, 11, 15, 16, 17]])
        assert np.abs(q[:, 18] - q_exact[:, 18]).max() < 1e-5
    assert (q_cpu[:, 18] > 0.3).all()


def test_u8_volume_upload_gives_identical_results(engine):
    ref, tar, z0, cpu, gpu = util.al_foam_crop()
    xyz = cpu[::40, 0:3].copy()
    xyz[:, 2] -= z0
    res = []
    for cast in (np.float32, np.uint8):
        q = ob.make_poi3d(xyz)
        f = ob.FFTCC3D(16, 16, 16, engine=engine)
        f.set_images(ref.astype(cast), tar.astype(cast))
        f.compute(q)
        icgn = ob.ICGN3D1(16, 16, 16, 0.001, 20, engine=engine)
        icgn.set_images(ref.astype(cast), tar.astype(cast))
        icgn.prepare()
        icgn.compute(q)
        res.append(q)
    assert np.array_equal(res[0], res[1])
    assert (res[0][:, 18] > 0.8).sum() >= 3  # some r=16 foam subvolumes do not converge (-4): same on both paths


def test_u8_upload_of_odd_sized_volume(engine):
    """101 x 99 x 97 voxels (not a multiple of 4): see test_gpu_2d.py::test_u8_upload_of_odd_sized_images."""
    ref, tar = synth.speckle_pair_3d(101, 99, 97)
    xyz = synth.grid_3d(30, 30, 30, 3, 3, 3, 18, 17, 16)
    res = []
    for cast in (np.float32, np.uint8):
        q = ob.make_poi3d(xyz)
        engine.set_images_3d(ref.astype(cast), tar.astype(cast))
        engine.fftcc3d(q, 8, 8, 8)
        engine.icgn3d_prepare()
        engine.icgn3d1(q, 8, 8, 8, 0.001, 20)
        res.append(q)
    assert np.array_equal(res[0], res[1])
    assert (res[0][:, 18] > 0.9).all()
