"""Acceptance: the reference's own example programs, compiled UNCHANGED against the C++ shim
(build() -> oracle/Makefile ref-examples -> oracle/_ref/bin/test_2d_dic_fftcc_icgn1, ..., from the OpenCorr
checkout), run on the GPU and reproduce the reference's shipped result tables;
this repo's own shim programs (examples/bin/) run on the committed example pair."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "examples", "bin")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "bin")
REF_MISSING = "reference example program not in oracle/_ref/bin/: build() found no OpenCorr checkout (oracle/Makefile, OPENCORR_REF)"


def _read_table(path):
    with open(path) as f:
        header = f.readline().strip().strip(",").split(",")
        rows = [[float(x) for x in line.strip().strip(",").split(",")] for line in f if line.strip()]
    return header, np.array(rows)


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_BIN, "test_2d_dic_fftcc_icgn1")), reason=REF_MISSING)
def test_reference_2d_example_runs_unchanged(tmp_path):
    data = tmp_path / "d:" / "dic_tests" / "2d_dic"  # the example hard-codes d:/dic_tests/2d_dic/...
    data.mkdir(parents=True)
    for name in ("oht_cfrp_0.bmp", "oht_cfrp_4.bmp"):
        shutil.copyfile(os.path.join(util.GOLDEN, name), data / name)
    out = subprocess.run([os.path.join(REF_BIN, "test_2d_dic_fftcc_icgn1")], cwd=tmp_path, stdin=subprocess.DEVNULL,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "30000 POIs" in out.stdout
    header, tab = _read_table(data / "oht_cfrp_4_fftcc_icgn1_r16.csv")
    assert header[:9] == ["x", "y", "u", "v", "u0", "v0", "ZNCC", "iteration", "convergence"]
    assert tab.shape[0] == 30000
    g = util.oht_cfrp_golden()
    gold, rows = g["table"], g["rows"]
    mine = tab[rows]
    assert np.array_equal(mine[:, 0:2], gold[:, 0:2])
    same_guess = (mine[:, 4] == gold[:, 4]) & (mine[:, 5] == gold[:, 5])
    assert same_guess.mean() > 0.998
    ok = same_guess & (gold[:, 7] < 10) & (mine[:, 7] == gold[:, 7])
    assert ok.sum() > 0.93 * len(gold)
    assert np.abs(mine[ok][:, 2:4] - gold[ok][:, 2:4]).max() < 1e-4
    assert np.abs(mine[ok, 6] - gold[ok, 6]).max() < 1e-5
    # the other files the example writes
    for suffix in ("_deformation.csv", "_u.csv", "_v.csv", "_time.csv"):
        assert (data / ("oht_cfrp_4_fftcc_icgn1_r16" + suffix)).exists()
    _, dtab = _read_table(data / "oht_cfrp_4_fftcc_icgn1_r16_deformation.csv")
    gd = g["deformation"]
    assert np.abs(dtab[rows][ok][:, [3, 4, 9, 10]] - gd[ok][:, [3, 4, 6, 7]]).max() < 2e-5  # ux uy vx vy


@pytest.mark.skipif(not os.path.exists(os.path.join(BIN, "dic_fftcc_icgn1_demo")), reason="demo binary not built")
def test_shim_demo(tmp_path):
    out_csv = tmp_path / "out.csv"
    out = subprocess.run([os.path.join(BIN, "dic_fftcc_icgn1_demo"), os.path.join(util.GOLDEN, "oht_cfrp_0.bmp"),
                          os.path.join(util.GOLDEN, "oht_cfrp_4.bmp"), str(out_csv), "16", "8"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    _, tab = _read_table(out_csv)
    assert tab.shape[0] > 1000 and (tab[:, 6] > 0.9).mean() > 0.9


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_BIN, "test_2d_dic_fftcc_iclm1")), reason=REF_MISSING)
def test_reference_2d_iclm_example_runs_unchanged(tmp_path):
    """examples/test_2d_dic_fftcc_iclm1.cpp of the reference, compiled unchanged against the shim."""
    data = tmp_path / "d:" / "dic_tests" / "2d_dic"
    data.mkdir(parents=True)
    for name in ("oht_cfrp_0.bmp", "oht_cfrp_4.bmp"):
        shutil.copyfile(os.path.join(util.GOLDEN, name), data / name)
    out = subprocess.run([os.path.join(REF_BIN, "test_2d_dic_fftcc_iclm1")], cwd=tmp_path, stdin=subprocess.DEVNULL,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    _, tab = _read_table(data / "oht_cfrp_4_fftcc_iclm1_r16.csv")
    g = util.oht_cfrp_iclm_golden()
    gold, rows = g["table"], g["rows"]
    mine = tab[rows]
    same = (mine[:, 4] == gold[:, 4]) & (mine[:, 5] == gold[:, 5])
    ok = same & (gold[:, 6] >= 0) & (mine[:, 7] == gold[:, 7])
    assert ok.sum() > 0.9 * len(gold)
    d = np.abs(mine[ok][:, 2:4] - gold[ok][:, 2:4]).max(1)
    assert np.percentile(d, 98) < 1e-4 and d.max() < 1.5e-3


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_BIN, "test_2d_dic_fftcc_nr1")), reason=REF_MISSING)
def test_reference_2d_nr_example_runs_unchanged(tmp_path):
    """examples/test_2d_dic_fftcc_nr1.cpp of the reference (FFTCC2D -> NR2D1 -> Strain), compiled unchanged."""
    data = tmp_path / "d:" / "dic_tests" / "2d_dic"
    data.mkdir(parents=True)
    for name in ("oht_cfrp_0.bmp", "oht_cfrp_4.bmp"):
        shutil.copyfile(os.path.join(util.GOLDEN, name), data / name)
    out = subprocess.run([os.path.join(REF_BIN, "test_2d_dic_fftcc_nr1")], cwd=tmp_path, stdin=subprocess.DEVNULL,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    header, tab = _read_table(data / "oht_cfrp_4_fftcc_nr1_r16.csv")
    assert header[:13] == ["x", "y", "u", "v", "u0", "v0", "ZNCC", "iteration", "convergence", "feature", "exx", "eyy", "exy"]
    assert tab.shape[0] == 30000
    g = util.oht_cfrp_nr_golden()
    gold, rows = g["table"], g["rows"]
    mine = tab[rows]
    assert np.array_equal(mine[:, 4:6], gold[:, 4:6])
    ok = (gold[:, 7] < 10) & (mine[:, 7] == gold[:, 7]) & (gold[:, 6] >= 0.9)
    assert ok.sum() > 0.9 * len(gold)
    assert np.abs(mine[ok][:, 2:4] - gold[ok][:, 2:4]).max() < 1e-4
    assert np.abs(mine[ok, 6] - gold[ok, 6]).max() < 1e-5
    # Strain ran on this table's own u, v, ZNCC: recompute it with the oracle from the printed values
    from oracle import oracle
    q = np.zeros((tab.shape[0], 25), np.float32)
    q[:, 0:2], q[:, 2], q[:, 8], q[:, 16] = tab[:, 0:2], tab[:, 2], tab[:, 3], tab[:, 6]
    oracle.strain(q, 20.0, 5, 0.9, 1, exact=True)
    # (a ZNCC printed as 0.90000000 may have been just below the threshold: allow a handful of such POIs and their
    # neighbours to differ)
    assert ((q[:, 20] == 0) != (tab[:, 10] == 0)).sum() <= 5
    assert np.percentile(np.abs(q[:, 20:23] - tab[:, 10:13]).max(1), 99) < 2e-7   # 8 printed decimals of u, v
    # and against the shipped strains, where the neighbourhood is the same as in the shipped run (the shipped table
    # predates the -4 code, so next to non-converged POIs the neighbour sets differ): the bulk agrees
    band, check = g["band"], g["band_check"]
    idx = {(int(x), int(y)): i for i, (x, y) in enumerate(tab[:, 0:2])}
    sel = np.array([idx[(int(x), int(y))] for x, y in band[:, 0:2]])
    mb = tab[sel]
    conv = check & (band[:, 4] >= 0.9) & (mb[:, 6] >= 0.9)
    assert np.percentile(np.abs(mb[conv][:, 10:13] - band[conv][:, 5:8]).max(1), 50) < 2e-5


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_BIN, "test_2d_dic_strain")), reason=REF_MISSING)
def test_reference_2d_strain_example_runs_unchanged(tmp_path):
    """examples/test_2d_dic_strain.cpp: loadTable2D -> Strain -> saveTable2D / saveMap2D, compiled unchanged.  Its input
    table is written here from the band fixture (the columns saveTable2D writes)."""
    data = tmp_path / "d:" / "dic_tests" / "2d_dic"
    data.mkdir(parents=True)
    shutil.copyfile(os.path.join(util.GOLDEN, "oht_cfrp_4.bmp"), data / "oht_cfrp_4.bmp")
    q, gold, check = util.strain_band_queue()
    with open(data / "oht_cfrp_4_fftcc_icgn1_r16.csv", "w") as f:
        f.write("x,y,u,v,u0,v0,ZNCC,iteration,convergence,feature,exx,eyy,exy,subset_rx,subset_ry,\n")
        for p in q:
            f.write("%g,%g,%.8f,%.8f,0,0,%.8f,3,0.0001,0,0,0,0,16,16,\n" % (p[0], p[1], p[2], p[8], p[16]))
    out = subprocess.run([os.path.join(REF_BIN, "test_2d_dic_strain")], cwd=tmp_path, stdin=subprocess.DEVNULL,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    _, tab = _read_table(data / "oht_cfrp_4_fftcc_icgn1_r16.csv")
    assert tab.shape[0] == q.shape[0] and np.array_equal(tab[:, 0:2], q[:, 0:2])
    good = check & (q[:, 16] >= 0.9)
    assert np.abs(tab[good][:, 10:13] - gold[good]).max() < 5e-7
    assert (data / "oht_cfrp_4_eyy.csv").exists()


def _write_tiff_stack(path, vol):
    """Minimal little-endian multi-page TIFF: 8-bit grayscale, uncompressed, one strip per page."""
    import struct
    nz, ny, nx = vol.shape
    out = bytearray(b"II*\x00\x00\x00\x00\x00")
    prev_next_field = 4
    for z in range(nz):
        data_off = len(out)
        out += vol[z].astype(np.uint8).tobytes()
        if len(out) % 2:
            out += b"\x00"
        ifd_off = len(out)
        struct.pack_into("<I", out, prev_next_field, ifd_off)
        tags = [(256, 4, 1, nx), (257, 4, 1, ny), (258, 3, 1, 8), (259, 3, 1, 1), (262, 3, 1, 1), (273, 4, 1, data_off),
                (277, 3, 1, 1), (278, 4, 1, ny), (279, 4, 1, nx * ny)]
        out += struct.pack("<H", len(tags))
        for tag, typ, cnt, val in tags:
            out += struct.pack("<HHI", tag, typ, cnt) + (struct.pack("<HH", val, 0) if typ == 3 else struct.pack("<I", val))
        prev_next_field = len(out)
        out += struct.pack("<I", 0)
    with open(path, "wb") as f:
        f.write(out)


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_BIN, "test_dvc_strain")), reason=REF_MISSING)
def test_reference_dvc_strain_example_runs_unchanged(tmp_path):
    """examples/test_dvc_strain.cpp: Image3D(.tif) for the dimensions, loadTable3D -> Strain -> saveTable3D."""
    data = tmp_path / "d:" / "dic_tests" / "dvc"
    data.mkdir(parents=True)
    _write_tiff_stack(data / "Torus_def.tif", (np.arange(4 * 6 * 8) % 251).reshape(4, 6, 8))
    q, gold, check = util.torus_queue()
    with open(data / "Torus_def_sift_icgn1_r16.csv", "w") as f:
        f.write(",".join("x,y,z,u,v,w,u0,v0,w0,ZNCC,iteration,convergence,feature,ux,uy,uz,vx,vy,vz,wx,wy,wz,exx,eyy,ezz,exy,eyz,ezx,"
                         "subset_rx,subset_ry,subset_rz".split(",")) + ",\n")
        for p in q:
            f.write("%g,%g,%g,%.8f,%.8f,%.8f,0,0,0,%.8f,5,0.0001,0," % (p[0], p[1], p[2], p[3], p[7], p[11], p[18])
                    + "0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,16,16,16,\n")
    out = subprocess.run([os.path.join(REF_BIN, "test_dvc_strain")], cwd=tmp_path, stdin=subprocess.DEVNULL,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    _, tab = _read_table(data / "Torus_def_sift_icgn1_r16.csv")
    assert tab.shape[0] == q.shape[0] and np.array_equal(tab[:, 0:3], q[:, 0:3])
    good = check & (q[:, 18] >= 0.9)
    assert np.abs(tab[good][:, 22:28] - gold[good]).max() < 5e-6
    assert (data / "Torus_def_strain_r30_time.csv").exists()


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_BIN, "test_3d_dic_strain")), reason=REF_MISSING)
def test_reference_stereo_strain_example_runs_unchanged(tmp_path):
    """examples/test_3d_dic_strain.cpp: Image2D(.tif) for the size, loadTable2DS -> Strain(POI2DS) -> saveTable2DS."""
    data = tmp_path / "d:" / "dic_tests" / "3d_dic"
    data.mkdir(parents=True)
    _write_tiff_stack(data / "GT4-0273_0.tif", (np.arange(12 * 16) % 251).reshape(1, 12, 16))
    q, gold, check = util.gt4_stereo_queue()
    cols = "x,y,u,v,w,r1r2 ZNCC,r1t1 ZNCC,r1t2 ZNCC,r2_x,r2_y,t1_x,t1_y,t2_x,t2_y,ref_x,ref_y,ref_z,tar_x,tar_y,tar_z,exx,eyy,ezz,exy,eyz,ezx,subset_rx,subset_ry"
    with open(data / "GT4-0273_0_epipolar_sift_r16.csv", "w") as f:
        f.write(cols + ",\n")
        for p in q:
            f.write(",".join("%.9g" % v for v in p[:20]) + ",0,0,0,0,0,0,16,16,\n")
    out = subprocess.run([os.path.join(REF_BIN, "test_3d_dic_strain")], cwd=tmp_path, stdin=subprocess.DEVNULL,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    header, tab = _read_table(data / "GT4-0273_0_epipolar_sift_r16.csv")
    assert header == cols.split(",")
    assert tab.shape[0] == q.shape[0] and np.array_equal(tab[:, 0:2], q[:, 0:2])
    good = check & np.all(q[:, 5:8] >= 0.9, axis=1)
    d = np.abs(tab[good][:, 20:26] - gold[good]).max(1)
    assert np.median(d) < 2e-5 and d.max() < 1e-3


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_BIN, "test_dvc_fftcc_icgn1")), reason=REF_MISSING)
def test_reference_dvc_example_runs_unchanged(tmp_path):
    """examples/test_dvc_fftcc_icgn1.cpp of the reference (north_star's second acceptance program: FFTCC3D -> ICGN3D1 with 61^3
    subvolumes on al_foam4_{0,1}.bin, 7 x 7 x 117 POIs), compiled unchanged against the shim.  The example hard-codes
    d:/dic_tests/dvc/al_foam4_{0,1}.bin (100 x 100 x 706 voxels); the committed fixture holds z-slices [18, 118) of that pair,
    so the volumes are rebuilt at full size with the remaining slices zero.  The POIs at z = 60..75 (the first four layers of
    the grid, 196 POIs) see only fixture data -- their 61^3 subvolumes, the 60^3 FFT-CC windows and the 15-tap prefilter stay
    inside [23, 112] -- and must reproduce the rows of the table the reference ships
    (examples/dvc/al_foam4_1_fftcc_icgn1_r30.csv); the other POIs reach into the zero padding and only have to come back."""
    ref, tar, z0, cpu_tab, _ = util.al_foam_crop()
    data = tmp_path / "d:" / "dic_tests" / "dvc"
    data.mkdir(parents=True)
    for name, crop in (("al_foam4_0.bin", ref), ("al_foam4_1.bin", tar)):
        vol = np.zeros((706, 100, 100), np.float32)
        vol[z0:z0 + crop.shape[0]] = crop
        with open(data / name, "wb") as f:
            np.array([100, 100, 706], np.int32).tofile(f)  # dim_x, dim_y, dim_z header, src/oc_image.cpp:76-110
            vol.tofile(f)
    out = subprocess.run([os.path.join(REF_BIN, "test_dvc_fftcc_icgn1")], cwd=tmp_path, stdin=subprocess.DEVNULL,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "5733 POIs" in out.stdout
    header, tab = _read_table(data / "al_foam4_1_fftcc_icgn1_r30.csv")
    assert header[:12] == ["x", "y", "z", "u", "v", "w", "u0", "v0", "w0", "ZNCC", "iteration", "convergence"]
    assert tab.shape[0] == 5733
    mine = tab[:196]  # the grid runs z-slowest: the first 4 x 49 rows are z = 60, 65, 70, 75
    assert np.array_equal(mine[:, 0:3], cpu_tab[:, 0:3])
    assert np.array_equal(mine[:, 6:9], cpu_tab[:, 6:9]), "FFT-CC guess differs from the shipped table"
    same_it = mine[:, 10] == cpu_tab[:, 10]
    assert same_it.mean() > 0.97
    # the shipped CPU table carries the float32 summation noise of the reference's sequential sums (61^3 samples):
    # ~3e-5 px / 2e-5 ZNCC away from exact arithmetic (DESIGN.md section 2); the GPU sums are trees
    assert np.abs(mine[same_it][:, 3:6] - cpu_tab[same_it][:, 3:6]).max() < 1e-4
    assert np.abs(mine[same_it, 9] - cpu_tab[same_it, 9]).max() < 5e-5
    assert (data / "al_foam4_1_fftcc_icgn1_r30_time.csv").exists()


@pytest.mark.skipif(not os.path.exists(os.path.join(BIN, "dic_fftcc_icgn1_demo")), reason="demo binary not built")
def test_shim_multi_device_matches_single_device(tmp_path):
    """The C++ shim with OPENCORR_B200_DEVICES=all (a GROUP context: FFTCC2D::compute / ICGN2D1::compute shard their
    std::vector<POI2D> over every visible GPU inside the C ABI) returns the same records as on one GPU: the shim demo (the 2D
    example's calls: FFTCC2D, ICGN2D1, IO2D::saveTable2D) writes byte-identical result tables either way.  (On a one-GPU box
    the group has one member.)"""
    tables = []
    for env_extra in ({"OPENCORR_B200_DEVICE": "0"}, {"OPENCORR_B200_DEVICES": "all"}):
        out_csv = tmp_path / ("run_%s.csv" % "_".join(env_extra.values()))
        env = dict(os.environ)
        env.pop("OPENCORR_B200_DEVICE", None)
        env.pop("OPENCORR_B200_DEVICES", None)
        env.update(env_extra)
        out = subprocess.run([os.path.join(BIN, "dic_fftcc_icgn1_demo"), os.path.join(util.GOLDEN, "oht_cfrp_0.bmp"),
                              os.path.join(util.GOLDEN, "oht_cfrp_4.bmp"), str(out_csv), "16", "2"],
                             stdin=subprocess.DEVNULL, capture_output=True, text=True, timeout=300, env=env)
        assert out.returncode == 0, out.stdout + out.stderr
        tables.append(out_csv.read_bytes())
    _, tab = _read_table(out_csv)
    assert tab.shape[0] > 30000 and (tab[:, 6] > 0.9).mean() > 0.9
    assert tables[0] == tables[1]
