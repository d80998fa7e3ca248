"""Regenerates the committed fixtures under tests/golden/ from the reference checkout.

Run where the OpenCorr checkout is (OPENCORR_REF, default /root/reference, as in oracle/Makefile):  python tests/golden/make_golden.py
Only DATA is copied (images, sub-sampled result tables the reference ships as its regression
fixtures, examples/2d_dic and examples/dvc); no reference source code.

Outputs
  oht_cfrp_0.bmp, oht_cfrp_4.bmp    the 2D example pair (280x900, 8-bit), verbatim
  oht_cfrp_4_fftcc_icgn1_r16.npz    every 23rd row of the shipped result table + deformation table, plus the three rows whose
                                    FFT-CC guess is an exact tie between two correlation bins (fftcc_tie_rows / fftcc_tie_table)
  oht_cfrp_4_fftcc_icgn1_r16_full.npz  all 30 000 rows of that table, the columns the oracle is checked on: x, y, u0, v0, iteration
                                    (int16 / int8) and u, v, ZNCC (float64, as printed)
  oht_cfrp_4_fftcc_iclm1_r16.npz    the same rows of the shipped ICLM2D1 table
  oht_cfrp_4_sift_icgn2_gpu_r16.npz every 23rd row of examples/2d_dic/oht_cfrp_4_sift_icgn2(gpu)_r16.csv (the reference's GPU ICGN2D2,
                                    SIFT-seeded): x,y,u,v,u0,v0,ZNCC,iteration,convergence.  u0, v0 are the seeds; the affine part
                                    of the seed is not in the table, so iteration counts agree on ~70 % of the rows only
  utn_30_self_adaptive_crop.npz     561 POIs (x in [1500,1700], y in [150,350], every third) of the shipped self-adaptive-subset table
                                    examples/2d_dic/utn_30_self_adaptive.csv (all 15 columns incl. the per-POI subset radii) and the
                                    parts of utn_00.bmp / utn_30.bmp they touch (the target window is ~480 px away: 30 % strain); the
                                    test pastes the crops into zero images of the full 3751x501 size -- checked here to give the
                                    oracle bit-identical results to the full images
  oht_cfrp_4_fftcc_nr1_r16.npz      every 23rd row of the shipped NR2D1 table (x,y,u,v,u0,v0,ZNCC,iteration,convergence)
                                    + a 96-row band (y in [370,560), all 100 columns, includes the specimen's hole)
                                    of x,y,u,v,ZNCC,exx,eyy,exy for the Strain test; rows with `band_check` have
                                    their whole 20-px neighbourhood inside the band
  torus_strain_crop.npz             a box of the shipped DVC table examples/dvc/Torus_def_sift_icgn1_r16.csv
                                    (x,y,z,u,v,w,ZNCC + 6 strains) for the 3D Strain test, same idea
  gt4_stereo_strain_crop.npz        the POIs with 600 <= x <= 1100, 400 <= y <= 800 of the shipped stereo-DIC table
                                    examples/3d_dic/GT4-0273_0_epipolar_sift_r16.csv (all 26 columns: x, y, u, v, w, three ZNCCs,
                                    matched positions, ref/tar 3D coordinates, 6 strains) for the POI2DS Strain test; `check` marks
                                    the POIs whose 20-px neighbourhood lies inside the crop
  step18_epipolar_crop.npz          stereo pair examples/3d_dic/"Step18 00,00-0005_{0,1}.tif" (2448x2048, 8-bit) cut down to what the
                                    60 POIs x = 1170..1215, y = 1000..1025 of test_3d_reconstruction_epipolar.cpp touch
                                    (view 1: the subsets; view 2: the +-150 px candidate sweep along the epipolar lines), the
                                    fundamental matrix of that example's calibration (float32, as updateFundementalMatrix
                                    forms it) and the shipped rows (x, y, ZNCC, r2_x, r2_y) of those POIs.  The test pastes the
                                    crops into zero images of the full size; make_golden checks that the oracle's results on
                                    the pasted images equal those on the full images bit for bit.
  al_foam4_crop.npz                 z-slices [18,118) of the DVC example pair as uint8 (values are
                                    integral, 52..202) + the shipped CPU and GPU result rows of the
                                    196 POIs with z in {60,65,70,75}.  The 15-tap prefilter and the
                                    subsets of those POIs never reach within 7 voxels of the cut, so
                                    results on the crop equal results on the full volume.
"""
import os
import shutil

import numpy as np

REF = os.path.join(os.environ.get("OPENCORR_REF", "/root/reference"), "examples")
OUT = os.path.dirname(os.path.abspath(__file__))


def step18_fundamental():
    """EpipolarSearch::updateFundementalMatrix (src/oc_epipolar_search.cpp:110-126) for the calibration hard-coded in
    examples/test_3d_reconstruction_epipolar.cpp:46-88, in float32."""
    f32 = np.float32

    def rot(rx, ry, rz):  # Calibration::updateRotationMatrix, src/oc_calibration.cpp:50-60 (Eigen AngleAxis)
        v = np.array([rx, ry, rz], f32)
        th = f32(np.linalg.norm(v))
        x, y, z = v / th
        c, s = f32(np.cos(th)), f32(np.sin(th))
        t = f32(1) - c
        return np.array([[t * x * x + c, t * x * y - s * z, t * x * z + s * y], [t * x * y + s * z, t * y * y + c, t * y * z - s * x],
                         [t * x * z - s * y, t * y * z + s * x, t * z * z + c]], f32)

    k1 = np.array([[10664.80664, 0, 1176.03418], [0, 10643.88965, 914.7337036], [0, 0, 1]], f32)
    k2 = np.array([[10749.53223, 0, 1034.707886], [0, 10726.52441, 1062.162842], [0, 0, 1]], f32)
    t2 = np.array([250.881488962793, -1.15469183120196, 37.4849858174401], f32)
    r2 = rot(0.01450813, -0.39152833, 0.01064092)
    tx = np.array([[0, -t2[2], t2[1]], [t2[2], 0, -t2[0]], [-t2[1], t2[0], 0]], f32)
    e = (tx @ r2).astype(f32)
    return (np.linalg.inv(k2.astype(np.float64)).T.astype(f32) @ e @ np.linalg.inv(k1.astype(np.float64)).astype(f32)).astype(f32)


def make_self_adaptive_fixture():
    """examples/test_2d_dic_self_adaptive_subset.cpp: ICGN2D1 with setSelfAdaptive(true) after SIFT + FeatureAffine.  The table
    keeps the seeds' translation (u0, v0) and the per-POI radii; the affine part of the seed is approximated by the table's
    strains (exx ~ ux, eyy ~ vy), which is enough for IC-GN to land on the same optimum."""
    import struct
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
    from oracle.oracle import Oracle2D

    def read_bmp8(path):
        with open(path, "rb") as f:
            b = f.read()
        off, w, h, bpp = struct.unpack_from("<I", b, 10)[0], struct.unpack_from("<i", b, 18)[0], struct.unpack_from("<i", b, 22)[0], struct.unpack_from("<H", b, 28)[0]
        assert bpp == 8
        stride = (w + 3) // 4 * 4
        img = np.frombuffer(b, np.uint8, stride * abs(h), off).reshape(abs(h), stride)[:, :w]
        return (img[::-1] if h > 0 else img).astype(np.float32)

    ref = read_bmp8(os.path.join(REF, "2d_dic", "utn_00.bmp"))
    tar = read_bmp8(os.path.join(REF, "2d_dic", "utn_30.bmp"))
    t = np.genfromtxt(os.path.join(REF, "2d_dic", "utn_30_self_adaptive.csv"), delimiter=",", skip_header=1)[:, :15]
    box = (t[:, 0] >= 1500) & (t[:, 0] <= 1700) & (t[:, 1] >= 150) & (t[:, 1] <= 350)
    tb = t[box][::3]

    def run(a, b):
        q = np.zeros((len(tb), 25), np.float32)
        q[:, 0:2] = tb[:, 0:2]
        q[:, 2], q[:, 8], q[:, 3], q[:, 10] = tb[:, 4], tb[:, 5], tb[:, 10], tb[:, 11]
        q[:, 23], q[:, 24] = tb[:, 13], tb[:, 14]
        Oracle2D(a, b).icgn2d_ex(1, q, 30, 30, 0.001, 10, None, True)
        return q

    m = int(max(tb[:, 13].max(), tb[:, 14].max())) + 8
    a0 = (max(0, int(tb[:, 1].min()) - m), min(ref.shape[0], int(tb[:, 1].max()) + m + 1),
          max(0, int(tb[:, 0].min()) - m), min(ref.shape[1], int(tb[:, 0].max()) + m + 1))
    tx, ty = tb[:, 0] + tb[:, 2], tb[:, 1] + tb[:, 3]
    m2 = int(m * 1.45) + 10
    b0 = (max(0, int(ty.min()) - m2), min(tar.shape[0], int(ty.max()) + m2 + 1), max(0, int(tx.min()) - m2), min(tar.shape[1], int(tx.max()) + m2 + 1))
    mr, mt = np.zeros_like(ref), np.zeros_like(tar)
    mr[a0[0]:a0[1], a0[2]:a0[3]] = ref[a0[0]:a0[1], a0[2]:a0[3]]
    mt[b0[0]:b0[1], b0[2]:b0[3]] = tar[b0[0]:b0[1], b0[2]:b0[3]]
    assert np.array_equal(run(mr, mt), run(ref, tar)), "crop changes the result"
    np.savez_compressed(os.path.join(OUT, "utn_30_self_adaptive_crop.npz"), shape=np.array(ref.shape),
                        ref=ref[a0[0]:a0[1], a0[2]:a0[3]].astype(np.uint8), ref_origin=np.array([a0[0], a0[2]]),
                        tar=tar[b0[0]:b0[1], b0[2]:b0[3]].astype(np.uint8), tar_origin=np.array([b0[0], b0[2]]), table=tb,
                        columns=np.array("x,y,u,v,u0,v0,ZNCC,iteration,convergence,feature,exx,eyy,exy,subset_rx,subset_ry".split(",")))


def make_epipolar_fixture():
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
    from oracle import oracle as orc
    from oracle.oracle import Oracle2D

    def load_tif(name):  # uncompressed 8-bit single-strip TIFF, pixel data at offset 8
        b = open(os.path.join(REF, "3d_dic", name), "rb").read()
        return np.frombuffer(b[8:8 + 2448 * 2048], np.uint8).reshape(2048, 2448).astype(np.float32)

    v1, v2 = load_tif("Step18 00,00-0005_0.tif"), load_tif("Step18 00,00-0005_1.tif")
    fm = step18_fundamental()
    tab = np.genfromtxt(os.path.join(REF, "3d_dic", "Step18 00,00-0005_1_reconstruction_epipolar.csv"), delimiter=",", skip_header=1)
    blk = tab.reshape(313, 313, 8)[150:156, 150:160].reshape(-1, 8)

    def run(a, b, legacy):
        orc.set_legacy_no_minus4(legacy)
        q = np.zeros((len(blk), 25), np.float32)
        q[:, 0:2] = blk[:, 0:2]
        o = Oracle2D(a, b)
        o.epipolar_search(q, fm, [0, 0, -30], [0, 0, -40], 150, 4, 20, 20, 0.05, 5)
        c = q.copy()
        o.icgn2d2(q, 9, 9, 0.001, 10)
        orc.set_legacy_no_minus4(0)
        return c, q

    c_full, q_full = run(v1, v2, 1)
    x, y = blk[:, 0], blk[:, 1]
    a0 = (int(y.min()) - 28, int(y.max()) + 29, int(x.min()) - 28, int(x.max()) + 29)
    cx, cy = c_full[:, 0] + c_full[:, 2], c_full[:, 1] + c_full[:, 8]
    b0 = (int(cy.min()) - 70, int(cy.max()) + 70, int(cx.min()) - 340, int(cx.max()) + 340)
    m1, m2 = np.zeros_like(v1), np.zeros_like(v2)
    m1[a0[0]:a0[1], a0[2]:a0[3]] = v1[a0[0]:a0[1], a0[2]:a0[3]]
    m2[b0[0]:b0[1], b0[2]:b0[3]] = v2[b0[0]:b0[1], b0[2]:b0[3]]
    for legacy in (1, 0):
        cf, qf = run(v1, v2, legacy)
        cm, qm = run(m1, m2, legacy)
        assert np.array_equal(cf, cm) and np.array_equal(qf, qm), "crop changes the result"
    np.savez_compressed(os.path.join(OUT, "step18_epipolar_crop.npz"), shape=np.array(v1.shape),
                        view1=v1[a0[0]:a0[1], a0[2]:a0[3]].astype(np.uint8), view1_origin=np.array([a0[0], a0[2]]),
                        view2=v2[b0[0]:b0[1], b0[2]:b0[3]].astype(np.uint8), view2_origin=np.array([b0[0], b0[2]]),
                        fundamental=fm, columns=np.array("x,y,r1r2 ZNCC,r2_x,r2_y".split(",")), table=blk[:, :5])


def make_full_2d_table():
    tab = np.genfromtxt(os.path.join(REF, "2d_dic", "oht_cfrp_4_fftcc_icgn1_r16.csv"), delimiter=",", skip_header=1)
    np.savez_compressed(os.path.join(OUT, "oht_cfrp_4_fftcc_icgn1_r16_full.npz"), xy=tab[:, 0:2].astype(np.int16),
                        u0v0=tab[:, 4:6].astype(np.int16), iteration=tab[:, 7].astype(np.int8), uv=tab[:, 2:4], zncc=tab[:, 6])


def main():
    for name in ("oht_cfrp_0.bmp", "oht_cfrp_4.bmp"):
        shutil.copyfile(os.path.join(REF, "2d_dic", name), os.path.join(OUT, name))
    tab = np.genfromtxt(os.path.join(REF, "2d_dic", "oht_cfrp_4_fftcc_icgn1_r16.csv"), delimiter=",", skip_header=1)
    dtab = np.genfromtxt(os.path.join(REF, "2d_dic", "oht_cfrp_4_fftcc_icgn1_r16_deformation.csv"), delimiter=",", skip_header=1)
    sel = np.arange(0, tab.shape[0], 23)
    # The three POIs (of 30 000) whose FFT-CC guess in the shipped table differs from the oracle's: in each, two bins of the
    # correlation map hold the SAME value (the subset lies in the specimen's featureless hole), so the arg-max is decided by
    # the rounding of the transform (FFTW there, the oracle's own FFT here).  Kept as full rows so that the tests can name them.
    ties = np.array([22154, 22472, 22557])
    np.savez_compressed(os.path.join(OUT, "oht_cfrp_4_fftcc_icgn1_r16.npz"),
                        columns=np.array("x,y,u,v,u0,v0,ZNCC,iteration,convergence".split(",")),
                        table=tab[sel, :9], deformation_columns=np.array("x,y,u,ux,uy,v,vx,vy".split(",")),
                        deformation=dtab[sel, :8], rows=sel, fftcc_tie_rows=ties, fftcc_tie_table=tab[ties, :9])
    make_full_2d_table()

    # ICLM2D1 table shipped by the reference (examples/2d_dic/oht_cfrp_4_fftcc_iclm1_r16.csv, same POIs)
    itab = np.genfromtxt(os.path.join(REF, "2d_dic", "oht_cfrp_4_fftcc_iclm1_r16.csv"), delimiter=",", skip_header=1)
    np.savez_compressed(os.path.join(OUT, "oht_cfrp_4_fftcc_iclm1_r16.npz"),
                        columns=np.array("x,y,u,v,u0,v0,ZNCC,iteration,convergence".split(",")), table=itab[sel, :9], rows=sel)

    # ICGN2D2 known-answer table (reference GPU build, SIFT / FeatureAffine seeds)
    gtab = np.genfromtxt(os.path.join(REF, "2d_dic", "oht_cfrp_4_sift_icgn2(gpu)_r16.csv"), delimiter=",", skip_header=1)
    np.savez_compressed(os.path.join(OUT, "oht_cfrp_4_sift_icgn2_gpu_r16.npz"),
                        columns=np.array("x,y,u,v,u0,v0,ZNCC,iteration,convergence".split(",")), table=gtab[sel, :9], rows=sel)

    make_self_adaptive_fixture()

    # NR2D1 + Strain table shipped by the reference (examples/2d_dic/oht_cfrp_4_fftcc_nr1_r16.csv)
    ntab = np.genfromtxt(os.path.join(REF, "2d_dic", "oht_cfrp_4_fftcc_nr1_r16.csv"), delimiter=",", skip_header=1)
    band = (ntab[:, 1] >= 370) & (ntab[:, 1] < 560)
    bt = ntab[band][:, [0, 1, 2, 3, 6, 10, 11, 12]].astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "oht_cfrp_4_fftcc_nr1_r16.npz"),
                        columns=np.array("x,y,u,v,u0,v0,ZNCC,iteration,convergence".split(",")), table=ntab[sel, :9], rows=sel,
                        band_columns=np.array("x,y,u,v,ZNCC,exx,eyy,exy".split(",")), band=bt,
                        band_check=(bt[:, 1] >= 390) & (bt[:, 1] < 540))

    # DVC table with strains (examples/dvc/Torus_def_sift_icgn1_r16.csv; strain radius 30, min 5 neighbours,
    # examples/test_dvc_strain.cpp:48-54)
    tt = np.genfromtxt(os.path.join(REF, "dvc", "Torus_def_sift_icgn1_r16.csv"), delimiter=",", skip_header=1)
    box = (tt[:, 0] >= 470) & (tt[:, 0] <= 630) & (tt[:, 2] >= 351) & (tt[:, 2] <= 501)
    tb = tt[box][:, [0, 1, 2, 3, 4, 5, 9, 22, 23, 24, 25, 26, 27]].astype(np.float32)
    inner = (tb[:, 0] >= 500) & (tb[:, 0] <= 600) & (tb[:, 2] >= 381) & (tb[:, 2] <= 471)
    np.savez_compressed(os.path.join(OUT, "torus_strain_crop.npz"),
                        columns=np.array("x,y,z,u,v,w,ZNCC,exx,eyy,ezz,exy,eyz,ezx".split(",")), table=tb, check=inner)

    make_epipolar_fixture()

    # stereo-DIC table with strains (examples/test_3d_dic_strain.cpp: radius 20, 5 neighbours)
    gt = np.genfromtxt(os.path.join(REF, "3d_dic", "GT4-0273_0_epipolar_sift_r16.csv"), delimiter=",", skip_header=1)
    box = (gt[:, 0] >= 600) & (gt[:, 0] <= 1100) & (gt[:, 1] >= 400) & (gt[:, 1] <= 800)
    gb = gt[box].astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "gt4_stereo_strain_crop.npz"), table=gb,
                        columns=np.array("x,y,u,v,w,r1r2 ZNCC,r1t1 ZNCC,r1t2 ZNCC,r2_x,r2_y,t1_x,t1_y,t2_x,t2_y,ref_x,ref_y,ref_z,tar_x,tar_y,tar_z,"
                                         "exx,eyy,ezz,exy,eyz,ezx".split(",")),
                        check=(gb[:, 0] >= 621) & (gb[:, 0] <= 1079) & (gb[:, 1] >= 421) & (gb[:, 1] <= 779))

    def load(p):
        d = np.fromfile(p, dtype=np.int32, count=3)
        v = np.fromfile(p, dtype=np.float32, offset=12)
        return v.reshape(d[2], d[1], d[0])

    z0, z1 = 18, 118
    ref = load(os.path.join(REF, "dvc", "al_foam4_0.bin"))[z0:z1]
    tar = load(os.path.join(REF, "dvc", "al_foam4_1.bin"))[z0:z1]
    assert np.all(ref == np.round(ref)) and ref.min() >= 0 and ref.max() <= 255
    assert np.all(tar == np.round(tar)) and tar.min() >= 0 and tar.max() <= 255
    cpu = np.genfromtxt(os.path.join(REF, "dvc", "al_foam4_1_fftcc_icgn1_r30.csv"), delimiter=",", skip_header=1)
    gpu = np.genfromtxt(os.path.join(REF, "dvc", "al_foam4_1_fftcc_icgn1(gpu)_r30.csv"), delimiter=",", skip_header=1)
    keep = cpu[:, 2] <= 75
    assert np.array_equal(cpu[keep, :3], gpu[keep, :3])
    np.savez_compressed(os.path.join(OUT, "al_foam4_crop.npz"), ref=ref.astype(np.uint8), tar=tar.astype(np.uint8),
                        z_offset=np.int32(z0),
                        cpu_columns=np.array("x,y,z,u,v,w,u0,v0,w0,ZNCC,iteration,convergence,ux,uy,uz,vx,vy,vz,wx,wy,wz".split(",")),
                        cpu_table=cpu[keep],
                        gpu_columns=np.array("x,y,z,u,v,w,u0,v0,w0,ZNCC,iteration,convergence,feature,ux,uy,uz,vx,vy,vz,wx,wy,wz".split(",")),
                        gpu_table=gpu[keep])
    for f in sorted(os.listdir(OUT)):
        print("%10d  %s" % (os.path.getsize(os.path.join(OUT, f)), f))


if __name__ == "__main__":
    main()
