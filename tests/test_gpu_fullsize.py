"""GPU parity at BASELINE.json's FULL sizes (configs B, E, D): the oracle on a random sample of the queue (tight
tolerances: 1e-4 px, 1e-5 ZNCC, integer outputs identical) plus size-independent properties over the WHOLE queue --
ground truth of the synthetic field, invariance to the order of the POIs, to splitting the queue into shards (what the
multi-GPU path does) and idempotence of a converged result."""
import numpy as np
import pytest

import opencorr_b200 as ob
from opencorr_b200 import synth
from oracle.oracle import Oracle2D, Oracle3D
import util

pytestmark = pytest.mark.gpu


def _pair(cfg):
    import torch
    dev = torch.device("cuda", 0)
    if cfg["kind"] == "2d":
        return synth.speckle_pair_2d(*cfg["size"], second_order=(cfg["order"] == 2), device=dev)
    return synth.speckle_pair_3d(*cfg["size"], device=dev)


@pytest.mark.parametrize("name", ["B", "E", "C"])
def test_full_size_2d(engine, name):
    cfg = synth.CONFIGS[name]
    ref, tar = _pair(cfg)
    r, order = cfg["r"], cfg["order"]
    xy = synth.grid_2d(*cfg["grid"])
    n = len(xy)
    assert n == {"B": 50000, "E": 500000, "C": 50000}[name]
    engine.set_images_2d(ref, tar)
    engine.icgn2d_prepare()
    icgn = engine.icgn2d1 if order == 1 else engine.icgn2d2

    def run(points):
        q = ob.make_poi2d(points)
        engine.fftcc2d(q, r, r)
        icgn(q, r, r, cfg["conv"], cfg["stop"])
        return q

    q = run(xy)
    # the specialisation each config exists to measure (the record is that of the last of the four pipelined chunks)
    want = dict(np=12, rc=20, wpp=1, tm=0) if order == 2 else dict(np=6, rc=16, wpp=1, tm=1)
    got = engine.last_launch()
    assert all(got.get(k) == v for k, v in want.items()), "config %s: expected %s, ran %s" % (name, want, got)
    # (1) every POI converged onto the analytic displacement field (loose: the field is not exactly affine per subset)
    assert (q[:, 16] > 0.9).all()
    u_true, v_true = synth.displacement_2d(xy[:, 0], xy[:, 1], cfg["size"][0], cfg["size"][1], second_order=(order == 2))
    assert np.abs(q[:, 2] - u_true).max() < 0.05 and np.abs(q[:, 8] - v_true).max() < 0.05
    # (2) order invariance: a shuffled queue gives bit-identical records (persistent warps pull POIs from a work counter)
    rng = np.random.default_rng(1)
    perm = rng.permutation(n)
    qp = run(xy[perm])
    assert np.array_equal(qp, q[perm])
    # (3) shard invariance: three uneven shards, as opencorr_b200.distributed splits them
    cuts = [0, n // 3 + 17, 2 * n // 3 - 5, n]
    qs = np.vstack([run(xy[a:b]) for a, b in zip(cuts[:-1], cuts[1:])])
    assert np.array_equal(qs, q)
    # (4) idempotence: restarting from the converged deformation stops after one iteration within conv of it
    q2 = q.copy()
    q2[:, 16] = 0
    icgn(q2, r, r, cfg["conv"], cfg["stop"])
    if order == 1:
        assert (q2[:, 17] == 1).mean() > 0.999
    else:  # ICGN2D2 drops the second-order terms of an incoming guess (src/oc_icgn.cpp:765-770): it has to find them again
        assert (q2[:, 17] <= 3).mean() > 0.999
    assert np.abs(q2[:, [2, 8]] - q[:, [2, 8]]).max() < 2 * cfg["conv"]
    # (5) the oracle on a random sample, tight tolerances
    sel = np.sort(rng.choice(n, 3000 if name != "E" else 2000, replace=False))
    qc = ob.make_poi2d(xy[sel])
    o = Oracle2D(ref, tar)
    o.fftcc2d(qc, r, r)
    (o.icgn2d1 if order == 1 else o.icgn2d2)(qc, r, r, cfg["conv"], cfg["stop"])
    stats = util.compare_2d(q[sel], qc, "full-size %s" % name, order=order)
    assert stats["n_compared"] > 0.98 * len(sel)


def test_full_size_dvc(engine):
    cfg = synth.CONFIGS["D"]
    ref, tar = _pair(cfg)
    r = cfg["r"]
    xyz = synth.grid_3d(*cfg["grid"])
    n = len(xyz)
    assert n == 20000
    engine.set_images_3d(ref, tar)
    engine.icgn3d_prepare()

    def run(points):
        q = ob.make_poi3d(points)
        engine.fftcc3d(q, r, r, r)
        engine.icgn3d1(q, r, r, r, cfg["conv"], cfg["stop"])
        return q

    q = run(xyz)
    assert (q[:, 18] > 0.9).all()
    ut, vt, wt = synth.displacement_3d(xyz[:, 0], xyz[:, 1], xyz[:, 2], *cfg["size"])
    assert max(np.abs(q[:, 3] - ut).max(), np.abs(q[:, 7] - vt).max(), np.abs(q[:, 11] - wt).max()) < 0.05
    rng = np.random.default_rng(2)
    perm = rng.permutation(n)
    assert np.array_equal(run(xyz[perm]), q[perm])                      # order invariance
    cuts = [0, n // 2 + 3, n]
    assert np.array_equal(np.vstack([run(xyz[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]), q)   # shard invariance
    sel = np.sort(rng.choice(n, 150, replace=False))
    qc = ob.make_poi3d(xyz[sel])
    o = Oracle3D(ref, tar)
    o.fftcc3d(qc, r, r, r, exact=True)
    o.icgn3d1(qc, r, r, r, cfg["conv"], cfg["stop"], exact=True)
    stats = util.compare_3d(q[sel], qc, "full-size D")
    assert stats["n_compared"] > 0.95 * len(sel)


def test_full_size_sibling_rows_config_b(engine):
    """The section-8(f) operators on the full config-B workload: ICLM2D1 and NR2D1 against the oracle on a sample, Strain
    against the oracle on all 50 000 POIs, order invariance of each."""
    from oracle import oracle
    cfg = synth.CONFIGS["B"]
    ref, tar = _pair(cfg)
    r = cfg["r"]
    xy = synth.grid_2d(*cfg["grid"])
    n = len(xy)
    engine.set_images_2d(ref, tar)
    engine.icgn2d_prepare()
    engine.nr2d_prepare()
    q0 = ob.make_poi2d(xy)
    engine.fftcc2d(q0, r, r)
    rng = np.random.default_rng(3)
    perm = rng.permutation(n)
    sel = np.sort(rng.choice(n, 1500, replace=False))
    o = Oracle2D(ref, tar)

    lm = q0.copy()
    engine.iclm2d(1, lm, r, r, 0.001, 10)
    lmp = q0[perm].copy()
    engine.iclm2d(1, lmp, r, r, 0.001, 10)
    assert np.array_equal(lmp, lm[perm])
    c = q0[sel].copy()
    o.iclm2d(1, c, r, r, 0.001, 10)
    same = lm[sel, 17] == c[:, 17]
    assert same.mean() > 0.97
    assert np.abs(lm[sel][same][:, [2, 8]] - c[same][:, [2, 8]]).max() < 1e-4
    assert np.abs(lm[sel][same, 16] - c[same, 16]).max() < 1e-5

    nr = q0.copy()
    engine.nr2d1(nr, r, r, 0.001, 10)
    nrp = q0[perm].copy()
    engine.nr2d1(nrp, r, r, 0.001, 10)
    assert np.array_equal(nrp, nr[perm])
    c = q0[sel].copy()
    o.nr2d1(c, r, r, 0.001, 10)
    same = nr[sel, 17] == c[:, 17]
    assert same.mean() > 0.97
    assert np.abs(nr[sel][same][:, [2, 8]] - c[same][:, [2, 8]]).max() < 1e-4
    assert np.abs(nr[sel][same, 16] - c[same, 16]).max() < 1e-5
    assert (nr[:, 16] > 0.9).all()

    st = nr.copy()
    engine.strain(st, 25.0, 5)
    cs = nr.copy()
    oracle.strain(cs, 25.0, 5, 0.9, 1, exact=True)
    assert np.abs(st[:, 20:23] - cs[:, 20:23]).max() < 1e-6
    assert (st[:, 20] != 0).all()
    # the fitted gradients recover the synthetic field's: u_x = 1.5e-3, v_y = 2.1e-3, (u_y + v_x) / 2 = -1e-4
    inner = (xy[:, 0] > 300) & (xy[:, 0] < 1700) & (xy[:, 1] > 300) & (xy[:, 1] < 1700)
    assert np.abs(st[inner, 20] - 1.5e-3).max() < 6e-4 and np.abs(st[inner, 21] - 2.1e-3).max() < 6e-4
    assert np.abs(st[inner, 22] + 1e-4).max() < 6e-4
    stp = nr[perm].copy()
    engine.strain(stp, 25.0, 5)
    assert np.abs(stp[:, 20:23] - st[perm][:, 20:23]).max() < 1e-9   # FP64 sums in sorted-cell order: independent of the queue order
