"""GPU: checked point ingestion (set_points(..., check=True) / mgb_set_points_checked) on sm_100a.  Valid sets of 2^20
points are accepted and stored exactly as mgb_set_points stores them; invalid points of every kind, at chunk boundaries
and lane positions of a 2^18 + 2^16 set, get the status byte the oracle gives (tests/point_checks.py)."""
import numpy as np
import pytest

import montgomery_b200 as m
from montgomery_b200 import inputs
from tests import point_checks as pc
from tests.helpers import OracleCurve, points_to_bytes

pytestmark = pytest.mark.gpu
CURVES = {"bls12-377": m.curves.BLS12_377, "pallas": m.curves.PALLAS, "ed-on-bls12-377": m.curves.ED_ON_BLS12_377,
          "bls12-381": m.curves.BLS12_381}


def closed_form(label, seed, sc):
    O = OracleCurve(label)
    return O.result_of(O.scale(inputs.dot_known_dlogs(sc, inputs.known_dlogs(seed, sc.shape[0])) % O.q, O.G))


def as_points(xy, z, cb):
    return [None if f else (int.from_bytes(r[:cb].tobytes(), "little"), int.from_bytes(r[cb:].tobytes(), "little")) for r, f in zip(xy, z)]


@pytest.mark.parametrize("label", list(CURVES))
def test_valid_2p20_accepted_and_unchanged(label):
    n = 1 << 20
    cv = CURVES[label]
    eng = m.MsmEngine(cv, 0, n)
    try:
        eng.random_points(n, seed=5)
        xy, z = eng.get_points(0, n)
        assert eng.set_points(xy, z, check=True) == n
        xy2, z2 = eng.get_points(0, n)
        assert np.array_equal(xy, xy2) and np.array_equal(z, z2)
        sc = inputs.random_scalars(cv.q, n, 6)
        assert eng.msm(sc)[0] == closed_form(label, 5, sc)
    finally:
        eng.close()


@pytest.mark.parametrize("label", list(CURVES))
def test_bad_points_at_chunk_boundaries_and_lanes(label):
    """2^18 + 2^16 points (two ingestion chunks): bad points at the chunk boundary, at lanes 0 / 31 / 17 of warps, at the
    first and the last index; status byte for byte, the count, the first index, and an engine left without points"""
    n = (1 << 18) + (1 << 16)
    cv = CURVES[label]
    cb = cv.coord_bytes
    eng = m.MsmEngine(cv, 0, n)
    try:
        eng.random_points(n, seed=9)
        xy, z = eng.get_points(0, n)
        good = as_points(xy[:16], z[:16], cb)
        bad = pc.bad_points(label, good)
        base = [0, (1 << 18) - 1, 1 << 18, (1 << 18) + 1, n - 1]
        positions = base + [4096 + 32 * (k // 3) + (0, 31, 17)[k % 3] for k in range(len(bad))]
        expected = np.zeros(n, np.uint8)
        xy = xy.copy()
        z = z.copy()
        for k, i in enumerate(positions):
            P = bad[k % len(bad)]
            bxy, bz = points_to_bytes([P], cb)
            xy[i] = bxy
            z[i] = bz[0]
            expected[i] = pc.expected_status(label, P)
        assert set(expected[positions].tolist()) == ({1, 2} if label == "pallas" else {1, 2, 4})
        with pytest.raises(m.InvalidPointsError) as ei:
            eng.set_points(xy, z, check=True)
        e = ei.value
        assert e.code == -1 and np.array_equal(e.status, expected)
        assert e.count == len(positions) and e.first == 0
        assert "%d invalid points; the first is point 0" % len(positions) in str(e)
        with pytest.raises(m.MsmError) as es:                  # no points held
            eng.msm(inputs.random_scalars(cv.q, 8, 1))
        assert es.value.code == -4
    finally:
        eng.close()


@pytest.mark.parametrize("label", list(CURVES))
def test_python_surfaces(label):
    """Parallel.pointsFromBytes(check=True): a valid set gives a PointSet whose MSM is right; an invalid one raises
    InvalidPointsError and gives none; status bit constants are exported"""
    assert (m.PT_NONCANONICAL, m.PT_OFF_CURVE, m.PT_NOT_IN_SUBGROUP) == (1, 2, 4)
    cv = CURVES[label]
    O = OracleCurve(label)
    mod = (m.Weierstrass if cv.kind == "weierstrass" else m.TwistedEdwards).create(cv)
    pts = [O.scale(int(a), O.G) for a in inputs.known_dlogs(3, 300)]
    xy, z = points_to_bytes(pts, cv.coord_bytes)
    ps = mod.Parallel.pointsFromBytes(xy, z, check=True)
    sc = inputs.random_scalars(cv.q, 300, 4)
    assert mod.Parallel.msm(sc, ps, 300)["result"] == closed_form(label, 3, sc)
    ps.close()
    bad = pc.bad_points(label, pts[:4])
    pts2 = list(pts)
    for k, P in enumerate(bad):
        pts2[100 + 2 * k] = P
    xy2, z2 = points_to_bytes(pts2, cv.coord_bytes)
    with pytest.raises(m.InvalidPointsError) as ei:
        mod.Parallel.pointsFromBytes(xy2, z2, check=True)
    assert ei.value.first == 100 and ei.value.count == len(bad)
    assert ei.value.status.tolist() == [pc.expected_status(label, P) for P in pts2]
    # the unchecked path is unchanged: it takes the same bytes
    mod.Parallel.pointsFromBytes(xy2, z2).close()


def test_multi_gpu_checked():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    label = "bls12-381"
    cv = CURVES[label]
    O = OracleCurve(label)
    mg = m.MultiGpuMsm(cv, [0, 1], 4096)
    try:
        pts = [O.scale(int(a), O.G) for a in inputs.known_dlogs(8, 1000)]
        xy, z = points_to_bytes(pts, cv.coord_bytes)
        assert mg.set_points(xy, z, check=True) == 1000
        sc = inputs.random_scalars(cv.q, 1000, 2)
        assert mg.msm(sc)[0] == closed_form(label, 8, sc)
        bad = pc.bad_points(label, pts[:4])
        pts2 = list(pts)
        for k, P in enumerate(bad):
            pts2[600 + k] = P                                  # all in the second shard
        xy2, z2 = points_to_bytes(pts2, cv.coord_bytes)
        with pytest.raises(m.InvalidPointsError) as ei:
            mg.set_points(xy2, z2, check=True)
        assert ei.value.first == 600 and ei.value.status.tolist() == [pc.expected_status(label, P) for P in pts2]
        with pytest.raises(m.MsmError) as es:
            mg.msm(sc)
        assert es.value.code == -4
    finally:
        mg.close()
