"""CPU: checked point ingestion (mgb_set_points_checked, mgb_multi_set_points_checked) through the whole emulated path --
msm.cu on the stand-in CUDA runtime, k_set_points<CV, true> and k_check_points on the lockstep SIMT emulator (see
tests/test_host_emu_pipeline.py, whose build this module shares).  Every status byte is compared with the Python mirror
of the device test (tests/point_checks.py).  Bad points sit at lane 0, lane 31 and a middle lane of otherwise valid warps,
so the rare branches of the complete formulas run inside generic warps, as in tests/test_gpu_units.py."""
import ctypes
import re

import numpy as np
import pytest

from montgomery_b200 import curves, inputs
from tests import point_checks as pc
from tests.helpers import OracleCurve, points_to_bytes
from tests.test_host_emu_pipeline import E_INVALID, E_STATE, _read_point, host, oracle_msm  # noqa: F401  (host: the module's fixture)

pytestmark = pytest.mark.timeout(900)
LABELS = ["bls12-377", "pallas", "ed-on-bls12-377", "bls12-381"]
REASON = {pc.NONCANONICAL: "non-canonical", pc.OFF_CURVE: "not on the curve", pc.NOT_IN_SUBGROUP: "not in the prime-order subgroup"}


def bind(lib):
    vp, sz = ctypes.c_void_p, ctypes.c_size_t
    lib.mgb_set_points_checked.argtypes = [vp, vp, vp, sz, vp, ctypes.POINTER(ctypes.c_uint64)]
    lib.mgb_multi_set_points_checked.argtypes = [vp, vp, vp, sz, vp, ctypes.POINTER(ctypes.c_uint64)]


def place(good, bad, positions):
    """good points with bad[k] at positions[k]"""
    pts = list(good)
    for k, i in enumerate(positions):
        pts[i] = bad[k % len(bad)]
    return pts


def lane_positions(count):
    """lane 0, lane 31 and lane 17 of consecutive warps"""
    return [32 * (k // 3) + (0, 31, 17)[k % 3] for k in range(count)]


def checked(lib, ctx_or_multi, pts, coord_bytes, with_status=True, multi=False):
    xy, z = points_to_bytes(pts, coord_bytes)
    xy.reshape(len(pts), -1)[z != 0] = 0xFF                  # a flagged point's coordinate bytes are not looked at
    st = np.full(len(pts), 0xEE, np.uint8)
    cnt = ctypes.c_uint64(12345)
    fn = lib.mgb_multi_set_points_checked if multi else lib.mgb_set_points_checked
    rc = fn(ctx_or_multi, xy.ctypes.data, z.ctypes.data, len(pts), st.ctypes.data if with_status else None, ctypes.byref(cnt))
    err = (lib.mgb_multi_last_error(ctx_or_multi) if multi else lib.mgb_last_error(ctx_or_multi)) or b""
    return rc, st, cnt.value, err.decode()


def check_message(err, expected):
    bad = [i for i, s in enumerate(expected) if s]
    m = re.match(r"(\d+) invalid points?; the first is point (\d+): (.*)$", err)
    assert m, err
    assert int(m.group(1)) == len(bad) and int(m.group(2)) == bad[0], err
    assert REASON[expected[bad[0]]] in m.group(3), err


@pytest.mark.parametrize("label", LABELS)
def test_checked_ingestion(host, label):
    """valid set: accepted, table identical to mgb_set_points, MSM equal to the oracle's; every kind of bad point at lane
    positions: MGB_E_INVALID, the status bytes, the count, the message, and a context left without points; the same
    without a status buffer"""
    bind(host.lib)
    ctx = host.create(label, 256)
    lib = ctx.lib
    try:
        good = ctx.random_points(200, seed=41)
        if label != "ed-on-bls12-377":
            good[5] = None                                     # a point flagged as zero
        rc, st, cnt, err = checked(lib, ctx.h, good, ctx.cv.coord_bytes)
        assert rc == 0 and cnt == 0 and not st.any(), err
        assert ctx.get_points(200) == good
        sc = inputs.random_scalars(ctx.cv.q, 200, 42)
        exp = oracle_msm(label, sc, good)
        assert ctx.msm(sc)[0] == exp
        ctx.set_points(good)                                   # unchecked ingestion of the same bytes: the same table
        assert ctx.get_points(200) == good

        bad = pc.bad_points(label, [P for P in good[:8] if P is not None])
        pts = place(good, bad, lane_positions(len(bad)))
        xy, _ = points_to_bytes(pts, ctx.cv.coord_bytes)
        expected = [pc.expected_status(label, P) for P in pts]
        assert sorted(set(expected)) == ([0, 1, 2] if label == "pallas" else [0, 1, 2, 4])
        rc, st, cnt, err = checked(lib, ctx.h, pts, ctx.cv.coord_bytes)
        assert rc == E_INVALID, err
        assert st.tolist() == expected
        assert cnt == sum(1 for s in expected if s)
        check_message(err, expected)
        ctx.msm(sc, expect_rc=E_STATE)                         # no points held
        assert lib.mgb_get_points(ctx.h, 0, 1, np.zeros(2 * ctx.cv.coord_bytes, np.uint8).ctypes.data, None) == E_INVALID

        rc, st, cnt, err = checked(lib, ctx.h, pts, ctx.cv.coord_bytes, with_status=False)
        assert rc == E_INVALID and cnt == sum(1 for s in expected if s) and (st == 0xEE).all()
        check_message(err, expected)
        ctx.msm(sc, expect_rc=E_STATE)

        # the context takes a valid set again after a rejected one
        rc, st, cnt, err = checked(lib, ctx.h, good, ctx.cv.coord_bytes)
        assert rc == 0, err
        assert ctx.msm(sc)[0] == exp
        # argument errors as mgb_set_points
        assert lib.mgb_set_points_checked(ctx.h, None, None, 3, None, None) == E_INVALID
        assert lib.mgb_set_points_checked(ctx.h, xy.ctypes.data, None, 257, None, None) == E_INVALID
        assert lib.mgb_set_points_checked(ctx.h, None, None, 0, None, None) == 0
        ctx.msm(sc, expect_rc=E_STATE)
    finally:
        ctx.close()


@pytest.mark.parametrize("label", ["bls12-381", "ed-on-bls12-377"])
def test_checked_ingestion_chunked(host, label, monkeypatch):
    """point sets above the chunk size (forced to 7 points): bad points on both sides of chunk boundaries keep their
    global index"""
    bind(host.lib)
    ctx = host.create(label, 64)
    try:
        good = ctx.random_points(60, seed=43)
        bad = pc.bad_points(label, good[:4])
        positions = [6, 7, 13, 14, 20, 27, 28, 59]
        pts = place(good, bad, positions)
        expected = [pc.expected_status(label, P) for P in pts]
        monkeypatch.setenv("MGB_DEBUG_INGEST_CHUNK", "7")
        rc, st, cnt, err = checked(ctx.lib, ctx.h, pts, ctx.cv.coord_bytes)
        assert rc == E_INVALID and st.tolist() == expected and cnt == len(positions), err
        check_message(err, expected)
        rc, st, cnt, err = checked(ctx.lib, ctx.h, good, ctx.cv.coord_bytes)
        assert rc == 0 and not st.any() and ctx.get_points(60) == good, err
    finally:
        ctx.close()


def test_multi_checked_ingestion(host):
    """mgb_multi_set_points_checked over three emulated devices: status and the first index are global, and one bad
    point in one shard leaves every device without points"""
    bind(host.lib)
    label = "bls12-377"
    cv = curves.BY_LABEL[label]
    lib = host.lib
    devs = (ctypes.c_int * 3)(0, 1, 2)
    m = ctypes.c_void_p()
    assert lib.mgb_multi_create(ctypes.byref(m), cv.curve_id, devs, 3, 40) == 0, lib.mgb_multi_last_error(None)
    try:
        O = OracleCurve(label)
        good = [O.scale(11 + 7 * i, O.G) for i in range(100)]        # shards of 34 / 34 / 32 points
        rc, st, cnt, err = checked(lib, m, good, cv.coord_bytes, multi=True)
        assert rc == 0 and cnt == 0 and not st.any(), err
        sc = inputs.random_scalars(cv.q, 100, 44)

        def msm(expect_rc=0):
            out, flag = np.zeros(2 * cv.coord_bytes, np.uint8), ctypes.c_int(0)
            rc = lib.mgb_multi_msm(m, sc.ctypes.data, 100, None, out.ctypes.data, ctypes.byref(flag), None)
            assert rc == expect_rc, (rc, lib.mgb_multi_last_error(m))
            return _read_point(cv, out, flag) if rc == 0 else None

        assert msm() == oracle_msm(label, sc, good)
        bad = pc.bad_points(label, good[:4])
        for positions in ([40, 41, 99], [70]):                      # the first bad point in the second / the third shard
            pts = place(good, bad, positions)
            expected = [pc.expected_status(label, P) for P in pts]
            rc, st, cnt, err = checked(lib, m, pts, cv.coord_bytes, multi=True)
            assert rc == E_INVALID and st.tolist() == expected and cnt == len(positions), err
            check_message(err, expected)
            msm(expect_rc=E_STATE)
            assert lib.mgb_multi_get_points(m, 0, 1, np.zeros(2 * cv.coord_bytes, np.uint8).ctypes.data, None) == E_INVALID
        rc, st, cnt, err = checked(lib, m, good, cv.coord_bytes, multi=True, with_status=False)
        assert rc == 0, err
        assert msm() == oracle_msm(label, sc, good)
    finally:
        lib.mgb_multi_destroy(m)
