"""Host-side mirror of the reference's MSM API, on top of the C ABI.

Reference surface reproduced here (same names, argument meaning and error behaviour):
  * `Weierstrass.create(params)` / `TwistedEdwards.create(params)` -> module with `.Parallel`
    (src/parallel.ts:40-177, :179-289)
  * `Parallel.pointsFromBytes`, `scalarsFromBytes`, `randomPointsFast`, `randomScalars`,
    `msm`, `msmUnsafe` (src/parallel.ts:97-145, :209-259)
  * `compute_msm(points, scalars)` (scripts/zprize23/submission-bls377.ts:20-65, submission.ts:19-35)
In the reference the arguments of `msm` are pointers into wasm memory; here they are a host byte
buffer of scalars and a `PointSet` handle naming points resident in HBM.  The reference has no
Node-free runtime in this image, so this layer is Python; INTEGRATION.md shows the N-API shim.
"""
import ctypes
import weakref

import numpy as np

from . import _native, curves, inputs


class MsmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("montgomery_b200 error %d: %s" % (code, msg))
        self.code = code


# status bits of a point checked on ingestion (set_points(..., check=True)); 0 = valid
PT_NONCANONICAL = _native.PT_NONCANONICAL          # x or y >= p
PT_OFF_CURVE = _native.PT_OFF_CURVE                # not on the curve
PT_NOT_IN_SUBGROUP = _native.PT_NOT_IN_SUBGROUP    # on the curve, not in the prime-order subgroup


class InvalidPointsError(MsmError):
    """set_points(..., check=True) found invalid points; the engine then holds no points.  `status` is the per-point
    np.uint8 array of PT_* bits, `count` the number of invalid points, `first` the index of the first one."""

    def __init__(self, code, msg, status, count, first):
        super().__init__(code, msg)
        self.status, self.count, self.first = status, count, first


def _set_points_checked(fn, handle, xy, zp, n, error_of):
    """mgb_set_points_checked / mgb_multi_set_points_checked -> None, or raises InvalidPointsError / MsmError"""
    status = np.zeros(n, dtype=np.uint8)
    count = ctypes.c_uint64(0)
    rc = fn(handle, _ptr(xy), zp, n, _ptr(status), ctypes.byref(count))
    if rc == _native.E_INVALID and count.value:
        raise InvalidPointsError(rc, error_of(), status, int(count.value), int(np.flatnonzero(status)[0]))
    if rc != 0:
        raise MsmError(rc, error_of())


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(ctypes.c_void_p)


def comm_unique_id() -> bytes:
    """mgb_comm_unique_id: the 128-byte NCCL id rank 0 draws and hands to the other ranks (needs no GPU)."""
    lib = _native.lib()
    buf = (ctypes.c_uint8 * _native.COMM_ID_BYTES)()
    rc = lib.mgb_comm_unique_id(buf)
    if rc != 0:
        raise MsmError(rc, lib.mgb_last_error(None).decode())
    return bytes(buf)


class MsmEngine:
    """One curve on one GPU: owns the device copy of the points and all scratch memory."""

    def __init__(self, curve: curves.CurveInfo, device: int = 0, max_points: int = 1 << 20):
        self.curve = curve
        self.lib = _native.lib()
        self._h = ctypes.c_void_p()
        rc = self.lib.mgb_create(ctypes.byref(self._h), curve.curve_id, device, max_points)
        if rc != 0:
            raise MsmError(rc, self.lib.mgb_last_error(None).decode())
        self.max_points = max_points
        self.n_points = 0
        self.device = device

    def _check(self, rc):
        if rc != 0:
            raise MsmError(rc, self.lib.mgb_last_error(self._h).decode())

    def close(self):
        if self._h:
            self.lib.mgb_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- points
    def set_points(self, xy_bytes, is_zero=None, check=False):
        """check=True: mgb_set_points_checked -- every point is checked on the device (canonical encoding, on the curve,
        in the prime-order subgroup); an invalid one raises InvalidPointsError and leaves the engine without points."""
        xy = np.ascontiguousarray(np.frombuffer(xy_bytes, dtype=np.uint8) if not isinstance(xy_bytes, np.ndarray) else xy_bytes.reshape(-1))
        pb = self.curve.point_bytes
        if xy.size % pb:
            raise ValueError("points buffer must be a multiple of %d bytes" % pb)
        n = xy.size // pb
        zp = None
        if is_zero is not None:
            z = np.ascontiguousarray(np.asarray(is_zero, dtype=np.uint8))
            assert z.size == n
            zp = _ptr(z)
        if check:
            self.n_points = 0
            _set_points_checked(self.lib.mgb_set_points_checked, self._h, xy, zp, n, lambda: self.lib.mgb_last_error(self._h).decode())
        else:
            self._check(self.lib.mgb_set_points(self._h, _ptr(xy), zp, n))
        self.n_points = n
        return n

    def random_points(self, n: int, seed: int):
        self._check(self.lib.mgb_random_points(self._h, seed, n))
        self.n_points = n

    def get_points(self, first: int, n: int):
        xy = np.empty(n * self.curve.point_bytes, dtype=np.uint8)
        z = np.empty(n, dtype=np.uint8)
        self._check(self.lib.mgb_get_points(self._h, first, n, _ptr(xy), _ptr(z)))
        return xy.reshape(n, self.curve.point_bytes), z

    # ---- msm
    def _opts(self, c, unsafe, projective=False, affine_reduction=False):
        return _native.MgbOpts(int(c or 0), int(bool(unsafe)), 0, int(bool(projective)), int(bool(affine_reduction)))

    def msm(self, scalars, n=None, c=None, unsafe=False, device_ptr=None, projective=False, affine_reduction=False):
        """scalars: (n, 32) uint8 host array (or bytes); or device_ptr = raw device pointer."""
        out = np.zeros(self.curve.point_bytes, dtype=np.uint8)
        is_zero = ctypes.c_int(0)
        tm = _native.MgbTiming()
        opts = self._opts(c, unsafe, projective, affine_reduction)
        if device_ptr is not None:
            if n is None:
                raise ValueError("msm(device_ptr=...): n is required (the length of a raw device buffer is unknown)")
            if int(device_ptr) % 16:
                raise ValueError("msm(device_ptr=...): the scalar buffer must be 16-byte aligned")
            self._check(self.lib.mgb_msm_device(self._h, ctypes.c_void_p(device_ptr), n, ctypes.byref(opts), _ptr(out),
                                                ctypes.byref(is_zero), ctypes.byref(tm)))
        else:
            sc = scalars if isinstance(scalars, np.ndarray) else np.frombuffer(scalars, dtype=np.uint8)
            sc = np.ascontiguousarray(sc.reshape(-1))
            if sc.size % 32:
                raise ValueError("scalars buffer must be a multiple of 32 bytes")
            if n is None:
                n = sc.size // 32
            if n < 0 or n * 32 > sc.size:
                raise ValueError("msm: n = %d exceeds the %d scalars in the buffer" % (n, sc.size // 32))
            self._check(self.lib.mgb_msm(self._h, _ptr(sc), n, ctypes.byref(opts), _ptr(out), ctypes.byref(is_zero), ctypes.byref(tm)))
        cb = self.curve.coord_bytes
        res = {
            "x": int.from_bytes(out[:cb].tobytes(), "little"),
            "y": int.from_bytes(out[cb:].tobytes(), "little"),
            "isZero": bool(is_zero.value),
        }
        return res, tm.as_dict()

    def prefetch(self, scalars, n=None):
        """Registers a host scalar set for upload ahead of its MSM (mgb_msm_prefetch): `scalars` is a C-contiguous uint8
        numpy array or a raw host address (then n is required).  The next msm call of this engine starts the copy behind
        its first tree round; the following msm / msm_sharded call with the SAME buffer and n uses the uploaded copy.
        Keep the buffer alive and unchanged until that call has returned."""
        if isinstance(scalars, np.ndarray):
            if not scalars.flags["C_CONTIGUOUS"] or scalars.dtype != np.uint8:
                raise ValueError("prefetch: a C-contiguous uint8 array is required (its address identifies the set)")
            if n is None:
                n = scalars.size // 32
            if n * 32 > scalars.size:
                raise ValueError("prefetch: n = %d exceeds the %d scalars in the buffer" % (n, scalars.size // 32))
            ptr = scalars.ctypes.data
        else:
            if n is None:
                raise ValueError("prefetch(address): n is required")
            ptr = int(scalars)
        self._check(self.lib.mgb_msm_prefetch(self._h, ctypes.c_void_p(ptr), n))

    def msm_partial(self, scalars_ptr, on_device, n, out_device_ptr, c=None):
        tm = _native.MgbTiming()
        opts = self._opts(c, False)
        self._check(self.lib.mgb_msm_partial(self._h, ctypes.c_void_p(scalars_ptr), int(on_device), n, ctypes.byref(opts),
                                             ctypes.c_void_p(out_device_ptr), ctypes.byref(tm)))
        return tm.as_dict()

    def combine_partials(self, partials_device_ptr, count):
        out = np.zeros(self.curve.point_bytes, dtype=np.uint8)
        is_zero = ctypes.c_int(0)
        self._check(self.lib.mgb_combine_partials(self._h, ctypes.c_void_p(partials_device_ptr), count, _ptr(out), ctypes.byref(is_zero)))
        cb = self.curve.coord_bytes
        return {"x": int.from_bytes(out[:cb].tobytes(), "little"), "y": int.from_bytes(out[cb:].tobytes(), "little"),
                "isZero": bool(is_zero.value)}

    @property
    def partial_bytes(self):
        return int(self.lib.mgb_partial_bytes(self._h))

    # ---- sharded msm: the context owns the NCCL communicator (mgb_comm_init) and runs the collective itself
    def comm_unique_id(self) -> bytes:
        return comm_unique_id()

    def comm_init(self, comm_id: bytes, rank: int, world: int):
        assert len(comm_id) == _native.COMM_ID_BYTES
        buf = (ctypes.c_uint8 * _native.COMM_ID_BYTES).from_buffer_copy(comm_id)
        self._check(self.lib.mgb_comm_init(self._h, buf, rank, world))

    def comm_info(self):
        r, w, v = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        self._check(self.lib.mgb_comm_info(self._h, ctypes.byref(r), ctypes.byref(w), ctypes.byref(v)))
        return {"rank": r.value, "world": w.value, "nccl_version": v.value}

    def msm_sharded(self, scalars_ptr, on_device, n_local, c=None):
        """This rank's shard of a sharded MSM; every rank gets the full result (mgb_msm_sharded)."""
        out = np.zeros(self.curve.point_bytes, dtype=np.uint8)
        is_zero = ctypes.c_int(0)
        tm = _native.MgbTiming()
        opts = self._opts(c, False)
        self._check(self.lib.mgb_msm_sharded(self._h, ctypes.c_void_p(scalars_ptr), int(on_device), n_local, ctypes.byref(opts),
                                             _ptr(out), ctypes.byref(is_zero), ctypes.byref(tm)))
        cb = self.curve.coord_bytes
        return {"x": int.from_bytes(out[:cb].tobytes(), "little"), "y": int.from_bytes(out[cb:].tobytes(), "little"),
                "isZero": bool(is_zero.value)}, tm.as_dict()


class MultiGpuMsm:
    """One host process driving several GPUs (mgb_multi_*): the shape a Node host uses (bindings/node)."""

    def __init__(self, curve: curves.CurveInfo, device_ids, max_points_per_device: int):
        self.curve = curve
        self.lib = _native.lib()
        self._h = ctypes.c_void_p()
        ids = (ctypes.c_int * len(device_ids))(*device_ids)
        rc = self.lib.mgb_multi_create(ctypes.byref(self._h), curve.curve_id, ids, len(device_ids), max_points_per_device)
        if rc != 0:
            raise MsmError(rc, self.lib.mgb_multi_last_error(None).decode())

    def _check(self, rc):
        if rc != 0:
            raise MsmError(rc, self.lib.mgb_multi_last_error(self._h).decode())

    def set_points(self, xy_bytes, is_zero=None, check=False):
        """check=True: mgb_multi_set_points_checked (see MsmEngine.set_points); status and `first` are global indices,
        and an invalid point in any shard leaves every device without points."""
        xy = np.ascontiguousarray(np.frombuffer(xy_bytes, dtype=np.uint8) if not isinstance(xy_bytes, np.ndarray) else xy_bytes.reshape(-1))
        n = xy.size // self.curve.point_bytes
        z = None if is_zero is None else np.ascontiguousarray(np.asarray(is_zero, dtype=np.uint8))
        zp = None if z is None else _ptr(z)
        if check:
            _set_points_checked(self.lib.mgb_multi_set_points_checked, self._h, xy, zp, n, lambda: self.lib.mgb_multi_last_error(self._h).decode())
        else:
            self._check(self.lib.mgb_multi_set_points(self._h, _ptr(xy), zp, n))
        return n

    def random_points(self, n, seed):
        self._check(self.lib.mgb_multi_random_points(self._h, seed, n))

    def get_points(self, first, n):
        xy = np.empty(n * self.curve.point_bytes, dtype=np.uint8)
        z = np.empty(n, dtype=np.uint8)
        self._check(self.lib.mgb_multi_get_points(self._h, first, n, _ptr(xy), _ptr(z)))
        return xy.reshape(n, self.curve.point_bytes), z

    def msm(self, scalars, n=None, c=None):
        sc = np.ascontiguousarray((scalars if isinstance(scalars, np.ndarray) else np.frombuffer(scalars, dtype=np.uint8)).reshape(-1))
        if n is None:
            n = sc.size // 32
        if n * 32 > sc.size:
            raise ValueError("msm: n = %d exceeds the %d scalars in the buffer" % (n, sc.size // 32))
        out = np.zeros(self.curve.point_bytes, dtype=np.uint8)
        is_zero = ctypes.c_int(0)
        tm = _native.MgbTiming()
        opts = _native.MgbOpts(int(c or 0), 0, 0, 0, 0)
        self._check(self.lib.mgb_multi_msm(self._h, _ptr(sc), n, ctypes.byref(opts), _ptr(out), ctypes.byref(is_zero), ctypes.byref(tm)))
        cb = self.curve.coord_bytes
        return {"x": int.from_bytes(out[:cb].tobytes(), "little"), "y": int.from_bytes(out[cb:].tobytes(), "little"),
                "isZero": bool(is_zero.value)}, tm.as_dict()

    def close(self):
        if self._h:
            self.lib.mgb_multi_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _log_from_timing(tm):
    """Same shape as the reference's `log` (list of printable rows, src/msm-common.ts:176-213)."""
    rows = [[{"n_pairs": tm["n_pairs"], "K": tm["K"], "c": tm["c"]}]]
    for label, key in (("copy scalars (H2D)", "h2d_scalars"), ("prepare points & scalars + slice scalars & count buckets", "decompose_slice"),
                       ("integrate bucket counts + sort points", "sort"), ("bucket accumulation", "accumulate"),
                       ("bucket reduction", "reduce"), ("partition sum + final sum", "final_sum"), ("msm total", "total")):
        rows.append(["%s... %.1fms" % (label, tm[key])])
    return rows


class _Parallel:
    """The `Parallel` member of a curve module (src/parallel.ts:135-145, :251-259)."""

    def __init__(self, module):
        self._m = module

    def _engine(self, n):
        return self._m._engine_for(n)

    def _new_point_set(self, n):
        eng = self._m._engine_for(n)
        ps = PointSet(eng, n)
        self._m._owner = weakref.ref(ps)
        return ps

    def pointsFromBytes(self, point_bytes, is_zero=None, check=False):
        """check=True: the points are checked on the device as they are ingested (the reference's isOnCurve /
        isInSubgroup); an invalid point raises InvalidPointsError and no PointSet is returned."""
        n = len(point_bytes) // self._m.curve.point_bytes
        ps = self._new_point_set(n)
        try:
            ps.engine.set_points(point_bytes, is_zero, check=check)
        except MsmError:
            ps.close()
            raise
        return ps

    def scalarsFromBytes(self, scalar_bytes):
        a = np.frombuffer(scalar_bytes, dtype=np.uint8) if not isinstance(scalar_bytes, np.ndarray) else scalar_bytes
        return np.ascontiguousarray(a.reshape(-1, 32))

    def randomPointsFast(self, n, seed=0x6D6F6E74):
        ps = self._new_point_set(n)
        ps.engine.random_points(n, seed)
        return ps

    def randomScalars(self, n, seed=0x6D6F6E74):
        return inputs.random_scalars(self._m.curve.q, n, seed)

    def msm(self, scalars, points, N, verboseTiming=False, options=None):
        options = options or {}
        points.engine.curve          # raises MsmError(MGB_E_STATE) on a closed handle
        if N > points.n:
            raise ValueError("msm: N = %d exceeds the %d points of the set" % (N, points.n))
        res, tm = points.engine.msm(scalars[:N] if isinstance(scalars, np.ndarray) else scalars, n=N, c=options.get("c"),
                                    unsafe=not options.get("useSafeAdditions", True), affine_reduction=bool(options.get("affineReduction")))
        log = _log_from_timing(tm)
        if verboseTiming:
            for row in log:
                print(*row)
        return {"result": res, "log": log, "timing": tm}

    def msmProjective(self, scalars, points, N, options=None):
        """msm-basic over projective coordinates, no GLV (src/parallel.ts:69-87); Weierstrass curves only."""
        assert self._m.curve.kind == "weierstrass"
        options = options or {}
        points.engine.curve          # raises MsmError(MGB_E_STATE) on a closed handle
        if N > points.n:
            raise ValueError("msmProjective: N = %d exceeds the %d points of the set" % (N, points.n))
        res, tm = points.engine.msm(scalars[:N] if isinstance(scalars, np.ndarray) else scalars, n=N, c=options.get("c"), projective=True)
        return {"result": res, "log": _log_from_timing(tm), "timing": tm}

    def msmUnsafe(self, scalars, points, N, verbose=False, options=None):
        options = dict(options or {})
        options["useSafeAdditions"] = False
        return self.msm(scalars, points, N, verbose, options)


class PointSet:
    """Handle to points resident in HBM (the analogue of a `pointPtr` into wasm memory).  As in the reference,
    where every pointPtr is its own memory (src/parallel.ts:97-116), every live PointSet has its own point table:
    the set keeps its engine (one context) alive, and a curve module hands an engine to a new set only when the
    set that used it before has been released (`close()` or garbage collection)."""

    def __init__(self, engine, n):
        self.engine = engine
        self.n = n

    def close(self):
        """Release the points: the module may give this set's engine (and its table) to the next set."""
        self.engine = _ReleasedEngine()

    def toBigints(self, first=0, n=None):
        n = self.n - first if n is None else n
        xy, z = self.engine.get_points(first, n)
        cb = self.engine.curve.coord_bytes
        return [{"x": int.from_bytes(r[:cb].tobytes(), "little"), "y": int.from_bytes(r[cb:].tobytes(), "little"), "isZero": bool(f)}
                for r, f in zip(xy, z)]


class _ReleasedEngine:
    def __getattr__(self, name):
        raise MsmError(_native_E_STATE, "this PointSet has been closed")


_native_E_STATE = -4   # MGB_E_STATE


class _CurveModule:
    def __init__(self, curve, device=0, max_points=None):
        self.curve = curve
        self.params = curve
        self.device = device
        self._engine = None
        self._owner = None          # weakref to the PointSet whose points sit in self._engine
        self._max_points = max_points
        self.Parallel = _Parallel(self)

    def _engine_for(self, n):
        """An engine whose point table is free for a new set of n points.  The cached engine is reused only when
        the PointSet that owned it is gone; otherwise that set keeps it and a new engine is created (two live
        PointSets never share a table), and an engine that is too small is left to its owner, not destroyed."""
        need = max(n, self._max_points or 0, 1)
        owner = self._owner() if self._owner is not None else None
        in_use = owner is not None and owner.engine is self._engine
        if self._engine is not None and not in_use and self._engine.max_points >= need:
            return self._engine
        if self._engine is not None and not in_use:
            self._engine.close()
        self._engine = MsmEngine(self.curve, self.device, need)
        return self._engine


class Weierstrass:
    @staticmethod
    def create(params, device=0, max_points=None):
        assert params.kind == "weierstrass", "only curves with a = 0 and an endomorphism are supported"
        return _CurveModule(params, device, max_points)


class TwistedEdwards:
    @staticmethod
    def create(params, device=0, max_points=None):
        assert params.kind == "twisted-edwards"
        return _CurveModule(params, device, max_points)


def make_compute_msm(curve: curves.CurveInfo, device=0, n_max=1 << 20):
    """`compute_msm(points, scalars)` of scripts/zprize23/submission-bls377.ts:20-65 (Weierstrass:
    bigint points `{x, y, isZero}` or 96-byte x||y; scalars bigint or 32-byte LE) and
    scripts/zprize23/submission.ts:19-35 (twisted Edwards, bytes).  Returns {x, y} (plus isZero)."""
    module = _CurveModule(curve, device, None)

    def compute_msm(input_points, input_scalars):
        cb = curve.coord_bytes
        raw_types = (bytes, bytearray, memoryview, np.ndarray)
        if not isinstance(input_scalars, raw_types) and len(input_scalars) and isinstance(input_scalars[0], int):
            sc = inputs.ints_to_le_bytes(input_scalars, 32)
        else:
            sc = np.frombuffer(bytes(input_scalars), dtype=np.uint8).reshape(-1, 32)
        n = sc.shape[0]
        is_zero = None
        if not isinstance(input_points, raw_types) and len(input_points) and isinstance(input_points[0], dict):
            xy = np.empty((n, 2 * cb), dtype=np.uint8)
            is_zero = np.zeros(n, dtype=np.uint8)
            for i, P in enumerate(input_points):
                xy[i, :cb] = np.frombuffer(int(P["x"]).to_bytes(cb, "little"), dtype=np.uint8)
                xy[i, cb:] = np.frombuffer(int(P["y"]).to_bytes(cb, "little"), dtype=np.uint8)
                is_zero[i] = 1 if P.get("isZero") else 0
            pts = module.Parallel.pointsFromBytes(xy.reshape(-1), is_zero)
        else:
            pts = module.Parallel.pointsFromBytes(np.frombuffer(bytes(input_points), dtype=np.uint8))
        out = module.Parallel.msm(sc, pts, n)
        return out["result"]

    return compute_msm
