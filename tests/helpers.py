"""Shared test helpers: oracle curve objects and conversions (tests may import oracle/)."""
import glob
import hashlib
import os
import subprocess

import numpy as np

from oracle.params import BLS12_377, BLS12_381, ED_ON_BLS12_377, PALLAS
from oracle.twisted_edwards import TwistedEdwardsCurve
from oracle.weierstrass import AffineCurve, ProjectiveCurve
from oracle.msm import msm as oracle_msm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_PARAMS = {"bls12-377": BLS12_377, "pallas": PALLAS, "ed-on-bls12-377": ED_ON_BLS12_377, "bls12-381": BLS12_381}


class OracleCurve:
    """Uniform view: points are affine (x, y) tuples or None (Weierstrass infinity)."""

    def __init__(self, label):
        self.prm = ORACLE_PARAMS[label]
        self.kind = self.prm.kind
        if self.kind == "weierstrass":
            self.A = AffineCurve(self.prm)
            self.P = ProjectiveCurve(self.prm)
        else:
            self.T = TwistedEdwardsCurve(self.prm)

    @property
    def q(self):
        return self.prm.q

    @property
    def G(self):
        return tuple(self.prm.G)

    def scale(self, s, P):
        if self.kind == "weierstrass":
            return self.P.to_affine(self.P.scale(s % self.q, self.P.from_affine(P)))
        return self.T.to_affine(self.T.scale(s % self.q, self.T.from_affine(P)))

    def msm(self, scalars, points):
        """Reference-shaped bigint Pippenger (src/bigint/msm.ts) -> result dict like the engine's."""
        if self.kind == "weierstrass":
            r = self.P.to_affine(oracle_msm(self.P, scalars, [self.P.from_affine(Q) for Q in points]))
            return {"x": 0, "y": 0, "isZero": True} if r is None else {"x": r[0], "y": r[1], "isZero": False}
        r = self.T.to_affine(oracle_msm(self.T, scalars, [self.T.from_affine(Q) for Q in points]))
        return {"x": r[0], "y": r[1], "isZero": r == (0, 1)}

    def result_of(self, P):
        if self.kind == "weierstrass":
            return {"x": 0, "y": 0, "isZero": True} if P is None else {"x": P[0], "y": P[1], "isZero": False}
        return {"x": P[0], "y": P[1], "isZero": tuple(P) == (0, 1)}


def points_to_bytes(points, coord_bytes):
    """affine tuples (None = infinity) -> (xy bytes array, is_zero flags)."""
    n = len(points)
    xy = np.zeros((n, 2 * coord_bytes), dtype=np.uint8)
    z = np.zeros(n, dtype=np.uint8)
    for i, P in enumerate(points):
        if P is None:
            z[i] = 1
            continue
        xy[i, :coord_bytes] = np.frombuffer(int(P[0]).to_bytes(coord_bytes, "little"), dtype=np.uint8)
        xy[i, coord_bytes:] = np.frombuffer(int(P[1]).to_bytes(coord_bytes, "little"), dtype=np.uint8)
    return xy.reshape(-1), z


def scalars_to_bytes(scalars):
    return np.frombuffer(b"".join(int(s).to_bytes(32, "little") for s in scalars), dtype=np.uint8).reshape(-1, 32).copy()


GPU_UNITS_SRC = os.path.join(ROOT, "tests", "gpu_units", "units.cu")


def gpu_units_flags():
    """The product library's code generation (montgomery_b200.build.NVCC_FLAGS + MGB_NVCC_EXTRA)."""
    from montgomery_b200 import build as b
    return b.NVCC_FLAGS + os.environ.get("MGB_NVCC_EXTRA", "").split()


def gpu_units_key():
    """Hash of the test harness tests/gpu_units/units.cu, every file of csrc/, the public header and the flags."""
    from montgomery_b200 import build as b
    h = hashlib.sha256()
    files = [GPU_UNITS_SRC] + sorted(glob.glob(os.path.join(b.CSRC, "*"))) + [os.path.join(ROOT, "include", "montgomery_b200.h")]
    for f in files:
        h.update(os.path.basename(f).encode() + b"\0")
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(gpu_units_flags()).encode())
    return h.hexdigest()[:20]


def compile_gpu_units(so_path):
    """nvcc tests/gpu_units/units.cu -> so_path (sm_100a, the product's flags); returns the compiler output."""
    from montgomery_b200 import build as b
    cmd = [b._nvcc()] + gpu_units_flags() + ["-shared", "-o", so_path, GPU_UNITS_SRC, "-lcudart"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed for tests/gpu_units/units.cu:\n" + (res.stdout + res.stderr)[-4000:])
    return res.stdout + res.stderr


def dumped_point(path, coord_bytes):
    """A result point written by `bench.py --dump-outputs` (float64 [x limbs, y limbs, isZero], 32-bit limbs) -> result dict."""
    v = np.load(path)
    nl = coord_bytes // 4
    assert v.dtype == np.float64 and v.shape == (2 * nl + 1,)
    assert all(0 <= w < 2**32 and w == int(w) for w in v[:-1]) and v[-1] in (0, 1)
    x, y = (sum(int(w) << (32 * i) for i, w in enumerate(v[k * nl:(k + 1) * nl])) for k in (0, 1))
    return {"x": x, "y": y, "isZero": bool(v[-1])}
