"""GPU unit tests of the device code above the field layer, bit-exact against Python integers and the oracle.

tests/gpu_units/units.cu runs the engine's routines and kernels on the B200 one unit at a time: the field operations on
stored (Montgomery-form) operands, the warp-cooperative arithmetic, the affine / XYZZ / extended-Edwards group law, the
quad-cooperative addition, the one-warp Horner steps, and the kernels k_batch_add, k_pair_add, k_final, k_normalize,
k_set_points / k_get_points.  Rare cases (doubling, P + (-P), neutral operands) are laid out among generic ones in the
same warp, because on the device they take data-dependent branches next to shuffles.  The last part runs whole MSMs
whose inputs make the rare paths common (one point, a few points and their negations, points at infinity, structured
scalars) against their closed form at several engine settings."""
import ctypes
import os
import random
import time
from functools import lru_cache

import numpy as np
import pytest

import montgomery_b200 as m
from montgomery_b200 import inputs
from oracle.params import BLS12_377, BLS12_381, ED_ON_BLS12_377, PALLAS
from oracle.twisted_edwards import TwistedEdwardsCurve
from oracle.weierstrass import AffineCurve
from tests.helpers import OracleCurve, compile_gpu_units, gpu_units_key, points_to_bytes, scalars_to_bytes

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = [(BLS12_377.p, 12), (BLS12_377.q, 8), (PALLAS.p, 8), (BLS12_381.p, 12)]
W_CURVES = [(0, BLS12_377, 12), (1, PALLAS, 8), (2, BLS12_381, 12)]
W_IDS = ["bls12-377", "pallas", "bls12-381"]
REF_NEG, REF_ENDO, REF_EMPTY = 0x80000000, 0x40000000, 0xFFFFFFFF
V_, I_, U_, S_ = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_size_t
SIGNATURES = {
    "gpu_fe_op": [I_, I_, V_, V_, V_, I_],
    "gpu_w_op": [I_, I_, V_, V_, V_, I_],
    "gpu_te_op": [I_, V_, V_, V_, I_],
    "gpu_warp_mul": [I_, V_, V_, V_, I_],
    "gpu_warp_mul2": [I_, V_, V_, V_, I_],
    "gpu_warp_addsub2": [I_, I_, V_, V_, V_, I_],
    "gpu_warp_finish": [I_, V_, V_, V_, I_],
    "gpu_warp_finish2": [I_, V_, V_, V_, V_, I_],
    "gpu_warp_inv": [I_, V_, V_, I_],
    "gpu_quad_add": [I_, V_, V_, V_, I_],
    "gpu_onewarp": [I_, I_, I_, V_, V_, V_, I_],
    "gpu_batch_add": [I_, I_, V_, S_, V_, U_, I_, I_, U_, V_, S_, V_, V_, S_, V_, S_, V_, S_, V_, U_, U_, I_],
    "gpu_pair_add_te": [I_, V_, S_, V_, U_, I_, V_, S_, V_, V_, S_, V_, S_, V_, S_, V_, U_, U_],
    "gpu_final": [I_, I_, I_, V_, V_, V_, V_],
    "gpu_set_get_points": [I_, U_, V_, V_, V_, V_, V_],
    "gpu_normalize": [I_, V_, I_, I_, V_, V_],
    "gpu_batch_add_emax": [],
    "gpu_batch_add_minb": [],
}


@pytest.fixture(scope="module")
def units(tmp_path_factory):
    """The harness, compiled once per content of units.cu + csrc/* + flags and cached under montgomery_b200/build/."""
    d = os.path.join(ROOT, "montgomery_b200", "build")
    try:
        os.makedirs(d, exist_ok=True)
        if not os.access(d, os.W_OK):
            raise OSError
    except OSError:                                   # read-only tree: compile into a temporary directory
        d = str(tmp_path_factory.mktemp("gpu_units"))
    so = os.path.join(d, "gpu_units_%s.so" % gpu_units_key())
    if not os.path.exists(so):
        t0 = time.time()
        tmp = "%s.%d.tmp" % (so, os.getpid())
        compile_gpu_units(tmp)
        os.replace(tmp, so)
        print("\ntests/gpu_units/units.cu compiled in %.1f s" % (time.time() - t0))
    lib = ctypes.CDLL(so)
    for name, args in SIGNATURES.items():
        getattr(lib, name).argtypes = args
        getattr(lib, name).restype = ctypes.c_int
    return lib


def call(fn, *args):
    rc = fn(*args)
    assert rc == 0, "%s returned cudaError %d" % (fn.__name__, rc)


def enc(vals, n):
    """ints -> n little-endian 32-bit limbs each, as one uint32 array"""
    return np.frombuffer(b"".join(int(v).to_bytes(4 * n, "little") for v in vals), dtype=np.uint32).copy()


def dec(arr, n):
    b = np.ascontiguousarray(arr).tobytes()
    return [int.from_bytes(b[i:i + 4 * n], "little") for i in range(0, len(b), 4 * n)]


def ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def layouts(rare, generic, width):
    """Cases in groups of `width` (a warp of per-lane cases, or the 8 quads of a warp): for every rare case and every
    position, a group with that rare case there and generic cases everywhere else; then a group entirely rare; then
    rare and generic cases alternating."""
    out = []
    for r in rare:
        for pos in range(width):
            g = [generic() for _ in range(width)]
            g[pos] = r
            out += g
    out += [rare[i % len(rare)] for i in range(width)]
    out += [rare[(i // 2) % len(rare)] if i % 2 == 0 else generic() for i in range(width)]
    return out


# ---------------------------------------------------------------- encodings of points in Montgomery form
class WCtx:
    def __init__(self, prm, n, seed):
        self.prm, self.n, self.p = prm, n, prm.p
        self.R = 1 << (32 * n)
        self.Ri = pow(self.R, -1, self.p)
        self.A = AffineCurve(prm)
        self.INF = 1 << (32 * n - 1)
        self.rnd = random.Random(seed)
        self.pool = pool_w(prm.p, prm.q)

    def M(self, x):
        return x * self.R % self.p

    def enc_aff(self, P):                             # 4 field elements: x | y | 0 | 0, infinity flag in x's top bit
        return [self.INF, 0, 0, 0] if P is None else [self.M(P[0]), self.M(P[1]), 0, 0]

    def dec_aff(self, v):
        return None if v[0] & self.INF else (v[0] * self.Ri % self.p, v[1] * self.Ri % self.p)

    def enc_x(self, P):
        p = self.p
        if P is None:
            return [0, self.M(1), 0, 0]
        z = self.rnd.randrange(1, p)
        return [self.M(P[0] * z * z % p), self.M(P[1] * z * z * z % p), self.M(z * z % p), self.M(z * z * z % p)]

    def dec_x(self, v):
        p = self.p
        X, Y, ZZ, ZZZ = [t * self.Ri % p for t in v]
        return None if ZZ == 0 else (X * pow(ZZ, -1, p) % p, Y * pow(ZZZ, -1, p) % p)

    def pt(self):
        return self.rnd.choice(self.pool)

    def generic_pair(self):
        while True:
            P, Q = self.pt(), self.pt()
            if P[0] != Q[0]:
                return (P, Q)

    def rare_pairs(self):
        P, Q = self.pt(), self.pt()
        return [(P, P), (Q, self.A.negate(Q)), (None, P), (Q, None), (None, None)]


class TCtx:
    def __init__(self, seed):
        self.prm = prm = ED_ON_BLS12_377
        self.n, self.p = 8, prm.p
        self.R = 1 << 256
        self.Ri = pow(self.R, -1, self.p)
        self.T = TwistedEdwardsCurve(prm)
        self.rnd = random.Random(seed)
        self.pool = pool_te()

    def M(self, x):
        return x * self.R % self.p

    def enc_e(self, P):
        z = self.rnd.randrange(1, self.p)
        x, y = self.T.to_affine(P)
        return [self.M(x * z % self.p), self.M(y * z % self.p), self.M(z), self.M(x * y * z % self.p)]

    def enc_a(self, P):                               # x | y | k t (k = 2d) | 0
        x, y = self.T.to_affine(P)
        return [self.M(x), self.M(y), self.M(2 * self.prm.d * x * y % self.p), 0]

    def dec_e(self, v):
        p = self.p
        X, Y, Z, Tt = [t * self.Ri % p for t in v]
        assert (X * Y - Tt * Z) % p == 0
        zi = pow(Z, -1, p)
        return (X * zi % p, Y * zi % p)

    def pt(self):
        return self.rnd.choice(self.pool)

    def generic_pair(self):
        while True:
            P, Q = self.pt(), self.pt()
            if self.T.to_affine(P) != self.T.to_affine(Q):
                return (P, Q)

    def rare_pairs(self):
        P, Q = self.pt(), self.pt()
        Z = self.T.zero
        return [(P, P), (Q, self.T.negate(Q)), (Z, P), (Q, Z), (Z, Z)]


@lru_cache(maxsize=None)
def pool_w(p, q):
    prm = next(c for _, c, _ in W_CURVES if c.p == p)
    A = AffineCurve(prm)
    rnd = random.Random(p % 1000)
    return [A.scale(rnd.randrange(1, q), prm.G) for _ in range(48)]


@lru_cache(maxsize=None)
def pool_te():
    T = TwistedEdwardsCurve(ED_ON_BLS12_377)
    rnd = random.Random(5)
    return [T.scale(rnd.randrange(1, ED_ON_BLS12_377.q), T.one) for _ in range(48)]


# ---------------------------------------------------------------- field layer on stored operands
def edge_values(p, n):
    """Stored operands where carry chains and the dedicated squaring go wrong: all-ones limbs, top bit set in every
    limb, single limbs, p - 1, 0, 1, R mod p, powers of two up to the top bit."""
    R = 1 << (32 * n)
    e = [0, 1, 2, p - 1, p - 2, (p - 1) // 2, (p + 1) // 2, R % p, (R - 1) % p, R * R % p]
    e += [((1 << (32 * k + 32)) - 1) % p for k in range(n)]
    e += [sum(0x80000000 << (32 * i) for i in range(n)) % p, sum(0xffffffff << (32 * i) for i in range(0, n, 2)) % p]
    e += [(0xffffffff << (32 * k)) % p for k in range(n)] + [(1 << (32 * k + 31)) % p for k in range(n)]
    e += [sum(0xffffffff << (32 * i) for i in range(n - 1)), p - (1 << 32), p - (1 << 64) + 1]
    e += [(p - 1) ^ (1 << k) for k in range(0, 32 * n, 29) if (p - 1) ^ (1 << k) < p]
    return sorted(set(e))


@pytest.mark.parametrize("fid", [0, 1, 2, 3])
def test_field_ops_stored_edges(units, fid):
    """Field:: mul, sqr, add, sub, neg, to / from Montgomery form and the three inverses (Fermat, binary gcd,
    division steps) on stored operands, one per thread, against a*b/R, a*a/R, ... mod p."""
    p, n = FIELDS[fid]
    R = 1 << (32 * n)
    Ri = pow(R, -1, p)
    rnd = random.Random(1000 + fid)
    edges = edge_values(p, n)
    pow2 = [1 << k for k in range(p.bit_length() - 1)]
    A = [x for x in edges for _ in edges] + pow2 + [rnd.randrange(p) for _ in range(3000)]
    B = [y for _ in edges for y in edges] + [rnd.randrange(p) for _ in pow2] + [rnd.randrange(p) for _ in range(3000)]
    a, b = enc(A, n), enc(B, n)

    def run(op, a_, b_, k):
        o = np.zeros(k * n, dtype=np.uint32)
        call(units.gpu_fe_op, fid, op, ptr(o), ptr(a_), ptr(b_), k)
        return dec(o, n)

    k = len(A)
    for op, f in [(0, lambda x, y: x * y * Ri % p), (1, lambda x, y: (x + y) % p), (2, lambda x, y: (x - y) % p),
                  (4, lambda x, y: x * R % p), (5, lambda x, y: x * Ri % p), (6, lambda x, y: x * x * Ri % p),
                  (7, lambda x, y: (-x) % p)]:
        got = run(op, a, b, k)
        bad = [(hex(x), hex(y)) for x, y, g in zip(A, B, got) if g != f(x, y)]
        assert not bad, (fid, op, len(bad), bad[:3])
    # inverses: every distinct operand (edges, powers of two with their long trailing-zero runs, random)
    U = sorted(set(A))
    u = enc(U, n)
    exp = [pow(x * Ri, -1, p) * R % p if x else 0 for x in U]
    for op in (9, 8, 3):
        vals = U if op != 3 else U[:1500]
        got = run(op, u, u, len(vals))
        bad = [hex(x) for x, g, e in zip(vals, got, exp) if g != e]
        assert not bad, (fid, op, len(bad), bad[:3])
    # the lane-parallel inverse the MSM runs (WarpField::inv_call), one element per warp: every lane holds the result
    o = np.zeros(len(U) * 32 * n, dtype=np.uint32)
    call(units.gpu_warp_inv, fid, ptr(o), ptr(u), len(U))
    lanes = o.reshape(len(U), 32, n)
    assert (lanes == lanes[:, :1, :]).all(), fid
    got = dec(lanes[:, 0, :], n)
    bad = [hex(x) for x, g, e in zip(U, got, exp) if g != e]
    assert not bad, (fid, len(bad), bad[:3])


@pytest.mark.parametrize("fid", [0, 1, 2, 3])
def test_field_op_warp_inverse_product_library(fid):
    """op 9 of mgb_field_op (WarpField::inv_call in the product library, plain values in and out)."""
    from montgomery_b200 import _native
    lib = _native.lib()
    p, n = FIELDS[fid]
    rnd = random.Random(1100 + fid)
    vals = edge_values(p, n) + [1 << k for k in range(p.bit_length() - 1)] + [rnd.randrange(p) for _ in range(1500)]
    a = np.frombuffer(b"".join(v.to_bytes(4 * n, "little") for v in vals), dtype=np.uint8).copy()
    out = np.zeros_like(a)
    rc = lib.mgb_field_op(0, fid, 9, ptr(a), ptr(a), ptr(out), len(vals))
    assert rc == 0
    got = [int.from_bytes(out[i * 4 * n:(i + 1) * 4 * n].tobytes(), "little") for i in range(len(vals))]
    bad = [hex(x) for x, g in zip(vals, got) if g != (pow(x, -1, p) if x else 0)]
    assert not bad, (fid, len(bad), bad[:3])


@pytest.mark.parametrize("fid", [0, 1, 2, 3])
def test_warp_mul_one_and_two_limbs_per_lane(units, fid):
    """WarpField::mul (16-lane groups) and WarpField2::mul (8-lane groups) on stored edge operands and random ones;
    the lanes above the top limb get garbage and must return 0; an odd count leaves part of the last warp idle."""
    p, n = FIELDS[fid]
    R = 1 << (32 * n)
    Ri = pow(R, -1, p)
    rnd = random.Random(1200 + fid)
    edges = edge_values(p, n)
    A = [x for x in edges for _ in edges] + [rnd.randrange(p) for _ in range(4001)]
    B = [y for _ in edges for y in edges] + [rnd.randrange(p) for _ in range(4001)]
    exp = [x * y * Ri % p for x, y in zip(A, B)]
    for fn in (units.gpu_warp_mul, units.gpu_warp_mul2):
        o = np.zeros(len(A) * 16, dtype=np.uint32)
        call(fn, fid, ptr(o), ptr(enc(A, n)), ptr(enc(B, n)), len(A))
        o = o.reshape(len(A), 16)
        assert not o[:, n:].any(), (fn.__name__, fid)
        got = dec(np.ascontiguousarray(o[:, :n]), n)
        bad = [(hex(x), hex(y)) for x, y, g, e in zip(A, B, got, exp) if g != e]
        assert not bad, (fn.__name__, fid, len(bad), bad[:3])


@pytest.mark.parametrize("fid", [0, 1, 2, 3])
def test_warp_distributed_add_sub(units, fid):
    """WarpField2 add / sub / dbl / is_zero with carries and borrows rippling across the lanes of a group."""
    p, n = FIELDS[fid]
    rnd = random.Random(1300 + fid)
    W64 = (1 << 64) - 1
    D = n // 2
    special = [0, 1, p - 1, p - 2, (p - 1) // 2, (p + 1) // 2, W64, 1 << 64, (1 << (64 * (D - 1))) - 1, 1 << (64 * (D - 1)),
               p - (1 << 64), p - W64, sum(W64 << (64 * i) for i in range(D - 1))]
    special = sorted(set(x % p for x in special + edge_values(p, n)))
    A = [x for x in special for _ in special] + [rnd.randrange(p) for _ in range(2000)] + special + special
    B = [y for _ in special for y in special] + [rnd.randrange(p) for _ in range(2000)] + special + [(p - x) % p for x in special]
    for op, f in ((0, lambda a, b: (a + b) % p), (1, lambda a, b: (a - b) % p), (2, lambda a, b: 2 * a % p), (3, lambda a, b: int(a == 0))):
        o = np.zeros(len(A) * 16, dtype=np.uint32)
        call(units.gpu_warp_addsub2, fid, op, ptr(o), ptr(enc(A, n)), ptr(enc(B, n)), len(A))
        got = dec(np.ascontiguousarray(o.reshape(len(A), 16)[:, :n]), n)
        if op == 3:
            got = [g & W64 for g in got]             # the flag comes back in every digit of the group
        bad = [(hex(a), hex(b)) for a, b, g in zip(A, B, got) if g != f(a, b)]
        assert not bad, (fid, op, len(bad), bad[:3])


@pytest.mark.parametrize("fid", [0, 1, 2, 3])
def test_warp_carry_and_borrow_lookahead(units, fid):
    """WarpField::finish and WarpField2::finish alone, on carries through runs of all-ones limbs / digits, borrows
    through limbs equal to the modulus's and pending carries at their maximum, many warps in one launch."""
    p, n = FIELDS[fid]
    rnd = random.Random(1400 + fid)
    plimbs = [(p >> (32 * i)) & 0xFFFFFFFF for i in range(n)]
    cases = []
    for lo_run in range(0, n - 1):
        for hi_run in range(lo_run, n - 1):
            for _ in range(3):
                t = [rnd.getrandbits(32) for _ in range(n)]
                c = [0] * n
                for i in range(lo_run, hi_run + 1):
                    t[i] = 0xFFFFFFFF
                t[n - 1] = rnd.randrange(plimbs[n - 1])
                c[lo_run] = rnd.choice([1, 2, (1 << 32) + 1, (1 << 33) + 8])
                if lo_run > 0:
                    t[lo_run - 1], c[lo_run - 1] = 0xFFFFFFFF, rnd.choice([1, 1 << 32])
                cases.append((t, c))
    for k in range(1, n):
        v = p + (1 << (32 * k)) - 1 - rnd.randrange(2)
        if v < 2 * p:
            cases.append(([(v >> (32 * i)) & 0xFFFFFFFF for i in range(n)], [0] * n))
    for v in (p, p - 1, p + 1, 2 * p - 1, 0, 1):
        cases.append(([(v >> (32 * i)) & 0xFFFFFFFF for i in range(n)], [0] * n))
    for _ in range(400):
        c = [rnd.randrange((1 << 33) + 9) for _ in range(n - 2)] + [rnd.randrange(4), 0]
        v = rnd.randrange(sum(ci << (32 * i) for i, ci in enumerate(c)), 2 * p)
        rest = v - sum(ci << (32 * i) for i, ci in enumerate(c))
        cases.append(([(rest >> (32 * i)) & 0xFFFFFFFF for i in range(n)], c))
    if len(cases) % 2:
        cases.append(cases[0])
    nw = len(cases) // 2
    t = np.zeros(nw * 32, dtype=np.uint32)
    c = np.zeros(nw * 32, dtype=np.uint64)
    for j, (tt, cc) in enumerate(cases):
        t[16 * j:16 * j + n] = tt
        c[16 * j:16 * j + n] = cc
    o = np.zeros(nw * 32, dtype=np.uint32)
    call(units.gpu_warp_finish, fid, ptr(o), ptr(t), ptr(c), nw)
    for j, (tt, cc) in enumerate(cases):
        v = sum((a + b) << (32 * i) for i, (a, b) in enumerate(zip(tt, cc)))
        got = sum(int(o[16 * j + i]) << (32 * i) for i in range(n))
        assert got == (v - p if v >= p else v) and not o[16 * j + n:16 * j + 16].any(), (fid, j, hex(v))
    # two limbs per lane
    D = n // 2
    W64 = (1 << 64) - 1
    pd = [(p >> (64 * i)) & W64 for i in range(D)]
    val2 = lambda t_, lo, hi: sum((a + b + (c_ << 64)) << (64 * i) for i, (a, b, c_) in enumerate(zip(t_, lo, hi)))
    cases2 = []
    for lo_run in range(0, D - 1):
        for hi_run in range(lo_run, D - 1):
            for _ in range(4):
                t_ = [rnd.getrandbits(64) for _ in range(D)]
                lo, hi = [0] * D, [0] * D
                for i in range(lo_run, hi_run + 1):
                    t_[i] = W64
                t_[D - 1] = rnd.randrange(pd[D - 1])
                lo[lo_run] = rnd.choice([1, 2, W64])
                if lo_run > 0:
                    t_[lo_run - 1], hi[lo_run - 1] = W64, rnd.choice([1, 2])
                if val2(t_, lo, hi) < 2 * p:
                    cases2.append((t_, lo, hi))
    for v in [p, p - 1, p + 1, 2 * p - 1, 0, 1] + [p + (1 << (64 * k)) - 1 for k in range(1, D)]:
        if v < 2 * p:
            cases2.append(([(v >> (64 * i)) & W64 for i in range(D)], [0] * D, [0] * D))
    for _ in range(400):
        lo = [rnd.getrandbits(64) for _ in range(D - 2)] + [rnd.randrange(4), 0]
        hi = [rnd.randrange(3) for _ in range(D - 2)] + [0, 0]
        low = val2([0] * D, lo, hi)
        v = rnd.randrange(low, 2 * p)
        cases2.append(([((v - low) >> (64 * i)) & W64 for i in range(D)], lo, hi))
    while len(cases2) % 4:
        cases2.append(cases2[0])
    nw = len(cases2) // 4
    t2 = np.zeros(nw * 32, dtype=np.uint64)
    lo2 = np.zeros(nw * 32, dtype=np.uint64)
    hi2 = np.zeros(nw * 32, dtype=np.uint32)
    for j, (a, b, c_) in enumerate(cases2):
        t2[8 * j:8 * j + D], lo2[8 * j:8 * j + D], hi2[8 * j:8 * j + D] = a, b, c_
    o2 = np.zeros(nw * 32, dtype=np.uint64)
    call(units.gpu_warp_finish2, fid, ptr(o2), ptr(t2), ptr(lo2), ptr(hi2), nw)
    for j, cs in enumerate(cases2):
        v = val2(*cs)
        got = sum(int(o2[8 * j + i]) << (64 * i) for i in range(D))
        assert got == (v - p if v >= p else v) and not o2[8 * j + D:8 * j + 8].any(), (fid, j, hex(v))


# ---------------------------------------------------------------- group law, rare lanes among generic ones
@pytest.mark.parametrize("cid,prm,n", W_CURVES, ids=W_IDS)
def test_weierstrass_ops_rare_lanes(units, cid, prm, n):
    """ec.cuh Weierstrass: affine add through prepare / invert / finish, madd, XYZZ add, dbl, to / from affine; one
    case per thread, rare cases at every lane position of a warp of generic ones, a warp of rare ones, alternating."""
    w = WCtx(prm, n, 2000 + cid)
    A = w.A
    two = layouts(w.rare_pairs(), w.generic_pair, 32)
    one = layouts([(None, None)], lambda: (w.pt(), None), 32)
    for op, cases, ea, eb, dec_, f in [
            (0, two, w.enc_aff, w.enc_aff, w.dec_aff, lambda P, Q: A.add(P, Q)),
            (1, two, w.enc_x, w.enc_aff, w.dec_x, lambda P, Q: A.add(P, Q)),
            (2, two, w.enc_x, w.enc_x, w.dec_x, lambda P, Q: A.add(P, Q)),
            (3, one + [(Q, None) for Q in w.pool], w.enc_x, w.enc_x, w.dec_x, lambda P, Q: A.double(P)),
            (4, one, w.enc_x, w.enc_x, w.dec_aff, lambda P, Q: P),
            (5, one, w.enc_aff, w.enc_aff, w.dec_x, lambda P, Q: P)]:
        a = enc([v for P, _ in cases for v in ea(P)], n)
        b = enc([v for _, Q in cases for v in eb(Q)], n)
        o = np.zeros_like(a)
        call(units.gpu_w_op, cid, op, ptr(o), ptr(a), ptr(b), len(cases))
        got = dec(o, n)
        for j, (P, Q) in enumerate(cases):
            assert dec_(got[4 * j:4 * j + 4]) == f(P, Q), (cid, op, j)


def test_twisted_edwards_ops_rare_lanes(units):
    """ec.cuh TwistedEdwards (ed-on-BLS12-377): add, madd, add_affine, dbl, to_affine with the same layouts."""
    t = TCtx(2100)
    T = t.T
    two = layouts(t.rare_pairs(), t.generic_pair, 32)
    one = layouts([(T.zero, T.zero)], lambda: (t.pt(), T.zero), 32)
    for op, cases, ea, eb, f in [
            (0, two, t.enc_e, t.enc_e, lambda P, Q: T.to_affine(T.add(P, Q))),
            (1, two, t.enc_e, t.enc_a, lambda P, Q: T.to_affine(T.add(P, Q))),
            (2, two, t.enc_a, t.enc_a, lambda P, Q: T.to_affine(T.add(P, Q))),
            (3, one, t.enc_e, t.enc_e, lambda P, Q: T.to_affine(T.double(P))),
            (4, one, t.enc_e, t.enc_e, lambda P, Q: T.to_affine(P))]:
        a = enc([v for P, _ in cases for v in ea(P)], 8)
        b = enc([v for _, Q in cases for v in eb(Q)], 8)
        o = np.zeros_like(a)
        call(units.gpu_te_op, op, ptr(o), ptr(a), ptr(b), len(cases))
        got = dec(o, 8)
        for j, (P, Q) in enumerate(cases):
            g = got[4 * j:4 * j + 4]
            res = tuple(v * t.Ri % t.p for v in g[:2]) if op == 4 else t.dec_e(g)
            assert res == f(P, Q), (op, j)


@pytest.mark.parametrize("cid,prm,n", W_CURVES, ids=W_IDS)
def test_quad_cooperative_addition_rare_quads(units, cid, prm, n):
    """QuadWeierstrass::add (8 additions per warp): a rare addition in each of the 8 quad positions of a warp of
    generic ones (the __any_sync branch with the serial formula on one lane of the quad), a warp of rare ones,
    alternating."""
    w = WCtx(prm, n, 2200 + cid)
    cases = layouts(w.rare_pairs(), w.generic_pair, 8)
    a = enc([v for P, _ in cases for v in w.enc_x(P)], n)
    b = enc([v for _, Q in cases for v in w.enc_x(Q)], n)
    o = np.zeros_like(a)
    call(units.gpu_quad_add, cid, ptr(o), ptr(a), ptr(b), len(cases) // 8)
    got = dec(o, n)
    for j, (P, Q) in enumerate(cases):
        assert w.dec_x(got[4 * j:4 * j + 4]) == w.A.add(P, Q), (cid, j)


@pytest.mark.parametrize("cid", [0, 1, 2, 3], ids=W_IDS + ["ed-on-bls12-377"])
def test_onewarp_horner_steps(units, cid):
    """onewarp.cuh (what k_final and k_window_assemble run), one case per warp, many warps per launch: runs of
    doublings, additions with every rare case, one Horner step 2^k P + Q including an empty top window."""
    if cid == 3:
        t = TCtx(2300)
        Tc = t.T
        zero, add, dbl, encp = Tc.zero, Tc.add, Tc.double, t.enc_e
        norm, neg = Tc.to_affine, Tc.negate
        decp = t.dec_e
        gen, rare, nl = t.generic_pair, t.rare_pairs, 8
    else:
        _, prm, nl = W_CURVES[cid]
        w = WCtx(prm, nl, 2300 + cid)
        zero, add, dbl, encp = None, w.A.add, w.A.double, w.enc_x
        norm, neg = (lambda P: P), w.A.negate
        decp = w.dec_x
        gen, rare = w.generic_pair, w.rare_pairs

    def dbl_k(P, k):
        for _ in range(k):
            P = dbl(P)
        return P

    def run(op, count, cases):
        a = enc([v for P, _ in cases for v in encp(P)], nl)
        b = enc([v for _, Q in cases for v in encp(Q)], nl)
        o = np.zeros_like(a)
        call(units.gpu_onewarp, cid, op, count, ptr(o), ptr(a), ptr(b), len(cases))
        got = dec(o, nl)
        return [decp(got[4 * j:4 * j + 4]) for j in range(len(cases))]

    adds = []
    for _ in range(24):
        adds += [gen(), gen()] + rare()
    assert run(1, 0, adds) == [norm(add(P, Q)) for P, Q in adds]
    for count in (0, 1, 2, 5, 13):
        cases = [gen() for _ in range(20)] + [(zero, zero)] * 3
        assert run(0, count, cases) == [norm(dbl_k(P, count)) for P, _ in cases], count
    # 2^4 P + Q with Q generic, an empty top window (P neutral), Q = 2^4 P (doubling), Q = -2^4 P, Q neutral
    steps = [gen() for _ in range(30)] + [(zero, gen()[1]) for _ in range(4)]
    for P, _ in [gen() for _ in range(3)]:
        steps += [(P, dbl_k(P, 4)), (P, neg(dbl_k(P, 4))), (P, zero)]
    assert run(2, 4, steps) == [norm(add(dbl_k(P, 4), Q)) for P, Q in steps]


# ---------------------------------------------------------------- kernels on synthetic buckets
def bucket_refs(rnd, npts, endo):
    """One bucket of 1..4 references; a third of them rare: doubling / cancellation in round 0 or in round 1, an
    infinite left or right operand in round 1."""
    def ref():
        return rnd.randrange(npts) | rnd.choice([0, REF_NEG]) | (rnd.choice([0, REF_ENDO]) if endo else 0)
    a, b, c, d = ref(), ref(), ref(), ref()
    kind = rnd.randrange(12)
    return [[a, a, c, d], [a, a ^ REF_NEG, c, d], [c, d, a, a ^ REF_NEG], [a, a ^ REF_NEG, b, b ^ REF_NEG],
            [a, b, a, b], [a, b, a ^ REF_NEG, b ^ REF_NEG], [a, a], [a, a ^ REF_NEG],
            [a], [a, b, c], [a, b], [a, b, c, d]][kind]


@pytest.mark.parametrize("e_big,blocks", [(1, 0), (8, 0), (64, 0), (2, 8)], ids=["E1", "E8", "E64", "E2-dynamic-tiles"])
@pytest.mark.parametrize("cid,prm,n", W_CURVES, ids=W_IDS)
def test_batch_add_two_rounds(units, cid, prm, n, e_big, blocks):
    """k_batch_add<CV, MGB_EMAX, MGB_MINB> on #SM x MINB blocks (blocks = 8: more tiles than warps, so most are handed
    out dynamically): two tree rounds over 4096 synthetic buckets with doublings and cancellations scattered through
    every tile.  Every written slot, and the next round's pair list (no duplicates, no holes)."""
    p = prm.p
    R = 1 << (32 * n)
    Ri = pow(R, -1, p)
    A = AffineCurve(prm)
    rnd = random.Random(3000 + 10 * cid + e_big)
    pts = pool_w(prm.p, prm.q)
    table = enc([v for x, y in pts for v in (x * R % p, y * R % p, prm.beta * x % p * R % p)], n)

    def ref_point(r_):
        x, y = pts[r_ & 0x3FFFFFFF]
        if r_ & REF_ENDO:
            x = prm.beta * x % p
        return (x, (-y) % p) if r_ & REF_NEG else (x, y)

    def add_all(refs):
        acc = None
        for r_ in refs:
            acc = A.add(acc, ref_point(r_))
        return acc

    buckets = [bucket_refs(rnd, len(pts), True) for _ in range(4096)]
    recs, lifes = [], []
    for refs in buckets:
        k = len(refs)
        recs += [refs[0], refs[1] if k > 1 else REF_EMPTY]
        lifes.append(2 if k > 2 else 1)
        recs += [refs[2], refs[3] if k > 3 else REF_EMPTY] if k > 2 else [REF_EMPTY, REF_EMPTY]
        lifes.append(1)
    npairs = 2 * len(buckets)
    recs = np.array(recs, dtype=np.uint32)
    lifes = np.array(lifes, dtype=np.uint8)
    offs = np.array([0, 2 * npairs], dtype=np.uint32)
    V = np.zeros(2 * npairs * 2 * n, dtype=np.uint32)
    pairs_a = np.zeros(2 * npairs, dtype=np.uint32)
    pairs_b = np.zeros(2 * npairs, dtype=np.uint32)
    cnt_a, cnt_b = np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.uint32)
    call(units.gpu_batch_add, cid, 1, ptr(V), V.size, None, 0, 0, e_big, 0xFFFFFFFF, ptr(pairs_a), npairs, ptr(cnt_a),
         ptr(recs), npairs, ptr(lifes), lifes.size, ptr(table), table.size, ptr(offs), 0, 1, blocks)

    def slot(s):
        w_ = V[s * 2 * n:(s + 1) * 2 * n]
        if int(w_[n - 1]) & 0x80000000:
            return None
        x, y = dec(w_, n)
        return (x * Ri % p, y * Ri % p)

    exp_pairs = []
    for j, refs in enumerate(buckets):
        assert slot(4 * j) == add_all(refs[:2]), ("round 0, first half of bucket", j, refs)
        if len(refs) > 2:
            assert slot(4 * j + 2) == add_all(refs[2:]), ("round 0, second half of bucket", j, refs)
            exp_pairs.append((4 * j, 2))
    got = [(int(pairs_a[2 * i]), int(pairs_a[2 * i + 1])) for i in range(int(cnt_a[0]))]
    assert len(got) == len(exp_pairs) and sorted(got) == exp_pairs
    call(units.gpu_batch_add, cid, 0, ptr(V), V.size, ptr(pairs_a), int(cnt_a[0]), 1, e_big, 0xFFFFFFFF, ptr(pairs_b), npairs,
         ptr(cnt_b), None, 0, None, 0, None, 0, None, 0, 0, blocks)
    for j, refs in enumerate(buckets):
        assert slot(4 * j) == add_all(refs), ("round 1, bucket", j, refs)
    assert cnt_b[0] == 0


def test_pair_add_two_rounds_twisted_edwards(units):
    """k_pair_add<CurveEd377> as msm.cu launches it: two tree rounds over 4096 buckets laid out back to back, with
    doublings and cancellations in both rounds; every written slot and the next round's pair list."""
    prm, n = ED_ON_BLS12_377, 8
    p = prm.p
    R = 1 << 256
    Ri = pow(R, -1, p)
    T = TwistedEdwardsCurve(prm)
    rnd = random.Random(3100)
    pts = pool_te()
    tab = []
    for P in pts:
        x, y = T.to_affine(P)
        tab += [x * R % p, y * R % p, x * y % p * R % p, 2 * prm.d * x * y % p * R % p]
    table = enc(tab, n)
    ref_point = lambda r_: T.negate(pts[r_ & 0x3FFFFFFF]) if r_ & REF_NEG else pts[r_ & 0x3FFFFFFF]

    def add_all(refs):
        acc = T.zero
        for r_ in refs:
            acc = T.add(acc, ref_point(r_))
        return T.to_affine(acc)

    buckets = []
    while len(buckets) < 4096:
        refs = bucket_refs(rnd, len(pts), False)
        if len(refs) >= 2:                            # the scatter never leaves a lone point in a pair of its own
            buckets.append(refs)
    recs, lifes, first_slot = [], [], []
    for refs in buckets:
        first_slot.append(len(recs))
        recs += [refs[0], refs[1]]
        lifes.append(2 if len(refs) > 2 else 1)
        if len(refs) > 2:
            recs += [refs[2], refs[3] if len(refs) > 3 else REF_EMPTY]
            lifes.append(1)
    npairs = len(lifes)
    recs = np.array(recs, dtype=np.uint32)
    lifes = np.array(lifes + [0] * (-len(lifes) % 4), dtype=np.uint8)
    offs = np.array([0, 2 * npairs], dtype=np.uint32)
    V = np.zeros(2 * npairs * 4 * n, dtype=np.uint32)
    pairs_a, pairs_b = np.zeros(2 * npairs, dtype=np.uint32), np.zeros(2 * npairs, dtype=np.uint32)
    cnt_a, cnt_b = np.zeros(1, dtype=np.uint32), np.zeros(1, dtype=np.uint32)
    call(units.gpu_pair_add_te, 1, ptr(V), V.size, None, 0, 0, ptr(pairs_a), npairs, ptr(cnt_a), ptr(recs), npairs,
         ptr(lifes), lifes.size, ptr(table), table.size, ptr(offs), 0, 1)

    def slot(s):
        X, Y, Z, Tt = [v * Ri % p for v in dec(V[s * 4 * n:(s + 1) * 4 * n], n)]
        assert (X * Y - Tt * Z) % p == 0
        zi = pow(Z, -1, p)
        return (X * zi % p, Y * zi % p)

    exp_pairs = []
    for refs, s0 in zip(buckets, first_slot):
        assert slot(s0) == add_all(refs[:2]), (s0, refs)
        if len(refs) > 2:
            assert slot(s0 + 2) == add_all(refs[2:]), (s0, refs)
            exp_pairs.append((s0, 2))
    got = [(int(pairs_a[2 * i]), int(pairs_a[2 * i + 1])) for i in range(int(cnt_a[0]))]
    assert len(got) == len(exp_pairs) and sorted(got) == exp_pairs
    call(units.gpu_pair_add_te, 0, ptr(V), V.size, ptr(pairs_a), int(cnt_a[0]), 1, ptr(pairs_b), npairs, ptr(cnt_b),
         None, 0, None, 0, None, 0, None, 0, 0)
    for refs, s0 in zip(buckets, first_slot):
        assert slot(s0) == add_all(refs), (s0, refs)
    assert cnt_b[0] == 0


@pytest.mark.parametrize("cid", [0, 1, 2, 3], ids=W_IDS + ["ed-on-bls12-377"])
def test_final_horner_kernel(units, cid):
    """k_final: sum_w 2^(c w) S_w over K window sums (an empty top window, a neutral one inside, two equal ones),
    with and without the fused normalisation, and a sum that is the neutral element."""
    if cid == 3:
        t = TCtx(3200)
        nl, zero, add, dbl, encp, norm = 8, t.T.zero, t.T.add, t.T.double, t.enc_e, t.T.to_affine
        decp, pt = t.dec_e, t.pt
    else:
        _, prm, nl = W_CURVES[cid]
        w = WCtx(prm, nl, 3200 + cid)
        zero, add, dbl, encp, norm = None, w.A.add, w.A.double, w.enc_x, (lambda P: P)
        decp, pt = w.dec_x, w.pt
    for K, c in ((7, 5), (3, 13), (2, 1)):
        S = [pt() for _ in range(K)]
        S[K - 1] = zero                              # empty top window
        if K > 3:
            S[1] = zero
            S[3] = S[2]
        exp = zero
        for s in reversed(S):
            for _ in range(c):
                exp = dbl(exp)
            exp = add(exp, s)
        words = enc([v for s in S for v in encp(s)], nl)
        acc = np.zeros(4 * nl, dtype=np.uint32)
        xy = np.zeros(2 * nl, dtype=np.uint32)
        flag = np.full(1, 7, dtype=np.uint32)
        call(units.gpu_final, cid, K, c, ptr(words), ptr(acc), ptr(xy), ptr(flag))
        assert decp(dec(acc, nl)) == norm(exp), (K, c)
        is_zero = exp is None if cid != 3 else norm(exp) == (0, 1)
        exp_xy = (0, 0) if exp is None else norm(exp)
        assert (tuple(dec(xy, nl)), int(flag[0])) == (exp_xy, int(is_zero)), (K, c)
        acc2 = np.zeros_like(acc)
        call(units.gpu_final, cid, K, c, ptr(words), ptr(acc2), None, None)
        assert (acc2 == acc).all()
    if cid != 3:
        words = enc([v for _ in range(3) for v in encp(None)], nl)
        call(units.gpu_final, cid, 3, 4, ptr(words), ptr(acc), ptr(xy), ptr(flag))
        assert flag[0] == 1 and not xy.any()


@pytest.mark.parametrize("cid,prm,n", W_CURVES, ids=W_IDS)
def test_normalize_partials(units, cid, prm, n):
    """k_normalize: 1, 2, 3, 8, 11 and 17 partial accumulators (the multi-GPU combine) with a neutral one, a duplicate
    and a cancelling pair among them, with and without the per-rank status words."""
    w = WCtx(prm, n, 3300 + cid)
    A = w.A
    for count in (1, 2, 3, 8, 11, 17):
        sel = [w.pt() for _ in range(count)]
        if count >= 3:
            sel[1] = None
        if count >= 8:
            sel[5] = sel[4]
            sel[7] = A.negate(sel[6])
        exp = None
        for P in sel:
            exp = A.add(exp, P)
        for status in (None, 3):
            stride = 4 * n if status is None else 4 * n + 4
            recs = []
            for k, P in enumerate(sel):
                recs.append(enc(w.enc_x(P), n))
                if status is not None:                # the rank's status word, padded to four limbs
                    recs.append(np.array([status if k == count // 2 else 0, 9, 9, 9], dtype=np.uint32))
            arr = np.concatenate(recs)
            assert arr.size == count * stride
            xy = np.zeros(2 * n, dtype=np.uint32)
            flag = np.full(2, 7, dtype=np.uint32)
            call(units.gpu_normalize, cid, ptr(arr), count, stride, ptr(xy), ptr(flag))
            assert (tuple(dec(xy, n)), int(flag[0])) == (((0, 0), 1) if exp is None else (exp, 0)), (count, status)
            assert (flag[1] != 0) == (status is not None), (count, status)


@pytest.mark.parametrize("cid", [0, 1, 2, 3], ids=W_IDS + ["ed-on-bls12-377"])
def test_set_get_points(units, cid):
    """k_set_points / k_get_points over 4101 points (a partly idle last block) with infinity flags at density 1/8 on
    the Weierstrass curves: the Montgomery table entry and the round trip."""
    rnd = random.Random(3400 + cid)
    npts = 4101
    if cid == 3:
        t = TCtx(3400)
        n, p, R = 8, t.p, t.R
        pts = [t.T.to_affine(t.pt()) for _ in range(npts)]
        flags = None
    else:
        _, prm, n = W_CURVES[cid]
        p, R = prm.p, 1 << (32 * n)
        pool = pool_w(prm.p, prm.q)
        pts = [rnd.choice(pool) for _ in range(npts)]
        flags = np.array([1 if rnd.randrange(8) == 0 else 0 for _ in range(npts)], dtype=np.uint8)
    xy = enc([v for x, y in pts for v in (x, y)], n)
    el = 3 * n if cid != 3 else 4 * n
    table = np.zeros(npts * el, dtype=np.uint32)
    back = np.zeros_like(xy)
    zback = np.zeros(npts, dtype=np.uint8)
    call(units.gpu_set_get_points, cid, npts, ptr(xy), None if flags is None else ptr(flags), ptr(table), ptr(back), ptr(zback))
    ents = table.reshape(npts, el)
    got = dec(back, n)
    for i, (x, y) in enumerate(pts):
        e = dec(ents[i], n)
        if flags is not None and flags[i]:
            assert e[0] >> (32 * n - 1) == 1 and zback[i] == 1 and got[2 * i:2 * i + 2] == [0, 0], i
            continue
        if cid == 3:
            assert e == [x * R % p, y * R % p, x * y % p * R % p, 2 * ED_ON_BLS12_377.d * x * y % p * R % p], i
        else:
            assert e == [x * R % p, y * R % p, W_CURVES[cid][1].beta * x % p * R % p], i
        assert (got[2 * i], got[2 * i + 1], int(zback[i])) == (x, y, 0), i


# ---------------------------------------------------------------- adversarial whole MSMs (closed form)
MSM_CURVES = {"bls12-377": m.curves.BLS12_377, "pallas": m.curves.PALLAS, "ed-on-bls12-377": m.curves.ED_ON_BLS12_377,
              "bls12-381": m.curves.BLS12_381}
NMSM = 1 << 16
# default plan, two explicit window sizes, the affine bucket reduction, tree depth 0 / 2, the finish kernel off / on
SETTINGS = [({}, {}), ({"c": 9}, {}), ({"c": 14}, {}), ({"affine_reduction": True}, {}), ({}, {"MGB_DEBUG_NROUNDS": "0"}),
            ({}, {"MGB_DEBUG_NROUNDS": "2"}), ({}, {"MGB_DEBUG_FINISH": "0"}), ({}, {"MGB_DEBUG_FINISH": "1"}),
            ({"affine_reduction": True}, {"MGB_DEBUG_NROUNDS": "2"})]


@pytest.fixture(scope="module")
def msm_engines():
    cache = {}

    def get(label):
        if label not in cache:
            cache[label] = m.MsmEngine(MSM_CURVES[label], 0, NMSM)
        return cache[label]

    yield get
    for e in cache.values():
        e.close()


def msm_all_settings(eng, sc, exp, what, monkeypatch):
    for kw, env in SETTINGS:
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            res, tm = eng.msm(sc, n=NMSM, **kw)
        assert res == exp, (what, kw, env, tm)


def neg_dlog(O, a):
    return (O.q - a) % O.q


@pytest.mark.parametrize("label", list(MSM_CURVES))
def test_msm_one_point_random_scalars(msm_engines, label, monkeypatch):
    """n = 2^16 copies of one point P with random scalars: (sum s_i mod q) P.  The GLV buckets hold P, -P, phi P and
    -phi P mixed (P and -P on the twisted-Edwards curve), so about half of round 0's additions are doublings or
    cancellations next to generic lanes, and the bucket sums collide in the reduction."""
    eng = msm_engines(label)
    O = OracleCurve(label)
    a = 0x1234567 + len(label)
    P = O.scale(a, O.G)
    xy, _ = points_to_bytes([P], eng.curve.coord_bytes)
    eng.set_points(np.tile(xy, NMSM))
    sc = inputs.random_scalars(O.q, NMSM, seed=5000 + len(label))
    k = sum(inputs.scalars_to_ints(sc)) * a % O.q
    msm_all_settings(eng, sc, O.result_of(O.scale(k, O.G)), "one point", monkeypatch)


@pytest.mark.parametrize("label", list(MSM_CURVES))
def test_msm_three_points_and_negations(msm_engines, label, monkeypatch):
    """P1, P2, P3, -P1, -P2, -P3 cycled over 2^16 inputs with random scalars."""
    eng = msm_engines(label)
    O = OracleCurve(label)
    d = [11, 2 ** 100 + 7, O.q // 3]
    d += [neg_dlog(O, x) for x in d]
    xy, _ = points_to_bytes([O.scale(x, O.G) for x in d], eng.curve.coord_bytes)
    eng.set_points(np.tile(xy, NMSM // 6 + 1)[:NMSM * eng.curve.point_bytes])
    sc = inputs.random_scalars(O.q, NMSM, seed=5100 + len(label))
    k = sum(s * d[i % 6] for i, s in enumerate(inputs.scalars_to_ints(sc))) % O.q
    msm_all_settings(eng, sc, O.result_of(O.scale(k, O.G)), "three points", monkeypatch)


@pytest.mark.parametrize("label", ["bls12-377", "pallas", "bls12-381"])
def test_msm_points_at_infinity(msm_engines, label, monkeypatch):
    """Known-dlog points with 1/8 of them set to infinity through set_points' flags, n = 2^16: sum s_i a_i with
    a_i = 0 for those points."""
    eng = msm_engines(label)
    O = OracleCurve(label)
    seed = 5200 + len(label)
    eng.random_points(NMSM, seed=seed)
    a = [int(v) for v in inputs.known_dlogs(seed, NMSM)]
    xy, _ = eng.get_points(0, NMSM)
    rng = np.random.default_rng(seed)
    z = (rng.integers(0, 8, NMSM) == 0).astype(np.uint8)
    eng.set_points(xy.reshape(-1).copy(), z)
    sc = inputs.random_scalars(O.q, NMSM, seed=seed + 1)
    k = sum(s * (0 if f else ai) for s, ai, f in zip(inputs.scalars_to_ints(sc), a, z)) % O.q
    msm_all_settings(eng, sc, O.result_of(O.scale(k, O.G)), "infinity", monkeypatch)


@pytest.mark.parametrize("label", list(MSM_CURVES))
def test_msm_structured_scalars(msm_engines, label, monkeypatch):
    """Structured scalars at the engine's own window size c, n = 2^16 known-dlog points: 0, 1, q - 1 (and q, 2^256 - 1
    on the GLV curves, which reduce any 256-bit scalar); multiples of 2^c; every c-bit digit equal to 2^(c-1), the
    carry boundary of the signed digits; lambda and lambda + 1, GLV halves with k1 = 0 or k2 = 0."""
    eng = msm_engines(label)
    O = OracleCurve(label)
    q = O.q
    seed = 5300 + len(label)
    eng.random_points(NMSM, seed=seed)
    a = [int(v) for v in inputs.known_dlogs(seed, NMSM)]
    probe = scalars_to_bytes([1] * NMSM)
    _, tm = eng.msm(probe, n=NMSM)
    c = tm["c"]
    rnd = random.Random(seed)
    glv = O.kind == "weierstrass"
    base = [0, 1, q - 1] + ([q, (1 << 256) - 1] if glv else [])
    half = sum(1 << (c - 1 + c * w) for w in range(q.bit_length() // c + 1))
    sets = {
        "edges": [base[i % len(base)] for i in range(NMSM)],
        "multiples of 2^c": [rnd.randrange(q >> c) << c for _ in range(NMSM)],
        "digits 2^(c-1)": [half % q if glv else half & ((1 << (q.bit_length() - 1)) - 1) for _ in range(NMSM)],
    }
    if glv:
        lam = O.prm.lam
        half128 = sum(1 << (c - 1 + c * w) for w in range(120 // c))
        sets["digits 2^(c-1), GLV halves"] = [(half128 + half128 * lam) % q] * NMSM
        sets["lambda, lambda + 1"] = [[lam, lam + 1, (rnd.randrange(1 << 100) * lam) % q, rnd.randrange(1 << 100)][i % 4] for i in range(NMSM)]
    for what, vals in sets.items():
        sc = scalars_to_bytes(vals)
        k = sum(s * ai for s, ai in zip(vals, a)) % q
        msm_all_settings(eng, sc, O.result_of(O.scale(k, O.G)), what, monkeypatch)
