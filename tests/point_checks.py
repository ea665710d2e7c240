"""Test inputs for checked point ingestion (mgb_set_points_checked), built on the oracle's curves, and a Python mirror of
the device's membership test.

Points are affine (x, y) tuples of Python integers, None for a point flagged as zero (as in tests/helpers.py).  The
coordinates of a non-canonical encoding are >= p; they still fit the 4N-byte format.

Status bits (include/montgomery_b200.h): NONCANONICAL = x or y >= p; OFF_CURVE = the curve equation fails (canonical
points only); NOT_IN_SUBGROUP = on the curve, outside the prime-order subgroup.
"""
import random

from tests.helpers import ORACLE_PARAMS, OracleCurve

NONCANONICAL, OFF_CURVE, NOT_IN_SUBGROUP = 1, 2, 4
COORD_BYTES = {"bls12-377": 48, "pallas": 32, "ed-on-bls12-377": 32, "bls12-381": 48}
# BLS12 parameter z and the power of the oracle's beta whose endomorphism sigma'(x, y) = (beta' x, y) has the eigenvalue
# z^2 - 1 on G1 (BLS12-381: the GLV lambda is z^2 - 1; BLS12-377: lambda is the other root, lambda^2 = z^2 - 1 mod q)
BLS_Z = {"bls12-377": 0x8508C00000000001, "bls12-381": -0xD201000000010000}
SIGMA_BETA_POWER = {"bls12-377": 2, "bls12-381": 1}
# primes dividing the cofactor h
COFACTOR_PRIMES = {"bls12-377": (2, 3, 7, 13, 499), "bls12-381": (3, 11, 10177, 859267, 52437899), "ed-on-bls12-377": (2,), "pallas": ()}


def on_curve(label, P):
    prm = ORACLE_PARAMS[label]
    x, y = P
    p = prm.p
    if prm.kind == "weierstrass":
        return (y * y - x * x * x - prm.b) % p == 0
    return (-x * x + y * y - 1 - prm.d * x * x * y * y) % p == 0


def scale_any(label, s, P):
    """[s] P for any integer s >= 0 (OracleCurve.scale reduces s mod q, which is wrong outside the subgroup)"""
    O = OracleCurve(label)
    if O.kind == "weierstrass":
        return O.P.to_affine(O.P.scale(s, O.P.from_affine(P)))
    return O.T.to_affine(O.T.scale(s, O.T.from_affine(P)))


def is_in_subgroup(label, P):
    """The oracle's definition: [q] P == O (AffineCurve.is_in_subgroup / TwistedEdwardsCurve.is_in_subgroup)"""
    O = OracleCurve(label)
    if O.kind == "weierstrass":
        return O.A.is_in_subgroup(P)
    return O.T.is_in_subgroup(O.T.from_affine(P))


def sigma(label, P):
    prm = ORACLE_PARAMS[label]
    return (pow(prm.beta, SIGMA_BETA_POWER[label], prm.p) * P[0] % prm.p, P[1])


def fast_in_subgroup(label, P):
    """The device's test for a point on the curve: Pallas h = 1; BLS12 sigma'(P) == [z^2 - 1] P; ed-on-BLS12-377 [q] P == O"""
    if label == "pallas":
        return True
    if label in BLS_Z:
        z = BLS_Z[label]
        return sigma(label, P) == scale_any(label, z * z - 1, P)
    return is_in_subgroup(label, P)


def expected_status(label, P):
    """the status byte mgb_set_points_checked reports for P (None = flagged as zero)"""
    if P is None:
        return 0
    p = ORACLE_PARAMS[label].p
    if P[0] >= p or P[1] >= p:
        return NONCANONICAL
    if not on_curve(label, P):
        return OFF_CURVE
    return 0 if fast_in_subgroup(label, P) else NOT_IN_SUBGROUP


def random_curve_point(label, rng):
    """a uniformly placed point of E(Fp): point_from_x without clearing the cofactor"""
    O = OracleCurve(label)
    prm = O.prm
    p = prm.p
    while True:
        x = rng.randrange(p)
        if O.kind == "weierstrass":
            y = O.A.Fp.sqrt((x * x * x + prm.b) % p)
        else:
            den = (1 - prm.d * x * x) % p
            y = O.T.Fp.sqrt((1 + x * x) * pow(den, -1, p) % p) if den else None
        if y is not None:
            return (x, y if rng.random() < 0.5 else (-y) % p)


def small_order_points(label, rng):
    """a point of every prime order l dividing the cofactor h; for ed-on-BLS12-377 every point of order 2 or 4 the affine
    format can hold: (0, -1) and (+-sqrt(-1), 0).  [h q / l] R alone is not enough: where the l-part of E(Fp) is not
    cyclic (BLS12-377 holds all of E[2], so its 2^92 part is), it is O for every R.  So T = [h q / l^v] R, l^v || h,
    lands in the l-part, and T is multiplied by l until the next multiple would be O."""
    prm = ORACLE_PARAMS[label]
    if label == "ed-on-bls12-377":
        p = prm.p
        i = OracleCurve(label).T.Fp.sqrt(p - 1)
        return [(0, p - 1), (i, 0), ((-i) % p, 0)]
    out = []
    for ell in COFACTOR_PRIMES[label]:
        v, h = 0, prm.h
        while h % ell == 0:
            h //= ell
            v += 1
        T = None
        while T is None:
            T = scale_any(label, prm.h * prm.q // ell**v, random_curve_point(label, rng))
        while (U := scale_any(label, ell, T)) is not None:
            T = U
        out.append(T)
    return out


def add(label, P, Q):
    O = OracleCurve(label)
    if O.kind == "weierstrass":
        return O.A.add(P, Q)
    return O.T.to_affine(O.T.add(O.T.from_affine(P), O.T.from_affine(Q)))


def bad_points(label, good, seed=1):
    """Invalid points of every kind for `label`, derived from the valid points `good` (affine, in the subgroup):
    non-canonical encodings x + p and y + p where they fit, off-curve points (y + 1), points on the curve outside the
    subgroup (random points of E(Fp), points of every small prime order, and mixes P1 + T).  Returns a list of points."""
    rng = random.Random(seed)
    prm = ORACLE_PARAMS[label]
    p, top = prm.p, 1 << (8 * COORD_BYTES[label])
    g = [P for P in good if P is not None]
    out = []
    for P in g[:2]:
        if P[0] + p < top:
            out.append((P[0] + p, P[1]))
        if P[1] + p < top:
            out.append((P[0], P[1] + p))
        out.append((P[0], (P[1] + 1) % p))
    if label != "pallas":
        out += [random_curve_point(label, rng) for _ in range(3)]
        small = small_order_points(label, rng)
        out += small
        out += [add(label, g[k % len(g)], T) for k, T in enumerate(small)]
    return out
