"""CPU: the facts the membership test of mgb_set_points_checked rests on (DESIGN.md "Checked point ingestion"), and the
Python mirror of that test (tests/point_checks.py) against the oracle's definition [q] P == O on crafted inputs."""
import importlib.util
import os
import random
from math import gcd

import pytest

from tests import point_checks as pc
from tests.helpers import ORACLE_PARAMS, ROOT, OracleCurve


def gen_constants():
    """montgomery_b200/gen_constants.py, the generator of the device constants (a script, not a module of the package)"""
    spec = importlib.util.spec_from_file_location("gen_constants", os.path.join(ROOT, "montgomery_b200", "gen_constants.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    return gen


def is_prime(n):
    return n > 1 and all(n % d for d in range(2, int(n**0.5) + 1))


@pytest.mark.parametrize("label", ["bls12-377", "bls12-381"])
def test_bls12_soundness_facts(label):
    prm = ORACLE_PARAMS[label]
    z = pc.BLS_Z[label]
    # E(Fp) = G1 + C, |C| = h: the decomposition needs gcd(h, q) = 1
    assert gcd(prm.h, prm.q) == 1
    # every prime dividing h divides z^2 - 1, so [z^2 - 1] kills every point of prime order in C
    primes = pc.COFACTOR_PRIMES[label]
    rest = prm.h
    for ell in primes:
        assert is_prime(ell) and rest % ell == 0
        while rest % ell == 0:
            rest //= ell
    assert rest == 1                                        # no other prime divides h
    assert all((z * z - 1) % ell == 0 for ell in primes)
    # sigma' has the eigenvalue z^2 - 1 on G1 (the generator), the other cube root of unity does not
    O = OracleCurve(label)
    G = O.G
    assert pc.sigma(label, G) == pc.scale_any(label, z * z - 1, G)
    other = (pow(prm.beta, 3 - pc.SIGMA_BETA_POWER[label], prm.p) * G[0] % prm.p, G[1])
    assert other != pc.scale_any(label, z * z - 1, G)
    # the device's constants (montgomery_b200/gen_constants.py) are the same z^2 and beta power
    gen = gen_constants()
    src = gen.subgroup_consts(abs(z), pc.SIGMA_BETA_POWER[label] == 2)
    assert "0x%016xull" % ((z * z) >> 64) in src and "0x%016xull" % ((z * z) & (2**64 - 1)) in src


def test_ed_naf_of_q():
    """the signed-digit chain of the twisted-Edwards test is q itself"""
    gen = gen_constants()
    q = ORACLE_PARAMS["ed-on-bls12-377"].q
    pos, neg = gen.naf_masks(q)
    assert pos - neg == q and pos & neg == 0 and (pos | neg) & ((pos | neg) >> 1) == 0


@pytest.mark.parametrize("label", ["bls12-377", "pallas", "ed-on-bls12-377", "bls12-381"])
def test_fast_check_agrees_with_oracle(label):
    """status of every crafted point: the fast test equals [q] P == O wherever the point is canonical and on the curve,
    and every kind of bad point gets its bit"""
    O = OracleCurve(label)
    good = [O.scale(5 + 7 * i, O.G) for i in range(4)]
    bad = pc.bad_points(label, good)
    kinds = set()
    for P in good + bad:
        st = pc.expected_status(label, P)
        kinds.add(st)
        p = O.prm.p
        if P[0] < p and P[1] < p and pc.on_curve(label, P):
            assert (st == 0) == pc.is_in_subgroup(label, P), (label, P)
    assert kinds == ({0, 1, 2} if label == "pallas" else {0, 1, 2, 4})
    # each small-order point, alone and added to a subgroup point, is rejected
    if label != "pallas":
        small = pc.small_order_points(label, random.Random(3))
        assert len(small) == len(pc.COFACTOR_PRIMES[label]) or label == "ed-on-bls12-377"
        for T in small:
            assert pc.expected_status(label, T) == pc.NOT_IN_SUBGROUP
            assert pc.expected_status(label, pc.add(label, good[0], T)) == pc.NOT_IN_SUBGROUP
    assert pc.expected_status(label, None) == 0
