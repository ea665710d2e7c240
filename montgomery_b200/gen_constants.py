#!/usr/bin/env python3
"""Generates csrc/constants_gen.cuh: per-field Montgomery constants and per-curve constants
(32-bit limbs, little-endian limb order) for the CUDA engine.

Stand-alone (plain Python ints, no imports from oracle/).  Parameter sources in the reference:
  src/concrete/bls12-377.params.ts:11-46, ed-on-bls12-377.params.ts:5-31, pasta.params.ts:10-46;
the GLV lattice follows src/glv/glv.ts:21-50 (egcdStopEarly) with the rounding constants of
src/wasm/glv.ts:45-50, re-derived for 32-bit limbs.

Run:  python montgomery_b200/gen_constants.py > montgomery_b200/csrc/constants_gen.cuh
"""
import sys


def limbs(x, n):
    assert 0 <= x < (1 << (32 * n)), (hex(x), n)
    return [(x >> (32 * i)) & 0xFFFFFFFF for i in range(n)]


def carr(name, x, n):
    body = ",".join("0x%08xu" % l for l in limbs(x, n))
    return ("  __host__ __device__ static constexpr uint32_t %s(int i) { constexpr uint32_t t[%d] = {%s}; return t[i]; }\n"
            % (name, n, body))


def field_struct(name, p, n, fid):
    R = 1 << (32 * n)
    assert 2 * p < R
    out = "struct %s {\n" % name
    out += "  static constexpr int ID = %d;   // index into the run-time table of Montgomery factors\n" % fid
    out += "  static constexpr int N = %d;\n" % n
    out += "  static constexpr int BITS = %d;\n" % p.bit_length()
    out += "  static constexpr uint32_t M0 = 0x%08xu;  // -p^-1 mod 2^32\n" % ((-pow(p, -1, 1 << 32)) % (1 << 32))
    out += carr("mod", p, n)
    out += carr("one", R % p, n)          # Montgomery form of 1
    out += carr("r2", R * R % p, n)       # to-Montgomery multiplier
    out += carr("r3", R * R * R % p, n)   # fixes up the plain binary inverse: mont(x, r3) = x*R^2
    out += carr("pm2", p - 2, n)          # Fermat exponent
    n30 = (p.bit_length() + 1 + 29) // 30 + (1 if (p.bit_length() + 1) % 30 == 0 else 0)
    n30 = max(n30, (32 * n + 29) // 30)   # must also hold any packed 32n-bit value
    out += "  static constexpr uint32_t MINV30 = 0x%08xu;  // p^-1 mod 2^30 (division-step inverse)\n" % pow(p, -1, 1 << 30)
    body = ",".join("0x%08x" % ((p >> (30 * i)) & 0x3FFFFFFF) for i in range(n30))
    out += "  static constexpr int N30 = %d;  // signed 30-bit limbs of the divsteps inverse\n" % n30
    out += ("  __host__ __device__ static constexpr int32_t mod30(int i) { constexpr int32_t t[%d] = {%s}; return t[i]; }\n" % (n30, body))
    out += "};\n\n"
    return out


def subgroup_consts(z_abs, beta_squared):
    """Membership test of G1 in mgb_set_points_checked: sigma'(P) + P == [z^2] P, sigma'(x, y) = (beta' x, y) with beta'
    the cube root of unity whose eigenvalue on G1 is z^2 - 1 (DESIGN.md, checked point ingestion).  z^2 is one binary
    chain of 127 or 128 bits.  Z2 = 0: the cofactor is 1 and every point on the curve is in the group."""
    z2 = z_abs * z_abs
    if z_abs:
        out = "  // z^2 of the BLS12 parameter (|z| = 0x%x) in two 64-bit halves, Z2_TOP = its top bit\n" % z_abs
    else:
        out = "  // cofactor 1: no subgroup chain\n"
    out += "  static constexpr uint64_t Z2_HI = 0x%016xull, Z2_LO = 0x%016xull;\n" % (z2 >> 64, z2 & (2**64 - 1))
    out += "  static constexpr int Z2_TOP = %d;\n" % (z2.bit_length() - 1)
    out += "  static constexpr bool SIGMA_BETA_SQUARED = %s;  // sigma'(x, y) = (beta^2 x, y) instead of (beta x, y)\n" % ("true" if beta_squared else "false")
    return out


def naf_masks(k):
    """non-adjacent form of k as two bit masks (positions of the +1 and of the -1 digits)"""
    pos = neg = 0
    i = 0
    while k:
        if k & 1:
            d = 2 - (k & 3)
            k -= d
            if d > 0:
                pos |= 1 << i
            else:
                neg |= 1 << i
        k >>= 1
        i += 1
    assert pos - neg > 0 and pos & neg == 0 and pos & (pos >> 1) == 0
    return pos, neg


def egcd_stop_early(l, p):
    r0, r1, t0, t1 = p, l, 0, 1
    while r1 * r1 > p:
        quo = r0 // r1
        r0, r1 = r1, r0 - quo * r1
        t0, t1 = t1, t0 - quo * t1
    quo = r0 // r1
    r2, t2 = r0 - quo * r1, t0 - quo * t1
    v00, v10 = r1, -t1
    if max(r0, abs(t0)) <= max(r2, abs(t2)):
        v01, v11 = r0, -t0
    else:
        v01, v11 = r2, -t2
    return v00, v01, v10, v11


def glv_struct(name, q, lam):
    """x_i = round(g_i * s / 2^SH) with g_i = round(2^SH * (+-v) / det); s0 = s - x0*v00 - x1*v01 ..."""
    v00, v01, v10, v11 = egcd_stop_early(lam, q)
    assert (v00 + lam * v10) % q == 0 and (v01 + lam * v11) % q == 0
    det = v00 * v11 - v10 * v01
    assert abs(det) == q
    # solve (s, 0) = x0*(v00, v10) + x1*(v01, v11) over the rationals:
    #   x0 = s*v11/det, x1 = -s*v10/det;  k0 = s - round(x0)*v00 - round(x1)*v01, k1 = -round(x0)*v10 - round(x1)*v11
    SH = 384  # s < 2^256, g < 2^(384-126) -> product < 2^(256+258); we keep bits [384, ...)
    num0, num1 = v11, -v10
    if det < 0:
        num0, num1, det = -num0, -num1, -det
    g0 = (abs(num0) << SH) // det
    g1 = (abs(num1) << SH) // det
    sg0 = 1 if num0 >= 0 else -1
    sg1 = 1 if num1 >= 0 else -1
    out = "struct %s {\n" % name
    out += "  // k0 = s - x0*v00 - x1*v01,  k1 = -x0*v10 - x1*v11,  x_i = sgn_i * ((g_i * s) >> 384 rounded)\n"
    out += "  static constexpr int GN = %d;  // limbs of g_i\n" % 9
    out += carr("g0", g0, 9)
    out += carr("g1", g1, 9)
    out += "  static constexpr int SG0 = %d, SG1 = %d;\n" % (sg0, sg1)
    for nm, v in (("v00", v00), ("v01", v01), ("v10", v10), ("v11", v11)):
        out += carr(nm, abs(v), 4)
        out += "  static constexpr int S_%s = %d;\n" % (nm.upper(), 1 if v >= 0 else -1)
    out += carr("q", q, 8)
    out += "};\n\n"
    return out, (v00, v01, v10, v11, g0, g1, sg0, sg1)


def main():
    p377 = 0x01AE3A4617C510EAC63B05C06CA1493B1A22D9F300F5138F1EF3622FBA094800170B5D44300000008508C00000000001
    q377 = 0x12AB655E9A2CA55660B44D1E5C37B00159AA76FED00000010A11800000000001
    lam377 = 0x12AB655E9A2CA55660B44D1E5C37B00114885F32400000000000000000000000
    beta377 = 0x1AE3A4617C510EABC8756BA8F8C524EB8882A75CC9BC8E359064EE822FB5BFFD1E945779FFFFFFFFFFFFFFFFFFFFFFF
    g377 = (0x008848DEFE740A67C8FC6225BF87FF5485951E2CAA9D41BB188282C8BD37CB5CD5481512FFCD394EEAB9B16EB21BE9EF,
            0x01914A69C5102EFF1F674F5D30AFEEC4BD7FB348CA3E52D96D182AD44FB82305C2FE3D3634A9591AFD82DE55559C8EA6)
    ppal = 0x40000000000000000000000000000000224698FC094CF91B992D30ED00000001
    qpal = 0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001
    lampal = pow(5, (qpal - 1) // 3, qpal)
    b2 = pow(5, (ppal - 1) // 3, ppal)
    betapal = b2 * b2 % ppal
    gpal = (1, 0x1B74B5A30A12937C53DFA9F06378EE548F655BD4333D477119CF7A23CAED2ABB)
    qed = 0x4AAD957A68B2955982D1347970DEC005293A3AFC43C8AFEB95AEE9AC33FD9FF
    ged = (0x9F1B5A5BAF6ACF06FED91C9AE9EBFA06068DD2835790980894E2328F3EBCA05,
           0x9A20DF36571AC3CD906B256080BA8454453C177AAF3131BB50A67BF1A806781)

    out = "// GENERATED by montgomery_b200/gen_constants.py -- do not edit.\n#pragma once\n#include <cstdint>\nnamespace mgb {\n\n"
    p381 = 0x1A0111EA397FE69A4B1BA7B6434BACD764774B84F38512BF6730D2A0F6B0F6241EABFFFEB153FFFFB9FEFFFFFFFFAAAB
    q381 = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
    lam381 = 0xD201000000010000 ** 2 - 1                                  # src/concrete/bls12-381.params.ts:24
    beta381 = 0x1A0111EA397FE699EC02408663D4DE85AA0D857D89759AD4897D29650FB85F9B409427EB4F49FFFD8BFD00000000AAAC
    g381 = (0x17F1D3A73197D7942695638C4FA9AC0FC3688C4F9774B905A14E3A3F171BAC586C55E83FF97A1AEFFB3AF00ADB22C6BB,
            0x08B3F481E3AAA0F1A09E30ED741D8AE4FCF5E095D5D00AF600DB18CB2C04B3EDD03CC744A2888AE40CAA232946C5E7E1)
    out += field_struct("Fp377", p377, 12, 0)
    out += field_struct("Fr377", q377, 8, 1)     # scalar field of BLS12-377 = base field of ed-on-BLS12-377
    out += field_struct("FpPallas", ppal, 8, 2)
    out += field_struct("Fp381", p381, 12, 3)
    out += "// -p^-1 mod 2^32 per field ID (loaded at run time, see field.cuh)\n"
    out += "#define MGB_MINV_TABLE {%s}\n\n" % ", ".join("0x%08xu" % ((-pow(pp, -1, 1 << 32)) % (1 << 32)) for pp in (p377, q377, ppal, p381))

    def mont(x, p, n):
        return x * (1 << (32 * n)) % p

    # curve constants in Montgomery form
    out += "struct Bls12377Consts {\n"
    out += carr("beta", mont(beta377, p377, 12), 12)
    out += carr("b3", mont(3 * 1, p377, 12), 12)
    out += carr("gx", mont(g377[0], p377, 12), 12)
    out += carr("gy", mont(g377[1], p377, 12), 12)
    out += "  static constexpr int SCALAR_BITS = 253;\n"
    out += subgroup_consts(0x8508C00000000001, beta_squared=True)      # beta^2: eigenvalue z^2 - 1 (the GLV lambda is the other root)
    out += "};\n\n"
    out += "struct PallasConsts {\n"
    out += carr("beta", mont(betapal, ppal, 8), 8)
    out += carr("b3", mont(3 * 5, ppal, 8), 8)
    out += carr("gx", mont(gpal[0], ppal, 8), 8)
    out += carr("gy", mont(gpal[1], ppal, 8), 8)
    out += "  static constexpr int SCALAR_BITS = 255;\n"
    out += subgroup_consts(0, beta_squared=False)                       # cofactor 1
    out += "};\n\n"
    out += "struct Bls12381Consts {\n"
    out += carr("beta", mont(beta381, p381, 12), 12)
    out += carr("b3", mont(3 * 4, p381, 12), 12)
    out += carr("gx", mont(g381[0], p381, 12), 12)
    out += carr("gy", mont(g381[1], p381, 12), 12)
    out += "  static constexpr int SCALAR_BITS = 255;\n"
    out += subgroup_consts(0xD201000000010000, beta_squared=False)     # beta: eigenvalue z^2 - 1 = the GLV lambda
    out += "};\n\n"
    out += "struct Ed377Consts {\n"
    out += carr("k", mont(2 * 3021, q377, 8), 8)     # k = 2d
    out += carr("gx", mont(ged[0], q377, 8), 8)
    out += carr("gy", mont(ged[1], q377, 8), 8)
    out += carr("q", qed, 8)
    pos, neg = naf_masks(qed)
    out += "  // [q]P == O test of mgb_set_points_checked: q in non-adjacent form, digit i = +1 / -1 where bit i of naf_pos / naf_neg is set\n"
    out += carr("naf_pos", pos, 8)
    out += carr("naf_neg", neg, 8)
    out += "  static constexpr int NAF_TOP = %d;  // the top digit, +1\n" % (pos.bit_length() - 1)
    out += "  static constexpr int SCALAR_BITS = 251;\n};\n\n"
    s, info377 = glv_struct("Glv377", q377, lam377)
    out += s
    s, infopal = glv_struct("GlvPallas", qpal, lampal)
    out += s
    s, info381 = glv_struct("Glv381", q381, lam381)
    out += s
    out += "}  // namespace mgb\n"
    sys.stdout.write(out)
    # self-check of the decomposition bound (stderr)
    import random
    rnd = random.Random(1)
    for (q, lam, info, nm) in ((q377, lam377, info377, "377"), (qpal, lampal, infopal, "pallas"), (q381, lam381, info381, "381")):
        v00, v01, v10, v11, g0, g1, sg0, sg1 = info
        mx = 0
        for _ in range(20000):
            s_ = rnd.randrange(q) if _ > 3 else (q - 1, 0, 1, (1 << 256) - 1)[_]
            x0 = sg0 * (((g0 * s_) >> 383) + 1 >> 1)
            x1 = sg1 * (((g1 * s_) >> 383) + 1 >> 1)
            k0 = s_ - x0 * v00 - x1 * v01
            k1 = -x0 * v10 - x1 * v11
            assert (k0 + k1 * lam - s_) % q == 0
            mx = max(mx, abs(k0).bit_length(), abs(k1).bit_length())
        print("glv", nm, "max half-scalar bits", mx, file=sys.stderr)


if __name__ == "__main__":
    main()
