// MSM pipeline kernels (sm_100a).  One template per curve family policy; see DESIGN.md for the
// data layout and the per-kernel rooflines.
//
// Pipeline (reference phases in brackets, src/msm-batched-affine.ts):
//   k_digits      GLV split + signed c-bit digits + bucket histogram         [:350-421, :175-205]
//   k_scan_*      exclusive scan of the histogram -> bucket offsets, exact size of every tree round [:423-447]
//   k_scatter     counting-sort scatter of point references (not points)     [:456-502]
//   k_batch_add   log-depth in-place tree per bucket: batched-affine additions, one lane-parallel inversion per
//                 warp tile of 32 * E additions (k_pair_add on the curves that add without inversion)
//                 [:243-283, src/curve-affine.ts:376-522, src/wasm/inverse.ts:220-271]
//   k_bucket_finish, k_group_partial, k_tree_*, k_digit_sums, k_window_assemble
//                 bucket reduction with the weight split into digits          [:504-583]
//   k_final       Horner over windows + affine normalisation, one warp       [:311-334, curve-projective.ts:335-349]
//   k_normalize   sum of the gathered partial accumulators (multi-GPU) + normalisation
#pragma once
#ifdef MGB_HOST_EMU
// host emulation (tests only): tests/host_emu/cuda_emu.h, included first, stands in for the CUDA built-ins used below
#ifndef MGB_CUDA_EMU
#error "MGB_HOST_EMU: include tests/host_emu/cuda_emu.h before engine.cuh"
#endif
#else
#include <cuda_runtime.h>
#endif
#include "ec.cuh"
#include "coop.cuh"
#include "onewarp.cuh"

namespace mgb {

// ---------------------------------------------------------------- vector loads / stores
template <class P>
MGB_DEV Fe<P> ld_fe(const uint32_t* p) {
  Fe<P> r;
  const uint4* q = reinterpret_cast<const uint4*>(p);
  _Pragma("unroll") for (int i = 0; i < P::N / 4; i++) {
    uint4 t = q[i];
    r.v[4 * i] = t.x; r.v[4 * i + 1] = t.y; r.v[4 * i + 2] = t.z; r.v[4 * i + 3] = t.w;
  }
  return r;
}
template <class P>
MGB_DEV Fe<P> ldg_fe(const uint32_t* p) {  // read-only path (point table)
  Fe<P> r;
  const uint4* q = reinterpret_cast<const uint4*>(p);
  _Pragma("unroll") for (int i = 0; i < P::N / 4; i++) {
    uint4 t = __ldg(q + i);
    r.v[4 * i] = t.x; r.v[4 * i + 1] = t.y; r.v[4 * i + 2] = t.z; r.v[4 * i + 3] = t.w;
  }
  return r;
}
template <class P>
MGB_DEV void st_fe(uint32_t* p, const Fe<P>& a) {
  uint4* q = reinterpret_cast<uint4*>(p);
  _Pragma("unroll") for (int i = 0; i < P::N / 4; i++) q[i] = make_uint4(a.v[4 * i], a.v[4 * i + 1], a.v[4 * i + 2], a.v[4 * i + 3]);
}

// reference bits of a sorted entry: point index | endo << 30 | negate << 31
static constexpr uint32_t REF_NEG = 0x80000000u;
static constexpr uint32_t REF_ENDO = 0x40000000u;
static constexpr uint32_t REF_IDX = 0x3fffffffu;
static constexpr uint32_t NO_BUCKET = 0xffffffffu;

// status bits of a point checked on ingestion (MGB_PT_* of include/montgomery_b200.h)
static constexpr uint32_t PT_NONCANONICAL = 1;
static constexpr uint32_t PT_OFF_CURVE = 2;
static constexpr uint32_t PT_NOT_IN_SUBGROUP = 4;

// ---------------------------------------------------------------- curve policies
template <class FP, class CC, class GL, int MAGB>
struct WeierstrassPolicy {
  typedef FP P;
  typedef Field<FP> F;
  typedef Weierstrass<FP> G;
  typedef typename G::acc acc;
  typedef typename G::affine vpoint;   // materialised bucket element
  typedef GL Glv;
  typedef OneWarpWeierstrass<FP> OneWarp;
  typedef QuadWeierstrass<FP> Quad;
  static constexpr int N = FP::N;
  static constexpr bool USE_GLV = true;
  static constexpr bool BATCH_AFFINE = true;
  static constexpr int HALVES = 2;
  static constexpr int MAG_LIMBS = 4;        // |k0|, |k1| < 2^128
  static constexpr int MAG_BITS = MAGB;      // bound on |k0|, |k1| in bits, plus one for the final carry
  static constexpr int ENTRY_LIMBS = 3 * N;  // x | y | beta*x
  static constexpr int V_LIMBS = 2 * N;
  static constexpr int ACC_LIMBS = 4 * N;
  static constexpr int COORD_BYTES = 4 * N;

  // table entry -> the point a sorted slot stands for (endomorphism / negation applied)
  MGB_DEV static vpoint load_entry(const uint32_t* table, uint32_t idx, bool endo, bool negate) {
    const uint32_t* e = table + (size_t)idx * ENTRY_LIMBS;
    vpoint r;
    r.x = ldg_fe<FP>(e + (endo ? 2 * N : 0));
    r.y = ldg_fe<FP>(e + N);
    if (negate) r.y = F::neg(r.y);
    return r;
  }
  MGB_DEV static vpoint load_v(const uint32_t* V, uint32_t slot) {
    const uint32_t* e = V + (size_t)slot * V_LIMBS;
    vpoint r; r.x = ld_fe<FP>(e); r.y = ld_fe<FP>(e + N); return r;
  }
  // x coordinate only (carries the infinity flag): all the first pass of a batched addition needs
  MGB_DEV static Fe<FP> load_v_x(const uint32_t* V, uint32_t slot) { return ld_fe<FP>(V + (size_t)slot * V_LIMBS); }
  MGB_DEV static void store_v(uint32_t* V, uint32_t slot, const vpoint& p) {
    uint32_t* e = V + (size_t)slot * V_LIMBS;
    st_fe<FP>(e, p.x); st_fe<FP>(e + N, p.y);
  }
  MGB_DEV static acc acc_zero() { return G::acc_zero(); }
  MGB_DEV static acc add(const acc& a, const acc& b) { return G::add(a, b); }
  MGB_DEV static acc dbl(const acc& a) { return G::dbl(a); }
  MGB_DEV static acc add_v(const acc& a, const vpoint& p) { return G::madd(a, p); }
  MGB_DEV static acc add_vv(const vpoint& p, const vpoint& q) { return G::mmadd(p, q); }   // two stored (affine) elements: 6 products, not 10
  // (add_refs -- the sum of two table entries -- is only needed by the paths that add without inversion: see the other policies)
  MGB_DEV static acc ld_acc(const uint32_t* p) { acc r; r.X = ld_fe<FP>(p); r.Y = ld_fe<FP>(p + N); r.ZZ = ld_fe<FP>(p + 2 * N); r.ZZZ = ld_fe<FP>(p + 3 * N); return r; }
  MGB_DEV static void st_acc(uint32_t* p, const acc& a) { st_fe<FP>(p, a.X); st_fe<FP>(p + N, a.Y); st_fe<FP>(p + 2 * N, a.ZZ); st_fe<FP>(p + 3 * N, a.ZZZ); }
  MGB_DEV static acc generator() {
    acc g; _Pragma("unroll") for (int i = 0; i < N; i++) { g.X.v[i] = CC::gx(i); g.Y.v[i] = CC::gy(i); }
    g.ZZ = F::one(); g.ZZZ = F::one(); return g;
  }
  // x||y canonical bytes -> table entry
  MGB_DEV static void make_entry(uint32_t* e, const Fe<FP>& x_plain, const Fe<FP>& y_plain, bool inf) {
    Fe<FP> x = F::to_mont(x_plain), y = F::to_mont(y_plain);
    Fe<FP> beta; _Pragma("unroll") for (int i = 0; i < N; i++) beta.v[i] = CC::beta(i);
    Fe<FP> bx = F::mul(x, beta);
    if (inf) { x = F::zero(); y = F::zero(); bx = F::zero(); x.v[N - 1] = G::INF_BIT; bx.v[N - 1] = G::INF_BIT; }
    st_fe<FP>(e, x); st_fe<FP>(e + N, y); st_fe<FP>(e + 2 * N, bx);
  }
  MGB_DEV static void make_entry_from_acc(uint32_t* e, const acc& a) {
    vpoint p = G::to_affine(a);
    bool inf = G::is_inf(p);
    make_entry(e, F::from_mont(p.x), F::from_mont(p.y), inf);
  }
  MGB_DEV static void entry_to_plain(const uint32_t* e, Fe<FP>& x, Fe<FP>& y, bool& inf) {
    Fe<FP> xm = ld_fe<FP>(e);
    inf = (xm.v[N - 1] & G::INF_BIT) != 0;
    if (inf) { x = F::zero(); y = F::zero(); return; }
    x = F::from_mont(xm); y = F::from_mont(ld_fe<FP>(e + N));
  }
  // final accumulator -> canonical plain coordinates
  MGB_DEV static void acc_to_plain(const acc& a, Fe<FP>& x, Fe<FP>& y, bool& inf) {
    vpoint p = G::to_affine(a);
    inf = G::is_inf(p);
    if (inf) { x = F::zero(); y = F::zero(); return; }
    x = F::from_mont(p.x); y = F::from_mont(p.y);
  }
  // Sum of `count` accumulators (the multi-GPU combine) by ONE warp; every lane returns the sum.  Quad q adds up the
  // partials q, q + 8, ..., then three levels of 4-lane additions (coop.cuh) combine the eight quads: 3 + count / 8
  // addition latencies of ~5 us instead of count - 1 serial 14-product additions (7 x 17 us at eight GPUs).
  MGB_DEV static acc sum_partials_warp(const uint32_t* accs, int count, int stride = ACC_LIMBS) {
    const int lane = threadIdx.x & 31, k = lane & 3, q = lane >> 2;
    Fe<FP> v = Quad::zero_coord(k);
    for (int base = 0; base < count; base += 8) {          // warp-uniform trip count
      Fe<FP> o = Quad::zero_coord(k);
      if (base + q < count) o = ld_fe<FP>(accs + (size_t)(base + q) * stride + k * N);
      v = Quad::add(v, o);
    }
    _Pragma("unroll 1") for (int dl = 4; dl >= 1; dl >>= 1) {
      const Fe<FP> o = Quad::shfl(v, (lane + 4 * dl) & 31);
      v = Quad::add(v, q < dl ? o : Quad::zero_coord(k));
    }
    acc r;
    r.X = Quad::shfl(v, 0); r.Y = Quad::shfl(v, 1); r.ZZ = Quad::shfl(v, 2); r.ZZZ = Quad::shfl(v, 3);
    return r;
  }
  // the same called by ALL 32 lanes of a warp with the same accumulator: the one inversion runs on the lane-parallel
  // division-step routine (warp.cuh, 20.6 us instead of 35.3 us on one lane); every lane returns the result
  MGB_DEV static void acc_to_plain_warp(const acc& a, Fe<FP>& x, Fe<FP>& y, bool& inf) {
    inf = G::acc_is_zero(a);                                  // warp-uniform
    if (inf) { x = F::zero(); y = F::zero(); return; }
    const Fe<FP> t = WarpField<FP>::inv_call(a.ZZZ);          // x = X / ZZ, y = Y / ZZZ: 1 / ZZ = t^2 ZZ^2 (ZZ^3 = ZZZ^2)
    const Fe<FP> izz = F::mul(F::sqr(t), F::sqr(a.ZZ));
    x = F::from_mont(F::mul(a.X, izz)); y = F::from_mont(F::mul(a.Y, t));
  }
  // Status bits (PT_*) of a table entry made from canonical coordinates: the curve equation 3(y^2 - x^3) == 3b, then
  // membership of the prime-order subgroup.  BLS12: sigma'(P) == [z^2 - 1] P (sigma' has the eigenvalue z^2 - 1 on G1;
  // DESIGN.md "Checked point ingestion" proves the test exact).  [z^2] P is one fixed double-and-add chain over the
  // 127/128-bit z^2 with mixed additions of the affine P, which is re-read from the table: one XYZZ accumulator is all
  // that lives across the chain (two chains over |z| would keep a second one and spill at 3 blocks per SM).  The chain
  // is a compile-time constant, so every lane of a warp runs the same instructions; the complete formulas branch only
  // on adversarial points.
  MGB_DEV static uint32_t check_entry(const uint32_t* e) {
    vpoint p = load_entry(e, 0, false, false);
    if (G::is_inf(p)) return 0;
    Fe<FP> b3; _Pragma("unroll") for (int i = 0; i < N; i++) b3.v[i] = CC::b3(i);
    const Fe<FP> t = F::sub(F::sqr(p.y), F::mul(F::sqr(p.x), p.x));
    if (!F::eq(F::add(F::dbl(t), t), b3)) return PT_OFF_CURVE;
    if (CC::Z2_TOP < 0) return 0;                                   // cofactor 1
    acc a = G::from_affine(p);                                      // the top bit of z^2
    _Pragma("unroll") for (int half = 1; half >= 0; half--) {
      const uint64_t word = half ? CC::Z2_HI : CC::Z2_LO;
      _Pragma("unroll 1") for (int bit = (half ? CC::Z2_TOP - 64 : 64) - 1; bit >= 0; bit--) {
        a = G::dbl(a);
        if ((word >> bit) & 1) a = G::madd(a, load_entry(e, 0, false, false));
      }
    }
    a = G::madd(a, load_entry(e, 0, false, true));                  // [z^2 - 1] P
    vpoint s = load_entry(e, 0, true, false);                       // sigma'(P) = (beta x, y) or (beta^2 x, y)
    if (CC::SIGMA_BETA_SQUARED) { Fe<FP> beta; _Pragma("unroll") for (int i = 0; i < N; i++) beta.v[i] = CC::beta(i); s.x = F::mul(s.x, beta); }
    // sigma'(P) (affine, never infinity) == [z^2 - 1] P (XYZZ) without inversion: x ZZ == X and y ZZZ == Y
    const bool same = !G::acc_is_zero(a) && F::eq(F::mul(s.x, a.ZZ), a.X) && F::eq(F::mul(s.y, a.ZZZ), a.Y);
    return same ? 0 : PT_NOT_IN_SUBGROUP;
  }
};

template <class FP, class CC>
struct TwistedEdwardsPolicy {
  typedef FP P;
  typedef Field<FP> F;
  typedef TwistedEdwards<FP, CC> G;
  typedef typename G::acc acc;
  typedef typename G::acc vpoint;
  typedef OneWarpTwistedEdwards<FP, CC> OneWarp;
  static constexpr int N = FP::N;
  static constexpr bool USE_GLV = false;
  static constexpr bool BATCH_AFFINE = false;
  static constexpr int HALVES = 1;
  static constexpr int MAG_LIMBS = 8;
  static constexpr int MAG_BITS = CC::SCALAR_BITS + 1;
  static constexpr int ENTRY_LIMBS = 4 * N;  // x | y | t = x*y | k*t (k = 2d: lets round 0 add two table entries with 7 products)
  static constexpr int V_LIMBS = 4 * N;
  static constexpr int ACC_LIMBS = 4 * N;
  static constexpr int COORD_BYTES = 4 * N;

  // Sum of two TABLE entries (round 0 of the bucket trees): both have Z = 1 and the second one's k*T is stored, so
  // add-2008-hwcd-3 needs A = (y1 - x1)(y2 - x2), B = (y1 + x1)(y2 + x2), C = t1 * (k t2), D = 2 and the four final
  // products: 7 instead of the 9 of the general unified addition.  Negation of an entry: -x, -t, -kt.
  MGB_DEV static vpoint add_refs(const uint32_t* table, uint32_t ra, uint32_t rb) {
    const uint32_t* ea = table + (size_t)(ra & REF_IDX) * ENTRY_LIMBS;
    const uint32_t* eb = table + (size_t)(rb & REF_IDX) * ENTRY_LIMBS;
    Fe<FP> x1 = ldg_fe<FP>(ea), y1 = ldg_fe<FP>(ea + N), t1 = ldg_fe<FP>(ea + 2 * N);
    Fe<FP> x2 = ldg_fe<FP>(eb), y2 = ldg_fe<FP>(eb + N), kt2 = ldg_fe<FP>(eb + 3 * N);
    if (ra & REF_NEG) { x1 = F::neg(x1); t1 = F::neg(t1); }
    if (rb & REF_NEG) { x2 = F::neg(x2); kt2 = F::neg(kt2); }
    const Fe<FP> A = F::mul(F::sub(y1, x1), F::sub(y2, x2));
    const Fe<FP> B = F::mul(F::add(y1, x1), F::add(y2, x2));
    const Fe<FP> Cc = F::mul(t1, kt2);
    const Fe<FP> D = F::dbl(F::one());
    const Fe<FP> E = F::sub(B, A), Ff = F::sub(D, Cc), Gg = F::add(D, Cc), H = F::add(B, A);
    vpoint r;
    r.X = F::mul(E, Ff); r.Y = F::mul(Gg, H); r.T = F::mul(E, H); r.Z = F::mul(Ff, Gg);
    return r;
  }

  // table entry (x, y, t = x*y) -> extended point with Z = 1 (negation: -x, -t)
  MGB_DEV static vpoint load_entry(const uint32_t* table, uint32_t idx, bool /*endo*/, bool negate) {
    const uint32_t* e = table + (size_t)idx * ENTRY_LIMBS;
    vpoint r; r.X = ldg_fe<FP>(e); r.Y = ldg_fe<FP>(e + N); r.Z = F::one(); r.T = ldg_fe<FP>(e + 2 * N);
    if (negate) { r.X = F::neg(r.X); r.T = F::neg(r.T); }
    return r;
  }
  MGB_DEV static vpoint load_v(const uint32_t* V, uint32_t slot) { return ld_acc(V + (size_t)slot * V_LIMBS); }
  MGB_DEV static void store_v(uint32_t* V, uint32_t slot, const vpoint& p) { st_acc(V + (size_t)slot * V_LIMBS, p); }
  MGB_DEV static acc acc_zero() { return G::acc_zero(); }
  MGB_DEV static acc add(const acc& a, const acc& b) { return G::add(a, b); }
  MGB_DEV static acc dbl(const acc& a) { return G::dbl(a); }
  MGB_DEV static acc add_v(const acc& a, const vpoint& p) { return G::add(a, p); }
  MGB_DEV static acc add_vv(const vpoint& p, const vpoint& q) { return G::add(p, q); }
  MGB_DEV static acc ld_acc(const uint32_t* p) { acc r; r.X = ld_fe<FP>(p); r.Y = ld_fe<FP>(p + N); r.Z = ld_fe<FP>(p + 2 * N); r.T = ld_fe<FP>(p + 3 * N); return r; }
  MGB_DEV static void st_acc(uint32_t* p, const acc& a) { st_fe<FP>(p, a.X); st_fe<FP>(p + N, a.Y); st_fe<FP>(p + 2 * N, a.Z); st_fe<FP>(p + 3 * N, a.T); }
  MGB_DEV static acc generator() {
    typename G::affine g; _Pragma("unroll") for (int i = 0; i < N; i++) { g.x.v[i] = CC::gx(i); g.y.v[i] = CC::gy(i); }
    return G::from_affine(g);
  }
  MGB_DEV static void make_entry(uint32_t* e, const Fe<FP>& x_plain, const Fe<FP>& y_plain, bool inf) {
    Fe<FP> x = F::to_mont(x_plain), y = F::to_mont(y_plain);
    if (inf) { x = F::zero(); y = F::one(); }
    const Fe<FP> t = F::mul(x, y);
    st_fe<FP>(e, x); st_fe<FP>(e + N, y); st_fe<FP>(e + 2 * N, t); st_fe<FP>(e + 3 * N, F::mul(t, G::k2d()));
  }
  MGB_DEV static void make_entry_from_acc(uint32_t* e, const acc& a) {
    Fe<FP> x, y; G::to_affine(a, x, y);
    make_entry(e, F::from_mont(x), F::from_mont(y), false);
  }
  MGB_DEV static void entry_to_plain(const uint32_t* e, Fe<FP>& x, Fe<FP>& y, bool& inf) {
    x = F::from_mont(ld_fe<FP>(e)); y = F::from_mont(ld_fe<FP>(e + N));
    Fe<FP> o = F::zero(); o.v[0] = 1;
    inf = F::is_zero(x) && F::eq(y, o);
  }
  MGB_DEV static void acc_to_plain(const acc& a, Fe<FP>& x, Fe<FP>& y, bool& inf) {
    Fe<FP> xm, ym; G::to_affine(a, xm, ym);
    x = F::from_mont(xm); y = F::from_mont(ym);
    Fe<FP> o = F::zero(); o.v[0] = 1;
    inf = F::is_zero(x) && F::eq(y, o);
  }
  // sum of `count` accumulators on every lane (unified additions, 9 products each; no quad form for this curve)
  MGB_DEV static acc sum_partials_warp(const uint32_t* accs, int count, int stride = ACC_LIMBS) {
    acc res = ld_acc(accs);
    for (int i = 1; i < count; i++) res = add(res, ld_acc(accs + (size_t)i * stride));
    return res;
  }
  // called by all 32 lanes of a warp with the same accumulator (lane-parallel inversion, see WeierstrassPolicy)
  MGB_DEV static void acc_to_plain_warp(const acc& a, Fe<FP>& x, Fe<FP>& y, bool& inf) {
    const Fe<FP> zi = WarpField<FP>::inv_call(a.Z);
    x = F::from_mont(F::mul(a.X, zi)); y = F::from_mont(F::mul(a.Y, zi));
    Fe<FP> o = F::zero(); o.v[0] = 1;
    inf = F::is_zero(x) && F::eq(y, o);
  }
  // Status bits (PT_*) of a table entry made from canonical coordinates: -x^2 + y^2 = 1 + d x^2 y^2, i.e.
  // 2(y^2 - x^2 - 1) == k x^2 y^2, then [q]P == O by the fixed signed-digit chain of q (constants_gen.cuh: 250
  // doublings, 87 mixed additions of +-P).  The neutral element (the entry of a point flagged as zero) passes both.
  MGB_DEV static uint32_t check_entry(const uint32_t* e) {
    typename G::affine p; p.x = ld_fe<FP>(e); p.y = ld_fe<FP>(e + N); p.kt = ld_fe<FP>(e + 3 * N);
    const Fe<FP> xx = F::sqr(p.x), yy = F::sqr(p.y);
    if (!F::eq(F::dbl(F::sub(F::sub(yy, xx), F::one())), F::mul(F::mul(xx, yy), G::k2d()))) return PT_OFF_CURVE;
    const typename G::affine np = G::neg(p);
    acc r = G::from_affine(p);                                      // the top digit is +1
    _Pragma("unroll") for (int w = CC::NAF_TOP / 32; w >= 0; w--) {
      const uint32_t pos = CC::naf_pos(w), neg = CC::naf_neg(w);
      _Pragma("unroll 1") for (int bit = (w == CC::NAF_TOP / 32 ? CC::NAF_TOP % 32 : 32) - 1; bit >= 0; bit--) {
        r = G::dbl(r);
        if ((pos >> bit) & 1) r = G::madd(r, p);
        if ((neg >> bit) & 1) r = G::madd(r, np);
      }
    }
    return F::is_zero(r.X) && !F::is_zero(r.Z) && F::eq(r.Y, r.Z) ? 0 : PT_NOT_IN_SUBGROUP;
  }
};

// The reference's `msmProjective` (src/parallel.ts:69-87): msm-basic over projective coordinates on a
// Weierstrass curve -- no GLV, no batched-affine additions.  Same table and accumulator types as the
// main policy, so it runs on the same context; kept as an independent path that the tests compare
// against the batched-affine one, as src/msm.test.ts:73-82 does.
template <class MAIN, int SCALAR_BITS>
struct WeierstrassBasicPolicy : MAIN {
  typedef typename MAIN::P FP;
  typedef typename MAIN::F F;
  typedef typename MAIN::G G;
  typedef typename MAIN::acc acc;
  typedef acc vpoint;
  static constexpr int N = MAIN::N;
  static constexpr bool USE_GLV = false;
  static constexpr bool BATCH_AFFINE = false;
  static constexpr int HALVES = 1;
  static constexpr int MAG_LIMBS = 8;
  static constexpr int MAG_BITS = SCALAR_BITS + 1;
  static constexpr int V_LIMBS = 4 * N;
  MGB_DEV static vpoint load_entry(const uint32_t* table, uint32_t idx, bool, bool negate) {
    return G::from_affine(MAIN::load_entry(table, idx, false, negate));
  }
  MGB_DEV static vpoint load_v(const uint32_t* V, uint32_t slot) { return MAIN::ld_acc(V + (size_t)slot * V_LIMBS); }
  MGB_DEV static void store_v(uint32_t* V, uint32_t slot, const vpoint& p) { MAIN::st_acc(V + (size_t)slot * V_LIMBS, p); }
  MGB_DEV static acc add_v(const acc& a, const vpoint& p) { return G::add(a, p); }
  MGB_DEV static acc add_vv(const vpoint& p, const vpoint& q) { return G::add(p, q); }
  // two table entries are both affine: mmadd (6 products) instead of the general XYZZ addition (14)
  MGB_DEV static vpoint add_refs(const uint32_t* table, uint32_t ra, uint32_t rb) {
    return G::mmadd(MAIN::load_entry(table, ra & REF_IDX, false, (ra & REF_NEG) != 0), MAIN::load_entry(table, rb & REF_IDX, false, (rb & REF_NEG) != 0));
  }
};

typedef WeierstrassPolicy<Fp377, Bls12377Consts, Glv377, 127> CurveBls377;     // |k| < 2^126 (gen_constants.py self-check; reference maxBits = 126)
typedef WeierstrassPolicy<FpPallas, PallasConsts, GlvPallas, 128> CurvePallas;  // |k| < 2^127
typedef TwistedEdwardsPolicy<Fr377, Ed377Consts> CurveEd377;
typedef WeierstrassPolicy<Fp381, Bls12381Consts, Glv381, 128> CurveBls381;      // |k| < 2^127; fourth curve of src/msm.test.ts:31
typedef WeierstrassBasicPolicy<CurveBls377, 253> CurveBls377Basic;
typedef WeierstrassBasicPolicy<CurvePallas, 255> CurvePallasBasic;
typedef WeierstrassBasicPolicy<CurveBls381, 255> CurveBls381Basic;

// ---------------------------------------------------------------- small multi-limb helpers (scalar side)
template <int NA, int NB>
MGB_DEV void mulw(uint32_t* out, const uint32_t* a, const uint32_t* b) {  // out[NA+NB] = a*b
  _Pragma("unroll") for (int i = 0; i < NA + NB; i++) out[i] = 0;
  _Pragma("unroll") for (int i = 0; i < NA; i++) {
    uint64_t carry = 0;
    _Pragma("unroll") for (int j = 0; j < NB; j++) {
      uint64_t t = (uint64_t)a[i] * b[j] + out[i + j] + carry;
      out[i + j] = (uint32_t)t;
      carry = t >> 32;
    }
    out[i + NB] = (uint32_t)carry;
  }
}
template <int NACC, int NT>
MGB_DEV void acc_addsub(uint32_t* acc, const uint32_t* t, bool subtract) {  // acc +-= t (two's complement, NACC limbs)
  uint64_t c = subtract ? 1 : 0;
  _Pragma("unroll") for (int i = 0; i < NACC; i++) {
    uint32_t ti = (i < NT) ? t[i] : 0u;
    if (subtract) ti = ~ti;
    uint64_t s = (uint64_t)acc[i] + ti + c;
    acc[i] = (uint32_t)s;
    c = s >> 32;
  }
}

// s (8 limbs) -> |k0|, |k1| (4 limbs each) and their signs, k0 + k1*lambda = s (mod q).
// Lattice rounding as in the reference (src/wasm/glv.ts:77-80), constants from gen_constants.py.
template <class GL>
MGB_DEV void glv_decompose(const uint32_t* s, uint32_t* k0, uint32_t* k1, bool& neg0, bool& neg1) {
  uint32_t g[9], prod[17], x0[5], x1[5];
  _Pragma("unroll") for (int h = 0; h < 2; h++) {
    _Pragma("unroll") for (int i = 0; i < 9; i++) g[i] = h ? GL::g1(i) : GL::g0(i);
    mulw<9, 8>(prod, g, s);
    // round: add 2^383, keep bits >= 384
    uint64_t c = (uint64_t)prod[11] + 0x80000000u;
    c >>= 32;
    uint32_t* x = h ? x1 : x0;
    _Pragma("unroll") for (int i = 0; i < 5; i++) { uint64_t t = (uint64_t)prod[12 + i] + c; x[i] = (uint32_t)t; c = t >> 32; }
  }
  uint32_t v[4], t[9], a0[10], a1[10];
  _Pragma("unroll") for (int i = 0; i < 10; i++) { a0[i] = (i < 8) ? s[i] : 0u; a1[i] = 0u; }
  // k0 = s - (SG0*S_V00) x0|v00| - (SG1*S_V01) x1|v01|
  _Pragma("unroll") for (int i = 0; i < 4; i++) v[i] = GL::v00(i);
  mulw<5, 4>(t, x0, v); acc_addsub<10, 9>(a0, t, GL::SG0 * GL::S_V00 > 0);
  _Pragma("unroll") for (int i = 0; i < 4; i++) v[i] = GL::v01(i);
  mulw<5, 4>(t, x1, v); acc_addsub<10, 9>(a0, t, GL::SG1 * GL::S_V01 > 0);
  // k1 = - (SG0*S_V10) x0|v10| - (SG1*S_V11) x1|v11|
  _Pragma("unroll") for (int i = 0; i < 4; i++) v[i] = GL::v10(i);
  mulw<5, 4>(t, x0, v); acc_addsub<10, 9>(a1, t, GL::SG0 * GL::S_V10 > 0);
  _Pragma("unroll") for (int i = 0; i < 4; i++) v[i] = GL::v11(i);
  mulw<5, 4>(t, x1, v); acc_addsub<10, 9>(a1, t, GL::SG1 * GL::S_V11 > 0);
  neg0 = (a0[9] >> 31) != 0;
  neg1 = (a1[9] >> 31) != 0;
  if (neg0) { _Pragma("unroll") for (int i = 0; i < 10; i++) a0[i] = ~a0[i]; uint32_t one1[1] = {1}; acc_addsub<10, 1>(a0, one1, false); }
  if (neg1) { _Pragma("unroll") for (int i = 0; i < 10; i++) a1[i] = ~a1[i]; uint32_t one1[1] = {1}; acc_addsub<10, 1>(a1, one1, false); }
  _Pragma("unroll") for (int i = 0; i < 4; i++) { k0[i] = a0[i]; k1[i] = a1[i]; }
}

struct MsmParams {
  uint32_t n;          // number of (scalar, point) pairs
  int c;               // window bits
  int K;               // windows
  uint32_t L;          // buckets per window = 2^(c-1)
  uint32_t nbuckets;   // K*L
  uint32_t nent;       // n * HALVES * K
  int top_sub;         // the top window's digit has few bits: its buckets are split 2^top_sub ways (by point index)
};

// ---------------------------------------------------------------- k_digits
// One thread per scalar.  Entry e = (h*K + w) of scalar i lives at [e*n + i] (coalesced).
template <class CV>
__global__ void __launch_bounds__(256) k_digits(MsmParams pr, uint32_t i_begin, uint32_t i_end, const uint32_t* __restrict__ scalars,
                                                uint32_t* __restrict__ ent_bucket, uint32_t* __restrict__ ent_rank,
                                                uint32_t* __restrict__ counts) {
  // scalars [i_begin, i_end): the host path launches one grid per uploaded chunk (see msm_core)
  uint32_t i = i_begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= i_end) return;
  uint32_t s[8];
  {
    const uint4* q = reinterpret_cast<const uint4*>(scalars + (size_t)i * 8);
    uint4 a = q[0], b = q[1];
    s[0] = a.x; s[1] = a.y; s[2] = a.z; s[3] = a.w; s[4] = b.x; s[5] = b.y; s[6] = b.z; s[7] = b.w;
  }
  constexpr int ML = CV::MAG_LIMBS;
  uint32_t mag[CV::HALVES][ML + 1];
  bool neg[CV::HALVES];
  if constexpr (CV::USE_GLV) {
    glv_decompose<typename CV::Glv>(s, mag[0], mag[1], neg[0], neg[1]);
    mag[0][ML] = 0; mag[1][ML] = 0;
  } else {
    _Pragma("unroll") for (int k = 0; k < ML; k++) mag[0][k] = s[k];
    mag[0][ML] = 0;
    neg[0] = false;
    // no reduction mod q on this path: the windows cover bits [0, MAG_BITS - 1) of the raw scalar, so a larger
    // one would be silently truncated -- flag it instead (msm_core returns MGB_E_INVALID; the reference's
    // scalars are field elements < q by construction, src/scalar-simple.ts)
    {
      constexpr int SB = CV::MAG_BITS - 1;
      uint32_t over = SB < 256 ? (s[SB >> 5] >> (SB & 31)) : 0u;
      _Pragma("unroll") for (int k = (SB >> 5) + 1; k < 8; k++) over |= s[k];
      if (over) atomicOr(&counts[pr.nbuckets], 2u);
    }
  }
  const int c = pr.c;
  const uint32_t L = pr.L, cmask = (1u << c) - 1;
  // digit w of half h -> bucket (NO_BUCKET for a zero digit) and "the digit is negative"
  auto digit = [&](int h, int w, uint32_t& carry, bool& dneg) -> uint32_t {
    const int bit = w * c;
    const int limb = bit >> 5, sh = bit & 31;
    uint32_t lo = 0, hi = 0;
    _Pragma("unroll") for (int k = 0; k <= ML; k++) { if (k == limb) lo = mag[h][k]; if (k == limb + 1) hi = mag[h][k]; }
    const uint32_t slice = (uint32_t)((((uint64_t)hi << 32) | lo) >> sh) & cmask;
    uint32_t l = slice + carry;
    dneg = false;
    if (l > L) { l = 2 * L - l; carry = 1; dneg = true; } else carry = 0;
    if (l == 0) return NO_BUCKET;
    uint32_t bucket = (uint32_t)w * L + (l - 1);
    if (w == pr.K - 1 && pr.top_sub) {
      // sparse top window: spread each digit over 2^top_sub buckets of equal weight
      if (l > (L >> pr.top_sub)) { atomicOr(&counts[pr.nbuckets], 1u); l = L >> pr.top_sub; }  // cannot happen for |k| < 2^(MAG_BITS-1)
      bucket = (uint32_t)w * L + (((l - 1) << pr.top_sub) | ((2 * i + h) & ((1u << pr.top_sub) - 1)));
    }
    return bucket;
  };
  constexpr int KU = 12;       // windows handled with all their histogram atomics in flight at once
  _Pragma("unroll") for (int h = 0; h < CV::HALVES; h++) {
    uint32_t carry = 0;
    if (pr.K <= KU) {
      // The rank of an entry is the value its histogram atomicAdd returns; issued one window at a time, a thread
      // waits for ~K dependent round trips to L2.  Here the digits of a half are formed first, then all atomics are
      // issued back to back, then the results are stored.
      uint32_t bk[KU], rk[KU];
      bool dn[KU];
      _Pragma("unroll") for (int w = 0; w < KU; w++) { bk[w] = NO_BUCKET; dn[w] = false; if (w < pr.K) bk[w] = digit(h, w, carry, dn[w]); }
      _Pragma("unroll") for (int w = 0; w < KU; w++) { rk[w] = 0; if (bk[w] != NO_BUCKET) rk[w] = atomicAdd(&counts[bk[w]], 1u); }
      _Pragma("unroll") for (int w = 0; w < KU; w++) {
        if (w >= pr.K) break;
        const size_t pos = (size_t)(h * pr.K + w) * pr.n + i;
        ent_bucket[pos] = bk[w];
        if (bk[w] != NO_BUCKET) ent_rank[pos] = rk[w] | ((dn[w] != neg[h]) ? REF_NEG : 0u);  // rank < 2^31
      }
    } else {
      for (int w = 0; w < pr.K; w++) {
        bool dneg;
        const uint32_t bucket = digit(h, w, carry, dneg);
        const size_t pos = (size_t)(h * pr.K + w) * pr.n + i;
        ent_bucket[pos] = bucket;
        if (bucket == NO_BUCKET) continue;
        const uint32_t rank = atomicAdd(&counts[bucket], 1u);
        ent_rank[pos] = rank | ((dneg != neg[h]) ? REF_NEG : 0u);  // rank < 2^31
      }
    }
  }
}

// ---------------------------------------------------------------- exclusive scan (uint32), 3 kernels
static constexpr int SCAN_T = 1024;
static constexpr int SCAN_ITEMS = 4;
static constexpr int SCAN_TILE = SCAN_T * SCAN_ITEMS;
static constexpr int SCAN_ROUNDS = 16;   // tree rounds whose exact size the scan reports

MGB_DEV uint32_t block_excl_scan(uint32_t val, uint32_t* total_out, uint32_t* sm /* 32 words */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t x = val;
  _Pragma("unroll") for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
  if (lane == 31) sm[wid] = x;
  __syncthreads();
  if (wid == 0) {
    uint32_t w = (lane < (int)(blockDim.x >> 5)) ? sm[lane] : 0;
    _Pragma("unroll") for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += y; }
    sm[lane] = w;  // inclusive scan of warp totals
  }
  __syncthreads();
  uint32_t base = wid ? sm[wid - 1] : 0;
  *total_out = sm[(blockDim.x >> 5) - 1];
  __syncthreads();
  return base + x - val;
}

// in: counts[n]; out: offs[n] (exclusive, tile-local), tile_sums[tile]; also global max of counts.
// Every bucket is given an EVEN number of slots (count rounded up), so that the round-0 pairs of the
// in-place bucket trees are the aligned slot pairs (2q, 2q+1) and need no pair list.
static __global__ void __launch_bounds__(SCAN_T) k_scan_tiles(const uint32_t* __restrict__ counts, uint32_t* __restrict__ offs,
                                                       uint32_t* __restrict__ tile_sums, uint32_t n, uint32_t* __restrict__ maxcount,
                                                       uint32_t* __restrict__ round_pairs /* [r] += additions of tree round r, r < SCAN_ROUNDS */) {
  __shared__ uint32_t sm[32];
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS], sum = 0, mx = 0, rp[SCAN_ROUNDS];
  _Pragma("unroll") for (int r = 0; r < SCAN_ROUNDS; r++) rp[r] = 0;
  _Pragma("unroll") for (int k = 0; k < SCAN_ITEMS; k++) {
    uint32_t cnt = (base + k < n) ? counts[base + k] : 0;
    mx = max(mx, cnt);
    // a bucket of cnt elements has ceil((cnt - 2^r) / 2^(r+1)) additions in round r of its tree
    _Pragma("unroll") for (int r = 0; r < SCAN_ROUNDS; r++) rp[r] += (cnt + (1u << r) - 1) >> (r + 1);
    v[k] = (cnt + 1) & ~1u;
    sum += v[k];
  }
  uint32_t total;
  uint32_t ex = block_excl_scan(sum, &total, sm);
  _Pragma("unroll") for (int k = 0; k < SCAN_ITEMS; k++) { if (base + k < n) offs[base + k] = ex; ex += v[k]; }
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
  mx = __reduce_max_sync(0xffffffffu, mx);
  if ((threadIdx.x & 31) == 0 && mx) atomicMax(maxcount, mx);
  _Pragma("unroll") for (int r = 0; r < SCAN_ROUNDS; r++) {
    uint32_t t = __reduce_add_sync(0xffffffffu, rp[r]);
    if ((threadIdx.x & 31) == 0 && t) atomicAdd(round_pairs + r, t);
  }
}
// single block: exclusive scan of tile_sums[ntiles] in place, total -> *grand
static __global__ void __launch_bounds__(SCAN_T) k_scan_sums(uint32_t* __restrict__ tile_sums, uint32_t ntiles, uint32_t* __restrict__ grand) {
  __shared__ uint32_t sm[32];
  uint32_t carry = 0;
  for (uint32_t base = 0; base < ntiles; base += SCAN_T) {
    uint32_t i = base + threadIdx.x;
    uint32_t v = (i < ntiles) ? tile_sums[i] : 0;
    uint32_t total;
    uint32_t ex = block_excl_scan(v, &total, sm);
    if (i < ntiles) tile_sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) *grand = carry;
}
// also writes (offset, count) of every bucket side by side: the scatter fetches both with ONE 8-byte gather per entry
static __global__ void __launch_bounds__(SCAN_T) k_scan_add(uint32_t* __restrict__ offs, const uint32_t* __restrict__ tile_sums,
                                                     uint32_t n, const uint32_t* __restrict__ grand,
                                                     const uint32_t* __restrict__ counts, uint2* __restrict__ offcnt) {
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t add = tile_sums[blockIdx.x];
  _Pragma("unroll") for (int k = 0; k < SCAN_ITEMS; k++) if (base + k < n) {
    const uint32_t o = offs[base + k] + add;
    offs[base + k] = o;
    offcnt[base + k] = make_uint2(o, counts[base + k]);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) offs[n] = *grand;
}

// ---------------------------------------------------------------- k_scatter
// Counting-sort scatter (the reference's sortPoints, msm-batched-affine.ts:456-502, copies the points
// into bucket order).  Here a sorted slot only records WHICH point it stands for:
//     ref(slot) = point index | endo << 30 | negate << 31,      slot = offs[bucket] + rank,
// kept per aligned slot pair: recs[slot / 2] = {ref(even), ref(odd)}, lifes[slot / 2] (see below);
// round 0 of the bucket trees gathers its operands straight from the point table and writes the
// sums to V[slot]: one write and one read of every sorted point (192 B per entry, ~1 ms at 2^20) are
// never done.  Buckets start at even slots (k_scan_tiles), so round 0 pairs slot 2q with 2q+1; the
// last element of an odd-sized bucket gets REF_EMPTY as its partner and is simply copied by round 0.
// With V != nullptr (no tree round follows -- tiny inputs: k_bucket_finish / k_group_partial then read V
// directly) the point is materialised here instead.
//
// The in-place bucket tree (msm-batched-affine.ts:243-263): in round r the element at local index j
// (multiple of 2^(r+1)) absorbs the element at j + 2^r if that is inside the bucket of size n.  The
// rounds in which a slot is a left operand are r = 0 .. life-1 with
//     life = min(ctz(j), floor(log2(n - j - 1)) + 1)        (0 if j is the last element),
// kept per even slot (lifes[slot / 2]); the pair lists of rounds >= 1 carry (slot, life),
// so no bucket lookup is needed later.
struct PairEnt {
  uint32_t slot;
  uint32_t life;
};
static constexpr uint32_t REF_EMPTY = 0xffffffffu;

MGB_DEV void emit_pair(bool active, PairEnt ent, PairEnt* __restrict__ pairs, uint32_t* __restrict__ npairs) {
  uint32_t m = __ballot_sync(0xffffffffu, active);
  if (m) {
    int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(npairs, (uint32_t)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (active) pairs[base + __popc(m & ((1u << lane) - 1))] = ent;
  }
}

// Grid: x covers the points in chunks of SCATTER_U * 256, y = (half, window of the group): no index division, and
// every thread has SCATTER_U independent entries in flight (the chain entry -> bucket offset / count -> scattered
// write is three dependent memory round trips; one entry per thread left the kernel latency-bound).
static constexpr int SCATTER_U = 4;
template <class CV>
__global__ void __launch_bounds__(256) k_scatter(MsmParams pr, int w_begin, int Kg, const uint32_t* __restrict__ ent_bucket, const uint32_t* __restrict__ ent_rank,
                                                 const uint2* __restrict__ offcnt /* (offset, count) per bucket */, const uint32_t* __restrict__ table,
                                                 uint32_t* __restrict__ V, uint32_t* __restrict__ recs /* 2 words per aligned slot pair */, uint8_t* __restrict__ lifes) {
  const uint32_t el = blockIdx.y;
  const uint32_t h = el / (uint32_t)Kg, w = (uint32_t)w_begin + el % (uint32_t)Kg;
  const size_t row = (size_t)(h * pr.K + w) * pr.n;
  const bool endo = h != 0;
  uint32_t i[SCATTER_U], b[SCATTER_U], rk[SCATTER_U], n[SCATTER_U], o[SCATTER_U];
  _Pragma("unroll") for (int u = 0; u < SCATTER_U; u++) {
    i[u] = (blockIdx.x * SCATTER_U + u) * blockDim.x + threadIdx.x;
    b[u] = NO_BUCKET; rk[u] = 0;
    if (i[u] < pr.n) { b[u] = ent_bucket[row + i[u]]; rk[u] = ent_rank[row + i[u]]; }
  }
  _Pragma("unroll") for (int u = 0; u < SCATTER_U; u++) {
    n[u] = 0; o[u] = 0;
    if (b[u] != NO_BUCKET) { const uint2 oc = offcnt[b[u]]; o[u] = oc.x; n[u] = oc.y; }
  }
  _Pragma("unroll") for (int u = 0; u < SCATTER_U; u++) {
    if (b[u] == NO_BUCKET) continue;
    const uint32_t j = rk[u] & ~REF_NEG;
    const uint32_t slot = o[u] + j;
    if (V) { CV::store_v(V, slot, CV::load_entry(table, i[u], endo, (rk[u] & REF_NEG) != 0)); continue; }
    uint32_t* rec = recs + (size_t)(slot >> 1) * 2;
    const uint32_t ref = i[u] | (endo ? REF_ENDO : 0u) | (rk[u] & REF_NEG);
    if (j & 1) { rec[1] = ref; continue; }
    const uint32_t rest = n[u] - j - 1;                 // elements after this one
    uint32_t life = 0;
    if (rest) {
      life = 32 - __clz(rest);                          // floor(log2(rest)) + 1
      if (j) life = min(life, (uint32_t)(__ffs(j) - 1));
    } else {
      rec[1] = REF_EMPTY;                               // padding slot of an odd-sized bucket
    }
    rec[0] = ref;
    lifes[slot >> 1] = (uint8_t)life;
  }
}

// Counters the host sizes the tree rounds from, written by the device into page-locked host memory:
// host[64] padded slots, [65] largest bucket, [66] range flags of k_digits, [68 + r] additions of tree round r
static __global__ void k_plan_to_host(const uint32_t* __restrict__ misc, const uint32_t* __restrict__ flags, uint32_t* host) {
  const int t = threadIdx.x;
  if (t < 2) host[64 + t] = misc[t];
  if (t == 2) host[66] = *flags;
  if (t < SCAN_ROUNDS) host[68 + t] = misc[512 + t];
  __threadfence_system();
}

// ---------------------------------------------------------------- k_batch_add (Weierstrass)
// Batched-affine additions with one field inversion per WARP tile of 32*E independent additions
// (reference: batchAddNew / batchAddUnsafeNew, src/curve-affine.ts:376-522, and the Montgomery
// trick of src/wasm/inverse.ts:220-271).  Warps are fully independent (no block barrier):
//   1. every lane walks E pairs, needing only the x coordinates, and keeps the running product of
//      the denominators; the prefix products go to a per-warp scratch area in global memory.  It
//      also counts the pairs whose sum goes on to the next round: one atomicAdd per TILE then
//      reserves their range in the next round's pair list;
//   2. warp-wide inclusive prefix and suffix products of the 32 lane totals by shuffles;
//   3. the warp inverts the grand total with the lane-parallel division-step inverse (warp.cuh; round 1 left it to
//      lane 0 while the other warps of the SM kept the multiplier pipe busy);
//   4. every lane gets the inverse of its own total (2 multiplications), then walks its pairs
//      backwards: recompute the denominator, peel off its inverse, finish the addition, store.
//      Continuing sums are appended to the reserved range (ballot + running offset, no atomic).
// 6 multiplications per addition + 13/E for the warp products.
//
// Operand staging.  The operands of a pair are two random 96-byte reads (a gather from the point
// table in round 0, from V later) that miss L1 and mostly L2; a warp has no registers to spare for
// loads in flight (128 registers, 4 blocks per SM), and L1 prefetches were evicted before use by the
// kernel's own streaming traffic (ncu: 29 % of the warp samples stalled on a long scoreboard).  So
// every global input of an iteration -- pair entry, operands, stored prefix product -- is copied
// asynchronously (cp.async, L2 -> shared memory, no registers, no L1) one iteration ahead (entries:
// two ahead, their content gives the operand addresses) into per-thread staging slots read back
// with conflict-free 16-byte shared-memory loads.  The backward pass goes further and keeps the
// coordinates IN those slots for the whole iteration, re-reading them where a formula needs them:
// Field::mul is an out-of-line call, and holding both points across its five calls does not fit
// in 128 registers (see the comment at the backward pass).
template <class P>
MGB_DEV Fe<P> shfl_fe(const Fe<P>& a, int src) {
  Fe<P> r;
  _Pragma("unroll") for (int i = 0; i < P::N; i++) r.v[i] = __shfl_sync(0xffffffffu, a.v[i], src);
  return r;
}

#ifdef MGB_HOST_EMU
// emulation: the copy completes at once, so the group bookkeeping has nothing to wait for
MGB_DEV void cp_async16(void* smem, const void* gmem) { memcpy(smem, gmem, 16); }
MGB_DEV void cp_async4(void* smem, const void* gmem) { memcpy(smem, gmem, 4); }
MGB_DEV void cp_async8(void* smem, const void* gmem) { memcpy(smem, gmem, 8); }
MGB_DEV void cp_async_commit() {}
MGB_DEV void cp_async_wait_all() {}
MGB_DEV void cp_async_wait_but_one() {}
#else
MGB_DEV void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
MGB_DEV void cp_async4(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem) : "memory");
}
MGB_DEV void cp_async8(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}
MGB_DEV void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
MGB_DEV void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
MGB_DEV void cp_async_wait_but_one() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }   // all but the most recent group
#endif

template <class CV>
MGB_DEV typename CV::vpoint load_ref(const uint32_t* table, uint32_t ref) {
  return CV::load_entry(table, ref & REF_IDX, (ref & REF_ENDO) != 0, (ref & REF_NEG) != 0);
}

// Round-0 record of the aligned slot pair (2q, 2q+1), written by k_scatter: recs[q] = (reference of
// the left point, reference of the right one or REF_EMPTY: none, the left point is only copied),
// lifes[q] = life of the left slot, one byte (only the backward pass needs it).
// FIRST = true is round 0: pair q of the window group's slot range [offs[b_begin], offs[b_end]) is
// recs[q]; operands come from the point table, V is only written, no pair list is read.
template <class CV, int EMAX, int MINB, bool FIRST>
__global__ void __launch_bounds__(128, MINB) k_batch_add(uint32_t* __restrict__ V, const PairEnt* __restrict__ pairs,
                                                         const uint32_t* __restrict__ npairs_ptr, int r, int E_big, int E_small, uint32_t n_big,
                                                         PairEnt* __restrict__ pairs_out, uint32_t* __restrict__ npairs_out,
                                                         uint32_t* __restrict__ tile_counter,
                                                         const uint2* __restrict__ recs, const uint8_t* __restrict__ lifes,
                                                         const uint32_t* __restrict__ table,
                                                         const uint32_t* __restrict__ offs, uint32_t b_begin, uint32_t b_end,
                                                         uint4* __restrict__ scratch) {
  typedef typename CV::P FP;
  typedef typename CV::F F;
  typedef typename CV::G G;
  typedef Fe<FP> fe;
  constexpr int N = CV::N;
  constexpr int CW = N / 4;             // 16-byte chunks per coordinate
  // staging slots, in chunks: A.x | B.x | A.y | B.y | prefix product | 3 pair entries: 18 chunks = 36 KB per block for a
  // 12-limb field (round 1 kept a second x buffer: 48 KB), four blocks per SM at 128 registers.  The multiplier pipe is
  // at 63 / 90 / 97 / 98 % of its rate with 1 / 2 / 3 / 4 warps of a scheduler inside a product at the same time
  // (profiles/r02_microbench_mul_vs_warps.jsonl) and a warp spends two thirds of its time there; the shared memory would
  // allow a fifth and sixth block, but at 96 / 80 registers those builds spill and were slower (MGB_MINB = 5, 6:
  // profiles/r02_ab_blocks_per_sm.txt).
  constexpr int ST_A = 0, ST_PRE = 4 * CW, ST_ENT = 5 * CW;
  constexpr int ST_TOTAL = ST_ENT + 3;
  __shared__ uint4 stage[ST_TOTAL][128];   // [chunk][thread]: conflict-free 16-byte accesses
  static_assert(sizeof(uint4) * ST_TOTAL * 128 <= 48 * 1024, "static shared memory limit");
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const uint32_t q0 = FIRST ? offs[b_begin] >> 1 : 0u;
  const uint32_t npairs = FIRST ? (offs[b_end] >> 1) - q0 : *npairs_ptr;
  // Tile sizes: the first n_big tiles hold E_big pairs per lane, the rest E_small (chosen by the host, see msm_core).
  const uint32_t TILE_BIG = 32u * (uint32_t)E_big, TILE_SMALL = 32u * (uint32_t)E_small;
  const uint32_t nbig = min(n_big, npairs / TILE_BIG);
  const uint32_t rest = npairs - nbig * TILE_BIG;
  const uint32_t ntiles = nbig + (rest + TILE_SMALL - 1) / TILE_SMALL;
  const uint32_t step = 1u << r;
  // prefix products of this warp's current tile: chunk c of pair e at [(e * CW + c) * 32 + lane]
  uint4* const my_pre = scratch + (size_t)(blockIdx.x * 4 + (tid >> 5)) * EMAX * CW * 32 + lane;

  auto stage_fe = [&](int c0) -> fe {
    fe x;
    _Pragma("unroll") for (int c = 0; c < CW; c++) {
      const uint4 q = stage[c0 + c][tid];
      x.v[4 * c] = q.x; x.v[4 * c + 1] = q.y; x.v[4 * c + 2] = q.z; x.v[4 * c + 3] = q.w;
    }
    return x;
  };
  // Tile hand-out.  Every warp first takes ONE statically assigned tile, then tiles are handed out
  // dynamically (warps drift apart -- inversion latency varies -- and a static split would leave the
  // tail of every round to a few warps).  The static first tile matters for the late rounds, which
  // have fewer tiles than warps: with a pure atomic hand-out the winners are random and some SM
  // sub-partitions run 3-4 tiles while others idle (ncu, round 6: sub-partitions active half of the
  // kernel's duration).  Blocks b, b + #SM, b + 2 #SM, .. share an SM and warp w of a block sits on
  // sub-partition w, so tile t goes to block t mod #blocks, warp (t / #blocks + b / #SM) mod 4:
  // tiles 0 .. #blocks-1 land one per block AND one per sub-partition of every SM.
  const uint32_t total_warps = gridDim.x * 4u;
  bool first_tile = true;
  while (true) {
    uint32_t tile = 0;
    if (first_tile) {
      const uint32_t k = ((uint32_t)(tid >> 5) + 4u - (blockIdx.x / (gridDim.x / (uint32_t)MINB)) % 4u) % 4u;
      tile = k * gridDim.x + blockIdx.x;
      first_tile = false;
      if (tile >= ntiles) continue;                  // nothing assigned: try the dynamic pool (empty when ntiles <= #warps)
    } else {
      if (lane == 0) tile = atomicAdd(tile_counter, 1u) + total_warps;
      tile = __shfl_sync(0xffffffffu, tile, 0);
      if (tile >= ntiles) break;
    }
    const int E = tile < nbig ? E_big : E_small;
    const uint32_t base = (tile < nbig ? tile * TILE_BIG : nbig * TILE_BIG + (tile - nbig) * TILE_SMALL) + lane;

    // pair entry e -> staging slot (e mod 3); x = REF_EMPTY marks "no pair"
    auto ent_slot = [&](int e) -> uint4* { return &stage[ST_ENT + (e + 3) % 3][tid]; };
    auto fetch_ent = [&](int e) {
      uint4* dst = ent_slot(e);
      const uint32_t idx = base + (uint32_t)e * 32u;
      if (e < 0 || e >= E || idx >= npairs) { dst->x = REF_EMPTY; return; }
      if (FIRST) {
        cp_async8(dst, recs + q0 + idx);
        cp_async4(&dst->z, reinterpret_cast<const uint32_t*>(lifes) + ((q0 + idx) >> 2));   // the word holding the byte
      } else {
        cp_async8(dst, pairs + idx);
      }
    };
    auto is_add = [&](const uint4& en) -> bool { return en.x != REF_EMPTY && !(FIRST && en.y == REF_EMPTY); };
    // global address of operand A / B of an entry (2N contiguous limbs: x | y as stored in V; round 0: a table
    // entry's x | y, or y | beta*x for an endomorphism image)
    auto addr_a = [&](const uint4& en) -> const uint32_t* {
      if (FIRST) return table + (size_t)(en.x & REF_IDX) * CV::ENTRY_LIMBS + ((en.x & REF_ENDO) ? N : 0);
      return V + (size_t)en.x * CV::V_LIMBS;
    };
    auto addr_b = [&](const uint4& en) -> const uint32_t* {
      if (FIRST) return table + (size_t)(en.y & REF_IDX) * CV::ENTRY_LIMBS + ((en.y & REF_ENDO) ? N : 0);
      return V + (size_t)(en.x + step) * CV::V_LIMBS;
    };
    auto full_a = [&](const uint4& en) -> typename CV::vpoint { return FIRST ? load_ref<CV>(table, en.x) : CV::load_v(V, en.x); };
    auto full_b = [&](const uint4& en) -> typename CV::vpoint { return FIRST ? load_ref<CV>(table, en.y) : CV::load_v(V, en.x + step); };

    // ---- forward pass: running product of the denominators
    auto issue_x = [&](int e) {   // x coordinates of pair e -> ST_A, ST_A + CW
      const uint4 en = *ent_slot(e);
      if (!is_add(en)) return;
      // round 0: x sits behind y in the operand of an endomorphism image
      const uint32_t* xa = addr_a(en) + ((FIRST && (en.x & REF_ENDO)) ? N : 0);
      const uint32_t* xb = addr_b(en) + ((FIRST && (en.y & REF_ENDO)) ? N : 0);
      _Pragma("unroll") for (int c = 0; c < CW; c++) {
        cp_async16(&stage[ST_A + c][tid], xa + 4 * c);
        cp_async16(&stage[ST_A + CW + c][tid], xb + 4 * c);
      }
    };
    fetch_ent(0);
    fetch_ent(1);
    cp_async_commit();
    cp_async_wait_all();
    issue_x(0);
    cp_async_commit();
    fe run = F::one();
    // does the sum written for this entry go on to the next round (is it a left operand there)?
    auto continues = [&](const uint4& en, int e) -> bool {
      if (en.x == REF_EMPTY) return false;
      const uint32_t life = FIRST ? (en.z >> (8 * ((q0 + base + (uint32_t)e * 32u) & 3))) & 0xffu : en.y;
      return (uint32_t)(r + 1) < life;
    };
    uint32_t n_emit = 0;                         // this lane's entries of the next round's pair list
    _Pragma("unroll 1") for (int e = 0; e < E; e++) {
      cp_async_wait_all();                       // x of pair e, entry e + 1
      const uint4 cur = *ent_slot(e);
      const fe xa = stage_fe(ST_A), xb = stage_fe(ST_A + CW);
      issue_x(e + 1);
      fetch_ent(e + 2);
      cp_async_commit();
      n_emit += continues(cur, e) ? 1u : 0u;
      fe d = F::one();
      if (is_add(cur)) {
        if (!G::prepare_x(xa, xb, d)) {  // rare: an operand is infinity or the x coordinates coincide
          typename CV::vpoint A = full_a(cur), B = full_b(cur);
          (void)G::add_prepare(A, B, d);
        }
      }
      _Pragma("unroll") for (int c = 0; c < CW; c++)
        my_pre[(e * CW + c) * 32] = make_uint4(run.v[4 * c], run.v[4 * c + 1], run.v[4 * c + 2], run.v[4 * c + 3]);
      run = F::mul(run, d);
    }
    cp_async_wait_all();
    __threadfence_block();                         // the prefix products are read back (by this thread) through cp.async
    // ONE reservation in the next round's pair list per tile (its size is known after the forward pass) instead of
    // one atomicAdd per warp and iteration of the backward pass: ptxas turns every such atomic into its own
    // warp-aggregated sequence whose result-distributing shuffle waits for the round trip to L2 on the spot
    // (ncu: 3.4 % of the samples of round 0), whichever way the source defers the use of the result.
    uint32_t tile_out = 0;
    {
      const uint32_t total = __reduce_add_sync(0xffffffffu, n_emit);
      if (lane == 0 && total) tile_out = atomicAdd(npairs_out, total);
      tile_out = __shfl_sync(0xffffffffu, tile_out, 0);
    }
    fetch_ent(E - 1);                        // first entries of the backward pass travel during the warp products
    fetch_ent(E - 2);
    cp_async_commit();
    // ---- warp products: pfx = c_0..c_lane, sfx = c_lane..c_31
    fe pfx = run, sfx = run;
    _Pragma("unroll 1") for (int dlt = 1; dlt < 32; dlt <<= 1) {
      fe up = shfl_fe<FP>(pfx, lane - dlt < 0 ? lane : lane - dlt);
      fe dn = shfl_fe<FP>(sfx, lane + dlt > 31 ? lane : lane + dlt);
      fe np = F::mul(pfx, up), ns = F::mul(sfx, dn);
      if (lane >= dlt) pfx = np;
      if (lane + dlt <= 31) sfx = ns;
    }
    fe inv = shfl_fe<FP>(pfx, 31);                  // -> 1 / (this warp's total)
    // Backward pass that keeps its operands in SHARED MEMORY instead of registers.  Field::mul is an out-of-line
    // call that needs ~70 registers of its own; the caller can keep few values across a call, and a version that
    // holds both points, the running inverse and the inverted denominator (72) spills, with every iteration waiting
    // for the reloads (ncu, round 1: 5 % of the samples of round 0).  Here only the running inverse and one
    // intermediate live across a call; coordinates are re-read from the staging slots when a formula needs them.
    // Prefetch of pair e - 1 (issued during iteration e, two groups):
    //   * X: x halves, prefix product (and, riding in the same group, entry e - 2): issued right after the last read
    //     of pair e's x halves -- just before the final product m (x1 - x3) -- so one product (~2.4 K issue cycles,
    //     several times that under contention) covers the trip to L2 / HBM;
    //   * Y: y halves, issued after the last read of pair e's y halves at the end of the iteration.
    // Iteration e waits for "all but the most recent group" at the top (X_e; Y_e may still be in flight) and for all
    // groups before the slope.
    constexpr int ST_AY = ST_A + 2 * CW, ST_BY = ST_A + 3 * CW;
    auto xslot = [&](int) -> int { return ST_A; };                           // A.x at xslot, B.x at xslot + CW
    auto issue_xpart = [&](int e) {   // x of both operands and the prefix product of pair e
      const uint4 en = *ent_slot(e);
      if (en.x == REF_EMPTY) return;
      const int xs = xslot(e);
      const uint32_t* pa = addr_a(en) + ((FIRST && (en.x & REF_ENDO)) ? N : 0);
      _Pragma("unroll") for (int c = 0; c < CW; c++) cp_async16(&stage[xs + c][tid], pa + 4 * c);
      if (is_add(en)) {
        const uint32_t* pb = addr_b(en) + ((FIRST && (en.y & REF_ENDO)) ? N : 0);
        _Pragma("unroll") for (int c = 0; c < CW; c++) cp_async16(&stage[xs + CW + c][tid], pb + 4 * c);
      }
      _Pragma("unroll") for (int c = 0; c < CW; c++) cp_async16(&stage[ST_PRE + c][tid], my_pre + (e * CW + c) * 32);
    };
    auto issue_ypart = [&](int e) {   // y of both operands (it comes first in the operand of an endomorphism image)
      const uint4 en = *ent_slot(e);
      if (en.x == REF_EMPTY) return;
      const uint32_t* pa = addr_a(en) + ((FIRST && (en.x & REF_ENDO)) ? 0 : N);
      _Pragma("unroll") for (int c = 0; c < CW; c++) cp_async16(&stage[ST_AY + c][tid], pa + 4 * c);
      if (is_add(en)) {
        const uint32_t* pb = addr_b(en) + ((FIRST && (en.y & REF_ENDO)) ? 0 : N);
        _Pragma("unroll") for (int c = 0; c < CW; c++) cp_async16(&stage[ST_BY + c][tid], pb + 4 * c);
      }
    };
    cp_async_wait_all();
    issue_xpart(E - 1);
    cp_async_commit();
    issue_ypart(E - 1);
    cp_async_commit();
    // all lanes share the inversion (lane-parallel division steps, warp.cuh): 20.6 us instead of 35.3 us on lane 0 alone,
    // and 32 instead of 1 active lanes in what was a tenth of the kernel's issue slots (A/B: profiles/r02_ab_winv_onewarp.jsonl)
    inv = WarpField<FP>::inv_call(inv);
    fe u = inv;                                   // -> 1 / (this lane's total)
    {
      const fe left = shfl_fe<FP>(pfx, lane == 0 ? 0 : lane - 1);
      if (lane > 0) u = F::mul(u, left);
      const fe right = shfl_fe<FP>(sfx, lane == 31 ? 31 : lane + 1);
      if (lane < 31) u = F::mul(u, right);
    }
    _Pragma("unroll 1") for (int e = E - 1; e >= 0; e--) {
      cp_async_wait_but_one();                   // X_e: x halves and prefix product of pair e, entry e - 1
      const uint4 cur = *ent_slot(e);
      const bool valid = cur.x != REF_EMPTY;
      const bool add = is_add(cur);
      const int xs = xslot(e);
      const fe pre = stage_fe(ST_PRE);
      fetch_ent(e - 2);                          // rides in group X_(e-1), committed below
      const fe inv_den = F::mul(u, pre);
      PairEnt out = {0u, 0u};
      if (valid) {
        out.slot = FIRST ? 2u * (q0 + base + (uint32_t)e * 32u) : cur.x;
        out.life = FIRST ? (cur.z >> (8 * ((q0 + base + (uint32_t)e * 32u) & 3))) & 0xffu : cur.y;
      }
      // kind of the addition (Weierstrass::add_prepare): 0 = generic, 1 = doubling, 2 / 3 = B / A is infinity,
      // 4 = P + (-P).  The generic case is decided from the x coordinates alone; in the rare other cases the
      // complete operands are fetched and written back into the staging slots, so that one straight-line formula
      // below serves both (the flow has no second copy of the products).
      int kind = 0;
      bool y_ready = false;                      // rare path: staged y already carries its sign
      if (add) {
        fe d;
        if (!G::prepare_x(stage_fe(xs), stage_fe(xs + CW), d)) {
          const typename CV::vpoint A = full_a(cur), B = full_b(cur);
          kind = G::add_prepare(A, B, d);
          cp_async_wait_all();                   // Y_e has landed: the slots can be overwritten
          _Pragma("unroll") for (int c = 0; c < CW; c++) {
            stage[xs + c][tid] = make_uint4(A.x.v[4 * c], A.x.v[4 * c + 1], A.x.v[4 * c + 2], A.x.v[4 * c + 3]);
            stage[xs + CW + c][tid] = make_uint4(B.x.v[4 * c], B.x.v[4 * c + 1], B.x.v[4 * c + 2], B.x.v[4 * c + 3]);
            stage[ST_AY + c][tid] = make_uint4(A.y.v[4 * c], A.y.v[4 * c + 1], A.y.v[4 * c + 2], A.y.v[4 * c + 3]);
            stage[ST_BY + c][tid] = make_uint4(B.y.v[4 * c], B.y.v[4 * c + 1], B.y.v[4 * c + 2], B.y.v[4 * c + 3]);
          }
          y_ready = true;
        }
        u = F::mul(u, d);
      }
      cp_async_wait_all();                       // Y_e (and entry e - 2)
      auto stage_y = [&](int c0, uint32_t ref) -> fe {
        const fe y = stage_fe(c0);
        return (FIRST && !y_ready && (ref & REF_NEG)) ? F::neg(y) : y;
      };
      // the x halves of pair e are read for the last time just before the final product: their slots then take pair e - 1
      auto prefetch_x = [&]() {
        if (e > 0) issue_xpart(e - 1);
        cp_async_commit();                       // group X_(e-1)
      };
      if (valid) {
        typename CV::vpoint R;
        if (add && kind < 2) {
          fe num;
          if (kind == 1) { const fe xx = F::sqr(stage_fe(xs)); num = F::add(F::dbl(xx), xx); }      // tangent: 3 x^2 / 2 y
          else num = F::sub(stage_y(ST_BY, cur.y), stage_y(ST_AY, cur.x));
          const fe m = F::mul(num, inv_den);
          R.x = F::sqr(m);
          const fe ax = stage_fe(xs);
          R.x = F::sub(F::sub(R.x, ax), stage_fe(xs + CW));      // doubling: B = A, so this is m^2 - 2x
          const fe t = F::sub(ax, R.x);
          prefetch_x();
          R.y = F::mul(m, t);
          R.y = F::sub(R.y, stage_y(ST_AY, cur.x));
        } else if (kind == 4) {
          R = G::affine_inf();
          prefetch_x();
        } else {                                 // no partner (round 0) or B infinite: A; A infinite: B
          R.x = stage_fe(kind == 3 ? xs + CW : xs);
          R.y = stage_y(kind == 3 ? ST_BY : ST_AY, kind == 3 ? cur.y : cur.x);
          prefetch_x();
        }
        CV::store_v(V, out.slot, R);
      } else {
        prefetch_x();
      }
      if (e > 0) issue_ypart(e - 1);
      cp_async_commit();                         // group Y_(e-1)
      {
        const bool em = valid && (uint32_t)(r + 1) < out.life;      // == continues(cur, e) of the forward pass
        const uint32_t mk = __ballot_sync(0xffffffffu, em);
        if (em) pairs_out[tile_out + __popc(mk & ((1u << lane) - 1u))] = out;
        tile_out += __popc(mk);
      }
    }
    cp_async_wait_all();
  }
}

// ---------------------------------------------------------------- k_pair_add (twisted Edwards: no inversion needed)
template <class CV, bool FIRST>
__global__ void __launch_bounds__(256) k_pair_add(uint32_t* __restrict__ V, const PairEnt* __restrict__ pairs,
                                                  const uint32_t* __restrict__ npairs_ptr, int r,
                                                  PairEnt* __restrict__ pairs_out, uint32_t* __restrict__ npairs_out,
                                                  const uint2* __restrict__ recs, const uint8_t* __restrict__ lifes,
                                                  const uint32_t* __restrict__ table, const uint32_t* __restrict__ offs,
                                                  uint32_t b_begin, uint32_t b_end) {
  const uint32_t q0 = FIRST ? offs[b_begin] >> 1 : 0u;
  const uint32_t npairs = FIRST ? (offs[b_end] >> 1) - q0 : *npairs_ptr;
  const uint32_t step = 1u << r;
  const uint32_t nround = (npairs + 31) & ~31u;   // whole warps iterate together (ballot in emit_pair)
  for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < nround; idx += gridDim.x * blockDim.x) {
    const bool valid = idx < npairs;
    PairEnt ent = {0u, 0u};
    if (valid) {
      if constexpr (FIRST) {
        const uint2 rr = recs[q0 + idx];
        ent.slot = 2u * (q0 + idx);
        ent.life = lifes[q0 + idx];
        const typename CV::vpoint A = rr.y != REF_EMPTY ? CV::add_refs(table, rr.x, rr.y) : load_ref<CV>(table, rr.x);
        CV::store_v(V, ent.slot, A);
      } else {
        ent = pairs[idx];
        CV::store_v(V, ent.slot, CV::add(CV::load_v(V, ent.slot), CV::load_v(V, ent.slot + step)));
      }
    }
    emit_pair(valid && (uint32_t)(r + 1) < ent.life, ent, pairs_out, npairs_out);
  }
}

// ---------------------------------------------------------------- bucket reduction
// Window sum S_w = sum_{l=1..L} l * B_l (reference: reduceBucketsColumnProjective, the running sum
// "triangle += row; row += B_l", msm-batched-affine.ts:556-583 -- 2L sequential additions per
// chunk).  A sequential walk is latency-bound on a GPU, so the weight is split into D digits of
// at most 5 bits instead:  idx = l - 1 = sum_d v_d * 2^(sh_d),  hence
//     S_w = sum_d 2^(sh_d) * ( sum_v v * G[w][d][v] ) + sum_l B_l,
//     G[w][d][v] = sum of the buckets of window w whose digit d equals v
// -- D plain sums per bucket, done as chunked partial sums plus a log-depth tree, then one warp
// per (w, d) forms sum_v v*G_v with a shuffle suffix scan (the "warp-shuffle running sum").
struct ReduceGeom {
  int D;            // digits
  int width[6];     // bits per digit
  int shift[6];     // bit position of each digit
  int NP;           // partial sums per group (power of two)
  int CH;           // buckets per partial sum
  int VB;           // NV = 2^VB group slots per (window, digit): 32, or 16 / 8 when no digit is wider than 4 / 3 bits (small
  int NV;           // windows: half of the groups -- and of the latency-bound tree work -- would be empty otherwise)
};

// Bucket sums after the last tree round: one thread per bucket adds whatever the bucket has left (the
// elements at stride 2^rounds) into an XYZZ accumulator.  Without it every one of the D digit passes of
// k_group_partial would walk the leftovers again; with it the batched-affine rounds can stop earlier
// (their late rounds are latency-bound, ~0.2 ms each for ever fewer additions) and hand 4-8 elements
// per bucket to this throughput-bound kernel instead.
template <class CV>
__global__ void __launch_bounds__(128) k_bucket_finish(uint32_t b_begin, uint32_t b_end, int rounds, const uint32_t* __restrict__ V,
                                                       const uint32_t* __restrict__ offs, const uint32_t* __restrict__ counts, uint32_t* __restrict__ Bsum) {
  const uint32_t b = b_begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= b_end) return;
  const uint32_t o = offs[b], n = counts[b], stride = 1u << rounds;
  if (n == 0) return;                                   // k_group_partial skips empty buckets by their count
  // the first two leftovers are both stored elements (affine on the batched-affine curves: 6 products instead of 10)
  typename CV::acc acc;
  if (n > stride) acc = CV::add_vv(CV::load_v(V, o), CV::load_v(V, o + stride));
  else acc = CV::add_v(CV::acc_zero(), CV::load_v(V, o));
  for (uint32_t q = 2 * stride; q < n; q += stride) acc = CV::add_v(acc, CV::load_v(V, o + q));
  CV::st_acc(Bsum + (size_t)b * CV::ACC_LIMBS, acc);
}

template <class CV>
__global__ void __launch_bounds__(128) k_group_partial(MsmParams pr, ReduceGeom gm, int w_begin, int Kg, int rounds, const uint32_t* __restrict__ V,
                                                       const uint32_t* __restrict__ offs, const uint32_t* __restrict__ counts,
                                                       const uint32_t* __restrict__ Bsum /* bucket sums of k_bucket_finish, or nullptr */, uint32_t* __restrict__ P) {
  // thread -> (window w, digit d, value v, chunk ch)
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t total = (uint32_t)Kg * gm.D * gm.NV * gm.NP;
  if (t >= total) return;
  t += (uint32_t)w_begin * gm.D * gm.NV * gm.NP;       // global (window, digit, value, chunk) index
  uint32_t ch = t % gm.NP, g = t / gm.NP;
  uint32_t v = g & (uint32_t)(gm.NV - 1), wd = g >> gm.VB;
  uint32_t d = wd % gm.D, w = wd / gm.D;
  typename CV::acc acc = CV::acc_zero();
  // digit d of the weight index idx = (bucket >> sub): bits [shift + sub, ...) of the bucket number
  const int sub = (w == (uint32_t)pr.K - 1) ? pr.top_sub : 0;
  const int nb = pr.c - 1;
  const int sh = min(gm.shift[d] + sub, nb);
  const int wdt = min(gm.width[d], nb - sh);
  const uint32_t gsize = pr.L >> wdt;                  // members of the group
  // a digit clipped to zero width (top window with sub-bucket spreading) has weight 0 everywhere:
  // its groups are only needed for digit 0, whose v = 0..: sum also yields the window total
  if (v < (1u << wdt) && !(wdt == 0 && d > 0)) {
    const uint32_t stride = 1u << rounds;
    const uint32_t chlen = (gsize + gm.NP - 1) / gm.NP;   // = CH except for clipped digits
    for (uint32_t k = 0; k < chlen; k++) {
      uint32_t m = ch * chlen + k;
      if (m >= gsize) break;
      uint32_t low = m & ((1u << sh) - 1), high = m >> sh;
      uint32_t idx = (high << (sh + wdt)) | (v << sh) | low;
      uint32_t b = w * pr.L + idx;
      uint32_t o = offs[b], n = counts[b];
      if (Bsum) {
        if (n) acc = CV::add(acc, CV::ld_acc(Bsum + (size_t)b * CV::ACC_LIMBS));
      } else {
        for (uint32_t q = 0; q < n; q += stride) acc = CV::add_v(acc, CV::load_v(V, o + q));
      }
    }
  }
  CV::st_acc(P + (size_t)t * CV::ACC_LIMBS, acc);
}

// ---- affine bucket reduction (SURVEY 8f-3; reference: reduceBucketsAffine, src/msm-batched-affine-single-thread.ts:522-700,
// doc/zprize22.md:317-358: "reducing buckets into one sum per partition, using only batch-affine additions").
// The reference splits every window into independent sub-sums so that the reduction, too, amortises one inversion over
// many additions.  The GPU form of the idea, on top of the digit decomposition above: the members of a group
// (window w, digit d, value v) are gathered side by side into a scratch array W, GS slots per group (bucket sums are
// single affine points once the bucket trees have run to completion; empty buckets and padding are the point at
// infinity), and every group is summed by the SAME in-place log-depth tree of batched-affine additions that sums the
// buckets (k_batch_add over pair lists: slot j of a group absorbs j + 2^r in round r).  All D K L additions that touch a
// bucket cost 6 multiplications instead of the 10 - 14 of the XYZZ formulas; what is left for XYZZ are the few hundred
// group sums themselves.  Opt-in (mgb_opts.affine_reduction): log2(GS) extra launches, each a round of at most
// 0.4 M additions, cost more latency than the multiplications they save (measured, profiles/r02_ab_affine_reduction.txt).
// Slots per group: GS0 for the windows below the top one, GS1 for the top window (its digits are clipped when the top
// window is sparse and spread over sub-buckets, MsmParams::top_sub, so its groups can be larger).  Groups lie back to back.
struct AffineRedGeom {
  int GS0, GS1;
  uint32_t g_top;        // first group of the top window = (K - 1) * D * NV
  uint32_t n0;           // slots of the groups below it = g_top * GS0
  uint32_t total;        // all slots
};
MGB_DEV uint32_t affine_group_base(const AffineRedGeom& ag, uint32_t g) {
  return g < ag.g_top ? g * (uint32_t)ag.GS0 : ag.n0 + (g - ag.g_top) * (uint32_t)ag.GS1;
}
template <class CV>
__global__ void __launch_bounds__(256) k_affine_gather(MsmParams pr, ReduceGeom gm, AffineRedGeom ag, const uint32_t* __restrict__ V,
                                                       const uint32_t* __restrict__ offs, const uint32_t* __restrict__ counts,
                                                       uint32_t* __restrict__ W, PairEnt* __restrict__ pairs, uint32_t* __restrict__ npairs) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ag.total) return;
  const bool top = t >= ag.n0;
  const int GS = top ? ag.GS1 : ag.GS0;
  const uint32_t tt = top ? t - ag.n0 : t;
  const uint32_t m = tt & (uint32_t)(GS - 1), g = (top ? ag.g_top : 0u) + tt / (uint32_t)GS;
  const uint32_t v = g & (uint32_t)(gm.NV - 1), wd = g >> gm.VB;
  const uint32_t d = wd % gm.D, w = wd / gm.D;
  const int sub = (w == (uint32_t)pr.K - 1) ? pr.top_sub : 0;
  const int nb = pr.c - 1;
  const int sh = min(gm.shift[d] + sub, nb);
  const int wdt = min(gm.width[d], nb - sh);
  const uint32_t gsize = pr.L >> wdt;
  typename CV::vpoint pt = CV::G::affine_inf();
  if (v < (1u << wdt) && !(wdt == 0 && d > 0) && m < gsize) {
    const uint32_t low = m & ((1u << sh) - 1), high = m >> sh;
    const uint32_t b = w * pr.L + ((high << (sh + wdt)) | (v << sh) | low);
    if (counts[b]) pt = CV::load_v(V, offs[b]);        // the bucket's sum sits in its first slot after the last tree round
  }
  CV::store_v(W, t, pt);
  if ((m & 1) == 0) {                                   // round 0 of the group trees: every even slot is a left operand
    int lg = 0;
    while ((1 << lg) < GS) lg++;
    const uint32_t life = m ? (uint32_t)(__ffs(m) - 1) : (uint32_t)lg;
    pairs[t >> 1] = PairEnt{t, life};
  }
  if (t == 0) *npairs = ag.total >> 1;
}
// group sums (first slot of every group in W) -> XYZZ partial sums P[g] (NP = 1) for k_digit_sums
template <class CV>
__global__ void __launch_bounds__(128) k_affine_group_sums(uint32_t ngroups, AffineRedGeom ag, const uint32_t* __restrict__ W, uint32_t* __restrict__ P) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ngroups) return;
  CV::st_acc(P + (size_t)g * CV::ACC_LIMBS, CV::G::from_affine(CV::load_v(W, affine_group_base(ag, g))));
}

// one tree level: P[g][i] += P[g][i + half] for i < half
template <class CV>
__global__ void __launch_bounds__(128) k_tree_round(uint32_t ngroups, int NP, int half, uint32_t* __restrict__ P) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ngroups * (uint32_t)half) return;
  uint32_t i = t % half, g = t / half;
  uint32_t* a = P + ((size_t)g * NP + i) * CV::ACC_LIMBS;
  CV::st_acc(a, CV::add(CV::ld_acc(a), CV::ld_acc(a + (size_t)half * CV::ACC_LIMBS)));
}

// the last tree levels of all groups in one launch: one warp per group, its <= 32 remaining partial
// sums reduced with shuffles
template <class CV>
MGB_DEV typename CV::acc shfl_acc(const typename CV::acc& a, int src);

template <class CV>
__global__ void __launch_bounds__(128) k_tree_tail(uint32_t ngroups, int NP, int remaining, uint32_t* __restrict__ P) {
  const int lane = threadIdx.x & 31;
  const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (g >= ngroups) return;
  uint32_t* base = P + (size_t)g * NP * CV::ACC_LIMBS;
  typename CV::acc a = lane < remaining ? CV::ld_acc(base + (size_t)lane * CV::ACC_LIMBS) : CV::acc_zero();
  _Pragma("unroll 1") for (int dl = 16; dl >= 1; dl >>= 1) {
    typename CV::acc o = shfl_acc<CV>(a, lane + dl > 31 ? lane : lane + dl);
    if (lane < dl && dl < remaining) a = CV::add(a, o);
  }
  if (lane == 0) CV::st_acc(base, a);
}

template <class CV>
MGB_DEV typename CV::acc shfl_acc(const typename CV::acc& a, int src) {
  typename CV::acc r;
  const uint32_t* pa = reinterpret_cast<const uint32_t*>(&a);
  uint32_t* pr = reinterpret_cast<uint32_t*>(&r);
  _Pragma("unroll") for (int i = 0; i < CV::ACC_LIMBS; i++) pr[i] = __shfl_sync(0xffffffffu, pa[i], src);
  return r;
}

// one-warp Horner: lane 8g + l holds 64-bit digit l of coordinate g of an accumulator (onewarp.cuh)
template <class FP>
MGB_DEV unsigned long long ow_load(const uint32_t* src) {
  const int g = (threadIdx.x & 31) >> 3, l = threadIdx.x & 7;
  return l < FP::N / 2 ? (((unsigned long long)src[g * FP::N + 2 * l + 1] << 32) | src[g * FP::N + 2 * l]) : 0ull;
}
template <class FP>
MGB_DEV void ow_store(uint32_t* dst, unsigned long long v) {
  const int g = (threadIdx.x & 31) >> 3, l = threadIdx.x & 7;
  if (l < FP::N / 2) { dst[g * FP::N + 2 * l] = (uint32_t)v; dst[g * FP::N + 2 * l + 1] = (uint32_t)(v >> 32); }
}

// block = one window, warp d = one digit: X_d = sum_v v * G_v by an inclusive suffix scan over the
// lanes (S_v = sum_{v' >= v} G_v', X = sum_{v >= 1} S_v), then thread 0 assembles
// S_w = sum_d 2^(sh_d) X_d + sum_l B_l.
template <class CV>
__global__ void __launch_bounds__(192) k_window_sums(MsmParams pr, ReduceGeom gm, int w_begin, const uint32_t* __restrict__ P, uint32_t* __restrict__ Sw) {
  __shared__ uint32_t sm[7 * CV::ACC_LIMBS];
  const int lane = threadIdx.x & 31, d = threadIdx.x >> 5, w = w_begin + blockIdx.x;
  if (d < gm.D) {
    typename CV::acc G = CV::acc_zero();
    if (lane < (1 << gm.width[d])) G = CV::ld_acc(P + ((size_t)((w * gm.D + d) * gm.NV + lane) * gm.NP) * CV::ACC_LIMBS);
    typename CV::acc S = G;
    _Pragma("unroll 1") for (int dl = 1; dl < 32; dl <<= 1) {
      typename CV::acc o = shfl_acc<CV>(S, lane + dl > 31 ? lane : lane + dl);
      if (lane + dl <= 31) S = CV::add(S, o);
    }
    typename CV::acc tot = shfl_acc<CV>(S, 0);       // sum of all buckets of the window
    typename CV::acc X = (lane >= 1) ? S : CV::acc_zero();
    _Pragma("unroll 1") for (int dl = 16; dl >= 1; dl >>= 1) {
      typename CV::acc o = shfl_acc<CV>(X, lane + dl > 31 ? lane : lane + dl);
      if (lane < dl) X = CV::add(X, o);
    }
    if (lane == 0) {
      CV::st_acc(sm + d * CV::ACC_LIMBS, X);
      if (d == 0) CV::st_acc(sm + 6 * CV::ACC_LIMBS, tot);
    }
  }
  __syncthreads();
  if (threadIdx.x < 32) {       // Horner over the digits with the point spread over the lanes of warp 0 (onewarp.cuh), as k_final does
    typedef typename CV::OneWarp OW;
    typedef typename CV::P FP;
    unsigned long long v = ow_load<FP>(sm + (gm.D - 1) * CV::ACC_LIMBS);
    for (int dd = gm.D - 2; dd >= 0; dd--) {
      for (int k = 0; k < gm.width[dd]; k++) v = OW::dbl(v);
      v = OW::add(v, ow_load<FP>(sm + dd * CV::ACC_LIMBS));
    }
    v = OW::add(v, ow_load<FP>(sm + 6 * CV::ACC_LIMBS));
    ow_store<FP>(Sw + (size_t)w * CV::ACC_LIMBS, v);
  }
}

// ---- quad-cooperative variants of the latency-bound reduction stages (Weierstrass, see coop.cuh) ----
// The last tree levels of one group (<= 32 partial sums left) in one 64-thread block: four lanes per
// addition, lane k moving coordinate k (N limbs) of the distributed point; block barrier between levels.
// (The earlier, throughput-bound levels stay with k_tree_round: one thread per addition.)
template <class CV>
__global__ void __launch_bounds__(64) k_tree_tail_quad(int NP, int remaining, uint32_t* P) {
  typedef typename CV::Quad Q;
  typedef Fe<typename CV::P> fe;
  constexpr int N = CV::N;
  const int k = threadIdx.x & 3, qd = threadIdx.x >> 2, wq = (threadIdx.x >> 5) * 8;   // quad of the block, first quad of the warp
  uint32_t* base = P + (size_t)blockIdx.x * NP * CV::ACC_LIMBS + k * N;
  for (int half = remaining >> 1; half >= 1; half >>= 1) {
    if (wq < half) {                                   // warp-uniform
      const bool act = qd < half;
      fe a = Q::zero_coord(k), b = a;
      if (act) { a = ld_fe<typename CV::P>(base + (size_t)qd * CV::ACC_LIMBS); b = ld_fe<typename CV::P>(base + (size_t)(qd + half) * CV::ACC_LIMBS); }
      const fe r = Q::add(a, b);
      if (act) st_fe<typename CV::P>(base + (size_t)qd * CV::ACC_LIMBS, r);
    }
    __syncthreads();
  }
}

// block = (window w, digit d), quad v = digit value: X_d = sum_v v * G_v by an inclusive suffix scan
// over the values (S_v = sum_{v' >= v} G_v', X = sum_{v >= 1} S_v) through shared memory.
// out[(w * D + d)] = X_d, out[K * D + w] = sum of all buckets of the window (from digit 0).
template <class CV>
__global__ void __launch_bounds__(128) k_digit_sums(MsmParams pr, ReduceGeom gm, int w_begin, const uint32_t* __restrict__ P, uint32_t* __restrict__ out) {
  typedef typename CV::Quad Q;
  typedef typename CV::P FP;
  typedef Fe<FP> fe;
  constexpr int N = CV::N;
  __shared__ uint32_t sm[32 * 4 * N];
  const int k = threadIdx.x & 3, v = threadIdx.x >> 2;
  const int d = blockIdx.x % gm.D, w = w_begin + blockIdx.x / gm.D;
  auto lds = [&](int vv) -> fe { fe r; _Pragma("unroll") for (int i = 0; i < N; i++) r.v[i] = sm[(vv * 4 + k) * N + i]; return r; };
  auto sts = [&](int vv, const fe& a) { _Pragma("unroll") for (int i = 0; i < N; i++) sm[(vv * 4 + k) * N + i] = a.v[i]; };
  fe S = Q::zero_coord(k);
  if (v < (1 << gm.width[d])) S = ld_fe<FP>(P + ((size_t)((w * gm.D + d) * gm.NV + v) * gm.NP) * CV::ACC_LIMBS + k * N);
  _Pragma("unroll 1") for (int dl = 1; dl < gm.NV; dl <<= 1) {        // values >= NV do not exist (zero): log2(NV) steps
    sts(v, S);
    __syncthreads();
    const fe o = (v + dl <= gm.NV - 1) ? lds(v + dl) : Q::zero_coord(k);
    __syncthreads();
    S = Q::add(S, o);
  }
  if (v == 0 && d == 0) st_fe<FP>(out + ((size_t)pr.K * gm.D + w) * CV::ACC_LIMBS + k * N, S);
  fe X = (v >= 1 && v < gm.NV) ? S : Q::zero_coord(k);
  _Pragma("unroll 1") for (int dl = gm.NV >> 1; dl >= 1; dl >>= 1) {
    sts(v, X);
    __syncthreads();
    const fe o = (v < dl) ? lds(v + dl) : Q::zero_coord(k);
    __syncthreads();
    X = Q::add(X, o);
  }
  if (v == 0) st_fe<FP>(out + ((size_t)w * gm.D + d) * CV::ACC_LIMBS + k * N, X);
}

// block = one window, ONE warp: S_w = sum_d 2^(sh_d) X_d + sum_l B_l by Horner over the digits, the point spread over the
// lanes (onewarp.cuh), as in k_final.
template <class CV>
__global__ void __launch_bounds__(32) k_window_assemble(MsmParams pr, ReduceGeom gm, int w_begin, const uint32_t* __restrict__ in, uint32_t* __restrict__ Sw) {
  typedef typename CV::P FP;
  typedef typename CV::OneWarp OW;
  const int w = w_begin + blockIdx.x;
  unsigned long long v = ow_load<FP>(in + ((size_t)w * gm.D + gm.D - 1) * CV::ACC_LIMBS);
  for (int dd = gm.D - 2; dd >= 0; dd--) {
    for (int k = 0; k < gm.width[dd]; k++) v = OW::dbl(v);
    v = OW::add(v, ow_load<FP>(in + ((size_t)w * gm.D + dd) * CV::ACC_LIMBS));
  }
  v = OW::add(v, ow_load<FP>(in + ((size_t)pr.K * gm.D + w) * CV::ACC_LIMBS));
  ow_store<FP>(Sw + (size_t)w * CV::ACC_LIMBS, v);
}

// result = sum_w 2^(c*w) S_w by Horner (msm-batched-affine.ts:322-334): (K-1)*c dependent doublings.
// out_xy != nullptr (single-GPU msm): the same warp also normalises -- canonical x || y and the is-zero flag, as
// k_normalize would -- so the result needs no further launch.
// One warp: the point is spread over the lanes (onewarp.cuh: 8-lane group g = coordinate g, one 64-bit digit per lane, the
// four products of a formula level are one WarpField2::mul; no shared memory, no barrier in the chain).  Round 1 ran the
// chain on a 128-thread block with a barrier per formula level: 0.370 -> 0.335 ms at 2^20 (profiles/r02_ab_winv_onewarp.jsonl),
// and 1.33 -> 0.31 ms for the 238 doublings of the twisted-Edwards curve at 2^18.
template <class CV>
__global__ void __launch_bounds__(32) k_final(int K, int c, const uint32_t* __restrict__ Sw, uint32_t* __restrict__ out_acc,
                                              uint32_t* __restrict__ out_xy, uint32_t* __restrict__ out_flag) {
  typedef typename CV::P FP;
  typedef typename CV::OneWarp OW;
  constexpr int N = CV::N;
  unsigned long long v = ow_load<FP>(Sw + (size_t)(K - 1) * CV::ACC_LIMBS);
  for (int w = K - 2; w >= 0; w--) {
    for (int d = 0; d < c; d++) v = OW::dbl(v);
    v = OW::add(v, ow_load<FP>(Sw + (size_t)w * CV::ACC_LIMBS));
  }
  ow_store<FP>(out_acc, v);
  if (out_xy) {
    Fe<FP> x, y;
    bool inf;
    CV::acc_to_plain_warp(OW::gather(v), x, y, inf);
    if (threadIdx.x == 0) {
      _Pragma("unroll") for (int i = 0; i < N; i++) { out_xy[i] = x.v[i]; out_xy[N + i] = y.v[i]; }
      *out_flag = inf ? 1u : 0u;
    }
  }
}

// sum `count` partial accumulators (multi-GPU combine) and/or normalise: out = canonical x||y + flag.  One warp: every
// lane forms the same sum, the inversion of the normalisation is lane-parallel.  The partials lie `stride` limbs apart;
// with stride > ACC_LIMBS each is followed by the status word of the rank that sent it (mgb_msm_sharded: non-zero = that
// rank could not compute its shard), and out_flag[1] tells the host whether any rank reported one.
template <class CV>
__global__ void __launch_bounds__(32) k_normalize(const uint32_t* __restrict__ accs, int count, int stride, uint32_t* __restrict__ out_xy, uint32_t* __restrict__ out_flag) {
  if (blockIdx.x != 0) return;
  const typename CV::acc res = count == 1 ? CV::ld_acc(accs) : CV::sum_partials_warp(accs, count, stride);
  Fe<typename CV::P> x, y;
  bool inf;
  CV::acc_to_plain_warp(res, x, y, inf);
  if (threadIdx.x == 0) {
    _Pragma("unroll") for (int i = 0; i < CV::N; i++) { out_xy[i] = x.v[i]; out_xy[CV::N + i] = y.v[i]; }
    out_flag[0] = inf ? 1u : 0u;
    uint32_t failed = 0;
    if (stride > CV::ACC_LIMBS)
      for (int i = 0; i < count; i++) failed |= accs[(size_t)i * stride + CV::ACC_LIMBS];
    out_flag[1] = failed;
  }
}

// ---------------------------------------------------------------- point ingestion / generation
template <class FP>
MGB_DEV bool below_modulus(const Fe<FP>& a) {   // a < p, on the raw limbs
  uint32_t borrow = 0;
  _Pragma("unroll") for (int i = 0; i < FP::N; i++) borrow = (uint32_t)(((uint64_t)a.v[i] - FP::mod(i) - borrow) >> 32) & 1u;
  return borrow != 0;
}
// CHECK (mgb_set_points_checked): also status[i] = PT_NONCANONICAL when x or y >= p, else 0 -- k_check_points then adds
// the curve and subgroup bits.  A point flagged as zero is valid whatever its coordinate bytes are.
template <class CV, bool CHECK = false>
__global__ void __launch_bounds__(128) k_set_points(uint32_t n, const uint32_t* __restrict__ xy, const uint8_t* __restrict__ is_zero, uint32_t* __restrict__ table,
                                                    uint8_t* __restrict__ status = nullptr) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fe<typename CV::P> x = ld_fe<typename CV::P>(xy + (size_t)i * 2 * CV::N), y = ld_fe<typename CV::P>(xy + (size_t)i * 2 * CV::N + CV::N);
  const bool inf = is_zero ? is_zero[i] != 0 : false;
  CV::make_entry(table + (size_t)i * CV::ENTRY_LIMBS, x, y, inf);
  if (CHECK) status[i] = inf || (below_modulus(x) && below_modulus(y)) ? 0 : (uint8_t)PT_NONCANONICAL;
}
// The curve and subgroup checks of mgb_set_points_checked over the resident table, one thread per point.  A point that
// k_set_points<CV, true> found non-canonical keeps that bit alone (its entry holds the coordinates mod p, not the input).
// counters[0] += number of invalid points; counters[1] = max(counters[1], ~index): the largest complement is that of
// the first invalid index (0: none).  The minimum of three blocks per SM keeps 12 warps resident (3 per scheduler):
// the chains are throughput-bound products (DESIGN.md §3).
template <class CV>
__global__ void __launch_bounds__(128, 3) k_check_points(uint32_t n, const uint32_t* __restrict__ table, uint8_t* __restrict__ status, uint32_t* __restrict__ counters) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t s = status[i];
  if (s == 0) {
    s = CV::check_entry(table + (size_t)i * CV::ENTRY_LIMBS);
    status[i] = (uint8_t)s;
  }
  if (s) {
    atomicAdd(&counters[0], 1u);
    atomicMax(&counters[1], ~i);
  }
}
template <class CV>
__global__ void __launch_bounds__(128) k_get_points(uint32_t first, uint32_t n, const uint32_t* __restrict__ table, uint32_t* __restrict__ xy, uint8_t* __restrict__ is_zero) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fe<typename CV::P> x, y;
  bool inf;
  CV::entry_to_plain(table + (size_t)(first + i) * CV::ENTRY_LIMBS, x, y, inf);
  st_fe<typename CV::P>(xy + (size_t)i * 2 * CV::N, x);
  st_fe<typename CV::P>(xy + (size_t)i * 2 * CV::N + CV::N, y);
  if (is_zero) is_zero[i] = inf ? 1 : 0;
}

MGB_DEV uint64_t splitmix64(uint64_t seed, uint64_t i) {
  uint64_t z = seed + (i + 1) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// P_i = a_i * G, a_i = splitmix64(seed, i) | 1-if-zero  (known discrete logs: closed-form checks)
template <class CV>
__global__ void __launch_bounds__(128) k_random_points(uint32_t n, uint64_t seed, uint32_t* __restrict__ table) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t a = splitmix64(seed, i);
  if (a == 0) a = 1;
  typename CV::acc g = CV::generator(), res = CV::acc_zero();
  for (int bit = 63; bit >= 0; bit--) {
    res = CV::dbl(res);
    if ((a >> bit) & 1) res = CV::add(res, g);
  }
  CV::make_entry_from_acc(table + (size_t)i * CV::ENTRY_LIMBS, res);
}

}  // namespace mgb
