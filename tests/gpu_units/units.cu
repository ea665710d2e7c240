// TEST-ONLY: the engine's device code (field.cuh, warp.cuh, ec.cuh, coop.cuh, onewarp.cuh, engine.cuh) run on the GPU one
// unit at a time, so that tests/test_gpu_units.py can check each against the oracle the way tests/host_emu checks the
// same source on the CPU.  Every entry point is the batched twin of an emu_* entry point of tests/host_emu/emu_lib.cpp or
// emu_kernels.cpp: the same operation codes and the same raw Montgomery-form operand layout, but n cases per launch (one
// per lane, 16- / 8-lane group, quad or warp, the way the engine uses the routine).  Each copies its inputs to device 0
// (cudaMalloc + cudaMemcpy), launches, synchronises, copies the results back and returns the cudaError_t as an int.
// Compiled with the product's nvcc flags (montgomery_b200.build.NVCC_FLAGS + MGB_NVCC_EXTRA); never linked into the
// product library.
#include <cstring>
#include <vector>
#include "../../montgomery_b200/csrc/engine.cuh"

// the production tile bounds of k_batch_add (same defaults and overrides as csrc/msm.cu)
#ifndef MGB_MINB
#define MGB_MINB 4
#endif
#ifndef MGB_EMAX
#define MGB_EMAX 64
#endif

using namespace mgb;

namespace {

#define CK(x) do { const cudaError_t e_ = (x); if (e_ != cudaSuccess) return (int)e_; } while (0)

// a device buffer, freed on every return path
struct Buf {
  void* d = nullptr;
  Buf() = default;
  Buf(const Buf&) = delete;
  ~Buf() { if (d) cudaFree(d); }
  template <class T> T* as() const { return reinterpret_cast<T*>(d); }
};
// `count` elements; from the host array h, or zero-filled when h is NULL
template <class T> int up(Buf& b, const T* h, size_t count) {
  const size_t bytes = std::max<size_t>(16, count * sizeof(T));
  CK(cudaMalloc(&b.d, bytes));
  if (h) CK(cudaMemcpy(b.d, h, count * sizeof(T), cudaMemcpyHostToDevice));
  else CK(cudaMemset(b.d, 0, bytes));
  return 0;
}
template <class T> int down(T* h, const Buf& b, size_t count) {
  if (h) CK(cudaMemcpy(h, b.d, count * sizeof(T), cudaMemcpyDeviceToHost));
  return 0;
}
int launched() {
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  return 0;
}
#define UP(b, h, n) do { const int rc_ = up(b, h, n); if (rc_) return rc_; } while (0)
#define DOWN(h, b, n) do { const int rc_ = down(h, b, n); if (rc_) return rc_; } while (0)
#define LAUNCHED() do { const int rc_ = launched(); if (rc_) return rc_; } while (0)

unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }
int sm_count() {
  int v = 0;
  cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, 0);
  return v > 0 ? v : 1;
}

template <class T> struct Tag { typedef T type; };
// field ids of emu_fe_op: 0 = BLS12-377 Fp, 1 = BLS12-377 Fr, 2 = Pallas Fp, 3 = BLS12-381 Fp
template <class Fn> int with_field(int f, Fn fn) {
  switch (f) {
    case 0: return fn(Tag<Fp377>());
    case 1: return fn(Tag<Fr377>());
    case 2: return fn(Tag<FpPallas>());
    case 3: return fn(Tag<Fp381>());
  }
  return (int)cudaErrorInvalidValue;
}
// Weierstrass curve ids of emu_w_op: 0 = BLS12-377, 1 = Pallas, 2 = BLS12-381 (base fields)
template <class Fn> int with_wfield(int c, Fn fn) {
  switch (c) {
    case 0: return fn(Tag<Fp377>());
    case 1: return fn(Tag<FpPallas>());
    case 2: return fn(Tag<Fp381>());
  }
  return (int)cudaErrorInvalidValue;
}
// curve policies of emu_kernels.cpp: 0 = BLS12-377, 1 = Pallas, 2 = BLS12-381, 3 = ed-on-BLS12-377
template <class Fn> int with_curve(int c, Fn fn) {
  switch (c) {
    case 0: return fn(Tag<CurveBls377>());
    case 1: return fn(Tag<CurvePallas>());
    case 2: return fn(Tag<CurveBls381>());
    case 3: return fn(Tag<CurveEd377>());
  }
  return (int)cudaErrorInvalidValue;
}

// ---------------------------------------------------------------- one case per thread
template <class P>
__global__ void __launch_bounds__(128) k_fe_op(int op, uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                                               uint32_t* __restrict__ out) {
  typedef Field<P> F;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Fe<P> x = ld_fe<P>(a + (size_t)i * P::N), y = ld_fe<P>(b + (size_t)i * P::N);
  Fe<P> r;
  switch (op) {
    case 0: r = F::mul(x, y); break;
    case 1: r = F::add(x, y); break;
    case 2: r = F::sub(x, y); break;
    case 3: r = F::inv(x); break;
    case 4: r = F::to_mont(x); break;
    case 5: r = F::from_mont(x); break;
    case 6: r = F::sqr(x); break;
    case 7: r = F::neg(x); break;
    case 8: r = F::inv_bgcd(x); break;
    case 9: r = F::inv_divsteps(x); break;
    default: r = F::zero();
  }
  st_fe<P>(out + (size_t)i * P::N, r);
}

// Weierstrass ops of emu_w_op; every operand and result takes 4N limbs (affine: x | y, infinity flag in x's top bit)
template <class P>
__global__ void __launch_bounds__(128) k_w_op(int op, uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                                              uint32_t* __restrict__ out) {
  typedef Weierstrass<P> W;
  typedef Field<P> F;
  constexpr int N = P::N;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* pa = a + (size_t)i * 4 * N;
  const uint32_t* pb = b + (size_t)i * 4 * N;
  uint32_t* po = out + (size_t)i * 4 * N;
  auto lda = [&](const uint32_t* p) { typename W::affine r; r.x = ld_fe<P>(p); r.y = ld_fe<P>(p + N); return r; };
  auto ldx = [&](const uint32_t* p) { typename W::acc r; r.X = ld_fe<P>(p); r.Y = ld_fe<P>(p + N); r.ZZ = ld_fe<P>(p + 2 * N); r.ZZZ = ld_fe<P>(p + 3 * N); return r; };
  auto sta = [&](const typename W::affine& r) { st_fe<P>(po, r.x); st_fe<P>(po + N, r.y); };
  auto stx = [&](const typename W::acc& r) { st_fe<P>(po, r.X); st_fe<P>(po + N, r.Y); st_fe<P>(po + 2 * N, r.ZZ); st_fe<P>(po + 3 * N, r.ZZZ); };
  switch (op) {
    case 0: {  // affine + affine through prepare / invert / finish
      const auto A = lda(pa), B = lda(pb);
      Fe<P> den;
      const int kind = W::add_prepare(A, B, den);
      sta(W::add_finish(kind, A, B, F::inv(den)));
      break;
    }
    case 1: stx(W::madd(ldx(pa), lda(pb))); break;
    case 2: stx(W::add(ldx(pa), ldx(pb))); break;
    case 3: stx(W::dbl(ldx(pa))); break;
    case 4: sta(W::to_affine(ldx(pa))); break;
    case 5: stx(W::from_affine(lda(pa))); break;
  }
}

// extended twisted-Edwards ops of emu_te_op (ed-on-BLS12-377); 4N limbs per operand and result (affine: x | y | k t)
__global__ void __launch_bounds__(128) k_te_op(int op, uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                                               uint32_t* __restrict__ out) {
  typedef Fr377 P;
  typedef TwistedEdwards<P, Ed377Consts> T;
  constexpr int N = P::N;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* pa = a + (size_t)i * 4 * N;
  const uint32_t* pb = b + (size_t)i * 4 * N;
  uint32_t* po = out + (size_t)i * 4 * N;
  auto lde = [&](const uint32_t* p) { typename T::acc r; r.X = ld_fe<P>(p); r.Y = ld_fe<P>(p + N); r.Z = ld_fe<P>(p + 2 * N); r.T = ld_fe<P>(p + 3 * N); return r; };
  auto lda = [&](const uint32_t* p) { typename T::affine r; r.x = ld_fe<P>(p); r.y = ld_fe<P>(p + N); r.kt = ld_fe<P>(p + 2 * N); return r; };
  auto ste = [&](const typename T::acc& r) { st_fe<P>(po, r.X); st_fe<P>(po + N, r.Y); st_fe<P>(po + 2 * N, r.Z); st_fe<P>(po + 3 * N, r.T); };
  switch (op) {
    case 0: ste(T::add(lde(pa), lde(pb))); break;
    case 1: ste(T::madd(lde(pa), lda(pb))); break;
    case 2: ste(T::add_affine(lda(pa), lda(pb))); break;
    case 3: ste(T::dbl(lde(pa))); break;
    case 4: { Fe<P> x, y; T::to_affine(lde(pa), x, y); st_fe<P>(po, x); st_fe<P>(po + N, y); break; }
  }
}

// ---------------------------------------------------------------- warp-cooperative field arithmetic (warp.cuh)
// one element per 16-lane group; out holds all 16 lanes of an element (lanes N..15 must return 0).  Lanes above the top
// limb pass garbage on purpose; groups past n run the shuffles on zeros.
template <class P>
__global__ void __launch_bounds__(128) k_warp_mul(uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out) {
  constexpr int N = P::N;
  const uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  const int l = threadIdx.x & 15;
  const bool live = e < n && l < N;
  const uint32_t x = live ? a[(size_t)e * N + l] : (e < n ? 0xdeadbeefu : 0u), y = live ? b[(size_t)e * N + l] : 0x12345678u;
  const uint32_t r = WarpField<P>::mul(x, y);
  if (e < n) out[(size_t)e * 16 + l] = r;
}

// one element per 8-lane group (two limbs per lane); out holds all 8 lanes (16 words) of an element
template <class P>
__global__ void __launch_bounds__(128) k_warp_mul2(uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out) {
  constexpr int N = P::N, D = N / 2;
  typedef unsigned long long u64;
  const uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int l = threadIdx.x & 7;
  const bool live = e < n && l < D;
  const u64 x = live ? (((u64)a[(size_t)e * N + 2 * l + 1] << 32) | a[(size_t)e * N + 2 * l]) : (e < n ? 0xdeadbeefcafef00dull : 0ull);
  const u64 y = live ? (((u64)b[(size_t)e * N + 2 * l + 1] << 32) | b[(size_t)e * N + 2 * l]) : 0x123456789abcdef0ull;
  const u64 r = WarpField2<P>::mul(x, y);
  if (e < n) { out[(size_t)e * 16 + 2 * l] = (uint32_t)r; out[(size_t)e * 16 + 2 * l + 1] = (uint32_t)(r >> 32); }
}

// op 0: a + b, 1: a - b, 2: 2a, 3: (a == 0) on elements spread over 8-lane groups; out as k_warp_mul2
template <class P>
__global__ void __launch_bounds__(128) k_warp_addsub2(int op, uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out) {
  constexpr int N = P::N, D = N / 2;
  typedef unsigned long long u64;
  typedef WarpField2<P> WF;
  const uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int l = threadIdx.x & 7;
  const bool live = e < n && l < D;
  const u64 x = live ? (((u64)a[(size_t)e * N + 2 * l + 1] << 32) | a[(size_t)e * N + 2 * l]) : 0ull;
  const u64 y = live ? (((u64)b[(size_t)e * N + 2 * l + 1] << 32) | b[(size_t)e * N + 2 * l]) : 0ull;
  const u64 r = op == 0 ? WF::add(x, y) : op == 1 ? WF::sub(x, y) : op == 2 ? WF::dbl(x) : (u64)WF::is_zero(x);
  if (e < n) { out[(size_t)e * 16 + 2 * l] = (uint32_t)r; out[(size_t)e * 16 + 2 * l + 1] = (uint32_t)(r >> 32); }
}

// the carry / borrow resolutions alone: thread t gets t[t] and c[t] (one warp = two or four elements)
template <class P>
__global__ void __launch_bounds__(128) k_warp_finish(uint32_t nthreads, const uint32_t* __restrict__ t, const uint64_t* __restrict__ c, uint32_t* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < nthreads;
  const uint32_t r = WarpField<P>::finish(live ? t[i] : 0u, live ? c[i] : 0ull);
  if (live) out[i] = r;
}
template <class P>
__global__ void __launch_bounds__(128) k_warp_finish2(uint32_t nthreads, const uint64_t* __restrict__ t, const uint64_t* __restrict__ clo,
                                                      const uint32_t* __restrict__ chi, uint64_t* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < nthreads;
  const uint64_t r = WarpField2<P>::finish(live ? t[i] : 0ull, live ? clo[i] : 0ull, live ? chi[i] : 0u);
  if (live) out[i] = r;
}

// one inversion per WARP through WarpField::inv_call (what k_batch_add and the normalisations run), every lane passing
// the same element; every lane's result is returned: out[(e * 32 + lane) * N]
template <class P>
__global__ void __launch_bounds__(128) k_warp_inv(uint32_t n, const uint32_t* __restrict__ a, uint32_t* __restrict__ out) {
  const uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const Fe<P> x = e < n ? ld_fe<P>(a + (size_t)e * P::N) : Field<P>::zero();
  const Fe<P> r = WarpField<P>::inv_call(x);
  if (e < n) st_fe<P>(out + ((size_t)e * 32 + (threadIdx.x & 31)) * P::N, r);
}

// ---------------------------------------------------------------- point arithmetic shared by lanes
// QuadWeierstrass::add: lane 4j + k of a warp holds coordinate k of its j-th addition; 32 elements per warp
template <class P>
__global__ void __launch_bounds__(128) k_quad_add(uint32_t nwarps, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if ((i >> 5) >= nwarps) return;                     // whole warps only
  const Fe<P> x = ld_fe<P>(a + (size_t)i * P::N), y = ld_fe<P>(b + (size_t)i * P::N);
  st_fe<P>(out + (size_t)i * P::N, QuadWeierstrass<P>::add(x, y));
}

// onewarp.cuh, one case per warp: op 0: P <- 2^count P, op 1: P <- P + Q, op 2: P <- 2^count P + Q (one Horner step).
// a, b, out: 4N limbs per case; a different lane of each warp stores its copy of the result.
template <class CV>
__global__ void __launch_bounds__(128) k_onewarp(int op, int count, uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                                                 uint32_t* __restrict__ out) {
  typedef typename CV::OneWarp OW;
  const uint32_t e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (e >= n) return;                                 // whole warps only
  auto v = OW::spread(CV::ld_acc(a + (size_t)e * CV::ACC_LIMBS));
  const auto q = OW::spread(CV::ld_acc(b + (size_t)e * CV::ACC_LIMBS));
  if (op == 0 || op == 2) for (int i = 0; i < count; i++) v = OW::dbl(v);
  if (op == 1 || op == 2) v = OW::add(v, q);
  const auto r = OW::gather(v);
  if ((threadIdx.x & 31) == ((e * 7u + 3u) & 31u)) CV::st_acc(out + (size_t)e * CV::ACC_LIMBS, r);
}

}  // namespace

extern "C" {

// ops 0-9 of emu_fe_op on n stored (Montgomery-form) operand pairs, one per thread
int gpu_fe_op(int field, int op, uint32_t* out, const uint32_t* a, const uint32_t* b, int n) {
  CK(cudaSetDevice(0));
  return with_field(field, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    const size_t w = (size_t)n * P::N;
    Buf da, db, dout;
    UP(da, a, w); UP(db, b, w); UP(dout, (const uint32_t*)nullptr, w);
    k_fe_op<P><<<cdiv(n, 128), 128>>>(op, (uint32_t)n, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, w);
    return 0;
  });
}

// emu_w_op with n cases; a, b, out: 4N limbs per case
int gpu_w_op(int curve, int op, uint32_t* out, const uint32_t* a, const uint32_t* b, int n) {
  CK(cudaSetDevice(0));
  return with_wfield(curve, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    const size_t w = (size_t)n * 4 * P::N;
    Buf da, db, dout;
    UP(da, a, w); UP(db, b, w); UP(dout, (const uint32_t*)nullptr, w);
    k_w_op<P><<<cdiv(n, 128), 128>>>(op, (uint32_t)n, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, w);
    return 0;
  });
}

// emu_te_op with n cases; a, b, out: 4N limbs per case
int gpu_te_op(int op, uint32_t* out, const uint32_t* a, const uint32_t* b, int n) {
  CK(cudaSetDevice(0));
  const size_t w = (size_t)n * 4 * Fr377::N;
  Buf da, db, dout;
  UP(da, a, w); UP(db, b, w); UP(dout, (const uint32_t*)nullptr, w);
  k_te_op<<<cdiv(n, 128), 128>>>(op, (uint32_t)n, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
  LAUNCHED();
  DOWN(out, dout, w);
  return 0;
}

// n products, one per 16-lane group; out: 16 words per product (lanes N..15 must come back 0)
int gpu_warp_mul(int field, uint32_t* out, const uint32_t* a, const uint32_t* b, int n) {
  CK(cudaSetDevice(0));
  return with_field(field, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    Buf da, db, dout;
    UP(da, a, (size_t)n * P::N); UP(db, b, (size_t)n * P::N); UP(dout, (const uint32_t*)nullptr, (size_t)n * 16);
    k_warp_mul<P><<<cdiv((size_t)n * 16, 128), 128>>>((uint32_t)n, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, (size_t)n * 16);
    return 0;
  });
}

// n products, one per 8-lane group (WarpField2); out: 16 words per product (digits D..7 must come back 0)
int gpu_warp_mul2(int field, uint32_t* out, const uint32_t* a, const uint32_t* b, int n) {
  CK(cudaSetDevice(0));
  return with_field(field, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    Buf da, db, dout;
    UP(da, a, (size_t)n * P::N); UP(db, b, (size_t)n * P::N); UP(dout, (const uint32_t*)nullptr, (size_t)n * 16);
    k_warp_mul2<P><<<cdiv((size_t)n * 8, 128), 128>>>((uint32_t)n, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, (size_t)n * 16);
    return 0;
  });
}

int gpu_warp_addsub2(int field, int op, uint32_t* out, const uint32_t* a, const uint32_t* b, int n) {
  CK(cudaSetDevice(0));
  return with_field(field, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    Buf da, db, dout;
    UP(da, a, (size_t)n * P::N); UP(db, b, (size_t)n * P::N); UP(dout, (const uint32_t*)nullptr, (size_t)n * 16);
    k_warp_addsub2<P><<<cdiv((size_t)n * 8, 128), 128>>>(op, (uint32_t)n, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, (size_t)n * 16);
    return 0;
  });
}

// emu_warp_finish over nwarps warps: t, c, out hold 32 entries per warp
int gpu_warp_finish(int field, uint32_t* out, const uint32_t* t, const uint64_t* c, int nwarps) {
  CK(cudaSetDevice(0));
  return with_field(field, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    const size_t m = (size_t)nwarps * 32;
    Buf dt, dc, dout;
    UP(dt, t, m); UP(dc, c, m); UP(dout, (const uint32_t*)nullptr, m);
    k_warp_finish<P><<<cdiv(m, 128), 128>>>((uint32_t)m, dt.as<uint32_t>(), dc.as<uint64_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, m);
    return 0;
  });
}

int gpu_warp_finish2(int field, uint64_t* out, const uint64_t* t, const uint64_t* clo, const uint32_t* chi, int nwarps) {
  CK(cudaSetDevice(0));
  return with_field(field, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    const size_t m = (size_t)nwarps * 32;
    Buf dt, dl, dh, dout;
    UP(dt, t, m); UP(dl, clo, m); UP(dh, chi, m); UP(dout, (const uint64_t*)nullptr, m);
    k_warp_finish2<P><<<cdiv(m, 128), 128>>>((uint32_t)m, dt.as<uint64_t>(), dl.as<uint64_t>(), dh.as<uint32_t>(), dout.as<uint64_t>());
    LAUNCHED();
    DOWN(out, dout, m);
    return 0;
  });
}

// n inversions through WarpField::inv_call, one per warp; out: 32 copies (one per lane) of N limbs per element
int gpu_warp_inv(int field, uint32_t* out, const uint32_t* a, int n) {
  CK(cudaSetDevice(0));
  return with_field(field, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    Buf da, dout;
    UP(da, a, (size_t)n * P::N); UP(dout, (const uint32_t*)nullptr, (size_t)n * 32 * P::N);
    k_warp_inv<P><<<cdiv((size_t)n * 32, 128), 128>>>((uint32_t)n, da.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, (size_t)n * 32 * P::N);
    return 0;
  });
}

// emu_quad_add over nwarps warps: 32 field elements (8 XYZZ points) per warp in a, b and out
int gpu_quad_add(int curve, uint32_t* out, const uint32_t* a, const uint32_t* b, int nwarps) {
  CK(cudaSetDevice(0));
  return with_wfield(curve, [&](auto tag) -> int {
    typedef typename decltype(tag)::type P;
    const size_t w = (size_t)nwarps * 32 * P::N;
    Buf da, db, dout;
    UP(da, a, w); UP(db, b, w); UP(dout, (const uint32_t*)nullptr, w);
    k_quad_add<P><<<cdiv((size_t)nwarps * 32, 128), 128>>>((uint32_t)nwarps, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, w);
    return 0;
  });
}

// emu_onewarp_w / emu_onewarp_te with n cases, one per warp (4N limbs per operand and result)
int gpu_onewarp(int curve, int op, int count, uint32_t* out, const uint32_t* a, const uint32_t* b, int n) {
  CK(cudaSetDevice(0));
  return with_curve(curve, [&](auto tag) -> int {
    typedef typename decltype(tag)::type CV;
    const size_t w = (size_t)n * CV::ACC_LIMBS;
    Buf da, db, dout;
    UP(da, a, w); UP(db, b, w); UP(dout, (const uint32_t*)nullptr, w);
    k_onewarp<CV><<<cdiv((size_t)n * 32, 128), 128>>>(op, count, (uint32_t)n, da.as<uint32_t>(), db.as<uint32_t>(), dout.as<uint32_t>());
    LAUNCHED();
    DOWN(out, dout, w);
    return 0;
  });
}

// One round of k_batch_add<CV, MGB_EMAX, MGB_MINB, FIRST> (curves 0-2) on the caller's buffers, launched the way msm.cu
// launches it: #SM x MINB blocks of 128 threads (blocks = 0), its shared-memory carve-out, per-warp scratch.  first = 1:
// round 0 over recs / lifes / table / offs; first = 0: round r over `pairs` (npairs_in entries).  V (v_words) and
// *npairs_out are read and written back; pairs_out has room for pairs_cap entries.
int gpu_batch_add(int curve, int first, uint32_t* V, size_t v_words, const uint32_t* pairs, uint32_t npairs_in, int r, int E_big,
                  uint32_t n_big, uint32_t* pairs_out, size_t pairs_cap, uint32_t* npairs_out, const uint32_t* recs, size_t nrecs,
                  const uint8_t* lifes, size_t nlifes, const uint32_t* table, size_t table_words, const uint32_t* offs, uint32_t b_begin,
                  uint32_t b_end, int blocks) {
  CK(cudaSetDevice(0));
  if (curve < 0 || curve > 2 || E_big < 1 || E_big > MGB_EMAX) return (int)cudaErrorInvalidValue;
  return with_curve(curve, [&](auto tag) -> int {
    typedef typename decltype(tag)::type CV;
    if constexpr (!CV::BATCH_AFFINE) {
      return (int)cudaErrorInvalidValue;
    } else {
      constexpr int EMAX = MGB_EMAX, MINB = MGB_MINB;
      const int nb = blocks > 0 ? blocks : sm_count() * MINB;
      if (nb % MINB) return (int)cudaErrorInvalidValue;       // the static first tile assumes MINB blocks per SM
      const size_t scratch_chunks = (size_t)nb * 4 * EMAX * (CV::N / 4) * 32;
      Buf dV, dpairs, dnin, dpout, dnout, dtiles, drecs, dlifes, dtable, doffs, dscratch;
      UP(dV, V, v_words);
      UP(dpout, (const uint32_t*)nullptr, 2 * pairs_cap);
      UP(dnout, npairs_out, 1);
      UP(dtiles, (const uint32_t*)nullptr, 1);
      UP(dscratch, (const uint4*)nullptr, scratch_chunks);
      const int E_small = E_big >= 16 ? E_big / 4 : E_big;
      if (first) {
        std::vector<uint8_t> lf(lifes, lifes + nlifes);
        lf.resize((nlifes + 3) & ~(size_t)3, 0);               // read as whole words
        UP(drecs, recs, 2 * nrecs); UP(dlifes, lf.data(), lf.size()); UP(dtable, table, table_words); UP(doffs, offs, (size_t)b_end + 1);
        auto kern = k_batch_add<CV, EMAX, MINB, true>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, MINB > 4 ? 90 : 75));
        kern<<<nb, 128>>>(dV.as<uint32_t>(), nullptr, nullptr, r, E_big, E_small, n_big, dpout.as<PairEnt>(), dnout.as<uint32_t>(),
                          dtiles.as<uint32_t>(), drecs.as<const uint2>(), dlifes.as<const uint8_t>(), dtable.as<const uint32_t>(),
                          doffs.as<const uint32_t>(), b_begin, b_end, dscratch.as<uint4>());
      } else {
        UP(dpairs, pairs, 2 * (size_t)npairs_in); UP(dnin, &npairs_in, 1);
        auto kern = k_batch_add<CV, EMAX, MINB, false>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, MINB > 4 ? 90 : 75));
        kern<<<nb, 128>>>(dV.as<uint32_t>(), dpairs.as<const PairEnt>(), dnin.as<const uint32_t>(), r, E_big, E_small, n_big,
                          dpout.as<PairEnt>(), dnout.as<uint32_t>(), dtiles.as<uint32_t>(), nullptr, nullptr, nullptr, nullptr, 0, 0,
                          dscratch.as<uint4>());
      }
      LAUNCHED();
      DOWN(V, dV, v_words);
      DOWN(npairs_out, dnout, 1);
      DOWN(pairs_out, dpout, 2 * pairs_cap);
      return 0;
    }
  });
}

// one tree round of k_pair_add<CurveEd377, FIRST>, launched as msm.cu does (#SM x 8 blocks of 256 threads); buffers as
// gpu_batch_add
int gpu_pair_add_te(int first, uint32_t* V, size_t v_words, const uint32_t* pairs, uint32_t npairs_in, int r, uint32_t* pairs_out,
                    size_t pairs_cap, uint32_t* npairs_out, const uint32_t* recs, size_t nrecs, const uint8_t* lifes, size_t nlifes,
                    const uint32_t* table, size_t table_words, const uint32_t* offs, uint32_t b_begin, uint32_t b_end) {
  CK(cudaSetDevice(0));
  typedef CurveEd377 CV;
  Buf dV, dpairs, dnin, dpout, dnout, drecs, dlifes, dtable, doffs;
  UP(dV, V, v_words);
  UP(dpout, (const uint32_t*)nullptr, 2 * pairs_cap);
  UP(dnout, npairs_out, 1);
  const unsigned nb = (unsigned)sm_count() * 8;
  if (first) {
    UP(drecs, recs, 2 * nrecs); UP(dlifes, lifes, nlifes); UP(dtable, table, table_words); UP(doffs, offs, (size_t)b_end + 1);
    k_pair_add<CV, true><<<nb, 256>>>(dV.as<uint32_t>(), nullptr, nullptr, r, dpout.as<PairEnt>(), dnout.as<uint32_t>(), drecs.as<const uint2>(),
                                      dlifes.as<const uint8_t>(), dtable.as<const uint32_t>(), doffs.as<const uint32_t>(), b_begin, b_end);
  } else {
    UP(dpairs, pairs, 2 * (size_t)npairs_in); UP(dnin, &npairs_in, 1);
    k_pair_add<CV, false><<<nb, 256>>>(dV.as<uint32_t>(), dpairs.as<const PairEnt>(), dnin.as<const uint32_t>(), r, dpout.as<PairEnt>(),
                                       dnout.as<uint32_t>(), nullptr, nullptr, nullptr, nullptr, 0, 0);
  }
  LAUNCHED();
  DOWN(V, dV, v_words);
  DOWN(npairs_out, dnout, 1);
  DOWN(pairs_out, dpout, 2 * pairs_cap);
  return 0;
}

// emu_final: k_final<CV> (one warp) over K window sums; out_xy (2N words) and out_flag (1 word) may be NULL
int gpu_final(int curve, int K, int c, const uint32_t* Sw, uint32_t* out_acc, uint32_t* out_xy, uint32_t* out_flag) {
  CK(cudaSetDevice(0));
  return with_curve(curve, [&](auto tag) -> int {
    typedef typename decltype(tag)::type CV;
    Buf dS, dacc, dxy;
    UP(dS, Sw, (size_t)K * CV::ACC_LIMBS); UP(dacc, (const uint32_t*)nullptr, CV::ACC_LIMBS);
    if (out_xy) UP(dxy, (const uint32_t*)nullptr, 2 * CV::N + 1);
    k_final<CV><<<1, 32>>>(K, c, dS.as<const uint32_t>(), dacc.as<uint32_t>(), out_xy ? dxy.as<uint32_t>() : nullptr,
                           out_xy ? dxy.as<uint32_t>() + 2 * CV::N : nullptr);
    LAUNCHED();
    DOWN(out_acc, dacc, CV::ACC_LIMBS);
    if (out_xy) {
      DOWN(out_xy, dxy, 2 * CV::N);
      std::vector<uint32_t> all(2 * CV::N + 1);
      DOWN(all.data(), dxy, all.size());
      if (out_flag) *out_flag = all[2 * CV::N];
    }
    return 0;
  });
}

// emu_set_get_points: k_set_points then k_get_points over n points (is_zero may be NULL)
int gpu_set_get_points(int curve, uint32_t n, const uint32_t* xy, const uint8_t* is_zero, uint32_t* table, uint32_t* xy_back, uint8_t* zero_back) {
  CK(cudaSetDevice(0));
  return with_curve(curve, [&](auto tag) -> int {
    typedef typename decltype(tag)::type CV;
    Buf dxy, dz, dtable, dback, dzback;
    UP(dxy, xy, (size_t)n * 2 * CV::N);
    if (is_zero) UP(dz, is_zero, n);
    UP(dtable, (const uint32_t*)nullptr, (size_t)n * CV::ENTRY_LIMBS);
    UP(dback, (const uint32_t*)nullptr, (size_t)n * 2 * CV::N);
    UP(dzback, (const uint8_t*)nullptr, n);
    k_set_points<CV><<<cdiv(n, 128), 128>>>(n, dxy.as<const uint32_t>(), is_zero ? dz.as<const uint8_t>() : nullptr, dtable.as<uint32_t>());
    LAUNCHED();
    k_get_points<CV><<<cdiv(n, 128), 128>>>(0, n, dtable.as<const uint32_t>(), dback.as<uint32_t>(), dzback.as<uint8_t>());
    LAUNCHED();
    DOWN(table, dtable, (size_t)n * CV::ENTRY_LIMBS);
    DOWN(xy_back, dback, (size_t)n * 2 * CV::N);
    DOWN(zero_back, dzback, n);
    return 0;
  });
}

// emu_normalize: k_normalize<CV> over `count` accumulators `stride` limbs apart; out_flag: 2 words
int gpu_normalize(int curve, const uint32_t* accs, int count, int stride, uint32_t* out_xy, uint32_t* out_flag) {
  CK(cudaSetDevice(0));
  return with_curve(curve, [&](auto tag) -> int {
    typedef typename decltype(tag)::type CV;
    Buf da, dxy, dflag;
    UP(da, accs, (size_t)count * stride);
    UP(dxy, (const uint32_t*)nullptr, 2 * CV::N);
    UP(dflag, (const uint32_t*)nullptr, 2);
    k_normalize<CV><<<1, 32>>>(da.as<const uint32_t>(), count, stride, dxy.as<uint32_t>(), dflag.as<uint32_t>());
    LAUNCHED();
    DOWN(out_xy, dxy, 2 * CV::N);
    DOWN(out_flag, dflag, 2);
    return 0;
  });
}

// the tile bounds this harness instantiated k_batch_add with
int gpu_batch_add_emax() { return MGB_EMAX; }
int gpu_batch_add_minb() { return MGB_MINB; }

}  // extern "C"
