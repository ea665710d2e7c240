// Host orchestration + C ABI of the MSM engine (see include/montgomery_b200.h).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include <mutex>
#include <thread>
#include <dlfcn.h>
#include <nccl.h>      // types only: the library is bound at run time (dlopen), see NcclApi
#include "engine.cuh"
#include "../../include/montgomery_b200.h"

using namespace mgb;

// k_batch_add shape: pairs per lane of the largest tile, resident blocks per SM (build-time knobs for experiments)
#ifndef MGB_MINB
#define MGB_MINB 4
#endif
#ifndef MGB_EMAX
#define MGB_EMAX 64
#endif

namespace {

thread_local std::string g_last_error;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

enum Ev { EV_START, EV_H2D, EV_DIGITS, EV_SORT, EV_ACC, EV_REDUCE, EV_FINAL, EV_COUNT };

}  // namespace

struct mgb_ctx {
  int curve = 0, device = 0;
  size_t max_points = 0, npoints = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t aux[3] = {};          // extra streams: window groups are pipelined against each other
  cudaEvent_t ev_fork = nullptr, ev_plan = nullptr, ev_join[3] = {}, ev_chunk[4] = {};
  cudaEvent_t ev[EV_COUNT] = {};
  DevBuf table, scalars, ent_bucket, ent_rank, counts, offs, offcnt, tile_sums, pairs, pairs2, V, W, recs, lifes, prebuf, bsum, redU[2], redW[2], misc, acc_out, out_xy, stage;
  DevBuf checks;                 // mgb_set_points_checked only: two counters, then one status byte per point
  uint32_t* h_pinned = nullptr;  // [0..31] out xy limbs + flag, [64..] misc readback
  int sm_count = 148;
  std::string err;
  // multi-GPU: the context owns its NCCL communicator (mgb_comm_init / mgb_multi_create)
  ncclComm_t comm = nullptr;
  int comm_rank = 0, comm_world = 1;
  DevBuf gathered;               // comm_world partial accumulators, rank order
  // scalar sets uploaded ahead of their MSM (mgb_msm_prefetch): two slots, so that the set of call i + 1 can travel while call i runs
  struct Prefetch { DevBuf buf; const void* host = nullptr; size_t n = 0; cudaEvent_t ev = nullptr; bool valid = false, issued = false; } pf[2];
  cudaStream_t pf_stream = nullptr;
};

// one host process, several GPUs (mgb_multi_*): one context per device, communicators from ncclCommInitAll
struct mgb_multi {
  std::vector<mgb_ctx*> ctxs;
  std::vector<size_t> lo, hi;     // shard g holds the pairs [lo, hi) of the point set
  size_t npoints = 0;
  std::string err;
};

namespace {

int fail(mgb_ctx* ctx, int code, const std::string& msg) {
  g_last_error = msg;
  if (ctx) ctx->err = msg;
  return code;
}

// NCCL is bound at run time: a single-GPU host never needs it, and a host that already carries an NCCL (PyTorch ships
// its own libnccl.so.2) must share that copy rather than load a second one -- dlopen by SONAME returns the loaded one.
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommGetAsyncError)(ncclComm_t, ncclResult_t*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string err;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {getenv("MGB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      if (!nm || !*nm) continue;
      api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
      api.err = dlerror();
    }
    if (!api.handle) return;
    bool ok = true;
    auto sym = [&](const char* nm) -> void* { void* f = dlsym(api.handle, nm); if (!f) { ok = false; api.err = std::string("missing symbol ") + nm; } return f; };
    api.GetVersion = (decltype(api.GetVersion))sym("ncclGetVersion");
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.CommGetAsyncError = (decltype(api.CommGetAsyncError))sym("ncclCommGetAsyncError");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    if (!ok) { dlclose(api.handle); api.handle = nullptr; }
  });
  return api.handle ? &api : nullptr;
}

#define NC(ctx, api, call)                                                                    \
  do {                                                                                        \
    ncclResult_t r_ = (call);                                                                 \
    if (r_ != ncclSuccess)                                                                    \
      return fail(ctx, MGB_E_COMM, std::string(#call) + ": " + (api)->GetErrorString(r_));    \
  } while (0)

#define CU(ctx, call)                                                                         \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? MGB_E_NOMEM : MGB_E_CUDA,            \
                  std::string(#call) + ": " + cudaGetErrorString(e_));                        \
  } while (0)

int ensure(mgb_ctx* ctx, DevBuf& b, size_t bytes) {
  if (b.cap >= bytes) return 0;
  if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
  size_t want = bytes + bytes / 8 + 256;
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, MGB_E_NOMEM, std::string("device memory overflow: cudaMalloc(") + std::to_string(want) + ") " + cudaGetErrorString(e));
  }
  b.cap = want;
  return 0;
}
#define ENS(ctx, buf, bytes) do { int r_ = ensure(ctx, buf, bytes); if (r_) return r_; } while (0)

// Window size, from sweeps on a B200 (profiles/r02_window_sweeps_*.txt).  Two things decide it: the accumulation cost
// falls with c (fewer windows, 2 n K entries), the reduction cost is a function of the bucket count K 2^(c-1) alone and
// does not shrink with n (0.36 / 0.48 / 0.78 / 0.89 / 1.6 / 2.4 / 4.0 / 7.8 ms for c = 12 .. 20, whatever n is).  For the
// GLV curves c = 16 is special: K = 8 windows cover the 127/128-bit half-scalars exactly, so it wins from 2^18 to
// 2^21 points (2^21: 10.4 ms against 11.9 ms at c = 17); below, the latency-bound reduction asks for few buckets, above,
// c = 18 (K = 8 again, sparse top window).  Curves without the decomposition (twisted Edwards, msmProjective: ~252-bit
// scalars) keep log2(n) - 4 from 2^18 on and log2(n) - 2 below (2^16 / 2^18 / 2^20: c = 14 / 14 / 16 measured best).
// A sparse top window is balanced by sub-bucket spreading (MsmParams::top_sub), not avoided.  The reference's own table
// (msm-common.ts:25-41) is tuned for 16 CPU threads and is not used here; opts.c overrides everything.
int default_window(bool glv, size_t n) {
  int lg = 0;
  while (((size_t)1 << lg) < n) lg++;
  int c;
  if (!glv || lg < 14) c = lg >= 18 ? lg - 4 : lg - 2;
  else if (lg <= 15) c = 12;
  else if (lg <= 17) c = 13;
  else if (lg <= 21) c = 16;
  else c = 18;
  return std::max(5, std::min(c, 22));
}

inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// Byte ingestion (SURVEY 8f-1: `pointsFromBytes` + `toMontgomery` as a device kernel overlapped with the host->device
// copies).  Large point sets travel in chunks through two staging halves: the copy of chunk k + 1 runs on the copy
// stream while k_set_points converts chunk k, and the staging memory stays bounded (2 x 2^18 points) instead of a second
// copy of the whole input.  Small sets are one copy and one launch.
// d_status (checked ingestion): k_set_points also writes the canonical-encoding bit of each point there.
template <class CV>
int set_points_impl(mgb_ctx* ctx, const uint8_t* xy, const uint8_t* is_zero, size_t n, uint8_t* d_status = nullptr) {
  const size_t pbytes = 2 * CV::COORD_BYTES;
  size_t chunk = (size_t)1 << 18;
  if (const char* ev = getenv("MGB_DEBUG_INGEST_CHUNK")) chunk = std::max(1, atoi(ev));   // (tests: several chunks of a small set)
  uint32_t* table = (uint32_t*)ctx->table.p;
  if (n <= chunk) {
    ENS(ctx, ctx->stage, n * pbytes + n);
    CU(ctx, cudaMemcpyAsync(ctx->stage.p, xy, n * pbytes, cudaMemcpyHostToDevice, ctx->stream));
    uint8_t* dz = nullptr;
    if (is_zero) {
      dz = (uint8_t*)ctx->stage.p + n * pbytes;
      CU(ctx, cudaMemcpyAsync(dz, is_zero, n, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (d_status) k_set_points<CV, true><<<cdiv(n, 128), 128, 0, ctx->stream>>>((uint32_t)n, (const uint32_t*)ctx->stage.p, dz, table, d_status);
    else k_set_points<CV><<<cdiv(n, 128), 128, 0, ctx->stream>>>((uint32_t)n, (const uint32_t*)ctx->stage.p, dz, table);
    CU(ctx, cudaGetLastError());
  } else {
    const size_t half = (chunk * (pbytes + 1) + 255) / 256 * 256;     // one staging half: the chunk's x||y bytes, then its flags
    ENS(ctx, ctx->stage, 2 * half);
    cudaStream_t cs = ctx->aux[2];
    cudaEvent_t* landed = ctx->ev_chunk;                              // [h]: the copy into half h has finished
    cudaEvent_t* drained = ctx->ev_join;                              // [h]: the kernel reading half h has finished
    size_t k = 0;
    for (size_t b = 0; b < n; b += chunk, k++) {
      const size_t cnt = std::min(chunk, n - b);
      const int h = (int)(k & 1);
      char* sp = (char*)ctx->stage.p + h * half;
      if (k >= 2) CU(ctx, cudaStreamWaitEvent(cs, drained[h], 0));
      CU(ctx, cudaMemcpyAsync(sp, xy + b * pbytes, cnt * pbytes, cudaMemcpyHostToDevice, cs));
      uint8_t* dz = nullptr;
      if (is_zero) {
        dz = (uint8_t*)sp + chunk * pbytes;
        CU(ctx, cudaMemcpyAsync(dz, is_zero + b, cnt, cudaMemcpyHostToDevice, cs));
      }
      CU(ctx, cudaEventRecord(landed[h], cs));
      CU(ctx, cudaStreamWaitEvent(ctx->stream, landed[h], 0));
      if (d_status) k_set_points<CV, true><<<cdiv(cnt, 128), 128, 0, ctx->stream>>>((uint32_t)cnt, (const uint32_t*)sp, dz, table + b * CV::ENTRY_LIMBS, d_status + b);
      else k_set_points<CV><<<cdiv(cnt, 128), 128, 0, ctx->stream>>>((uint32_t)cnt, (const uint32_t*)sp, dz, table + b * CV::ENTRY_LIMBS);
      CU(ctx, cudaGetLastError());
      CU(ctx, cudaEventRecord(drained[h], ctx->stream));
    }
  }
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->npoints = n;
  return 0;
}

// Checked ingestion (mgb_set_points_checked): the ingestion above with the canonical-encoding bit, then k_check_points
// over the whole table.  found = {number of invalid points, index of the first, its status byte}.  The context keeps
// the points only when every one is valid.
template <class CV>
int set_points_checked_impl(mgb_ctx* ctx, const uint8_t* xy, const uint8_t* is_zero, size_t n, uint8_t* status, uint32_t* found) {
  static_assert(PT_NONCANONICAL == MGB_PT_NONCANONICAL && PT_OFF_CURVE == MGB_PT_OFF_CURVE && PT_NOT_IN_SUBGROUP == MGB_PT_NOT_IN_SUBGROUP, "status bits");
  ENS(ctx, ctx->checks, 8 + n);
  uint32_t* counters = (uint32_t*)ctx->checks.p;
  uint8_t* d_status = (uint8_t*)ctx->checks.p + 8;
  int rc = set_points_impl<CV>(ctx, xy, is_zero, n, d_status);
  ctx->npoints = 0;                                                 // (set_points_impl stored n)
  if (rc) return rc;
  CU(ctx, cudaMemsetAsync(counters, 0, 8, ctx->stream));
  k_check_points<CV><<<cdiv(n, 128), 128, 0, ctx->stream>>>((uint32_t)n, (const uint32_t*)ctx->table.p, d_status, counters);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(found, counters, 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (status) CU(ctx, cudaMemcpyAsync(status, d_status, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  found[1] = ~found[1];                                             // k_check_points keeps the complement of the index
  found[2] = 0;
  if (found[0]) {
    uint8_t why = 0;
    CU(ctx, cudaMemcpyAsync(&why, d_status + found[1], 1, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    found[2] = why;
  } else {
    ctx->npoints = n;
  }
  return 0;
}

template <class CV>
int random_points_impl(mgb_ctx* ctx, uint64_t seed, size_t n) {
  k_random_points<CV><<<cdiv(n, 128), 128, 0, ctx->stream>>>((uint32_t)n, seed, (uint32_t*)ctx->table.p);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->npoints = n;
  return 0;
}

template <class CV>
int get_points_impl(mgb_ctx* ctx, size_t first, size_t n, uint8_t* xy, uint8_t* is_zero) {
  const size_t pbytes = 2 * CV::COORD_BYTES;
  ENS(ctx, ctx->stage, n * pbytes + n);
  uint8_t* dz = (uint8_t*)ctx->stage.p + n * pbytes;
  k_get_points<CV><<<cdiv(n, 128), 128, 0, ctx->stream>>>((uint32_t)first, (uint32_t)n, (const uint32_t*)ctx->table.p, (uint32_t*)ctx->stage.p, dz);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(xy, ctx->stage.p, n * pbytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (is_zero) CU(ctx, cudaMemcpyAsync(is_zero, dz, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

// Starts the uploads of the scalar sets registered by mgb_msm_prefetch.  Called by msm_core behind the launch of tree
// round 0: the copy then overlaps the multiplier-bound accumulation instead of the bandwidth-bound digit / sort kernels.
int issue_prefetches(mgb_ctx* ctx) {
  for (auto& q : ctx->pf)
    if (q.valid && !q.issued) {
      CU(ctx, cudaMemcpyAsync(q.buf.p, q.host, q.n * 32, cudaMemcpyHostToDevice, ctx->pf_stream));
      CU(ctx, cudaEventRecord(q.ev, ctx->pf_stream));
      q.issued = true;
    }
  return 0;
}

// Runs the pipeline; leaves the un-normalised result accumulator in ctx->acc_out.
template <class CV>
int msm_core(mgb_ctx* ctx, const void* scalars, bool on_device, size_t n, const mgb_opts* opts, mgb_timing* tm, bool normalize = false) {
  cudaStream_t st = ctx->stream;
  uint32_t launches = 0;
  int c = (opts && opts->c > 0) ? opts->c : default_window(CV::USE_GLV, n);
  if (c < 2 || c > 24) return fail(ctx, MGB_E_INVALID, "window size c must be in [2, 24]");
  MsmParams pr;
  pr.n = (uint32_t)n;
  pr.c = c;
  pr.K = (CV::MAG_BITS + c - 1) / c;
  pr.L = 1u << (c - 1);
  pr.nbuckets = (uint32_t)pr.K * pr.L;
  pr.nent = (uint32_t)(n * CV::HALVES * pr.K);
  {
    const int top_bits = CV::MAG_BITS - (pr.K - 1) * c;   // the top digit is at most 2^top_bits
    pr.top_sub = std::max(0, (c - 1) - top_bits);
  }
  if ((size_t)n * CV::HALVES * pr.K >= (1ull << 31)) return fail(ctx, MGB_E_INVALID, "n * windows exceeds 2^31 entries");
  // geometry of the bucket reduction: c-1 index bits in D digits of <= 5 bits
  ReduceGeom gm;
  {
    const int nb = c - 1;
    gm.D = std::max(1, (nb + 4) / 5);
    int pos = 0, minw = 32;
    for (int d = 0; d < 6; d++) { gm.width[d] = 0; gm.shift[d] = 0; }
    for (int d = 0; d < gm.D; d++) {
      gm.width[d] = nb / gm.D + (d < nb % gm.D ? 1 : 0);
      gm.shift[d] = pos;
      pos += gm.width[d];
      minw = std::min(minw, gm.width[d]);
    }
    const uint32_t gmax = pr.L >> minw;        // largest group
    // buckets per partial sum: more of the (throughput-bound) first tree level folded into k_group_partial
    // when there are buckets enough to keep every SM busy anyway (measured at 2^18 / 2^20 / 2^22 points: 2 / 4 / 4 best)
    // (profiles/r02_ab_reduction_chunk.txt: CH = 1 / 2 / 4 at 2^16, c = 13: reduce 0.46 / 0.48 / 0.55 ms; 2^18, c = 16: 1.08 / 1.01 / 0.96 ms)
    gm.CH = pr.nbuckets >= (1u << 18) ? 4 : (pr.nbuckets >= (1u << 15) ? 1 : 2);
    if (const char* ev = getenv("MGB_DEBUG_CH")) gm.CH = std::max(1, atoi(ev));
    gm.NP = 1;
    while ((uint32_t)gm.NP * gm.CH < gmax) gm.NP <<= 1;
    gm.VB = 3;
    for (int d = 0; d < gm.D; d++) gm.VB = std::max(gm.VB, gm.width[d]);
    if (const char* ev = getenv("MGB_DEBUG_NV32")) { if (atoi(ev)) gm.VB = 5; }
    gm.NV = 1 << gm.VB;
  }
  const uint32_t ngroups = (uint32_t)pr.K * gm.D * gm.NV;
  ENS(ctx, ctx->acc_out, CV::ACC_LIMBS * 4);
  CU(ctx, cudaEventRecord(ctx->ev[EV_START], st));
  // Host scalars travel in chunks on a second stream; the digit kernel of a chunk starts as soon as that chunk has
  // landed, so only the last chunk's digits are not hidden behind the PCIe transfer.
  const uint32_t* d_scalars;
  mgb_ctx::Prefetch* pf = nullptr;               // host scalars that mgb_msm_prefetch already put on their way
  if (!on_device)
    for (auto& q : ctx->pf)
      if (q.valid && q.host == scalars && q.n == n) {
        if (q.issued) pf = &q;
        else q.valid = false;                    // never started: this call uploads the set itself
      }
  const int n_chunks = (!on_device && !pf && n >= (1u << 16)) ? 4 : 1;
  if (on_device) {
    d_scalars = (const uint32_t*)scalars;
  } else if (pf) {
    d_scalars = (const uint32_t*)pf->buf.p;
    CU(ctx, cudaStreamWaitEvent(st, pf->ev, 0));
    pf->valid = false;                           // the slot is free again once this call has returned
  } else {
    ENS(ctx, ctx->scalars, n * 32);
    d_scalars = (const uint32_t*)ctx->scalars.p;
    if (n_chunks == 1) {
      CU(ctx, cudaMemcpyAsync(ctx->scalars.p, scalars, n * 32, cudaMemcpyHostToDevice, st));
    } else {
      cudaStream_t cs = ctx->aux[2];
      CU(ctx, cudaStreamWaitEvent(cs, ctx->ev[EV_START], 0));
      for (int k = 0; k < n_chunks; k++) {
        const size_t b = n * (size_t)k / n_chunks, e = n * (size_t)(k + 1) / n_chunks;
        CU(ctx, cudaMemcpyAsync((char*)ctx->scalars.p + b * 32, (const char*)scalars + b * 32, (e - b) * 32, cudaMemcpyHostToDevice, cs));
        CU(ctx, cudaEventRecord(ctx->ev_chunk[k], cs));
      }
    }
  }
  CU(ctx, cudaEventRecord(ctx->ev[EV_H2D], st));

  ENS(ctx, ctx->ent_bucket, (size_t)pr.nent * 4);
  ENS(ctx, ctx->ent_rank, (size_t)pr.nent * 4);
  ENS(ctx, ctx->counts, ((size_t)pr.nbuckets + 1) * 4);
  ENS(ctx, ctx->offs, ((size_t)pr.nbuckets + 1) * 4);
  ENS(ctx, ctx->offcnt, ((size_t)pr.nbuckets + 1) * 8);
  const uint32_t ntiles = cdiv(pr.nbuckets, SCAN_TILE);
  ENS(ctx, ctx->tile_sums, (size_t)ntiles * 4);
  // every non-empty bucket occupies an even number of slots (k_scan_tiles)
  const size_t max_slots = std::min<size_t>((size_t)pr.nent + pr.nbuckets, 2 * (size_t)pr.nent) + 2;
  ENS(ctx, ctx->pairs, ((size_t)pr.nent / 4 + 8) * sizeof(PairEnt));           // pair lists of rounds 1, 3, ..
  ENS(ctx, ctx->pairs2, ((size_t)pr.nent / 8 + 8) * sizeof(PairEnt));    // rounds 2, 4, ..
  ENS(ctx, ctx->V, max_slots * CV::V_LIMBS * 4);
  ENS(ctx, ctx->redU[0], (size_t)ngroups * gm.NP * CV::ACC_LIMBS * 4);
  ENS(ctx, ctx->redW[0], (size_t)pr.K * CV::ACC_LIMBS * 4);
  ENS(ctx, ctx->redW[1], (size_t)pr.K * (gm.D + 1) * CV::ACC_LIMBS * 4);
  ENS(ctx, ctx->misc, 1024 * 4);
  // misc: [0] grand total of (padded) slots, [1] max bucket, [512 + r] exact number of additions of tree round r, [8 + 64 g + r] pair count of round r of window group g,
  //       [264 + 64 g + r] tile counter of that round
  uint32_t* misc = (uint32_t*)ctx->misc.p;
  CU(ctx, cudaMemsetAsync(ctx->counts.p, 0, ((size_t)pr.nbuckets + 1) * 4, st));
  CU(ctx, cudaMemsetAsync(misc, 0, 1024 * 4, st));

  // ---- digits + histogram
  for (int k = 0; k < n_chunks; k++) {
    const size_t b = n * (size_t)k / n_chunks, e = n * (size_t)(k + 1) / n_chunks;
    if (n_chunks > 1) CU(ctx, cudaStreamWaitEvent(st, ctx->ev_chunk[k], 0));
    k_digits<CV><<<cdiv(e - b, 256), 256, 0, st>>>(pr, (uint32_t)b, (uint32_t)e, d_scalars, (uint32_t*)ctx->ent_bucket.p, (uint32_t*)ctx->ent_rank.p, (uint32_t*)ctx->counts.p);
    launches++;
  }
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaEventRecord(ctx->ev[EV_DIGITS], st));

  // ---- bucket offsets; the totals come back to the host to size the rounds
  k_scan_tiles<<<ntiles, SCAN_T, 0, st>>>((const uint32_t*)ctx->counts.p, (uint32_t*)ctx->offs.p, (uint32_t*)ctx->tile_sums.p, pr.nbuckets, misc + 1, misc + 512);
  k_scan_sums<<<1, SCAN_T, 0, st>>>((uint32_t*)ctx->tile_sums.p, ntiles, misc);
  k_scan_add<<<ntiles, SCAN_T, 0, st>>>((uint32_t*)ctx->offs.p, (const uint32_t*)ctx->tile_sums.p, pr.nbuckets, misc, (const uint32_t*)ctx->counts.p, (uint2*)ctx->offcnt.p);
  launches += 3;
  CU(ctx, cudaGetLastError());
  // A kernel stores the counters straight into the page-locked host buffer (mapped into the device's address space under
  // unified addressing).  Three cudaMemcpyAsync did this before; they queue on a copy engine -- behind the upload of the
  // NEXT call's scalars when mgb_msm_prefetch is in use, which left the GPU idle until that upload had finished
  // (pipelined end-to-end step +0.2 ms on one GPU, +0.6 ms with eight GPUs sharing the host's memory bandwidth).
  k_plan_to_host<<<1, 32, 0, st>>>(misc, (const uint32_t*)ctx->counts.p + pr.nbuckets, ctx->h_pinned);
  launches++;
  CU(ctx, cudaEventRecord(ctx->ev_plan, st));
  // The host needs the counters above to size the tree rounds.  For inputs that certainly have a round 0 the scatter
  // does not depend on them, so it is launched FIRST and the host waits for the counters (an event, not the stream)
  // while it runs: the round trip no longer idles the GPU.  Should the plan come out without a round 0 after all
  // (only possible for tiny buckets), the scatter is simply run again in its materialising form.
  int G = 1;   // window groups pipelined on separate streams; measured on B200: 2 groups change the total by < 1 %; the mechanism stays for tuning
  if (const char* ev = getenv("MGB_DEBUG_GROUPS")) G = std::max(1, std::min(4, atoi(ev)));
  G = std::min(G, pr.K);
  const bool early_scatter = G == 1 && pr.nent >= (1u << 19) && !getenv("MGB_DEBUG_NROUNDS");
  if (early_scatter) {
    ENS(ctx, ctx->recs, (max_slots / 2 + 1) * 8);
    ENS(ctx, ctx->lifes, max_slots / 2 + 8);
    k_scatter<CV><<<dim3(cdiv(n, 256 * SCATTER_U), (unsigned)(CV::HALVES * pr.K)), 256, 0, st>>>(
        pr, 0, pr.K, (const uint32_t*)ctx->ent_bucket.p, (const uint32_t*)ctx->ent_rank.p, (const uint2*)ctx->offcnt.p,
        (const uint32_t*)ctx->table.p, nullptr, (uint32_t*)ctx->recs.p, (uint8_t*)ctx->lifes.p);
    launches++;
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaEventRecord(ctx->ev[EV_SORT], st));
  }
  CU(ctx, cudaEventSynchronize(ctx->ev_plan));
  const uint32_t maxcount = ctx->h_pinned[65];
  const uint32_t* round_pairs = ctx->h_pinned + 68;
  if (ctx->h_pinned[66] & 2u)
    return fail(ctx, MGB_E_INVALID, "a scalar is out of range: this path takes scalars below 2^" + std::to_string(CV::MAG_BITS - 1) + " (reduce them mod q first)");
  if (ctx->h_pinned[66]) return fail(ctx, MGB_E_INVALID, "internal: a half-scalar exceeded its bound");

  // Depth of the bucket trees.  Full depth is ceil(log2(max bucket)).  A round costs at least one batch latency
  // (~0.2 ms: prefix products, inversion, back-substitution) however few additions it holds, and below ~0.3-0.5 M
  // additions it is cheaper to leave them to k_bucket_finish (mixed XYZZ additions, 10 instead of 6
  // multiplications each, but throughput-bound): measured best depth at 2^16 / 2^18 / 2^20 points = 2 / 3 / 4-5
  // rounds.  Buckets far above the typical size (skewed scalars) force more rounds: at most 16 elements of
  // any bucket are left to the finish kernel.
  int r_full = 0;
  while ((1u << r_full) < maxcount) r_full++;
  int rounds = 0;
  uint32_t min_pairs = CV::BATCH_AFFINE ? 300000u : 20000u;   // rounds without an inversion have a much lower floor
  if (const char* ev = getenv("MGB_DEBUG_MINPAIRS")) min_pairs = (uint32_t)atoi(ev);
  while (rounds < r_full && rounds < SCAN_ROUNDS && round_pairs[rounds] >= min_pairs) rounds++;
  rounds = std::max(rounds, r_full - 4);
  if (opts && opts->verbose > 1) rounds = r_full;
  // affine bucket reduction (opt-in, SURVEY 8f-3): the bucket trees run to completion, every bucket sum is one affine point
  const bool affine_red = CV::BATCH_AFFINE && opts && opts->affine_reduction && G == 1;
  if (const char* ev = getenv("MGB_DEBUG_NROUNDS")) rounds = std::max(0, std::min(r_full, atoi(ev)));   // tuning aid
  if (affine_red) rounds = r_full;               // (after the tuning knob: the group trees need complete bucket sums)
  // Elements a bucket has left after the last round are summed once by k_bucket_finish when there are many of them
  // (otherwise k_group_partial adds the single leftover directly as a mixed addition, which is cheaper).
  uint64_t left = 0;
  for (int r = rounds; r < SCAN_ROUNDS; r++) left += round_pairs[r];
  bool use_finish = rounds < r_full && 4 * left >= pr.nbuckets;
  if (const char* ev = getenv("MGB_DEBUG_FINISH")) use_finish = atoi(ev) != 0 && rounds < r_full;
  // round 0 gathers its operands from the point table (see k_scatter); without a round 0 the sorted
  // points are materialised by the scatter as the reduction expects
  const bool fuse = rounds > 0;
  if (fuse) { ENS(ctx, ctx->recs, (max_slots / 2 + 1) * 8); ENS(ctx, ctx->lifes, max_slots / 2 + 8); }
  uint32_t* recs = fuse ? (uint32_t*)ctx->recs.p : nullptr;
  uint8_t* lifes = fuse ? (uint8_t*)ctx->lifes.p : nullptr;
  const uint32_t* table = (const uint32_t*)ctx->table.p;
  const uint32_t* offs = (const uint32_t*)ctx->offs.p;
  const uint32_t* counts = (const uint32_t*)ctx->counts.p;

  // ---- window groups, pipelined on separate streams: every round ends with a tail in which few
  // tiles are left (and the late rounds and the reduction are latency-bound throughout); the
  // kernels of another, independent group of windows fill the SMs meanwhile.
  CU(ctx, cudaEventRecord(ctx->ev_fork, st));
  size_t pair_off = 0, pair2_off = 0;
  for (int g = 0; g < G; g++) {
    cudaStream_t sg = g == 0 ? st : ctx->aux[g - 1];
    if (g > 0) CU(ctx, cudaStreamWaitEvent(sg, ctx->ev_fork, 0));
    const int w_begin = (int)((long long)pr.K * g / G), w_end = (int)((long long)pr.K * (g + 1) / G), Kg = w_end - w_begin;
    const size_t nent_g = (size_t)n * CV::HALVES * Kg;
    // round r reads pl[r & 1] and writes pl[(r & 1) ^ 1]; round 0 reads no list
    PairEnt* pl[2] = {(PairEnt*)ctx->pairs2.p + pair2_off, (PairEnt*)ctx->pairs.p + pair_off};
    pair_off += nent_g / 4 + 1;
    pair2_off += nent_g / 8 + 1;
    const uint32_t b_begin = (uint32_t)w_begin * pr.L, b_end = (uint32_t)w_end * pr.L;
    uint32_t* cnt = misc + 8 + 64 * g;
    uint32_t* tcnt = misc + 264 + 64 * g;
    if (!(early_scatter && fuse)) {
      k_scatter<CV><<<dim3(cdiv(n, 256 * SCATTER_U), (unsigned)(CV::HALVES * Kg)), 256, 0, sg>>>(pr, w_begin, Kg, (const uint32_t*)ctx->ent_bucket.p, (const uint32_t*)ctx->ent_rank.p,
                                                      (const uint2*)ctx->offcnt.p, table, fuse ? nullptr : (uint32_t*)ctx->V.p, recs, lifes);
      launches++;
      if (g == 0) CU(ctx, cudaEventRecord(ctx->ev[EV_SORT], st));
    }
    for (int r = 0; r < rounds; r++) {
      PairEnt* pin = pl[r & 1];
      PairEnt* pout = pl[(r & 1) ^ 1];
      if constexpr (CV::BATCH_AFFINE) {
        constexpr int EMAX = MGB_EMAX, MINB = MGB_MINB;
        // pairs this launch walks (exact over all windows, from the scan): round 0 walks every aligned slot pair, the
        // partner-less last elements of odd buckets included (they are copied); later rounds walk their pair list
        const uint64_t est = (r == 0 ? (uint64_t)(ctx->h_pinned[64] / 2) : (r < SCAN_ROUNDS ? (uint64_t)round_pairs[r] : 0)) * Kg / pr.K;
        const uint64_t warps = (uint64_t)ctx->sm_count * MINB * 4;
        // Tile shape: every tile holds E pairs per lane, with E chosen so that the round is an (almost) whole number
        // k of tiles per resident warp:  per lane p = est / (32 * warps) additions, k = ceil(p / EMAX) tiles,
        // E = ceil(p / k).  A batch (warp products + inversion) costs the same however small, so few, large tiles
        // win -- but a power-of-two E leaves up to a quarter of the warps without a second tile (or without any
        // tile) while the others finish.  Measured at 2^20 (profiles/r02_tile_sweep.txt): E = 64/64/32/16/8 ->
        // 56/28/28/14/7 takes the accumulation from 4.78 to 4.37 ms, and round 0 alone is 2.07 ms at E = 56 against
        // 2.13 - 2.27 ms at 48, 52, 54, 58 or 60.  Rounds with more than 32 pairs per lane get two tiles per warp (the
        // dynamic hand-out of the second one takes the warps out of lockstep: one tile of 111 pairs per lane with
        // EMAX = 128 was slower, 2.54 ms), smaller rounds one.
        const uint64_t per_lane = std::max<uint64_t>(1, (est + 32 * warps - 1) / (32 * warps));
        uint64_t ktiles = (per_lane + EMAX - 1) / EMAX;
        if (per_lane > 32 && ktiles < 2) ktiles = 2;
        if (const char* ev = getenv("MGB_DEBUG_KTILES")) ktiles = std::max(1, atoi(ev));
        int emin = 4;
        if (const char* ev = getenv("MGB_DEBUG_EMIN")) emin = std::max(1, atoi(ev));
        int E = (int)std::min<uint64_t>(EMAX, std::max<uint64_t>((uint64_t)emin, (per_lane + ktiles - 1) / ktiles));
        uint32_t n_big = 0xffffffffu;            // all tiles have E pairs per lane (the E/4 tail tiles are not needed when balanced)
        if (const char* ev = getenv("MGB_DEBUG_E")) {   // tuning aid: comma-separated E per round
          int k = 0; const char* q = ev;
          while (k < r && (q = strchr(q, ',')) != nullptr) { q++; k++; }
          if (q && k == r && atoi(q) != 0) E = std::min(EMAX, std::abs(atoi(q)));
        }
        if (const char* ev = getenv("MGB_DEBUG_NBIG")) n_big = (uint32_t)(atof(ev) * warps);
        int E_small = E >= 16 ? E / 4 : E;          // only used when n_big cuts the tile list (tuning knobs)
        // per-warp scratch for the prefix products of a tile (see k_batch_add)
        const size_t pre_bytes = (size_t)ctx->sm_count * MINB * 4 * EMAX * (CV::N / 4) * 32 * 16;
        ENS(ctx, ctx->prebuf, pre_bytes * 4);     // one area per window group (at most 4)
        uint4* scratch = (uint4*)((char*)ctx->prebuf.p + pre_bytes * g);
        if (r == 0) {
          auto kern = k_batch_add<CV, EMAX, MINB, true>;
          cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, MINB > 4 ? 90 : 75);   // MINB blocks x 36 KB of staging
          kern<<<ctx->sm_count * MINB, 128, 0, sg>>>((uint32_t*)ctx->V.p, nullptr, nullptr, r, E, E_small, n_big, pout, cnt + r + 1, tcnt + r,
                                                    (const uint2*)recs, lifes, table, offs, b_begin, b_end, scratch);
        } else {
          auto kern = k_batch_add<CV, EMAX, MINB, false>;
          cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, MINB > 4 ? 90 : 75);
          kern<<<ctx->sm_count * MINB, 128, 0, sg>>>((uint32_t*)ctx->V.p, pin, cnt + r, r, E, E_small, n_big, pout, cnt + r + 1, tcnt + r,
                                                    nullptr, nullptr, nullptr, nullptr, 0, 0, scratch);
        }
      } else {
        if (r == 0) k_pair_add<CV, true><<<ctx->sm_count * 8, 256, 0, sg>>>((uint32_t*)ctx->V.p, nullptr, nullptr, r, pout, cnt + r + 1, (const uint2*)recs, lifes, table, offs, b_begin, b_end);
        else k_pair_add<CV, false><<<ctx->sm_count * 8, 256, 0, sg>>>((uint32_t*)ctx->V.p, pin, cnt + r, r, pout, cnt + r + 1, nullptr, nullptr, nullptr, nullptr, 0, 0);
      }
      launches += 1;
      if (r == 0) { int rc_ = issue_prefetches(ctx); if (rc_) return rc_; }
      if (G == 1 && getenv("MGB_DEBUG_ROUNDS")) {   // tuning aid: per-round wall time (synchronises!)
        cudaEvent_t e1; cudaEventCreate(&e1);
        cudaEventRecord(e1, st); cudaEventSynchronize(e1);
        static thread_local float last = 0; float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[EV_SORT], e1);
        fprintf(stderr, "  round %d: +%.3f ms (cum %.3f)\n", r, ms - (r ? last : 0), ms); last = ms;
        cudaEventDestroy(e1);
      }
    }
    if (g == 0) CU(ctx, cudaEventRecord(ctx->ev[EV_ACC], st));
    // bucket reduction of the group's windows (digit-decomposed weights, see engine.cuh)
    const uint32_t ngroups_g = (uint32_t)Kg * gm.D * gm.NV;
    uint32_t* Pg = (uint32_t*)ctx->redU[0].p + (size_t)w_begin * gm.D * gm.NV * gm.NP * CV::ACC_LIMBS;
    const uint32_t* bsum = nullptr;
    bool reduced_affine = false;
    if constexpr (CV::BATCH_AFFINE) {
      if (affine_red) {
        constexpr int EMAX = MGB_EMAX, MINB = MGB_MINB;
        int minw = 32, minw_top = 32;
        for (int d = 0; d < gm.D; d++) {
          minw = std::min(minw, gm.width[d]);
          const int nbits = c - 1, shd = std::min(gm.shift[d] + pr.top_sub, nbits), wdt = std::min(gm.width[d], nbits - shd);
          if (!(wdt == 0 && d > 0)) minw_top = std::min(minw_top, wdt);
        }
        AffineRedGeom ag;
        ag.GS0 = 2;                                                          // at least two slots: every even slot is a pair-list entry
        while ((uint32_t)ag.GS0 < (pr.L >> minw)) ag.GS0 <<= 1;               // slots per group (largest group, power of two)
        ag.GS1 = 2;
        while ((uint32_t)ag.GS1 < (pr.L >> minw_top)) ag.GS1 <<= 1;           // the same for the (possibly clipped) top window
        ag.g_top = (uint32_t)(pr.K - 1) * gm.D * gm.NV;
        ag.n0 = ag.g_top * (uint32_t)ag.GS0;
        const size_t nslots = (size_t)ag.n0 + (size_t)gm.D * gm.NV * ag.GS1;
        if (nslots >= (1ull << 31)) return fail(ctx, MGB_E_INVALID, "affine_reduction: too many group slots for this window size");
        ag.total = (uint32_t)nslots;
        const int GSmax = std::max(ag.GS0, ag.GS1);
        ENS(ctx, ctx->W, nslots * CV::V_LIMBS * 4);
        ENS(ctx, ctx->pairs, (nslots / 2 + 8) * sizeof(PairEnt));
        ENS(ctx, ctx->pairs2, (nslots / 4 + 8) * sizeof(PairEnt));
        PairEnt* apl[2] = {(PairEnt*)ctx->pairs.p, (PairEnt*)ctx->pairs2.p};   // round r reads apl[r & 1], writes apl[(r & 1) ^ 1]
        uint32_t* acnt = misc + 700;                                           // pair counts of the group-tree rounds
        uint32_t* atcnt = misc + 800;                                          // their tile counters
        k_affine_gather<CV><<<cdiv(nslots, 256), 256, 0, sg>>>(pr, gm, ag, (const uint32_t*)ctx->V.p, offs, counts, (uint32_t*)ctx->W.p, apl[0], acnt);
        launches++;
        const uint64_t warps = (uint64_t)ctx->sm_count * MINB * 4;
        const size_t pre_bytes = (size_t)ctx->sm_count * MINB * 4 * EMAX * (CV::N / 4) * 32 * 16;
        ENS(ctx, ctx->prebuf, pre_bytes * 4);
        int r = 0;
        for (size_t np = nslots / 2; np >= 1 && (1 << r) < GSmax; np >>= 1, r++) {
          const uint64_t per_lane = std::max<uint64_t>(1, (np + 32 * warps - 1) / (32 * warps));
          const uint64_t kt = std::max<uint64_t>((per_lane + EMAX - 1) / EMAX, per_lane > 32 ? 2 : 1);
          const int E = (int)std::min<uint64_t>(EMAX, std::max<uint64_t>(4, (per_lane + kt - 1) / kt));
          auto kern = k_batch_add<CV, EMAX, MINB, false>;
          cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, MINB > 4 ? 90 : 75);
          kern<<<ctx->sm_count * MINB, 128, 0, sg>>>((uint32_t*)ctx->W.p, apl[r & 1], acnt + r, r, E, E, 0xffffffffu, apl[(r & 1) ^ 1], acnt + r + 1, atcnt + r,
                                                    nullptr, nullptr, nullptr, nullptr, 0, 0, (uint4*)ctx->prebuf.p);
          launches++;
        }
        k_affine_group_sums<CV><<<cdiv(ngroups_g, 128), 128, 0, sg>>>(ngroups_g, ag, (const uint32_t*)ctx->W.p, (uint32_t*)ctx->redU[0].p);
        launches++;
        reduced_affine = true;
      }
    }
    ReduceGeom gmr = gm;                       // geometry seen by the digit sums: one partial sum per group after the affine trees
    if (reduced_affine) gmr.NP = 1;
    if (!reduced_affine) {
    if (use_finish) {
      ENS(ctx, ctx->bsum, (size_t)pr.nbuckets * CV::ACC_LIMBS * 4);
      k_bucket_finish<CV><<<cdiv(b_end - b_begin, 128), 128, 0, sg>>>(b_begin, b_end, rounds, (const uint32_t*)ctx->V.p, offs, counts, (uint32_t*)ctx->bsum.p);
      launches++;
      bsum = (const uint32_t*)ctx->bsum.p;
    }
    k_group_partial<CV><<<cdiv(ngroups_g * gm.NP, 128), 128, 0, sg>>>(pr, gm, w_begin, Kg, rounds, (const uint32_t*)ctx->V.p, offs, counts, bsum,
                                                                     (uint32_t*)ctx->redU[0].p);
    launches++;
    }
    int remaining = gmr.NP;
    for (; remaining > 32; remaining >>= 1) {
      k_tree_round<CV><<<cdiv((size_t)ngroups_g * (remaining / 2), 128), 128, 0, sg>>>(ngroups_g, gm.NP, remaining / 2, Pg);
      launches++;
    }
    if constexpr (CV::BATCH_AFFINE) {
      // latency-bound stages, four lanes per point addition (coop.cuh): last tree levels, digit sums, per-window assembly
      if (remaining > 1) { k_tree_tail_quad<CV><<<ngroups_g, 64, 0, sg>>>(gm.NP, remaining, Pg); launches++; }
      k_digit_sums<CV><<<Kg * gm.D, 128, 0, sg>>>(pr, gmr, w_begin, (const uint32_t*)ctx->redU[0].p, (uint32_t*)ctx->redW[1].p);
      k_window_assemble<CV><<<Kg, 32, 0, sg>>>(pr, gm, w_begin, (const uint32_t*)ctx->redW[1].p, (uint32_t*)ctx->redW[0].p);
      launches += 2;
    } else {
      if (remaining > 1) {
        k_tree_tail<CV><<<cdiv((size_t)ngroups_g * 32, 128), 128, 0, sg>>>(ngroups_g, gm.NP, remaining, Pg);
        launches++;
      }
      k_window_sums<CV><<<Kg, 192, 0, sg>>>(pr, gm, w_begin, (const uint32_t*)ctx->redU[0].p, (uint32_t*)ctx->redW[0].p);
      launches++;
    }
    if (g > 0) CU(ctx, cudaEventRecord(ctx->ev_join[g - 1], sg));
  }
  for (int g = 1; g < G; g++) CU(ctx, cudaStreamWaitEvent(st, ctx->ev_join[g - 1], 0));
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaEventRecord(ctx->ev[EV_REDUCE], st));
  uint32_t* d_xy = nullptr;
  if (normalize) { ENS(ctx, ctx->out_xy, 64 * 4); d_xy = (uint32_t*)ctx->out_xy.p; }
  k_final<CV><<<1, 32, 0, st>>>(pr.K, pr.c, (const uint32_t*)ctx->redW[0].p, (uint32_t*)ctx->acc_out.p, d_xy, d_xy ? d_xy + 2 * CV::N : nullptr);
  launches++;
  CU(ctx, cudaGetLastError());
  { int rc_ = issue_prefetches(ctx); if (rc_) return rc_; }   // inputs too small for a tree round: start the upload here
  if (tm) {
    tm->c = c; tm->K = pr.K; tm->rounds = rounds; tm->max_bucket = maxcount; tm->n_launches = launches;
    tm->n_pairs = 0;  // filled after the final sync (needs the per-round counters)
  }
  return 0;
}

int finish_timing(mgb_ctx* ctx, mgb_timing* tm) {
  if (!tm) return 0;
  auto el = [&](int a, int b) { float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]); return ms; };
  tm->h2d_scalars = el(EV_START, EV_H2D);
  tm->decompose_slice = el(EV_H2D, EV_DIGITS);
  tm->sort = el(EV_DIGITS, EV_SORT);
  tm->accumulate = el(EV_SORT, EV_ACC);
  tm->reduce = el(EV_ACC, EV_REDUCE);
  tm->final_sum = el(EV_REDUCE, EV_FINAL);
  tm->total = el(EV_START, EV_FINAL);
  // additions done by the tree rounds: exact per-round counts from the scan (rounds beyond SCAN_ROUNDS -- heavily
  // skewed inputs only -- from the pair-list counters)
  uint64_t s = 0;
  const uint32_t* round_pairs = ctx->h_pinned + 68;      // read back by msm_core before the rounds were sized
  for (int r = 0; r < tm->rounds && r < SCAN_ROUNDS; r++) s += round_pairs[r];
  if (tm->rounds > SCAN_ROUNDS) {                        // heavily skewed inputs only: a blocking copy of the counters
    uint32_t h[1024];
    CU(ctx, cudaMemcpy(h, (uint32_t*)ctx->misc.p, sizeof(h), cudaMemcpyDeviceToHost));
    for (int g = 0; g < 4; g++)
      for (int r = SCAN_ROUNDS; r < tm->rounds && r < 63; r++) s += h[8 + 64 * g + r];
  }
  tm->n_pairs = s;
  return 0;
}

// d_accs == nullptr: k_final has normalised already (msm_core with normalize = true), only the read-back is left.
// stride_limbs > ACC_LIMBS: the partials are the gathered records of mgb_msm_sharded, each followed by its rank's status
// word; *peer_failed then tells whether any rank reported that it could not compute its shard.
template <class CV>
int normalize_out(mgb_ctx* ctx, const void* d_accs, int count, uint8_t* out_xy, int* out_is_zero, int stride_limbs = CV::ACC_LIMBS, bool* peer_failed = nullptr) {
  ENS(ctx, ctx->out_xy, 64 * 4);
  uint32_t* d = (uint32_t*)ctx->out_xy.p;
  const bool with_status = d_accs && stride_limbs > CV::ACC_LIMBS;
  if (d_accs) {
    k_normalize<CV><<<1, 32, 0, ctx->stream>>>((const uint32_t*)d_accs, count, stride_limbs, d, d + 2 * CV::N);
    CU(ctx, cudaGetLastError());
  }
  CU(ctx, cudaMemcpyAsync(ctx->h_pinned, d, (2 * CV::N + (with_status ? 2 : 1)) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaEventRecord(ctx->ev[EV_FINAL], ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  if (out_xy) memcpy(out_xy, ctx->h_pinned, 2 * CV::COORD_BYTES);
  if (out_is_zero) *out_is_zero = (int)ctx->h_pinned[2 * CV::N];
  if (peer_failed) *peer_failed = with_status && ctx->h_pinned[2 * CV::N + 1] != 0;
  return 0;
}

template <class CV>
int msm_impl(mgb_ctx* ctx, const void* scalars, bool on_device, size_t n, const mgb_opts* opts, uint8_t* out_xy, int* out_is_zero, mgb_timing* tm) {
  if (tm) memset(tm, 0, sizeof(*tm));
  if (n == 0) {  // neutral element without touching the device pipeline
    memset(out_xy, 0, 2 * CV::COORD_BYTES);
    if (!CV::BATCH_AFFINE) out_xy[CV::COORD_BYTES] = 1;  // twisted Edwards neutral (0, 1)
    if (out_is_zero) *out_is_zero = 1;
    return 0;
  }
  int r = msm_core<CV>(ctx, scalars, on_device, n, opts, tm, true);     // k_final normalises as well
  if (r) return r;
  r = normalize_out<CV>(ctx, nullptr, 1, out_xy, out_is_zero);
  if (r) return r;
  return finish_timing(ctx, tm);
}

template <class CV>
__global__ void k_acc_neutral(uint32_t* out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) CV::st_acc(out, CV::acc_zero());
}

template <class CV>
int msm_partial_impl(mgb_ctx* ctx, const void* scalars, bool on_device, size_t n, const mgb_opts* opts, void* d_out, mgb_timing* tm) {
  if (tm) memset(tm, 0, sizeof(*tm));
  if (n == 0) {   // an empty shard (fewer pairs than ranks) contributes the neutral element
    ENS(ctx, ctx->acc_out, CV::ACC_LIMBS * 4);
    k_acc_neutral<CV><<<1, 32, 0, ctx->stream>>>((uint32_t*)d_out);
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
  }
  int r = msm_core<CV>(ctx, scalars, on_device, n, opts, tm);
  if (r) return r;
  CU(ctx, cudaMemcpyAsync(d_out, ctx->acc_out.p, CV::ACC_LIMBS * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  CU(ctx, cudaEventRecord(ctx->ev[EV_FINAL], ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return finish_timing(ctx, tm);
}


// One rank of the sharded MSM (SURVEY 8e): partial sum of the local shard, ONE ncclAllGather of the un-normalised
// partial accumulators on the engine's own stream straight behind k_final, sum + normalisation of the comm_world
// partials in one kernel, one device->host copy, one synchronisation.  An empty shard contributes the neutral element.
// A rank whose shard fails (a scalar out of range, a window size that does not fit, no memory) must not leave its peers
// waiting in the collective: every rank sends its accumulator followed by a status word, the failing rank joins the
// all-gather with the neutral element and a non-zero status, returns its own error, and the others return MGB_E_COMM
// instead of a sum that misses a shard.  (The reference's workers share one address space and one exception,
// src/threads/threads.ts:319-330; ranks in different processes need the status to travel with the data.)
template <class CV>
int msm_sharded_impl(mgb_ctx* ctx, const void* scalars, bool on_device, size_t n, const mgb_opts* opts, uint8_t* out_xy, int* out_is_zero, mgb_timing* tm,
                     int pre_rc /* a rank-local argument error found by mgb_msm_sharded (message in ctx->err): join flagged, compute nothing */) {
  if (tm) memset(tm, 0, sizeof(*tm));
  constexpr int REC_LIMBS = CV::ACC_LIMBS + 4;              // accumulator + status word, padded to 16 bytes
  const size_t acc_bytes = CV::ACC_LIMBS * 4, rec_bytes = REC_LIMBS * 4;
  const bool collective = ctx->comm_world > 1;
  ENS(ctx, ctx->acc_out, rec_bytes);
  int local_rc = pre_rc;
  std::string local_err;
  if (local_rc) {
    // nothing to compute
  } else if (n == 0) {
    k_acc_neutral<CV><<<1, 32, 0, ctx->stream>>>((uint32_t*)ctx->acc_out.p);
    CU(ctx, cudaGetLastError());
  } else {
    local_rc = msm_core<CV>(ctx, scalars, on_device, n, opts, tm, !collective);
  }
  if (local_rc && !collective) return local_rc;
  const void* partials = (!collective && n) ? nullptr : ctx->acc_out.p;
  bool peer_failed = false;
  if (collective) {
    NcclApi* api = nccl_api();
    if (!api || !ctx->comm) return fail(ctx, MGB_E_STATE, "sharded msm: the context has no communicator (mgb_comm_init)");
    if (local_rc) {                                         // join the collective all the same, flagged
      local_err = ctx->err;
      ENS(ctx, ctx->acc_out, rec_bytes);                    // (msm_core may have failed before it got that far)
      k_acc_neutral<CV><<<1, 32, 0, ctx->stream>>>((uint32_t*)ctx->acc_out.p);
      CU(ctx, cudaGetLastError());
    }
    CU(ctx, cudaMemsetAsync((char*)ctx->acc_out.p + acc_bytes, local_rc ? 0xff : 0, rec_bytes - acc_bytes, ctx->stream));
    ENS(ctx, ctx->gathered, rec_bytes * ctx->comm_world);
    NC(ctx, api, api->AllGather(ctx->acc_out.p, ctx->gathered.p, rec_bytes, ncclUint8, ctx->comm, ctx->stream));
    partials = ctx->gathered.p;
    if (tm) tm->n_launches += 1;
  }
  int r = normalize_out<CV>(ctx, partials, ctx->comm_world, out_xy, out_is_zero, collective ? REC_LIMBS : CV::ACC_LIMBS, &peer_failed);
  if (r) return r;
  if (tm && partials) tm->n_launches += 1;
  if (ctx->comm) {     // asynchronous NCCL failures (a peer died, a transport error) surface here, not as a hang later
    NcclApi* api = nccl_api();
    ncclResult_t async = ncclSuccess;
    NC(ctx, api, api->CommGetAsyncError(ctx->comm, &async));
    if (async != ncclSuccess) return fail(ctx, MGB_E_COMM, std::string("NCCL asynchronous error: ") + api->GetErrorString(async));
  }
  if (local_rc) return fail(ctx, local_rc, local_err);
  if (peer_failed) return fail(ctx, MGB_E_COMM, "sharded msm: another rank could not compute its shard (its own error says why); no result");
  return n ? finish_timing(ctx, tm) : 0;
}

#define DISPATCH(ctx, fn, ...)                                              \
  switch ((ctx)->curve) {                                                   \
    case MGB_BLS12_377_G1: return fn<CurveBls377>(__VA_ARGS__);             \
    case MGB_PALLAS: return fn<CurvePallas>(__VA_ARGS__);                   \
    case MGB_ED_ON_BLS12_377: return fn<CurveEd377>(__VA_ARGS__);           \
    case MGB_BLS12_381_G1: return fn<CurveBls381>(__VA_ARGS__);             \
    default: return fail(ctx, MGB_E_INVALID, "unknown curve");              \
  }

size_t entry_bytes(int curve) {
  switch (curve) {
    case MGB_BLS12_377_G1: return CurveBls377::ENTRY_LIMBS * 4;
    case MGB_PALLAS: return CurvePallas::ENTRY_LIMBS * 4;
    case MGB_BLS12_381_G1: return CurveBls381::ENTRY_LIMBS * 4;
    default: return CurveEd377::ENTRY_LIMBS * 4;
  }
}

size_t point_bytes(int curve) {   // x||y little-endian bytes of one point in the caller's format
  switch (curve) {
    case MGB_BLS12_377_G1: return 2 * CurveBls377::COORD_BYTES;
    case MGB_PALLAS: return 2 * CurvePallas::COORD_BYTES;
    case MGB_BLS12_381_G1: return 2 * CurveBls381::COORD_BYTES;
    default: return 2 * CurveEd377::COORD_BYTES;
  }
}

int msm_common(mgb_ctx* ctx, const void* scalars, bool dev, size_t n, const mgb_opts* opts, uint8_t* out_xy, int* out_is_zero, mgb_timing* tm) {
  if (!ctx || !out_xy || (!scalars && n)) return fail(ctx, MGB_E_INVALID, "mgb_msm: NULL argument");
  if (n > ctx->npoints) return fail(ctx, ctx->npoints ? MGB_E_INVALID : MGB_E_STATE, "mgb_msm: n exceeds the number of points set");
  if (dev && ((uintptr_t)scalars & 15)) return fail(ctx, MGB_E_INVALID, "mgb_msm_device: the device scalar buffer must be 16-byte aligned");
  CU(ctx, cudaSetDevice(ctx->device));
  if (opts && opts->projective) {
    if (ctx->curve == MGB_BLS12_377_G1) return msm_impl<CurveBls377Basic>(ctx, scalars, dev, n, opts, out_xy, out_is_zero, tm);
    if (ctx->curve == MGB_PALLAS) return msm_impl<CurvePallasBasic>(ctx, scalars, dev, n, opts, out_xy, out_is_zero, tm);
    if (ctx->curve == MGB_BLS12_381_G1) return msm_impl<CurveBls381Basic>(ctx, scalars, dev, n, opts, out_xy, out_is_zero, tm);
  }
  DISPATCH(ctx, msm_impl, ctx, scalars, dev, n, opts, out_xy, out_is_zero, tm);
}

// argument checks + checked ingestion of one context (found: see set_points_checked_impl)
int set_points_checked_ctx(mgb_ctx* ctx, const uint8_t* xy_le, const uint8_t* is_zero, size_t n, uint8_t* status, uint32_t* found) {
  found[0] = found[1] = found[2] = 0;
  if (n > ctx->max_points) return fail(ctx, MGB_E_INVALID, "mgb_set_points_checked: n exceeds max_points");
  CU(ctx, cudaSetDevice(ctx->device));
  ctx->npoints = 0;
  if (n == 0) return 0;
  DISPATCH(ctx, set_points_checked_impl, ctx, xy_le, is_zero, n, status, found);
}

std::string invalid_points_message(uint64_t count, uint64_t first, uint32_t why) {
  const char* reason = (why & MGB_PT_NONCANONICAL) ? "non-canonical encoding (x or y >= p)"
                       : (why & MGB_PT_OFF_CURVE)  ? "not on the curve"
                                                   : "not in the prime-order subgroup";
  return std::to_string(count) + (count == 1 ? " invalid point" : " invalid points") + "; the first is point " + std::to_string(first) + ": " + reason;
}

int multi_fail(mgb_multi* m, int code, const std::string& msg) {
  if (m) m->err = msg;
  g_last_error = msg;
  return code;
}

// contiguous split, the rule of the reference's range() (src/threads/threads.ts:354-359)
void multi_shards(mgb_multi* m, size_t n) {
  const size_t G = m->ctxs.size(), per = (n + G - 1) / G;
  for (size_t g = 0; g < G; g++) { m->lo[g] = std::min(n, per * g); m->hi[g] = std::min(n, m->lo[g] + per); }
  m->npoints = n;
}

// run fn(g) for every device on its own host thread; first non-zero code wins
template <class Fn>
int multi_each(mgb_multi* m, Fn fn) {
  const size_t G = m->ctxs.size();
  std::vector<int> rc(G, 0);
  std::vector<std::thread> th;
  for (size_t g = 1; g < G; g++) th.emplace_back([&, g] { rc[g] = fn(g); });
  rc[0] = fn(0);
  for (auto& t : th) t.join();
  // the root cause first: when one device fails its shard the others report MGB_E_COMM ("another rank could not ...")
  for (int pass = 0; pass < 2; pass++)
    for (size_t g = 0; g < G; g++)
      if (rc[g] && (pass == 1 || rc[g] != MGB_E_COMM)) return multi_fail(m, rc[g], "device " + std::to_string(m->ctxs[g]->device) + ": " + m->ctxs[g]->err);
  return 0;
}

}  // namespace

extern "C" {

int mgb_create(mgb_ctx** out, int curve, int device, size_t max_points) {
  if (!out) return fail(nullptr, MGB_E_INVALID, "mgb_create: out is NULL");
  if (curve < 0 || curve > 3) return fail(nullptr, MGB_E_INVALID, "mgb_create: unknown curve");
  if (max_points == 0 || max_points > (1ull << 28)) return fail(nullptr, MGB_E_INVALID, "mgb_create: max_points must be in [1, 2^28]");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(nullptr, MGB_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(nullptr, MGB_E_INVALID, "mgb_create: bad device index");
  mgb_ctx* ctx = new mgb_ctx();
  ctx->curve = curve;
  ctx->device = device;
  ctx->max_points = max_points;
  int rc = [&]() -> int {
    CU(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(ctx, cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    CU(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    for (int i = 0; i < 3; i++) { CU(ctx, cudaStreamCreateWithFlags(&ctx->aux[i], cudaStreamNonBlocking)); CU(ctx, cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming)); }
    CU(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&ctx->ev_plan, cudaEventDisableTiming));
    for (int i = 0; i < 4; i++) CU(ctx, cudaEventCreateWithFlags(&ctx->ev_chunk[i], cudaEventDisableTiming));
    CU(ctx, cudaStreamCreateWithFlags(&ctx->pf_stream, cudaStreamNonBlocking));
    for (auto& q : ctx->pf) CU(ctx, cudaEventCreateWithFlags(&q.ev, cudaEventDisableTiming));
    for (int i = 0; i < EV_COUNT; i++) CU(ctx, cudaEventCreate(&ctx->ev[i]));
    CU(ctx, cudaMallocHost((void**)&ctx->h_pinned, 256 * 4));
    return ensure(ctx, ctx->table, max_points * entry_bytes(curve));
  }();
  if (rc) { std::string m = ctx->err; mgb_destroy(ctx); return fail(nullptr, rc, m); }
  *out = ctx;
  return 0;
}

int mgb_set_points(mgb_ctx* ctx, const uint8_t* xy_le, const uint8_t* is_zero, size_t n) {
  if (!ctx || (!xy_le && n)) return fail(ctx, MGB_E_INVALID, "mgb_set_points: NULL argument");
  if (n > ctx->max_points) return fail(ctx, MGB_E_INVALID, "mgb_set_points: n exceeds max_points");
  CU(ctx, cudaSetDevice(ctx->device));
  if (n == 0) { ctx->npoints = 0; return 0; }
  DISPATCH(ctx, set_points_impl, ctx, xy_le, is_zero, n);
}

int mgb_set_points_checked(mgb_ctx* ctx, const uint8_t* xy_le, const uint8_t* is_zero, size_t n, uint8_t* status, uint64_t* n_invalid) {
  if (!ctx || (!xy_le && n)) return fail(ctx, MGB_E_INVALID, "mgb_set_points_checked: NULL argument");
  uint32_t found[3];
  int rc = set_points_checked_ctx(ctx, xy_le, is_zero, n, status, found);
  if (rc) return rc;
  if (n_invalid) *n_invalid = found[0];
  if (found[0]) return fail(ctx, MGB_E_INVALID, invalid_points_message(found[0], found[1], found[2]));
  return 0;
}

int mgb_random_points(mgb_ctx* ctx, uint64_t seed, size_t n) {
  if (!ctx) return fail(ctx, MGB_E_INVALID, "mgb_random_points: NULL ctx");
  if (n > ctx->max_points) return fail(ctx, MGB_E_INVALID, "mgb_random_points: n exceeds max_points");
  CU(ctx, cudaSetDevice(ctx->device));
  if (n == 0) { ctx->npoints = 0; return 0; }
  DISPATCH(ctx, random_points_impl, ctx, seed, n);
}

int mgb_get_points(mgb_ctx* ctx, size_t first, size_t n, uint8_t* xy_le, uint8_t* is_zero) {
  if (!ctx || (!xy_le && n)) return fail(ctx, MGB_E_INVALID, "mgb_get_points: NULL argument");
  if (first + n > ctx->npoints) return fail(ctx, MGB_E_INVALID, "mgb_get_points: range exceeds stored points");
  CU(ctx, cudaSetDevice(ctx->device));
  if (n == 0) return 0;
  DISPATCH(ctx, get_points_impl, ctx, first, n, xy_le, is_zero);
}

int mgb_msm(mgb_ctx* ctx, const uint8_t* scalars_le32, size_t n, const mgb_opts* opts, uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing) {
  return msm_common(ctx, scalars_le32, false, n, opts, out_xy_le, out_is_zero, timing);
}
int mgb_msm_device(mgb_ctx* ctx, const void* d_scalars_le32, size_t n, const mgb_opts* opts, uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing) {
  return msm_common(ctx, d_scalars_le32, true, n, opts, out_xy_le, out_is_zero, timing);
}

size_t mgb_partial_bytes(const mgb_ctx* ctx) {
  if (!ctx) return 0;
  switch (ctx->curve) {
    case MGB_BLS12_377_G1: return CurveBls377::ACC_LIMBS * 4;
    case MGB_PALLAS: return CurvePallas::ACC_LIMBS * 4;
    case MGB_BLS12_381_G1: return CurveBls381::ACC_LIMBS * 4;
    default: return CurveEd377::ACC_LIMBS * 4;
  }
}

int mgb_msm_partial(mgb_ctx* ctx, const void* scalars, int scalars_on_device, size_t n, const mgb_opts* opts, void* d_partial_out, mgb_timing* timing) {
  if (!ctx || !d_partial_out || (!scalars && n)) return fail(ctx, MGB_E_INVALID, "mgb_msm_partial: NULL argument");
  if (n > ctx->npoints) return fail(ctx, ctx->npoints ? MGB_E_INVALID : MGB_E_STATE, "mgb_msm_partial: n exceeds the number of points set");
  if (scalars_on_device && ((uintptr_t)scalars & 15)) return fail(ctx, MGB_E_INVALID, "mgb_msm_partial: the device scalar buffer must be 16-byte aligned");
  CU(ctx, cudaSetDevice(ctx->device));
  DISPATCH(ctx, msm_partial_impl, ctx, scalars, scalars_on_device != 0, n, opts, d_partial_out, timing);
}

int mgb_combine_partials(mgb_ctx* ctx, const void* d_partials, int count, uint8_t* out_xy_le, int* out_is_zero) {
  if (!ctx || !d_partials || !out_xy_le || count < 1) return fail(ctx, MGB_E_INVALID, "mgb_combine_partials: bad argument");
  CU(ctx, cudaSetDevice(ctx->device));
  DISPATCH(ctx, normalize_out, ctx, d_partials, count, out_xy_le, out_is_zero);
}

int mgb_comm_unique_id(uint8_t* id_out) {
  if (!id_out) return fail(nullptr, MGB_E_INVALID, "mgb_comm_unique_id: NULL argument");
  NcclApi* api = nccl_api();
  if (!api) return fail(nullptr, MGB_E_COMM, "NCCL library not found (libnccl.so.2; set MGB_NCCL_LIB)");
  static_assert(sizeof(ncclUniqueId) == MGB_COMM_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id;
  NC(nullptr, api, api->GetUniqueId(&id));
  memcpy(id_out, &id, sizeof(id));
  return 0;
}

int mgb_comm_init(mgb_ctx* ctx, const uint8_t* id, int rank, int world) {
  if (!ctx || !id) return fail(ctx, MGB_E_INVALID, "mgb_comm_init: NULL argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, MGB_E_INVALID, "mgb_comm_init: need 0 <= rank < world");
  if (ctx->comm) return fail(ctx, MGB_E_STATE, "mgb_comm_init: the context already has a communicator");
  NcclApi* api = nccl_api();
  if (!api) return fail(ctx, MGB_E_COMM, "NCCL library not found (libnccl.so.2; set MGB_NCCL_LIB)");
  CU(ctx, cudaSetDevice(ctx->device));
  ncclUniqueId uid;
  memcpy(&uid, id, sizeof(uid));
  NC(ctx, api, api->CommInitRank(&ctx->comm, world, uid, rank));
  ctx->comm_rank = rank;
  ctx->comm_world = world;
  return 0;
}

int mgb_comm_info(const mgb_ctx* ctx, int* rank, int* world, int* nccl_version) {
  if (!ctx) return fail(nullptr, MGB_E_INVALID, "mgb_comm_info: NULL ctx");
  if (rank) *rank = ctx->comm_rank;
  if (world) *world = ctx->comm_world;
  if (nccl_version) {
    *nccl_version = 0;
    NcclApi* api = nccl_api();
    if (api) api->GetVersion(nccl_version);
  }
  return 0;
}

int mgb_msm_prefetch(mgb_ctx* ctx, const uint8_t* scalars_le32, size_t n) {
  if (!ctx) return fail(nullptr, MGB_E_INVALID, "null context");
  if (!scalars_le32 || n == 0 || n > ctx->max_points) return fail(ctx, MGB_E_INVALID, "prefetch: scalars must be n <= max_points 32-byte words");
  CU(ctx, cudaSetDevice(ctx->device));
  mgb_ctx::Prefetch* slot = nullptr;
  for (auto& q : ctx->pf)
    if (q.valid && q.host == scalars_le32) slot = &q;          // the same host buffer again: upload it again (contents may have changed)
  if (slot) CU(ctx, cudaEventSynchronize(slot->ev));
  for (auto& q : ctx->pf)
    if (!slot && !q.valid) slot = &q;
  if (!slot) return fail(ctx, MGB_E_INVALID, "prefetch: two scalar sets are already waiting for their MSM");
  ENS(ctx, slot->buf, n * 32);
  slot->host = scalars_le32;
  slot->n = n;
  slot->valid = true;
  slot->issued = false;
  // The upload itself is started by the NEXT MSM call of this context, right behind the launch of its first tree round
  // (issue_prefetches): started here, at once, it would run next to that call's digit / sort phase and slow it down
  // (measured at 4 GPUs, 2^20 per GPU: pipelined step 6.05 ms against 5.93 ms; the device-resident step takes 5.91 ms).
  return 0;
}

int mgb_msm_sharded(mgb_ctx* ctx, const void* scalars, int scalars_on_device, size_t n_local, const mgb_opts* opts,
                    uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing) {
  if (!ctx || !out_xy_le || (!scalars && n_local)) return fail(ctx, MGB_E_INVALID, "mgb_msm_sharded: NULL argument");
  if (opts && opts->projective) return fail(ctx, MGB_E_INVALID, "mgb_msm_sharded: the projective cross-check path is single-GPU only");   // (the same on every rank)
  // argument errors that only THIS rank may have: with a communicator the rank still joins the collective, flagged, so
  // that its peers return MGB_E_COMM instead of waiting for it (msm_sharded_impl)
  int pre = 0;
  if (n_local > ctx->npoints) pre = fail(ctx, ctx->npoints ? MGB_E_INVALID : MGB_E_STATE, "mgb_msm_sharded: n_local exceeds the number of points set");
  else if (scalars_on_device && ((uintptr_t)scalars & 15)) pre = fail(ctx, MGB_E_INVALID, "mgb_msm_sharded: the device scalar buffer must be 16-byte aligned");
  if (pre && ctx->comm_world == 1) return pre;
  CU(ctx, cudaSetDevice(ctx->device));
  DISPATCH(ctx, msm_sharded_impl, ctx, scalars, scalars_on_device != 0, n_local, opts, out_xy_le, out_is_zero, timing, pre);
}

/* ---- one host process driving several GPUs (SURVEY 8b: `device_ids, n_devices`) ---- */
int mgb_multi_create(mgb_multi** out, int curve, const int* device_ids, int n_devices, size_t max_points_per_device) {
  if (!out || !device_ids || n_devices < 1) return multi_fail(nullptr, MGB_E_INVALID, "mgb_multi_create: bad argument");
  mgb_multi* m = new mgb_multi();
  m->lo.assign(n_devices, 0);
  m->hi.assign(n_devices, 0);
  for (int g = 0; g < n_devices; g++) {
    mgb_ctx* c = nullptr;
    int rc = mgb_create(&c, curve, device_ids[g], max_points_per_device);
    if (rc) { std::string e = g_last_error; mgb_multi_destroy(m); return multi_fail(nullptr, rc, e); }
    m->ctxs.push_back(c);
  }
  if (n_devices > 1) {
    NcclApi* api = nccl_api();
    if (!api) { mgb_multi_destroy(m); return multi_fail(nullptr, MGB_E_COMM, "NCCL library not found (libnccl.so.2; set MGB_NCCL_LIB)"); }
    std::vector<ncclComm_t> comms(n_devices);
    ncclResult_t r = api->CommInitAll(comms.data(), n_devices, device_ids);
    if (r != ncclSuccess) { std::string e = api->GetErrorString(r); mgb_multi_destroy(m); return multi_fail(nullptr, MGB_E_COMM, "ncclCommInitAll: " + e); }
    for (int g = 0; g < n_devices; g++) { m->ctxs[g]->comm = comms[g]; m->ctxs[g]->comm_rank = g; m->ctxs[g]->comm_world = n_devices; }
  }
  *out = m;
  return 0;
}

int mgb_multi_set_points(mgb_multi* m, const uint8_t* xy_le, const uint8_t* is_zero, size_t n) {
  if (!m || (!xy_le && n)) return multi_fail(m, MGB_E_INVALID, "mgb_multi_set_points: NULL argument");
  multi_shards(m, n);
  const size_t pb = point_bytes(m->ctxs[0]->curve);              // x||y bytes of one point
  return multi_each(m, [&](size_t g) {
    return mgb_set_points(m->ctxs[g], xy_le + m->lo[g] * pb, is_zero ? is_zero + m->lo[g] : nullptr, m->hi[g] - m->lo[g]);
  });
}

int mgb_multi_set_points_checked(mgb_multi* m, const uint8_t* xy_le, const uint8_t* is_zero, size_t n, uint8_t* status, uint64_t* n_invalid) {
  if (!m || (!xy_le && n)) return multi_fail(m, MGB_E_INVALID, "mgb_multi_set_points_checked: NULL argument");
  multi_shards(m, n);
  const size_t G = m->ctxs.size(), pb = point_bytes(m->ctxs[0]->curve);
  std::vector<uint32_t> found(3 * G, 0);
  int rc = multi_each(m, [&](size_t g) {
    return set_points_checked_ctx(m->ctxs[g], xy_le + m->lo[g] * pb, is_zero ? is_zero + m->lo[g] : nullptr, m->hi[g] - m->lo[g],
                                  status ? status + m->lo[g] : nullptr, &found[3 * g]);
  });
  uint64_t count = 0, first = 0;
  uint32_t why = 0;
  for (size_t g = G; g-- > 0;)                                      // the lowest shard with an invalid point names the first
    if (found[3 * g]) { count += found[3 * g]; first = m->lo[g] + found[3 * g + 1]; why = found[3 * g + 2]; }
  if (rc || count) {                                                // no device keeps its shard
    for (mgb_ctx* c : m->ctxs) c->npoints = 0;
    m->npoints = 0;
  }
  if (rc) return rc;
  if (n_invalid) *n_invalid = count;
  if (count) return multi_fail(m, MGB_E_INVALID, invalid_points_message(count, first, why));
  return 0;
}

int mgb_multi_random_points(mgb_multi* m, uint64_t seed, size_t n) {
  if (!m) return multi_fail(m, MGB_E_INVALID, "mgb_multi_random_points: NULL argument");
  multi_shards(m, n);
  // shard g is the point set of seed + g (as the one-process-per-GPU host layer does): the union is the global set
  return multi_each(m, [&](size_t g) { return mgb_random_points(m->ctxs[g], seed + g, m->hi[g] - m->lo[g]); });
}

int mgb_multi_get_points(mgb_multi* m, size_t first, size_t n, uint8_t* xy_le, uint8_t* is_zero) {
  if (!m || (!xy_le && n)) return multi_fail(m, MGB_E_INVALID, "mgb_multi_get_points: NULL argument");
  if (first + n > m->npoints) return multi_fail(m, MGB_E_INVALID, "mgb_multi_get_points: range exceeds stored points");
  const size_t pb = point_bytes(m->ctxs[0]->curve);
  for (size_t g = 0; g < m->ctxs.size(); g++) {
    const size_t a = std::max(first, m->lo[g]), b = std::min(first + n, m->hi[g]);
    if (a >= b) continue;
    int rc = mgb_get_points(m->ctxs[g], a - m->lo[g], b - a, xy_le + (a - first) * pb, is_zero ? is_zero + (a - first) : nullptr);
    if (rc) return multi_fail(m, rc, m->ctxs[g]->err);
  }
  return 0;
}

int mgb_multi_msm(mgb_multi* m, const uint8_t* scalars_le32, size_t n, const mgb_opts* opts, uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing) {
  if (!m || !out_xy_le || (!scalars_le32 && n)) return multi_fail(m, MGB_E_INVALID, "mgb_multi_msm: NULL argument");
  if (n > m->npoints) return multi_fail(m, m->npoints ? MGB_E_INVALID : MGB_E_STATE, "mgb_multi_msm: n exceeds the number of points set");
  // every device takes the pairs of ITS point shard that lie below n; every rank ends with the full sum, device 0 reports it
  std::vector<std::vector<uint8_t>> scratch(m->ctxs.size(), std::vector<uint8_t>(256));
  std::vector<int> zero(m->ctxs.size(), 0);
  return multi_each(m, [&](size_t g) {
    const size_t lo = std::min(n, m->lo[g]), hi = std::min(n, m->hi[g]);
    return mgb_msm_sharded(m->ctxs[g], scalars_le32 + lo * 32, 0, hi - lo, opts, g == 0 ? out_xy_le : scratch[g].data(),
                           g == 0 ? out_is_zero : &zero[g], g == 0 ? timing : nullptr);
  });
}

const char* mgb_multi_last_error(const mgb_multi* m) { return m ? m->err.c_str() : g_last_error.c_str(); }

void mgb_multi_destroy(mgb_multi* m) {
  if (!m) return;
  for (mgb_ctx* c : m->ctxs) mgb_destroy(c);
  delete m;
}

const char* mgb_last_error(const mgb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

void mgb_destroy(mgb_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->comm) { if (NcclApi* api = nccl_api()) api->CommDestroy(ctx->comm); ctx->comm = nullptr; }
  if (ctx->gathered.p) cudaFree(ctx->gathered.p);
  DevBuf* bufs[] = {&ctx->table, &ctx->scalars, &ctx->ent_bucket, &ctx->ent_rank, &ctx->counts, &ctx->offs, &ctx->offcnt, &ctx->tile_sums, &ctx->pairs, &ctx->pairs2, &ctx->V, &ctx->W, &ctx->recs, &ctx->lifes, &ctx->prebuf, &ctx->bsum, &ctx->redU[0], &ctx->redU[1], &ctx->redW[0], &ctx->redW[1], &ctx->misc,
                    &ctx->acc_out, &ctx->out_xy, &ctx->stage, &ctx->checks};
  for (DevBuf* b : bufs) if (b->p) cudaFree(b->p);
  for (auto& q : ctx->pf) { if (q.buf.p) cudaFree(q.buf.p); if (q.ev) cudaEventDestroy(q.ev); }
  if (ctx->pf_stream) cudaStreamDestroy(ctx->pf_stream);
  if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
  for (int i = 0; i < EV_COUNT; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  for (int i = 0; i < 3; i++) { if (ctx->aux[i]) cudaStreamDestroy(ctx->aux[i]); if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]); }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_plan) cudaEventDestroy(ctx->ev_plan);
  for (int i = 0; i < 4; i++) if (ctx->ev_chunk[i]) cudaEventDestroy(ctx->ev_chunk[i]);
  delete ctx;
}

}  // extern "C"
