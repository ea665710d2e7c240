/* montgomery_b200 -- C ABI of the B200-native MSM engine.
 *
 * This is the drop-in boundary for the MSM hot path of mitschabaude/montgomery.  The reference has
 * no FFI: its seam is the TypeScript object built by `createMsm` / `createMsmBasic` and registered
 * as `Parallel.msm / msmUnsafe` (src/msm-batched-affine.ts:45-51,585-599, src/msm-basic.ts:34-43,
 * src/parallel.ts:135-145,251-259), plus the value-typed `compute_msm(points, scalars)` wrappers
 * (scripts/zprize23/submission-bls377.ts:20-65, scripts/zprize23/submission.ts:19-35).  Each entry
 * point below names the reference interface it replaces.  INTEGRATION.md shows the N-API / ctypes
 * bindings that sit on top.
 *
 * Conventions: every function returns 0 on success and a negative MGB_E_* code on failure (never
 * throws or aborts across the ABI); `mgb_last_error` gives the message.  The caller owns all host
 * buffers; the context owns all device memory and its stream.  One in-flight call per context.
 * Byte formats are the reference's (src/parallel.ts:97-133,209-249): scalar = 32 bytes little
 * endian; Weierstrass point = x||y, each ceil(bits/8) bytes LE (2*48 for BLS12-377 / BLS12-381, 2*32 for
 * Pallas); twisted-Edwards point = x||y, 2*32 bytes LE.  The result is the canonical affine point
 * (coordinates in [0,p), LE) plus an is_zero flag (Weierstrass infinity -> x = y = 0, flag 1, as
 * src/curve-affine.ts:369-371; twisted-Edwards neutral -> (0,1), flag 1).
 */
#ifndef MONTGOMERY_B200_H
#define MONTGOMERY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mgb_ctx mgb_ctx;

enum mgb_curve {
  MGB_BLS12_377_G1 = 0,     /* src/concrete/bls12-377.params.ts, msm-batched-affine + GLV   */
  MGB_PALLAS = 1,           /* src/concrete/pasta.params.ts, msm-batched-affine + GLV       */
  MGB_ED_ON_BLS12_377 = 2,  /* src/concrete/ed-on-bls12-377.params.ts, msm-basic, no GLV    */
  MGB_BLS12_381_G1 = 3      /* src/concrete/bls12-381.params.ts, msm-batched-affine + GLV   */
};

enum mgb_error {
  MGB_OK = 0,
  MGB_E_INVALID = -1,   /* bad argument (null pointer, n > capacity, unknown curve, c out of range) */
  MGB_E_CUDA = -2,      /* a CUDA runtime call failed; message has the CUDA error string             */
  MGB_E_NOMEM = -3,     /* device memory exhausted (the reference's "memory overflow" error,
                           src/wasm/memory-helpers.ts:225-236)                                         */
  MGB_E_STATE = -4,     /* msm called before points were set / sharded msm without a communicator     */
  MGB_E_COMM = -5       /* NCCL: library not found, communicator set-up or collective failed, an asynchronous
                           error reported by ncclCommGetAsyncError, or (mgb_msm_sharded) ANOTHER rank could not
                           compute its shard -- that rank returns its own error code                    */
};

/* Per-call options; mirrors `{c?, useSafeAdditions?}` of msm-batched-affine.ts:74-77 and
 * `{c?}` of msm-basic.ts:35-41.  c = 0 picks the engine's window size.  `unsafe` is accepted for
 * API parity with `msmUnsafe`; the engine's additions are always complete, so it changes nothing.
 * `projective` = 1 selects the reference's `msmProjective` variant on Weierstrass curves
 * (src/parallel.ts:69-87: msm-basic over projective coordinates, no GLV, no batched-affine
 * additions) -- an independent path used as a cross-check, as in src/msm.test.ts:73-82. */
typedef struct mgb_opts {
  int c;
  int unsafe;
  int verbose;
  int projective;
  int affine_reduction;   /* 1: bucket reduction by batched-affine additions (the reference's `reduceBucketsAffine`
                             experiment, src/msm-batched-affine-single-thread.ts:522-700); batched-affine curves only,
                             same result, slower on a B200 than the default (kept as a measured alternative) */
} mgb_opts;

/* Per-phase device times in milliseconds (CUDA events on the context's stream); the analogue of
 * the `log` array returned by msm() (src/msm-common.ts:176-213) with the same phase boundaries. */
typedef struct mgb_timing {
  float h2d_scalars;        /* host->device copy of the scalars when it is one copy on the main stream (n < 2^16); larger
                               inputs upload in chunks overlapped with decompose_slice, which then includes the transfer */
  float decompose_slice;    /* "prepare points & scalars" + "slice scalars & count buckets"          */
  float sort;               /* "integrate bucket counts" + "sort points"                             */
  float accumulate;         /* "bucket accumulation"                                                  */
  float reduce;             /* "normalize bucket storage" + "bucket reduction" (incl. the sums of the bucket leftovers) */
  float final_sum;          /* "partition sum" + "final sum" + affine normalisation                   */
  float total;              /* whole call on the device, first kernel to result available             */
  int c, K, rounds;         /* window bits, number of windows, accumulation rounds                    */
  uint32_t max_bucket;      /* largest bucket (maxBucketSize, msm-batched-affine.ts:208)             */
  uint64_t n_pairs;         /* additions performed by the tree rounds of the accumulation phase      */
  uint32_t n_launches;      /* kernels launched by this call                                          */
} mgb_timing;

/* Replaces `Weierstrass.create(params)` / `TwistedEdwards.create(params)` + `startThreads()`
 * (src/parallel.ts:40,179,291): builds the engine for one curve on one GPU.  `max_points` bounds n
 * of later calls (the reference bounds it by its 4 GiB wasm memory, src/field-msm.ts:55-56). */
int mgb_create(mgb_ctx** out, int curve, int device, size_t max_points);

/* Replaces `Parallel.pointsFromBytes` (src/parallel.ts:97-116, :209-232): uploads n points given as
 * x||y LE bytes and converts them to the device layout (Montgomery form).  `is_zero` is optional
 * (NULL = no point at infinity, as in the reference's byte format); a non-zero byte marks point i
 * as the neutral element (the reference's `isNonZero` flag, src/curve-affine.ts:20-52). */
int mgb_set_points(mgb_ctx* ctx, const uint8_t* xy_le, const uint8_t* is_zero, size_t n);

/* mgb_set_points for points from outside (SRS files, another library's output, bytes off the wire): the same
 * ingestion, and every point is checked on the device as it is ingested -- the reference's `isOnCurve` and
 * `isInSubgroup` of its curve types (src/curve-projective.ts, src/curve-twisted-edwards.ts), one thread per point.
 * Each point gets a status byte, a mask of the MGB_PT_* bits below (0 = valid; a point flagged in is_zero is valid
 * whatever its coordinate bytes are).  A non-canonical encoding gets MGB_PT_NONCANONICAL alone; the curve equation is
 * checked on canonical points, and MGB_PT_NOT_IN_SUBGROUP is set only for points on the curve.  Subgroup tests:
 * Pallas has cofactor 1; BLS12-377 / BLS12-381 G1 test sigma'(P) + P == [z^2] P with the endomorphism of eigenvalue
 * z^2 - 1 (exact, DESIGN.md "Checked point ingestion"); ed-on-BLS12-377 tests [q] P == O.
 * All points valid: returns MGB_OK and stores the table mgb_set_points would store from the same bytes.
 * Any point invalid: returns MGB_E_INVALID, mgb_last_error names the count and the first invalid index with its reason,
 * and the context holds NO points afterwards (mgb_msm returns MGB_E_STATE, as on a fresh context).
 * `status` (n bytes) and `n_invalid` may be NULL; the count and the first index are kept on the device either way.
 * Device memory: one byte per point plus 8 bytes, allocated by the first call and kept by the context. */
#define MGB_PT_NONCANONICAL 1      /* x or y >= p (from the raw bytes)                                       */
#define MGB_PT_OFF_CURVE 2         /* the point does not satisfy the curve equation                          */
#define MGB_PT_NOT_IN_SUBGROUP 4   /* on the curve, not in the prime-order subgroup                          */
int mgb_set_points_checked(mgb_ctx* ctx, const uint8_t* xy_le, const uint8_t* is_zero, size_t n,
                           uint8_t* status /* n bytes, may be NULL */, uint64_t* n_invalid /* may be NULL */);

/* Replaces `Parallel.randomPointsFast(n)` (src/curve-random.ts:24-92): fills the context with n
 * points a_i*G, a_i a seeded 64-bit value (splitmix64 of seed and i), built on the device from
 * a 64-step double-and-add of the generator, one thread per point.  Deterministic; used for benchmarks
 * and closed-form checks. */
int mgb_random_points(mgb_ctx* ctx, uint64_t seed, size_t n);

/* Reads back points [first, first+n) as canonical x||y LE bytes (`Affine.toBigint`,
 * src/curve-affine.ts:220-233); is_zero may be NULL. */
int mgb_get_points(mgb_ctx* ctx, size_t first, size_t n, uint8_t* xy_le, uint8_t* is_zero);

/* Replaces `Parallel.msm / msmUnsafe(scalarPtr, pointPtr, N)` followed by `Projective.toAffine` +
 * `Affine.toBigint` (src/msm-batched-affine.ts:69-340, scripts/msm-weierstrass.ts:90-92), or
 * `msmBasic` + `toAffine` for the twisted-Edwards curve (src/msm-basic.ts:45-164).  Scalars are n
 * host values of 32 bytes LE, paired with the first n points of the context.  n = 0 gives the
 * neutral element.  opts and timing may be NULL. */
int mgb_msm(mgb_ctx* ctx, const uint8_t* scalars_le32, size_t n, const mgb_opts* opts,
            uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing);

/* Registers a host scalar set for upload AHEAD of its MSM and returns at once.  The copy is started by the next MSM call
 * of this context, behind the launch of its first tree round, and runs on its own stream while that MSM computes (started
 * any earlier it would slow the bandwidth-bound digit / sort phase down).  The following mgb_msm / mgb_msm_partial /
 * mgb_msm_sharded call whose host pointer and n are the ones given here uses the uploaded copy instead of transferring
 * again; if no MSM ran in between, that call simply uploads the set itself.  The reference has no counterpart (its
 * scalars already live in the Wasm memory, src/msm-batched-affine.ts:69-75); a prover that calls `msm` for one polynomial
 * after another calls mgb_msm_prefetch(set i + 1) before mgb_msm(set i).  The buffer must stay unchanged until the MSM
 * call that consumes it returns (page-locked memory for a truly asynchronous copy); at most two sets wait at a time
 * (MGB_E_INVALID beyond that); registering the same pointer again replaces the earlier registration. */
int mgb_msm_prefetch(mgb_ctx* ctx, const uint8_t* scalars_le32, size_t n);

/* Same with scalars already in device memory (device pointer), for kernel-only timing.
 * Contract for caller-owned device scalars (here and in mgb_msm_partial / mgb_msm_sharded with
 * scalars_on_device): the pointer must be 16-byte aligned (128-bit loads) and the data must be
 * complete before the call -- the engine reads it on its own non-blocking stream, which is not
 * ordered after the stream that produced it, so synchronise the producer first. */
int mgb_msm_device(mgb_ctx* ctx, const void* d_scalars_le32, size_t n, const mgb_opts* opts,
                   uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing);

/* Multi-GPU building blocks for a host layer that runs the collective itself: each rank runs the
 * MSM on its shard and leaves the partial sum, un-normalised, in a caller-provided DEVICE buffer of
 * mgb_partial_bytes() bytes; mgb_combine_partials adds `count` gathered partials (device buffer)
 * and normalises.  n = 0 writes the neutral element.  (mgb_msm_sharded below does all of it inside
 * the library and is what the bench uses.) */
size_t mgb_partial_bytes(const mgb_ctx* ctx);
int mgb_msm_partial(mgb_ctx* ctx, const void* scalars, int scalars_on_device, size_t n,
                    const mgb_opts* opts, void* d_partial_out, mgb_timing* timing);
int mgb_combine_partials(mgb_ctx* ctx, const void* d_partials, int count,
                         uint8_t* out_xy_le, int* out_is_zero);

/* Sharded MSM with the collective inside the library (SURVEY 8b/8e: "ctx owns ... the NCCL
 * communicator").  Replaces the SPMD split of src/threads/threads.ts:354-359 plus the sum of the
 * per-thread partial results on the main thread (src/msm-batched-affine.ts:311-320).
 *
 * One process per GPU: rank 0 calls mgb_comm_unique_id and hands the MGB_COMM_ID_BYTES bytes to the other
 * ranks by any host channel (MPI, a TCP store, torch.distributed's broadcast, a worker message);
 * every rank then calls mgb_comm_init(ctx, id, rank, world) on its own context (collective: returns
 * when all ranks have joined).  mgb_msm_sharded runs the MSM of the rank's shard (n_local pairs:
 * the rank's scalars against the first n_local points of ITS context; 0 is allowed and contributes
 * the neutral element), then -- on the engine's stream, with no host round trip in between -- ONE
 * ncclAllGather of the un-normalised partial accumulators and one kernel that adds them and
 * normalises.  Every rank receives the same canonical result.  NCCL is bound at run time
 * (dlopen of libnccl.so.2, or the path in MGB_NCCL_LIB): single-GPU hosts do not need it.
 * A context with no communicator (world 1) computes the plain MSM.
 * Failure of one rank (a scalar out of range, a window size that does not fit, device memory): the
 * status travels with the data -- the failing rank still joins the all-gather (neutral element,
 * flagged) and returns its own error; every other rank returns MGB_E_COMM and no result.  Nobody
 * is left waiting in the collective, and nobody gets a sum that misses a shard.  The same holds for
 * the argument errors a single rank can make (n_local above the points it holds, a misaligned device
 * buffer); only NULL pointers and the `projective` option -- identical on all ranks -- return at once.  The reference's workers share one exception through the
 * barrier timeout of src/threads/threads.ts:319-330. */
#define MGB_COMM_ID_BYTES 128
int mgb_comm_unique_id(uint8_t* id_out /* MGB_COMM_ID_BYTES */);
int mgb_comm_init(mgb_ctx* ctx, const uint8_t* id /* MGB_COMM_ID_BYTES */, int rank, int world);
int mgb_comm_info(const mgb_ctx* ctx, int* rank, int* world, int* nccl_version);   /* any out pointer may be NULL */
int mgb_msm_sharded(mgb_ctx* ctx, const void* scalars, int scalars_on_device, size_t n_local,
                    const mgb_opts* opts, uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing);

/* One host process driving several GPUs (the shape a Node / TypeScript host needs: it cannot reach
 * an MPI-style launcher).  mgb_multi_create builds one context per listed device and the
 * communicators (ncclCommInitAll); the point set is split contiguously over the devices by the
 * reference's `range()` rule (src/threads/threads.ts:354-359); mgb_multi_msm pairs the first n
 * scalars with the first n points, each device working on the part of its shard below n (one
 * host thread per device), and returns the canonical sum.  mgb_multi_random_points gives shard g
 * the known-dlog points of seed + g. */
typedef struct mgb_multi mgb_multi;
int mgb_multi_create(mgb_multi** out, int curve, const int* device_ids, int n_devices, size_t max_points_per_device);
int mgb_multi_set_points(mgb_multi* m, const uint8_t* xy_le, const uint8_t* is_zero, size_t n);
/* mgb_set_points_checked over the shards (isOnCurve / isInSubgroup of the reference): every device checks its shard at
 * the same time; status, the count and the first index in the message are global.  If any shard holds an invalid point,
 * returns MGB_E_INVALID and EVERY device is left without points. */
int mgb_multi_set_points_checked(mgb_multi* m, const uint8_t* xy_le, const uint8_t* is_zero, size_t n,
                                 uint8_t* status /* n bytes, may be NULL */, uint64_t* n_invalid /* may be NULL */);
int mgb_multi_random_points(mgb_multi* m, uint64_t seed, size_t n);
int mgb_multi_get_points(mgb_multi* m, size_t first, size_t n, uint8_t* xy_le, uint8_t* is_zero);
int mgb_multi_msm(mgb_multi* m, const uint8_t* scalars_le32, size_t n, const mgb_opts* opts,
                  uint8_t* out_xy_le, int* out_is_zero, mgb_timing* timing /* device 0's phases */);
const char* mgb_multi_last_error(const mgb_multi* m);
void mgb_multi_destroy(mgb_multi* m);

/* Test hooks for the field layer (the analogue of the Wasm exports checked by src/field.test.ts):
 * applies op elementwise on the device to n elements given as canonical LE bytes in/out.
 * field: 0 = BLS12-377 Fp, 1 = BLS12-377 Fr (= ed-on-377 base field), 2 = Pallas Fp, 3 = BLS12-381 Fp.
 * op: 0 mul, 1 add, 2 sub, 3 inverse (Fermat), 4 square, 5 inverse (binary gcd), 6 negate,
 * 7 inverse (division steps, the one the MSM uses), 8 mul by the warp-cooperative routine (one limb per
 * lane, csrc/warp.cuh; b is the second factor), 9 inverse by the lane-parallel division-step routine of
 * csrc/warp.cuh (the one every tile of the accumulation and the final normalisation use). */
int mgb_field_op(int device, int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);

/* Integer-pipe microbenchmarks (roofline denominator).  mode: 0 = mad.lo.u32 (IMAD), 1 = mad.hi.u32,
 * 2 = mad.wide.u32 with 64-bit accumulate, 3 = mad.lo.cc/madc.hi.cc carry chain (IMAD.WIDE.U32.X:
 * the full 32x32+64->64 multiply-accumulate the field multiplication is made of), 4/5 = Fp377 /
 * Fr377 Montgomery multiplications through the out-of-line call, 6/7 = the same inlined, 8/9 = chains
 * of Fp377 division-step inversions on all lanes / on lane 0 of each warp (threads <= 128), 10/11 = a
 * dependent chain of Fp377 products on a warp running alone: lane 0 with the per-thread routine / all
 * lanes with the warp-cooperative one (ms / (2 iters) = latency of one product), 12 = like 9 with the
 * lane-parallel inverse (one inversion per warp, all lanes working), 13 = Fp377 products two per call, their
 * instruction streams free to interleave (instruction-level parallelism for a warp that runs alone).  All
 * multiplicands change every iteration (a loop-invariant product would be hoisted by ptxas).
 * Returns operations per second (lane operations for modes 0-3, field multiplications for 4-7) in
 * *ops_per_s and the kernel time in *ms. */
int mgb_microbench(int device, int mode, int blocks_per_sm, int threads, int iters, double* ops_per_s, float* ms);

const char* mgb_last_error(const mgb_ctx* ctx);   /* ctx may be NULL: last error of a ctx-less call */
void mgb_destroy(mgb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* MONTGOMERY_B200_H */
