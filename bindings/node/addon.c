/* N-API addon over include/montgomery_b200.h -- the "thin C-ABI N-API addon" between montgomery's
 * TypeScript API and the CUDA engine.  Plain C, node_api.h only (no node-addon-api, no C++).
 *
 * NOT BUILT IN THIS REPOSITORY'S IMAGE: there is no Node.js (nor its headers) in it.  A maintainer builds it
 * with node-gyp (binding.gyp next to this file); index.ts is the TypeScript face that mirrors the reference's
 * Parallel.msm / compute_msm on top of these exports.
 *
 * Exports (all take the context handle returned by create):
 *   create(curve, device, maxPoints) -> External            mgb_create        (Weierstrass.create + startThreads)
 *   setPoints(ctx, Uint8Array xy, n[, check])                mgb_set_points    (Parallel.pointsFromBytes); check = 1:
 *                                                            mgb_set_points_checked (isOnCurve / isInSubgroup of every
 *                                                            point on the GPU), throws its message on an invalid point
 *   randomPoints(ctx, seed, n)                               mgb_random_points (Parallel.randomPointsFast)
 *   msm(ctx, Uint8Array scalars, n, c, projective) -> Promise<{xy: Uint8Array, isZero, log}>
 *                                                            mgb_msm on a libuv worker thread, so the event loop is
 *                                                            never blocked (the reference's msm is async as well)
 *   createMulti(curve, Int32Array deviceIds, maxPointsPerDevice) -> External      mgb_multi_create: ONE Node process drives
 *   setPointsMulti(mctx, Uint8Array xy, n) / randomPointsMulti(mctx, seed, n)      several GPUs (contexts + NCCL communicators
 *   msmSharded(mctx, Uint8Array scalars, n, c) -> Promise<{xy, isZero, log}>       inside the library; replaces startThreads(n) +
 *                                                            the per-thread split of src/threads/threads.ts:354-359)
 * The context is released by its finaliser (mgb_destroy, the analogue of stopThreads) when the handle is collected.
 * Errors become JS exceptions / rejected promises carrying mgb_last_error's text.  One in-flight msm per context.
 */
#include <node_api.h>
#include <stdlib.h>
#include <string.h>
#include "montgomery_b200.h"

#define CHECK(call) do { if ((call) != napi_ok) { napi_throw_error(env, NULL, "N-API call failed: " #call); return NULL; } } while (0)

static mgb_ctx* ctx_of(napi_env env, napi_value v) {
  void* p = NULL;
  if (napi_get_value_external(env, v, &p) != napi_ok || !p) { napi_throw_type_error(env, NULL, "expected an engine handle"); return NULL; }
  return (mgb_ctx*)p;
}
static void ctx_finalize(napi_env env, void* data, void* hint) { (void)env; (void)hint; mgb_destroy((mgb_ctx*)data); }

static napi_value Create(napi_env env, napi_callback_info info) {
  size_t argc = 3; napi_value argv[3]; int32_t curve, device; int64_t max_points; mgb_ctx* ctx = NULL; napi_value out;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  CHECK(napi_get_value_int32(env, argv[0], &curve));
  CHECK(napi_get_value_int32(env, argv[1], &device));
  CHECK(napi_get_value_int64(env, argv[2], &max_points));
  if (mgb_create(&ctx, curve, device, (size_t)max_points) != MGB_OK) { napi_throw_error(env, NULL, mgb_last_error(NULL)); return NULL; }
  CHECK(napi_create_external(env, ctx, ctx_finalize, NULL, &out));
  return out;
}

static napi_value SetPoints(napi_env env, napi_callback_info info) {
  size_t argc = 4, len; napi_value argv[4]; void* data; int64_t n; int32_t check = 0; napi_typedarray_type ty; mgb_ctx* ctx;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (argc >= 4) CHECK(napi_get_value_int32(env, argv[3], &check));
  if (!(ctx = ctx_of(env, argv[0]))) return NULL;
  CHECK(napi_get_typedarray_info(env, argv[1], &ty, &len, &data, NULL, NULL));
  CHECK(napi_get_value_int64(env, argv[2], &n));
  if (ty != napi_uint8_array) { napi_throw_type_error(env, NULL, "points: Uint8Array of x||y little-endian"); return NULL; }
  if (n < 0 || len % 64 != 0 || (n > 0 && len / (size_t)n != 64 && len / (size_t)n != 96) || len % (size_t)(n > 0 ? n : 1) != 0) {
    napi_throw_range_error(env, NULL, "points: the buffer must hold exactly n points of 2 * 32 or 2 * 48 bytes");   /* never read past the array */
    return NULL;
  }
  if ((check ? mgb_set_points_checked(ctx, (const uint8_t*)data, NULL, (size_t)n, NULL, NULL)
             : mgb_set_points(ctx, (const uint8_t*)data, NULL, (size_t)n)) != MGB_OK)
    napi_throw_error(env, NULL, mgb_last_error(ctx));
  return NULL;
}

static napi_value RandomPoints(napi_env env, napi_callback_info info) {
  size_t argc = 3; napi_value argv[3]; int64_t seed, n; mgb_ctx* ctx;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (!(ctx = ctx_of(env, argv[0]))) return NULL;
  CHECK(napi_get_value_int64(env, argv[1], &seed));
  CHECK(napi_get_value_int64(env, argv[2], &n));
  if (mgb_random_points(ctx, (uint64_t)seed, (size_t)n) != MGB_OK) napi_throw_error(env, NULL, mgb_last_error(ctx));
  return NULL;
}

/* ---- msm on a worker thread */
typedef struct {
  napi_async_work work; napi_deferred deferred; napi_ref scalars_ref;
  mgb_ctx* ctx; mgb_multi* multi; const uint8_t* scalars; size_t n; mgb_opts opts;
  uint8_t out[96]; int is_zero; mgb_timing tm; int rc; char err[256];
} msm_job;

static void msm_execute(napi_env env, void* data) {
  msm_job* j = (msm_job*)data; (void)env;
  j->rc = mgb_msm(j->ctx, j->scalars, j->n, &j->opts, j->out, &j->is_zero, &j->tm);
  if (j->rc != MGB_OK) { strncpy(j->err, mgb_last_error(j->ctx), sizeof j->err - 1); j->err[sizeof j->err - 1] = 0; }
}
static void set_num(napi_env env, napi_value obj, const char* k, double v) { napi_value x; napi_create_double(env, v, &x); napi_set_named_property(env, obj, k, x); }
static void msm_complete(napi_env env, napi_status status, void* data) {
  msm_job* j = (msm_job*)data; napi_value res, xy, log, flag, msg, errv; void* buf; (void)status;
  if (j->rc != MGB_OK) {
    napi_create_string_utf8(env, j->err, NAPI_AUTO_LENGTH, &msg); napi_create_error(env, NULL, msg, &errv);
    napi_reject_deferred(env, j->deferred, errv);
  } else {
    napi_value ab;
    napi_create_object(env, &res);
    napi_create_arraybuffer(env, 96, &buf, &ab); memcpy(buf, j->out, 96);
    napi_create_typedarray(env, napi_uint8_array, 96, ab, 0, &xy);       /* x||y LE, coordinates padded to 48 bytes */
    napi_set_named_property(env, res, "xy", xy);
    napi_get_boolean(env, j->is_zero != 0, &flag); napi_set_named_property(env, res, "isZero", flag);
    napi_create_object(env, &log);                                        /* the phase log of src/msm-common.ts:176-213 */
    set_num(env, log, "decomposeSlice", j->tm.decompose_slice); set_num(env, log, "sort", j->tm.sort);
    set_num(env, log, "accumulate", j->tm.accumulate); set_num(env, log, "reduce", j->tm.reduce);
    set_num(env, log, "finalSum", j->tm.final_sum); set_num(env, log, "total", j->tm.total);
    set_num(env, log, "c", j->tm.c); set_num(env, log, "K", j->tm.K);
    napi_set_named_property(env, res, "log", log);
    napi_resolve_deferred(env, j->deferred, res);
  }
  napi_delete_reference(env, j->scalars_ref);
  napi_delete_async_work(env, j->work);
  free(j);
}

static napi_value Msm(napi_env env, napi_callback_info info) {
  size_t argc = 5, len; napi_value argv[5], promise, name; void* data; int64_t n; int32_t c = 0, projective = 0; napi_typedarray_type ty; mgb_ctx* ctx; msm_job* j;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (!(ctx = ctx_of(env, argv[0]))) return NULL;
  CHECK(napi_get_typedarray_info(env, argv[1], &ty, &len, &data, NULL, NULL));
  CHECK(napi_get_value_int64(env, argv[2], &n));
  if (argc > 3) napi_get_value_int32(env, argv[3], &c);
  if (argc > 4) napi_get_value_int32(env, argv[4], &projective);
  if (ty != napi_uint8_array || len < 32 * (size_t)n) { napi_throw_type_error(env, NULL, "scalars: Uint8Array of n * 32 bytes, little-endian"); return NULL; }
  j = (msm_job*)calloc(1, sizeof *j);
  j->ctx = ctx; j->scalars = (const uint8_t*)data; j->n = (size_t)n; j->opts.c = c; j->opts.projective = projective;
  CHECK(napi_create_reference(env, argv[1], 1, &j->scalars_ref));       /* keeps the scalar buffer alive during the call */
  CHECK(napi_create_promise(env, &j->deferred, &promise));
  CHECK(napi_create_string_utf8(env, "mgb_msm", NAPI_AUTO_LENGTH, &name));
  CHECK(napi_create_async_work(env, NULL, name, msm_execute, msm_complete, j, &j->work));
  CHECK(napi_queue_async_work(env, j->work));
  return promise;
}

/* prefetch(ctx, scalars, n): starts the upload of the scalars of the NEXT msm call (mgb_msm_prefetch).  The caller keeps the
 * Uint8Array alive and unchanged until the msm(ctx, scalars, n) call that consumes it has resolved; a JS heap buffer is
 * pageable, so the driver stages the copy (the call returns once the staging is done, the transfer itself still overlaps). */
static napi_value Prefetch(napi_env env, napi_callback_info info) {
  size_t argc = 3, len; napi_value argv[3], undef; void* data; int64_t n; napi_typedarray_type ty; mgb_ctx* ctx;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (!(ctx = ctx_of(env, argv[0]))) return NULL;
  CHECK(napi_get_typedarray_info(env, argv[1], &ty, &len, &data, NULL, NULL));
  CHECK(napi_get_value_int64(env, argv[2], &n));
  if (ty != napi_uint8_array || n < 0 || len < 32 * (size_t)n) { napi_throw_type_error(env, NULL, "scalars: Uint8Array of n * 32 bytes, little-endian"); return NULL; }
  if (mgb_msm_prefetch(ctx, (const uint8_t*)data, (size_t)n) != 0) { napi_throw_error(env, NULL, mgb_last_error(ctx)); return NULL; }
  CHECK(napi_get_undefined(env, &undef));
  return undef;
}

/* ---- one process, several GPUs: mgb_multi_* (contexts, shards and the NCCL all-gather live inside the library) */
static mgb_multi* multi_of(napi_env env, napi_value v) {
  void* p = NULL;
  if (napi_get_value_external(env, v, &p) != napi_ok || !p) { napi_throw_type_error(env, NULL, "expected a multi-GPU engine handle"); return NULL; }
  return (mgb_multi*)p;
}
static void multi_finalize(napi_env env, void* data, void* hint) { (void)env; (void)hint; mgb_multi_destroy((mgb_multi*)data); }

static napi_value CreateMulti(napi_env env, napi_callback_info info) {
  size_t argc = 3, len; napi_value argv[3], out; int32_t curve; int64_t max_points; void* data; napi_typedarray_type ty; mgb_multi* m = NULL;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  CHECK(napi_get_value_int32(env, argv[0], &curve));
  CHECK(napi_get_typedarray_info(env, argv[1], &ty, &len, &data, NULL, NULL));
  CHECK(napi_get_value_int64(env, argv[2], &max_points));
  if (ty != napi_int32_array || len == 0) { napi_throw_type_error(env, NULL, "deviceIds: non-empty Int32Array"); return NULL; }
  if (mgb_multi_create(&m, curve, (const int*)data, (int)len, (size_t)max_points) != MGB_OK) { napi_throw_error(env, NULL, mgb_multi_last_error(NULL)); return NULL; }
  CHECK(napi_create_external(env, m, multi_finalize, NULL, &out));
  return out;
}

static napi_value SetPointsMulti(napi_env env, napi_callback_info info) {
  size_t argc = 3, len; napi_value argv[3]; void* data; int64_t n; napi_typedarray_type ty; mgb_multi* m;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (!(m = multi_of(env, argv[0]))) return NULL;
  CHECK(napi_get_typedarray_info(env, argv[1], &ty, &len, &data, NULL, NULL));
  CHECK(napi_get_value_int64(env, argv[2], &n));
  if (ty != napi_uint8_array || n <= 0 || len % (size_t)n != 0 || (len / (size_t)n != 64 && len / (size_t)n != 96)) {
    napi_throw_range_error(env, NULL, "points: Uint8Array of exactly n points, x||y little-endian (2 * 32 or 2 * 48 bytes each)");
    return NULL;
  }
  if (mgb_multi_set_points(m, (const uint8_t*)data, NULL, (size_t)n) != MGB_OK) napi_throw_error(env, NULL, mgb_multi_last_error(m));
  return NULL;
}

static napi_value RandomPointsMulti(napi_env env, napi_callback_info info) {
  size_t argc = 3; napi_value argv[3]; int64_t seed, n; mgb_multi* m;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (!(m = multi_of(env, argv[0]))) return NULL;
  CHECK(napi_get_value_int64(env, argv[1], &seed));
  CHECK(napi_get_value_int64(env, argv[2], &n));
  if (mgb_multi_random_points(m, (uint64_t)seed, (size_t)n) != MGB_OK) napi_throw_error(env, NULL, mgb_multi_last_error(m));
  return NULL;
}

static void msm_sharded_execute(napi_env env, void* data) {
  msm_job* j = (msm_job*)data; (void)env;
  j->rc = mgb_multi_msm(j->multi, j->scalars, j->n, &j->opts, j->out, &j->is_zero, &j->tm);
  if (j->rc != MGB_OK) { strncpy(j->err, mgb_multi_last_error(j->multi), sizeof j->err - 1); j->err[sizeof j->err - 1] = 0; }
}

static napi_value MsmSharded(napi_env env, napi_callback_info info) {
  size_t argc = 4, len; napi_value argv[4], promise, name; void* data; int64_t n; int32_t c = 0; napi_typedarray_type ty; mgb_multi* m; msm_job* j;
  CHECK(napi_get_cb_info(env, info, &argc, argv, NULL, NULL));
  if (!(m = multi_of(env, argv[0]))) return NULL;
  CHECK(napi_get_typedarray_info(env, argv[1], &ty, &len, &data, NULL, NULL));
  CHECK(napi_get_value_int64(env, argv[2], &n));
  if (argc > 3) napi_get_value_int32(env, argv[3], &c);
  if (ty != napi_uint8_array || n < 0 || len < 32 * (size_t)n) { napi_throw_type_error(env, NULL, "scalars: Uint8Array of n * 32 bytes, little-endian"); return NULL; }
  j = (msm_job*)calloc(1, sizeof *j);
  j->multi = m; j->scalars = (const uint8_t*)data; j->n = (size_t)n; j->opts.c = c;
  CHECK(napi_create_reference(env, argv[1], 1, &j->scalars_ref));
  CHECK(napi_create_promise(env, &j->deferred, &promise));
  CHECK(napi_create_string_utf8(env, "mgb_multi_msm", NAPI_AUTO_LENGTH, &name));
  CHECK(napi_create_async_work(env, NULL, name, msm_sharded_execute, msm_complete, j, &j->work));
  CHECK(napi_queue_async_work(env, j->work));
  return promise;
}

static napi_value Init(napi_env env, napi_value exports) {
  napi_property_descriptor d[] = {
    {"create", NULL, Create, NULL, NULL, NULL, napi_default, NULL},
    {"setPoints", NULL, SetPoints, NULL, NULL, NULL, napi_default, NULL},
    {"randomPoints", NULL, RandomPoints, NULL, NULL, NULL, napi_default, NULL},
    {"msm", NULL, Msm, NULL, NULL, NULL, napi_default, NULL},
    {"prefetch", NULL, Prefetch, NULL, NULL, NULL, napi_default, NULL},
    {"createMulti", NULL, CreateMulti, NULL, NULL, NULL, napi_default, NULL},
    {"setPointsMulti", NULL, SetPointsMulti, NULL, NULL, NULL, napi_default, NULL},
    {"randomPointsMulti", NULL, RandomPointsMulti, NULL, NULL, NULL, napi_default, NULL},
    {"msmSharded", NULL, MsmSharded, NULL, NULL, NULL, napi_default, NULL},
  };
  napi_define_properties(env, exports, sizeof d / sizeof d[0], d);
  return exports;
}
NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
