/*
 * N-API shim over the C ABI of libntru_b200.so (include/ntru_b200.h).
 *
 * NOT RUN IN THIS REPOSITORY'S IMAGE: node, npm and node_api.h are absent (SURVEY.md section 8c).  The file is
 * syntax- and type-checked against a stub of node_api.h (tests/napi_stub, tests/test_host.py).  It is the binding a
 * maintainer of numtel/ntru-circom would add next to index.js; build with
 *     gcc -shared -fPIC -I<node>/include/node -I../../include ntru_napi.c -L../../ntru-circom_b200 -lntru_b200 -o ntru_b200.node
 *
 * Every call is synchronous, like the reference.  The context is an external handle; N, p, q are read back from it
 * (ntru_get_params), never taken from JavaScript, and every typed array is checked for its element type and for
 * holding at least the B x width elements the library will read or write -- a short array throws a RangeError
 * (what expandArray throws upstream, index.js:98,126), a wrong type a TypeError.
 *
 *   create(N, p, q, device) -> handle          destroy(handle)              params(handle) -> {N, p, q, pitch}
 *   setOption(handle, key, value)              setRngKey(handle, key: Uint8Array(32), firstRow)   rngNextRow(handle)
 *   setPublicKey(handle, h: Uint16Array)       setPrivateKey(handle, f: Int8Array, fp: Uint8Array)
 *   encryptBatch(handle, B, r: Uint8Array | null, m: Uint8Array | Uint16Array[, h: Uint16Array])
 *        -> {value, quotientE, remainderE, r}      r == null: the device draws r (needs setOption(OPT_DR, dr));
 *                                                   a Uint16Array m takes the wide path (index.js:91); h: one key per row
 *   decryptBatch(handle, B, e: Uint16Array[, f: Int8Array, fp: Uint8Array])
 *        -> {value, quotient1, remainder1, quotient2, remainder2}
 *   encryptBatchPacked(handle, B, r: Uint32Array | null, m: Uint32Array) / decryptBatchPacked(handle, B, e: Uint32Array):
 *        the same with every array as rows of BN254 field elements (packOutput form), B x packedElems x 8 words
 *   verifyKeysBatch(handle, B, f, fq, fp, g)   keygenBatch(handle, B, f, g)
 *   checkEncryptBatch(handle, B, h, keyShared, r, m, quotientE, remainderE) -> Uint8Array(B) verdicts
 *   checkDecryptBatch(handle, B, f, fp, keyShared, e, quotient1, remainder1, quotient2, remainder2) -> Uint8Array(B)
 *   checkInverseBatch(handle, B, modP, x, y, quotientI, remainderI) -> Uint8Array(B)
 *        witness checks (VerifyEncrypt / VerifyDecrypt / VerifyInverse): bit 1 satisfied, 2 canonical, 4 not evaluated;
 *        keyShared: h (f, fp) is one row of N; y, quotientI, remainderI are Uint8Array when modP
 *   packOutput(handle, B, maxVal, data: Uint8Array | Uint16Array, dataLen) -> Uint32Array(B x outputSize x 8)
 *   unpackInput(handle, B, maxVal, packedBits, data: Uint32Array, nElems, wide: bool) -> Uint8Array | Uint16Array
 *   packGeometry(maxVal, dataLen) -> {maxInputBits, inputsPerOutput, arrLen, outputSize}
 *   sum(handle, B, e: Uint16Array) -> Uint16Array(N)
 *   xchgCreate(handle, world, rank) -> Uint8Array(64)   xchgConnect(handle, handles: Uint8Array(world x 64))
 *   sumAllreduce(handle, B, e: Uint16Array) -> Uint16Array(N)            xchgDestroy(handle)
 * Trimming / expandArray / {value, inputs, params} assembly stay in JavaScript (bindings/node/index.mjs).
 * The device-pointer entry points (*_dev) are for hosts that own device memory (the ctypes harness); a JavaScript
 * caller has none, so they are not bound.
 */
#include <node_api.h>
#include <stdbool.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "ntru_b200.h"

/* ---- error plumbing ------------------------------------------------------------------------------------------ */
#define NAPI_TRY(env, call)                                             \
  do {                                                                  \
    if ((call) != napi_ok) {                                            \
      napi_throw_error((env), NULL, "N-API call failed: " #call);       \
      return NULL;                                                      \
    }                                                                   \
  } while (0)

#define NTRU_TRY(env, ctx, call)                                                          \
  do {                                                                                    \
    int rc_ = (call);                                                                     \
    if (rc_ != NTRU_OK) {                                                                 \
      const char *msg_ = (ctx) ? ntru_last_error(ctx) : ntru_strerror(rc_);               \
      if (!msg_ || !*msg_) msg_ = ntru_strerror(rc_);                                     \
      if (rc_ == NTRU_E_LENGTH) napi_throw_range_error((env), NULL, msg_);                \
      else if (rc_ == NTRU_E_NOKEY) napi_throw_type_error((env), NULL, msg_);             \
      else napi_throw_error((env), NULL, msg_);                                           \
      return NULL;                                                                        \
    }                                                                                     \
  } while (0)

static void finalize_ctx(napi_env env, void *data, void *hint) {
  (void)env; (void)hint;
  if (data) ntru_destroy(*(ntru_ctx **)data);
  free(data);
}

/* the external holds a pointer to the context pointer, so that destroy() can clear it before the finalizer runs */
static ntru_ctx *get_ctx(napi_env env, napi_value v) {
  void *p = NULL;
  if (napi_get_value_external(env, v, &p) != napi_ok || !p || !*(ntru_ctx **)p) {
    napi_throw_type_error(env, NULL, "not a live ntru_b200 context");
    return NULL;
  }
  return *(ntru_ctx **)p;
}

/* typed array of exactly `type` with at least `need` elements; NULL (and a pending exception) otherwise */
static void *typed_arg(napi_env env, napi_value v, napi_typedarray_type type, size_t need, const char *what) {
  bool is_ta = false;
  if (napi_is_typedarray(env, v, &is_ta) != napi_ok || !is_ta) {
    napi_throw_type_error(env, NULL, what);
    return NULL;
  }
  napi_typedarray_type t;
  size_t len = 0, off = 0;
  void *data = NULL;
  napi_value ab;
  if (napi_get_typedarray_info(env, v, &t, &len, &data, &ab, &off) != napi_ok || t != type) {
    napi_throw_type_error(env, NULL, what);
    return NULL;
  }
  if (len < need) {
    napi_throw_range_error(env, NULL, "Invalid array length");      /* what expandArray throws upstream */
    return NULL;
  }
  return data;
}

static bool is_nullish(napi_env env, napi_value v) {
  napi_valuetype t;
  return napi_typeof(env, v, &t) == napi_ok && (t == napi_null || t == napi_undefined);
}

static bool typed_kind(napi_env env, napi_value v, napi_typedarray_type *t) {
  bool is_ta = false;
  size_t len, off;
  void *data;
  napi_value ab;
  return napi_is_typedarray(env, v, &is_ta) == napi_ok && is_ta &&
         napi_get_typedarray_info(env, v, t, &len, &data, &ab, &off) == napi_ok;
}

static napi_value make_typed(napi_env env, napi_typedarray_type t, size_t count, size_t elem, void **data) {
  napi_value ab, ta;
  if (napi_create_arraybuffer(env, count * elem, data, &ab) != napi_ok || napi_create_typedarray(env, t, count, ab, 0, &ta) != napi_ok) {
    napi_throw_error(env, NULL, "out of memory");
    *data = NULL;
    return NULL;
  }
  return ta;
}

static bool get_u32(napi_env env, napi_value v, uint32_t *out, const char *what) {
  if (napi_get_value_uint32(env, v, out) != napi_ok) {
    napi_throw_type_error(env, NULL, what);
    return false;
  }
  return true;
}

static bool ctx_N(ntru_ctx *ctx, size_t *N) {
  int n = 0;
  if (ntru_get_params(ctx, &n, NULL, NULL) != NTRU_OK) return false;
  *N = (size_t)n;
  return true;
}

#define ARGS(n)                                                                  \
  size_t argc = (n);                                                             \
  napi_value argv[(n)];                                                          \
  NAPI_TRY(env, napi_get_cb_info(env, info, &argc, argv, NULL, NULL));           \
  for (size_t i_ = argc; i_ < (n); ++i_) NAPI_TRY(env, napi_get_undefined(env, &argv[i_]))

#define SET(obj, name, val) NAPI_TRY(env, napi_set_named_property(env, obj, name, val))

/* ---- context ------------------------------------------------------------------------------------------------- */
static napi_value Create(napi_env env, napi_callback_info info) {
  ARGS(4);
  int32_t a[4] = {0, 3, 0, 0};
  for (int i = 0; i < 4; ++i)
    if (!is_nullish(env, argv[i])) NAPI_TRY(env, napi_get_value_int32(env, argv[i], &a[i]));
  ntru_ctx **box = (ntru_ctx **)calloc(1, sizeof *box);
  if (!box) { napi_throw_error(env, NULL, "out of memory"); return NULL; }
  int rc = ntru_create(box, a[0], a[1], a[2], a[3]);
  if (rc != NTRU_OK) {
    free(box);
    napi_throw_error(env, NULL, rc == NTRU_E_CUDA ? "no usable CUDA device (this engine has no CPU fallback)" : ntru_strerror(rc));
    return NULL;
  }
  napi_value ext;
  if (napi_create_external(env, box, finalize_ctx, NULL, &ext) != napi_ok) {
    ntru_destroy(*box);
    free(box);
    napi_throw_error(env, NULL, "napi_create_external failed");
    return NULL;
  }
  return ext;
}

static napi_value Destroy(napi_env env, napi_callback_info info) {
  ARGS(1);
  void *p = NULL;
  if (napi_get_value_external(env, argv[0], &p) == napi_ok && p && *(ntru_ctx **)p) {
    ntru_destroy(*(ntru_ctx **)p);
    *(ntru_ctx **)p = NULL;
  }
  return NULL;
}

static napi_value Params(napi_env env, napi_callback_info info) {
  ARGS(1);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  if (!ctx) return NULL;
  int N, p, q;
  NTRU_TRY(env, ctx, ntru_get_params(ctx, &N, &p, &q));
  napi_value out, v;
  NAPI_TRY(env, napi_create_object(env, &out));
  NAPI_TRY(env, napi_create_int32(env, N, &v)); SET(out, "N", v);
  NAPI_TRY(env, napi_create_int32(env, p, &v)); SET(out, "p", v);
  NAPI_TRY(env, napi_create_int32(env, q, &v)); SET(out, "q", v);
  NAPI_TRY(env, napi_create_int32(env, ntru_pitch(ctx), &v)); SET(out, "pitch", v);
  return out;
}

static napi_value SetOption(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  if (!ctx) return NULL;
  int32_t key;
  int64_t value;
  NAPI_TRY(env, napi_get_value_int32(env, argv[1], &key));
  NAPI_TRY(env, napi_get_value_int64(env, argv[2], &value));
  NTRU_TRY(env, ctx, ntru_set_option(ctx, key, (long)value));
  return NULL;
}

static napi_value SetRngKey(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  if (!ctx) return NULL;
  const uint8_t *key = (const uint8_t *)typed_arg(env, argv[1], napi_uint8_array, NTRU_RNG_KEY_BYTES, "key: Uint8Array(32)");
  if (!key) return NULL;
  int64_t first = 0;
  if (!is_nullish(env, argv[2])) NAPI_TRY(env, napi_get_value_int64(env, argv[2], &first));
  NTRU_TRY(env, ctx, ntru_set_rng_key(ctx, key, (uint64_t)first));
  return NULL;
}

static napi_value RngNextRow(napi_env env, napi_callback_info info) {
  ARGS(1);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  if (!ctx) return NULL;
  napi_value v;
  NAPI_TRY(env, napi_create_int64(env, (int64_t)ntru_rng_next_row(ctx), &v));
  return v;
}

static napi_value SetPublicKey(napi_env env, napi_callback_info info) {
  ARGS(2);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  if (!ctx || !ctx_N(ctx, &N)) return NULL;
  const uint16_t *h = (const uint16_t *)typed_arg(env, argv[1], napi_uint16_array, N, "h: Uint16Array(N)");
  if (!h) return NULL;
  NTRU_TRY(env, ctx, ntru_set_public_key(ctx, h));
  return NULL;
}

static napi_value SetPrivateKey(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  if (!ctx || !ctx_N(ctx, &N)) return NULL;
  const int8_t *f = (const int8_t *)typed_arg(env, argv[1], napi_int8_array, N, "f: Int8Array(N)");
  if (!f) return NULL;
  const uint8_t *fp = (const uint8_t *)typed_arg(env, argv[2], napi_uint8_array, N, "fp: Uint8Array(N)");
  if (!fp) return NULL;
  NTRU_TRY(env, ctx, ntru_set_private_key(ctx, f, fp));
  return NULL;
}

/* ---- encryptBits / decryptBits for B rows ---------------------------------------------------------------------- */
static napi_value EncryptBatch(napi_env env, napi_callback_info info) {
  ARGS(5);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  const size_t rows = (size_t)B * N, wit = (size_t)B * (N + 1);
  const uint8_t *r = NULL;
  if (!is_nullish(env, argv[2])) {
    r = (const uint8_t *)typed_arg(env, argv[2], napi_uint8_array, rows, "r: Uint8Array(B x N) or null");
    if (!r) return NULL;
  }
  napi_typedarray_type mt;
  if (!typed_kind(env, argv[3], &mt) || (mt != napi_uint8_array && mt != napi_uint16_array)) {
    napi_throw_type_error(env, NULL, "m: Uint8Array(B x N), or Uint16Array(B x N) for coefficients above 255");
    return NULL;
  }
  const void *m = typed_arg(env, argv[3], mt, rows, "m");
  if (!m) return NULL;
  const uint16_t *h = NULL;
  if (!is_nullish(env, argv[4])) {
    h = (const uint16_t *)typed_arg(env, argv[4], napi_uint16_array, rows, "h: Uint16Array(B x N) (one key per row)");
    if (!h) return NULL;
    if (mt != napi_uint8_array) {
      napi_throw_type_error(env, NULL, "per-row keys take byte messages");
      return NULL;
    }
  }
  void *value, *quo, *rem, *r_out;
  napi_value v0 = make_typed(env, napi_uint16_array, rows, 2, &value), v1 = make_typed(env, napi_uint16_array, wit, 2, &quo),
             v2 = make_typed(env, napi_uint16_array, wit, 2, &rem), v3 = make_typed(env, napi_uint8_array, rows, 1, &r_out);
  if (!value || !quo || !rem || !r_out) return NULL;
  if (h) NTRU_TRY(env, ctx, ntru_encrypt_batch_keys(ctx, B, h, r, (const uint8_t *)m, value, quo, rem, r_out));
  else if (mt == napi_uint16_array) NTRU_TRY(env, ctx, ntru_encrypt_batch_wide(ctx, B, r, (const uint16_t *)m, value, quo, rem, r_out));
  else NTRU_TRY(env, ctx, ntru_encrypt_batch(ctx, B, r, (const uint8_t *)m, value, quo, rem, r_out));
  napi_value out;
  NAPI_TRY(env, napi_create_object(env, &out));
  SET(out, "value", v0);
  SET(out, "quotientE", v1);
  SET(out, "remainderE", v2);
  SET(out, "r", v3);
  return out;
}

static napi_value DecryptBatch(napi_env env, napi_callback_info info) {
  ARGS(5);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  const size_t rows = (size_t)B * N, wit = (size_t)B * (N + 1);
  const uint16_t *e = (const uint16_t *)typed_arg(env, argv[2], napi_uint16_array, rows, "e: Uint16Array(B x N)");
  if (!e) return NULL;
  const int8_t *f = NULL;
  const uint8_t *fp = NULL;
  if (!is_nullish(env, argv[3]) || !is_nullish(env, argv[4])) {
    f = (const int8_t *)typed_arg(env, argv[3], napi_int8_array, rows, "f: Int8Array(B x N) (one key per row)");
    if (!f) return NULL;
    fp = (const uint8_t *)typed_arg(env, argv[4], napi_uint8_array, rows, "fp: Uint8Array(B x N) (one key per row)");
    if (!fp) return NULL;
  }
  void *value, *q1, *r1, *q2, *r2;
  napi_value v0 = make_typed(env, napi_uint8_array, rows, 1, &value), v1 = make_typed(env, napi_uint16_array, wit, 2, &q1),
             v2 = make_typed(env, napi_uint16_array, wit, 2, &r1), v3 = make_typed(env, napi_uint8_array, wit, 1, &q2),
             v4 = make_typed(env, napi_uint8_array, wit, 1, &r2);
  if (!value || !q1 || !r1 || !q2 || !r2) return NULL;
  if (f) NTRU_TRY(env, ctx, ntru_decrypt_batch_keys(ctx, B, f, fp, e, value, q1, r1, q2, r2));
  else NTRU_TRY(env, ctx, ntru_decrypt_batch(ctx, B, e, value, q1, r1, q2, r2));
  napi_value out;
  NAPI_TRY(env, napi_create_object(env, &out));
  SET(out, "value", v0);
  SET(out, "quotient1", v1);
  SET(out, "remainder1", v2);
  SET(out, "quotient2", v3);
  SET(out, "remainder2", v4);
  return out;
}

/* ---- the same two calls with BN254 field elements on the wire (packOutput form, index.js:572-596) ---------------------
 * encryptBatchPacked(handle, B, r: Uint32Array | null, m: Uint32Array) -> {value, quotientE, remainderE, r}
 * decryptBatchPacked(handle, B, e: Uint32Array) -> {value, quotient1, remainder1, quotient2, remainder2}
 * every array: B x packedElems x 8 little-endian 32-bit words per row (BigInt = sum of word[i] << 32 i). */
static napi_value EncryptBatchPacked(napi_env env, napi_callback_info info) {
  ARGS(4);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  const size_t small = (size_t)B * (size_t)ntru_packed_elems(ctx, 0, (int)N) * 8, val = (size_t)B * (size_t)ntru_packed_elems(ctx, 1, (int)N) * 8,
               wit = (size_t)B * (size_t)ntru_packed_elems(ctx, 1, (int)N + 1) * 8;
  const void *r = NULL;
  if (!is_nullish(env, argv[2])) {
    r = typed_arg(env, argv[2], napi_uint32_array, small, "r: Uint32Array(B x packedElems x 8) or null");
    if (!r) return NULL;
  }
  const void *m = typed_arg(env, argv[3], napi_uint32_array, small, "m: Uint32Array(B x packedElems x 8)");
  if (!m) return NULL;
  void *value, *quo, *rem, *r_out;
  napi_value v0 = make_typed(env, napi_uint32_array, val, 4, &value), v1 = make_typed(env, napi_uint32_array, wit, 4, &quo),
             v2 = make_typed(env, napi_uint32_array, wit, 4, &rem), v3 = make_typed(env, napi_uint32_array, small, 4, &r_out);
  if (!value || !quo || !rem || !r_out) return NULL;
  NTRU_TRY(env, ctx, ntru_encrypt_batch_packed(ctx, B, r, m, value, quo, rem, r_out));
  napi_value out;
  NAPI_TRY(env, napi_create_object(env, &out));
  SET(out, "value", v0);
  SET(out, "quotientE", v1);
  SET(out, "remainderE", v2);
  SET(out, "r", v3);
  return out;
}

static napi_value DecryptBatchPacked(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  const size_t e_len = (size_t)B * (size_t)ntru_packed_elems(ctx, 1, (int)N) * 8, wq = (size_t)B * (size_t)ntru_packed_elems(ctx, 1, (int)N + 1) * 8,
               vs = (size_t)B * (size_t)ntru_packed_elems(ctx, 0, (int)N) * 8, ws = (size_t)B * (size_t)ntru_packed_elems(ctx, 0, (int)N + 1) * 8;
  const void *e = typed_arg(env, argv[2], napi_uint32_array, e_len, "e: Uint32Array(B x packedElems x 8)");
  if (!e) return NULL;
  void *value, *q1, *r1, *q2, *r2;
  napi_value v0 = make_typed(env, napi_uint32_array, vs, 4, &value), v1 = make_typed(env, napi_uint32_array, wq, 4, &q1),
             v2 = make_typed(env, napi_uint32_array, wq, 4, &r1), v3 = make_typed(env, napi_uint32_array, ws, 4, &q2),
             v4 = make_typed(env, napi_uint32_array, ws, 4, &r2);
  if (!value || !q1 || !r1 || !q2 || !r2) return NULL;
  NTRU_TRY(env, ctx, ntru_decrypt_batch_packed(ctx, B, e, value, q1, r1, q2, r2));
  napi_value out;
  NAPI_TRY(env, napi_create_object(env, &out));
  SET(out, "value", v0);
  SET(out, "quotient1", v1);
  SET(out, "remainder1", v2);
  SET(out, "quotient2", v3);
  SET(out, "remainder2", v4);
  return out;
}

/* verifyKeysBatch(handle, B, f: Int8Array, fq: Uint16Array, fp: Uint8Array, g: Int8Array) -- index.js:141-197 for B keys */
static napi_value VerifyKeysBatch(napi_env env, napi_callback_info info) {
  ARGS(6);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: key count")) return NULL;
  const size_t rows = (size_t)B * N, wit = (size_t)B * (N + 1);
  const int8_t *f = (const int8_t *)typed_arg(env, argv[2], napi_int8_array, rows, "f: Int8Array(B x N)");
  if (!f) return NULL;
  const uint16_t *fq = (const uint16_t *)typed_arg(env, argv[3], napi_uint16_array, rows, "fq: Uint16Array(B x N)");
  if (!fq) return NULL;
  const uint8_t *fp = (const uint8_t *)typed_arg(env, argv[4], napi_uint8_array, rows, "fp: Uint8Array(B x N)");
  if (!fp) return NULL;
  const int8_t *g = (const int8_t *)typed_arg(env, argv[5], napi_int8_array, rows, "g: Int8Array(B x N)");
  if (!g) return NULL;
  void *o[6];
  static const char *names[6] = {"quotientFq", "remainderFq", "quotientFp", "remainderFp", "quotientH", "remainderH"};
  napi_value v[6];
  for (int i = 0; i < 6; ++i) {
    const int bytes = (i == 2 || i == 3) ? 1 : 2;
    v[i] = make_typed(env, bytes == 1 ? napi_uint8_array : napi_uint16_array, wit, (size_t)bytes, &o[i]);
    if (!o[i]) return NULL;
  }
  NTRU_TRY(env, ctx, ntru_verify_keys_batch(ctx, B, f, fq, fp, g, o[0], o[1], o[2], o[3], o[4], o[5]));
  napi_value out;
  NAPI_TRY(env, napi_create_object(env, &out));
  for (int i = 0; i < 6; ++i) SET(out, names[i], v[i]);
  return out;
}

/* keygenBatch(handle, B, f: Int8Array, g: Int8Array) -> {fq, fp, h, valid} -- index.js:30-79 for B keys */
static napi_value KeygenBatch(napi_env env, napi_callback_info info) {
  ARGS(4);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: key count")) return NULL;
  const size_t rows = (size_t)B * N;
  const int8_t *f = (const int8_t *)typed_arg(env, argv[2], napi_int8_array, rows, "f: Int8Array(B x N)");
  if (!f) return NULL;
  const int8_t *g = (const int8_t *)typed_arg(env, argv[3], napi_int8_array, rows, "g: Int8Array(B x N)");
  if (!g) return NULL;
  void *fq, *fp, *h, *valid;
  napi_value v0 = make_typed(env, napi_uint16_array, rows, 2, &fq), v1 = make_typed(env, napi_uint8_array, rows, 1, &fp),
             v2 = make_typed(env, napi_uint16_array, rows, 2, &h), v3 = make_typed(env, napi_uint8_array, B, 1, &valid);
  if (!fq || !fp || !h || !valid) return NULL;
  NTRU_TRY(env, ctx, ntru_keygen_batch(ctx, B, f, g, fq, fp, h, valid));
  napi_value out;
  NAPI_TRY(env, napi_create_object(env, &out));
  SET(out, "fq", v0);
  SET(out, "fp", v1);
  SET(out, "h", v2);
  SET(out, "valid", v3);
  return out;
}

/* ---- witness checks: VerifyEncrypt / VerifyDecrypt / VerifyInverse (circuits/ntru.circom:155-256) ----------------- */
static bool get_flag(napi_env env, napi_value v, bool *out) {
  *out = false;
  return is_nullish(env, v) || napi_get_value_bool(env, v, out) == napi_ok;
}

static napi_value CheckEncryptBatch(napi_env env, napi_callback_info info) {
  ARGS(8);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  bool shared;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  if (!get_flag(env, argv[3], &shared)) { napi_throw_type_error(env, NULL, "keyShared: boolean"); return NULL; }
  const size_t rows = (size_t)B * N, wit = (size_t)B * (N + 1);
  const uint16_t *h = (const uint16_t *)typed_arg(env, argv[2], napi_uint16_array, shared ? N : rows, "h: Uint16Array(N or B x N)");
  if (!h) return NULL;
  const uint8_t *r = (const uint8_t *)typed_arg(env, argv[4], napi_uint8_array, rows, "r: Uint8Array(B x N)");
  if (!r) return NULL;
  const uint16_t *m = (const uint16_t *)typed_arg(env, argv[5], napi_uint16_array, rows, "m: Uint16Array(B x N)");
  if (!m) return NULL;
  const uint16_t *qe = (const uint16_t *)typed_arg(env, argv[6], napi_uint16_array, wit, "quotientE: Uint16Array(B x (N+1))");
  if (!qe) return NULL;
  const uint16_t *re = (const uint16_t *)typed_arg(env, argv[7], napi_uint16_array, wit, "remainderE: Uint16Array(B x (N+1))");
  if (!re) return NULL;
  void *verdict;
  napi_value out = make_typed(env, napi_uint8_array, B, 1, &verdict);
  if (!verdict) return NULL;
  NTRU_TRY(env, ctx, ntru_check_encrypt_batch(ctx, B, h, shared, r, m, qe, re, verdict));
  return out;
}

static napi_value CheckDecryptBatch(napi_env env, napi_callback_info info) {
  ARGS(10);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  bool shared;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  if (!get_flag(env, argv[4], &shared)) { napi_throw_type_error(env, NULL, "keyShared: boolean"); return NULL; }
  const size_t rows = (size_t)B * N, wit = (size_t)B * (N + 1), key = shared ? N : rows;
  const uint16_t *f = (const uint16_t *)typed_arg(env, argv[2], napi_uint16_array, key, "f: Uint16Array(N or B x N), -1 as q-1");
  if (!f) return NULL;
  const uint8_t *fp = (const uint8_t *)typed_arg(env, argv[3], napi_uint8_array, key, "fp: Uint8Array(N or B x N)");
  if (!fp) return NULL;
  const uint16_t *e = (const uint16_t *)typed_arg(env, argv[5], napi_uint16_array, rows, "e: Uint16Array(B x N)");
  if (!e) return NULL;
  const uint16_t *q1 = (const uint16_t *)typed_arg(env, argv[6], napi_uint16_array, wit, "quotient1: Uint16Array(B x (N+1))");
  if (!q1) return NULL;
  const uint16_t *r1 = (const uint16_t *)typed_arg(env, argv[7], napi_uint16_array, wit, "remainder1: Uint16Array(B x (N+1))");
  if (!r1) return NULL;
  const uint8_t *q2 = (const uint8_t *)typed_arg(env, argv[8], napi_uint8_array, wit, "quotient2: Uint8Array(B x (N+1))");
  if (!q2) return NULL;
  const uint8_t *r2 = (const uint8_t *)typed_arg(env, argv[9], napi_uint8_array, wit, "remainder2: Uint8Array(B x (N+1))");
  if (!r2) return NULL;
  void *verdict;
  napi_value out = make_typed(env, napi_uint8_array, B, 1, &verdict);
  if (!verdict) return NULL;
  NTRU_TRY(env, ctx, ntru_check_decrypt_batch(ctx, B, f, fp, shared, e, q1, r1, q2, r2, verdict));
  return out;
}

static napi_value CheckInverseBatch(napi_env env, napi_callback_info info) {
  ARGS(7);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  bool mod_p;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  if (!get_flag(env, argv[2], &mod_p)) { napi_throw_type_error(env, NULL, "modP: boolean"); return NULL; }
  const size_t rows = (size_t)B * N, wit = (size_t)B * (N + 1);
  const napi_typedarray_type t = mod_p ? napi_uint8_array : napi_uint16_array;
  const uint16_t *x = (const uint16_t *)typed_arg(env, argv[3], napi_uint16_array, rows, "x: Uint16Array(B x N)");
  if (!x) return NULL;
  const void *y = typed_arg(env, argv[4], t, rows, "y: Uint16Array(B x N), Uint8Array when modP");
  if (!y) return NULL;
  const void *qi = typed_arg(env, argv[5], t, wit, "quotientI: Uint16Array(B x (N+1)), Uint8Array when modP");
  if (!qi) return NULL;
  const void *ri = typed_arg(env, argv[6], t, wit, "remainderI: Uint16Array(B x (N+1)), Uint8Array when modP");
  if (!ri) return NULL;
  void *verdict;
  napi_value out = make_typed(env, napi_uint8_array, B, 1, &verdict);
  if (!verdict) return NULL;
  NTRU_TRY(env, ctx, ntru_check_inverse_batch(ctx, B, mod_p, x, y, qi, ri, verdict));
  return out;
}

/* ---- packOutput / unpackInput (index.js:572-620) ----------------------------------------------------------------- */
static napi_value PackGeometry(napi_env env, napi_callback_info info) {
  ARGS(2);
  uint32_t max_val, data_len;
  if (!get_u32(env, argv[0], &max_val, "maxVal") || !get_u32(env, argv[1], &data_len, "dataLen")) return NULL;
  int bits, n, arr, outs;
  NTRU_TRY(env, NULL, ntru_pack_geometry(max_val, (int)data_len, &bits, &n, &arr, &outs));
  napi_value out, v;
  NAPI_TRY(env, napi_create_object(env, &out));
  NAPI_TRY(env, napi_create_int32(env, bits, &v)); SET(out, "maxInputBits", v);
  NAPI_TRY(env, napi_create_int32(env, n, &v)); SET(out, "inputsPerOutput", v);
  NAPI_TRY(env, napi_create_int32(env, arr, &v)); SET(out, "arrLen", v);
  NAPI_TRY(env, napi_create_int32(env, outs, &v)); SET(out, "outputSize", v);
  return out;
}

static napi_value PackOutput(napi_env env, napi_callback_info info) {
  ARGS(5);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  uint32_t B, max_val, data_len;
  if (!ctx || !get_u32(env, argv[1], &B, "B") || !get_u32(env, argv[2], &max_val, "maxVal") || !get_u32(env, argv[4], &data_len, "dataLen"))
    return NULL;
  napi_typedarray_type t;
  if (!typed_kind(env, argv[3], &t) || (t != napi_uint8_array && t != napi_uint16_array)) {
    napi_throw_type_error(env, NULL, "data: Uint8Array or Uint16Array (B x dataLen)");
    return NULL;
  }
  const void *data = typed_arg(env, argv[3], t, (size_t)B * data_len, "data");
  if (!data) return NULL;
  int outs;
  NTRU_TRY(env, ctx, ntru_pack_geometry(max_val, (int)data_len, NULL, NULL, NULL, &outs));
  void *words;
  napi_value out = make_typed(env, napi_uint32_array, (size_t)B * (size_t)outs * 8, 4, &words);
  if (!words) return NULL;
  NTRU_TRY(env, ctx, ntru_pack_output(ctx, B, data, t == napi_uint8_array ? 1 : 2, (int)data_len, max_val, words));
  return out;
}

static napi_value UnpackInput(napi_env env, napi_callback_info info) {
  ARGS(7);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  uint32_t B, max_val, packed_bits, n_elems;
  bool wide = true;
  if (!ctx || !get_u32(env, argv[1], &B, "B") || !get_u32(env, argv[2], &max_val, "maxVal") || !get_u32(env, argv[3], &packed_bits, "packedBits") ||
      !get_u32(env, argv[5], &n_elems, "nElems"))
    return NULL;
  if (!is_nullish(env, argv[6])) NAPI_TRY(env, napi_get_value_bool(env, argv[6], &wide));
  const uint32_t *data = (const uint32_t *)typed_arg(env, argv[4], napi_uint32_array, (size_t)B * n_elems * 8, "data: Uint32Array(B x nElems x 8)");
  if (!data) return NULL;
  int bits = 0;
  for (uint32_t v = max_val; v; v >>= 1) ++bits;
  if (bits == 0 || packed_bits < (uint32_t)bits) {
    napi_throw_range_error(env, NULL, "maxVal / packedBits");
    return NULL;
  }
  const size_t width = (size_t)(packed_bits / (uint32_t)bits) * n_elems;
  void *coef;
  napi_value out = make_typed(env, wide ? napi_uint16_array : napi_uint8_array, (size_t)B * width, wide ? 2 : 1, &coef);
  if (!coef) return NULL;
  NTRU_TRY(env, ctx, ntru_unpack_input(ctx, B, data, (int)n_elems, max_val, (int)packed_bits, coef, wide ? 2 : 1));
  return out;
}

/* ---- homomorphic sum: one GPU, and over the ranks of an exchange --------------------------------------------------- */
static napi_value Sum(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  const uint16_t *e = (const uint16_t *)typed_arg(env, argv[2], napi_uint16_array, (size_t)B * N, "e: Uint16Array(B x N)");
  if (!e) return NULL;
  void *out_data;
  napi_value out = make_typed(env, napi_uint16_array, N, 2, &out_data);
  if (!out_data) return NULL;
  NTRU_TRY(env, ctx, ntru_sum(ctx, B, e, out_data));
  return out;
}

static napi_value XchgCreate(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  uint32_t world, rank;
  if (!ctx || !get_u32(env, argv[1], &world, "world") || !get_u32(env, argv[2], &rank, "rank")) return NULL;
  void *handle;
  napi_value out = make_typed(env, napi_uint8_array, NTRU_XCHG_HANDLE_BYTES, 1, &handle);
  if (!handle) return NULL;
  NTRU_TRY(env, ctx, ntru_xchg_create(ctx, (int)world, (int)rank, (unsigned char *)handle));
  return out;
}

static napi_value XchgConnect(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  uint32_t world;
  if (!ctx || !get_u32(env, argv[2], &world, "world")) return NULL;
  const unsigned char *handles =
      (const unsigned char *)typed_arg(env, argv[1], napi_uint8_array, (size_t)world * NTRU_XCHG_HANDLE_BYTES, "handles: Uint8Array(world x 64)");
  if (!handles) return NULL;
  NTRU_TRY(env, ctx, ntru_xchg_connect(ctx, handles));
  return NULL;
}

static napi_value XchgDestroy(napi_env env, napi_callback_info info) {
  ARGS(1);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  if (!ctx) return NULL;
  NTRU_TRY(env, ctx, ntru_xchg_destroy(ctx));
  return NULL;
}

static napi_value SumAllreduce(napi_env env, napi_callback_info info) {
  ARGS(3);
  ntru_ctx *ctx = get_ctx(env, argv[0]);
  size_t N;
  uint32_t B;
  if (!ctx || !ctx_N(ctx, &N) || !get_u32(env, argv[1], &B, "B: row count")) return NULL;
  const uint16_t *e = NULL;
  if (B > 0) {
    e = (const uint16_t *)typed_arg(env, argv[2], napi_uint16_array, (size_t)B * N, "e: Uint16Array(B x N)");
    if (!e) return NULL;
  }
  void *out_data;
  napi_value out = make_typed(env, napi_uint16_array, N, 2, &out_data);
  if (!out_data) return NULL;
  NTRU_TRY(env, ctx, ntru_sum_allreduce(ctx, B, e, out_data));
  return out;
}

static napi_value Init(napi_env env, napi_value exports) {
#define FN(name, fn) {name, 0, fn, 0, 0, 0, napi_default, 0}
  napi_property_descriptor d[] = {
      FN("create", Create), FN("destroy", Destroy), FN("params", Params), FN("setOption", SetOption), FN("setRngKey", SetRngKey),
      FN("rngNextRow", RngNextRow), FN("setPublicKey", SetPublicKey), FN("setPrivateKey", SetPrivateKey),
      FN("encryptBatch", EncryptBatch), FN("decryptBatch", DecryptBatch), FN("encryptBatchPacked", EncryptBatchPacked),
      FN("decryptBatchPacked", DecryptBatchPacked), FN("verifyKeysBatch", VerifyKeysBatch),
      FN("keygenBatch", KeygenBatch), FN("packGeometry", PackGeometry), FN("packOutput", PackOutput), FN("unpackInput", UnpackInput),
      FN("sum", Sum), FN("xchgCreate", XchgCreate), FN("xchgConnect", XchgConnect), FN("xchgDestroy", XchgDestroy),
      FN("sumAllreduce", SumAllreduce), FN("checkEncryptBatch", CheckEncryptBatch), FN("checkDecryptBatch", CheckDecryptBatch),
      FN("checkInverseBatch", CheckInverseBatch),
  };
#undef FN
  if (napi_define_properties(env, exports, sizeof d / sizeof d[0], d) != napi_ok) {
    napi_throw_error(env, NULL, "napi_define_properties failed");
    return NULL;
  }
  return exports;
}

NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
