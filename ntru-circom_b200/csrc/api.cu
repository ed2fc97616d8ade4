// C ABI of libntru_b200.so (include/ntru_b200.h): context, keys, host-buffer pipeline and
// device-resident entry points.  No CPU compute path exists in this library.

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <sys/random.h>

#include <new>
#include <string>

#include "ntru_internal.cuh"

namespace ntru {

int fail(ntru_ctx *ctx, int code, const std::string &msg) {
  if (ctx) ctx->err = msg;
  return code;
}

int cuda_fail(ntru_ctx *ctx, cudaError_t e, const char *what) {
  if (ctx) ctx->err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
  return NTRU_E_CUDA;
}

static cudaEvent_t pool_get(ntru_ctx *ctx) {
  if (!ctx->event_pool.empty()) {
    cudaEvent_t e = ctx->event_pool.back();
    ctx->event_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

LaunchTimer::LaunchTimer(ntru_ctx *c, int k) : ctx(c), kind(k) {
  ctx->launches++;
  if (!ctx->timing) return;
  a = pool_get(ctx);
  b = pool_get(ctx);
  cudaEventRecord(a, ctx->stream);
}

LaunchTimer::~LaunchTimer() {
  if (!a) return;
  cudaEventRecord(b, ctx->stream);
  ctx->timed.push_back({kind, a, b});
}

namespace {

// One array of a host-buffer call: packed on the host (row = width elements), pitched on the device.
struct HostArr {
  const void *in = nullptr;   // host source (inputs)
  void *out = nullptr;        // host destination (outputs)
  size_t elem = 1;            // bytes per element
  size_t width = 0;           // packed elements per row on the host
  bool used = false;
  // field-element wire format (ntru_*_batch_packed): the host row is fe_elems BN254 field elements of 32 bytes,
  // packOutput(maxVal, width, row).expected -- fe_n coefficients of fe_bits bits each per element; 0 = plain rows
  int fe_bits = 0, fe_n = 0, fe_elems = 0;
  // flat: one value per row (the verdict bytes of the witness checks): the kernel works on the packed staging itself
  bool flat = false;
  size_t host_row_bytes() const { return fe_bits ? (size_t)fe_elems * 32 : width * elem; }
};

constexpr int kMaxArr = 10;

// Runs `launch(rows, dev[])` over B rows in chunks, overlapping H2D, kernels and D2H on three streams.
// Every array moves over PCIe as a packed 1-D copy; k_repitch converts to / from the pitched device layout.
template <class Launch>
int run_pipeline(ntru_ctx *ctx, size_t B, HostArr (&arr)[kMaxArr], Launch launch) {
  const size_t chunk = ctx->chunk_rows;
  const size_t P = (size_t)ctx->P;
  const size_t rows_alloc = B < chunk ? B : chunk;
  for (int s = 0; s < kNumSlots; ++s)
    for (int a = 0; a < kMaxArr; ++a)
      if (arr[a].used) {
        if (!arr[a].flat) NTRU_CUDA(ctx, ctx->slot_bufs[s][a].reserve(rows_alloc * P * arr[a].elem));
        NTRU_CUDA(ctx, ctx->slot_packed[s][a].reserve(rows_alloc * arr[a].host_row_bytes()));
      }
  size_t ci = 0;
  for (size_t row0 = 0; row0 < B; row0 += chunk, ++ci) {
    const size_t rows = (B - row0) < chunk ? (B - row0) : chunk;
    const int s = (int)(ci % kNumSlots);
    void *dev[kMaxArr];
    for (int a = 0; a < kMaxArr; ++a)
      dev[a] = arr[a].used ? (arr[a].flat ? ctx->slot_packed[s][a].ptr : ctx->slot_bufs[s][a].ptr) : nullptr;
    // inputs: packed 1-D H2D on s_in (the slot's packed staging is free once the previous unpack ran)
    if (ci >= (size_t)kNumSlots) NTRU_CUDA(ctx, cudaStreamWaitEvent(ctx->s_in, ctx->ev_comp[s], 0));
    for (int a = 0; a < kMaxArr; ++a) {
      if (!arr[a].used || !arr[a].in) continue;
      const size_t wb = arr[a].host_row_bytes();
      NTRU_CUDA(ctx, cudaMemcpyAsync(ctx->slot_packed[s][a].ptr, (const char *)arr[a].in + row0 * wb, rows * wb,
                                     cudaMemcpyHostToDevice, ctx->s_in));
    }
    NTRU_CUDA(ctx, cudaEventRecord(ctx->ev_in[s], ctx->s_in));
    NTRU_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_in[s], 0));
    if (ci >= (size_t)kNumSlots) NTRU_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_out[s], 0));
    for (int a = 0; a < kMaxArr; ++a) {
      if (!arr[a].used || !arr[a].in) continue;
      int rc = arr[a].fe_bits
                   ? launch_wire_unpack(ctx, rows, (const uint32_t *)ctx->slot_packed[s][a].ptr, arr[a].fe_elems, arr[a].fe_bits,
                                        arr[a].fe_n, (int)arr[a].width, dev[a], (int)arr[a].elem)
                   : launch_repitch(ctx, ctx->slot_packed[s][a].ptr, dev[a], rows, (int)arr[a].width, (int)arr[a].elem, true);
      if (rc != NTRU_OK) return rc;
    }
    int rc = launch(rows, dev);
    if (rc != NTRU_OK) return rc;
    for (int a = 0; a < kMaxArr; ++a) {
      if (!arr[a].used || !arr[a].out || arr[a].flat) continue;
      rc = arr[a].fe_bits
               ? launch_pack_fields(ctx, rows, dev[a], (int)arr[a].elem, (int)arr[a].width, (size_t)ctx->P, arr[a].fe_bits, arr[a].fe_n,
                                    arr[a].fe_elems, (uint32_t *)ctx->slot_packed[s][a].ptr)
               : launch_repitch(ctx, dev[a], ctx->slot_packed[s][a].ptr, rows, (int)arr[a].width, (int)arr[a].elem, false);
      if (rc != NTRU_OK) return rc;
    }
    NTRU_CUDA(ctx, cudaEventRecord(ctx->ev_comp[s], ctx->stream));
    NTRU_CUDA(ctx, cudaStreamWaitEvent(ctx->s_out, ctx->ev_comp[s], 0));
    for (int a = 0; a < kMaxArr; ++a) {
      if (!arr[a].used || !arr[a].out) continue;
      const size_t wb = arr[a].host_row_bytes();
      NTRU_CUDA(ctx, cudaMemcpyAsync((char *)arr[a].out + row0 * wb, ctx->slot_packed[s][a].ptr, rows * wb,
                                     cudaMemcpyDeviceToHost, ctx->s_out));
    }
    NTRU_CUDA(ctx, cudaEventRecord(ctx->ev_out[s], ctx->s_out));
  }
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->s_out));
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NTRU_OK;
}

void set_in(HostArr &a, const void *p, size_t elem, size_t width) {
  a.in = p; a.elem = elem; a.width = width; a.used = p != nullptr;
}
void set_out(HostArr &a, void *p, size_t elem, size_t width) {
  a.out = p; a.elem = elem; a.width = width; a.used = p != nullptr;
}

int bit_length(uint32_t v) {   // floor(log2(v) + 1) for v >= 1 (index.js:573, 601)
  int b = 0;
  while (v) { ++b; v >>= 1; }
  return b;
}
// the array crosses the host link as packOutput(max_val, width, row).expected (index.js:572-596)
void set_fe(HostArr &a, uint32_t max_val) {
  if (!a.used) return;
  a.fe_bits = bit_length(max_val);
  a.fe_n = 252 / a.fe_bits;
  int outs = ((int)a.width + a.fe_n - 1) / a.fe_n;
  a.fe_elems = outs < 3 ? 3 : outs;
}

int packed_elems(uint32_t max_val, int width) {
  const int n = 252 / bit_length(max_val);
  const int outs = (width + n - 1) / n;
  return outs < 3 ? 3 : outs;
}

// Below this many rows the tcgen05 schedule cannot fill the chip (one CTA pair per 256 rows, 74 pairs) and the
// one-warp-per-ciphertext IMMA schedule finishes sooner (scripts/bench_latency.py: 1024 rows at N = 821 take 1.7 ms
// against 0.55 ms): NTRU_OPT_PATH = 0 picks the IMMA schedule there.
constexpr size_t kSmallBatchRows = 4096;

bool want_tensor(ntru_ctx *ctx, bool same_key, bool ready, size_t B, int *rc) {
  *rc = NTRU_OK;
  if (ctx->opt_path == 1 || ctx->opt_path == 3) return false;
  if (ctx->opt_path == 0 && B < kSmallBatchRows && ctx->tensor_ok && imma_supported(ctx)) return false;
  const bool ok = same_key && ctx->tensor_ok && ready;
  if (ctx->opt_path == 2 && !ok) {
    *rc = fail(ctx, NTRU_E_UNSUPPORTED, "tensor schedule forced but not available for this call");
    return false;
  }
  return ok;
}

// register-fragment (IMMA) schedule: the default whenever the tcgen05 same-key schedule does not apply
bool want_imma(ntru_ctx *ctx, bool wide_message, int *rc) {
  *rc = NTRU_OK;
  if (ctx->opt_path == 1) return false;
  const bool ok = ctx->tensor_ok && imma_supported(ctx) && !wide_message;
  if (ctx->opt_path == 3 && !ok) {
    *rc = fail(ctx, NTRU_E_UNSUPPORTED, "register-fragment schedule forced but not available for this call");
    return false;
  }
  return ok;
}

int encrypt_dispatch(ntru_ctx *ctx, size_t B, const uint16_t *h_rows, const uint8_t *r, const void *m, int m_wide,
                     uint16_t *value, uint16_t *quo, uint16_t *rem) {
  int rc;
  const bool same_key = h_rows == nullptr;
  if (same_key && !ctx->has_pub) return fail(ctx, NTRU_E_NOKEY, "public key h is not set");
  if (want_tensor(ctx, same_key && !m_wide, ctx->km_h.ready, B, &rc)) {
    ctx->last_path = 2;
    return umma_encrypt(ctx, B, r, (const uint8_t *)m, value, quo, rem);
  }
  if (rc != NTRU_OK) return rc;
  if (want_imma(ctx, m_wide != 0, &rc)) {
    ctx->last_path = 3;
    return launch_encrypt_imma(ctx, B, same_key ? (const uint16_t *)ctx->d_h.ptr : h_rows, same_key ? 0 : (size_t)ctx->P, r,
                               (const uint8_t *)m, value, quo, rem);
  }
  if (rc != NTRU_OK) return rc;
  ctx->last_path = 1;
  return launch_encrypt_generic(ctx, B, same_key ? (const uint16_t *)ctx->d_h.ptr : h_rows,
                                same_key ? 0 : (size_t)ctx->P, r, m, m_wide, value, quo, rem);
}

int decrypt_dispatch(ntru_ctx *ctx, size_t B, const int8_t *f_rows, const uint8_t *fp_rows, const uint16_t *e,
                     uint8_t *value, uint16_t *q1, uint16_t *r1, uint8_t *q2, uint8_t *r2) {
  int rc;
  const bool same_key = f_rows == nullptr && fp_rows == nullptr;
  if ((f_rows == nullptr) != (fp_rows == nullptr)) return fail(ctx, NTRU_E_PARAM, "f_rows and fp_rows must be given together");
  if (same_key && !ctx->has_priv) return fail(ctx, NTRU_E_NOKEY, "private key f/fp is not set");
  if (want_tensor(ctx, same_key, ctx->km_f.ready && ctx->km_fp.ready, B, &rc)) {
    ctx->last_path = 2;
    return umma_decrypt(ctx, B, e, value, q1, r1, q2, r2);
  }
  if (rc != NTRU_OK) return rc;
  if (want_imma(ctx, false, &rc)) {
    ctx->last_path = 3;
    return launch_decrypt_imma(ctx, B, same_key ? (const int8_t *)ctx->d_f.ptr : f_rows,
                               same_key ? (const uint8_t *)ctx->d_fp.ptr : fp_rows, same_key ? 0 : (size_t)ctx->P, e, value, q1,
                               r1, q2, r2);
  }
  if (rc != NTRU_OK) return rc;
  ctx->last_path = 1;
  return launch_decrypt_generic(ctx, B, same_key ? (const int8_t *)ctx->d_f.ptr : f_rows,
                                same_key ? (const uint8_t *)ctx->d_fp.ptr : fp_rows,
                                same_key ? 0 : (size_t)ctx->P, e, value, q1, r1, q2, r2);
}

int check(ntru_ctx *ctx) {
  if (!ctx) return NTRU_E_PARAM;
  cudaError_t e = cudaSetDevice(ctx->device);
  if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaSetDevice");
  return NTRU_OK;
}

}  // namespace
}  // namespace ntru

using namespace ntru;

extern "C" {

const char *ntru_strerror(int code) {
  switch (code) {
    case NTRU_OK: return "ok";
    case NTRU_E_PARAM: return "bad parameter";
    case NTRU_E_LENGTH: return "bad length";
    case NTRU_E_NOKEY: return "key not set";
    case NTRU_E_CUDA: return "CUDA error";
    case NTRU_E_NCCL: return "NCCL error";
    case NTRU_E_NOMEM: return "out of memory";
    case NTRU_E_UNSUPPORTED: return "unsupported";
    default: return "unknown error";
  }
}

const char *ntru_last_error(const ntru_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int ntru_create(ntru_ctx **out, int N, int p, int q, int device) {
  if (!out) return NTRU_E_PARAM;
  *out = nullptr;
  if (p != 3) return NTRU_E_PARAM;
  if (N < 8 || N > kMaxN) return NTRU_E_PARAM;
  // q <= 8192: the tcgen05 schedule keeps 5 bits in its high limb and folds a lifted coefficient <= q into one byte
  // (umma_pair.cuh), and BASELINE's largest modulus is 8192; larger moduli are refused instead of being routed silently
  if (q < 4 || q > 8192 || (q & (q - 1)) != 0) return NTRU_E_PARAM;
  // fp32 exactness bound of the CUDA-core schedule: N * 2 * (q-1) < 2^24
  if ((long long)N * 2 * (q - 1) >= (1ll << 24)) return NTRU_E_PARAM;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) return NTRU_E_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return NTRU_E_CUDA;
  ntru_ctx *ctx = new (std::nothrow) ntru_ctx();
  if (!ctx) return NTRU_E_NOMEM;
  ctx->N = N; ctx->p = p; ctx->q = q; ctx->device = device;
  ctx->logq = 0;
  while ((1 << ctx->logq) < q) ctx->logq++;
  ctx->P = ((N + 1 + 15) / 16) * 16;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess;
  ctx->own_stream = ok;
  ok = ok && cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking) == cudaSuccess;
  for (int s = 0; ok && s < kNumSlots; ++s) {
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_in[s], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_comp[s], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_out[s], cudaEventDisableTiming) == cudaSuccess;
  }
  ok = ok && ctx->d_h.reserve((size_t)ctx->P * 2) == cudaSuccess;
  ok = ok && ctx->d_f.reserve((size_t)ctx->P) == cudaSuccess;
  ok = ok && ctx->d_fp.reserve((size_t)ctx->P) == cudaSuccess;
  ok = ok && ctx->d_partial.reserve((size_t)ctx->P * 4) == cudaSuccess;
  if (!ok) {
    ntru_destroy(ctx);
    return NTRU_E_CUDA;
  }
  // key of the device CSPRNG that draws r (index.js:89 uses crypto.getRandomValues): 256 bits of OS entropy
  {
    size_t got = 0;
    unsigned char *kb = reinterpret_cast<unsigned char *>(ctx->rng_key);
    while (got < sizeof ctx->rng_key) {
      ssize_t n = getrandom(kb + got, sizeof ctx->rng_key - got, 0);
      if (n <= 0) break;
      got += (size_t)n;
    }
    if (got < sizeof ctx->rng_key) {
      FILE *fh = fopen("/dev/urandom", "rb");
      if (fh) {
        got += fread(kb + got, 1, sizeof ctx->rng_key - got, fh);
        fclose(fh);
      }
    }
    ctx->rng_keyed = got == sizeof ctx->rng_key;   // without entropy r == NULL is refused (no silent weak key)
  }
  umma_init(ctx);
  *out = ctx;
  return NTRU_OK;
}

static int xchg_release(ntru_ctx *ctx);
static int xchg_check(ntru_ctx *ctx);

void ntru_destroy(ntru_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (int s = 0; s < kNumSlots; ++s) {
    if (ctx->ev_in[s]) cudaEventDestroy(ctx->ev_in[s]);
    if (ctx->ev_comp[s]) cudaEventDestroy(ctx->ev_comp[s]);
    if (ctx->ev_out[s]) cudaEventDestroy(ctx->ev_out[s]);
    for (auto &b : ctx->slot_bufs[s]) b.release();
    for (auto &b : ctx->slot_packed[s]) b.release();
  }
  xchg_release(ctx);
  ctx->d_h.release(); ctx->d_f.release(); ctx->d_fp.release(); ctx->d_b.release(); ctx->d_partial.release(); ctx->d_sum_scratch.release();
  ctx->km_h.mat.release(); ctx->km_f.mat.release(); ctx->km_fp.mat.release();
  for (auto &b : ctx->kg_bufs) b.release();
  for (auto &b : ctx->check_key) b.release();
  for (auto &t : ctx->timed) {
    cudaEventDestroy(t.a);
    cudaEventDestroy(t.b);
  }
  for (auto e : ctx->event_pool) cudaEventDestroy(e);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
  if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
  delete ctx;
}

int ntru_set_option(ntru_ctx *ctx, int key, long value) {
  if (!ctx) return NTRU_E_PARAM;
  switch (key) {
    case NTRU_OPT_PATH:
      if (value < 0 || value > 3) return fail(ctx, NTRU_E_PARAM, "NTRU_OPT_PATH must be 0, 1, 2 or 3");
      ctx->opt_path = (int)value;
      return NTRU_OK;
    case NTRU_OPT_CHUNK_ROWS:
      if (value < 128) return fail(ctx, NTRU_E_PARAM, "NTRU_OPT_CHUNK_ROWS must be >= 128");
      ctx->chunk_rows = (size_t)value;
      return NTRU_OK;
    case NTRU_OPT_TIMING:
      ctx->timing = value != 0;
      return NTRU_OK;
    case NTRU_OPT_SCHEDULE:
      if (value < 0 || value > 1) return fail(ctx, NTRU_E_PARAM, "NTRU_OPT_SCHEDULE must be 0 or 1");
      ctx->opt_lohi = (int)value;
      return NTRU_OK;
    case NTRU_OPT_EPILOGUE:
      if (value < 0 || value > 2) return fail(ctx, NTRU_E_PARAM, "NTRU_OPT_EPILOGUE must be 0, 1 or 2");
      ctx->opt_epilogue = (int)value;
      if (ctx->tensor_ok) {       // the chunk tables depend on it: rebuild the operand matrices
        if (ctx->has_pub) { int rc = umma_prepare_public(ctx); if (rc) return rc; }
        if (ctx->has_priv) { int rc = umma_prepare_private(ctx); if (rc) return rc; }
      }
      return NTRU_OK;
    case NTRU_OPT_IMMA_FORM:
      if (value < 0 || value > 1) return fail(ctx, NTRU_E_PARAM, "NTRU_OPT_IMMA_FORM must be 0 or 1");
      ctx->opt_imma_form = (int)value;
      return NTRU_OK;
    case NTRU_OPT_DEC1_FORM:
      if (value < 0 || value > 2) return fail(ctx, NTRU_E_PARAM, "NTRU_OPT_DEC1_FORM must be 0, 1 or 2");
      ctx->opt_dec1_form = (int)value;
      if (ctx->has_priv && ctx->tensor_ok) return umma_prepare_private(ctx);   // rebuild the operand matrix of f in the other form
      return NTRU_OK;
    case NTRU_OPT_DR:
      // index.js:462-464
      if (value < 0 || 2 * value > ctx->N) return fail(ctx, NTRU_E_PARAM, "The total of 1s and -1s cannot exceed the array length.");
      ctx->opt_dr = (int)value;
      return NTRU_OK;
    default:
      return fail(ctx, NTRU_E_PARAM, "unknown option");
  }
}

int ntru_pitch(const ntru_ctx *ctx) { return ctx ? ctx->P : 0; }
uint64_t ntru_launch_count(const ntru_ctx *ctx) { return ctx ? ctx->launches : 0; }
int ntru_last_path(const ntru_ctx *ctx) { return ctx ? ctx->last_path : 0; }

int ntru_timing_reset(ntru_ctx *ctx) {
  int rc = check(ctx);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto &t : ctx->timed) {
    ctx->event_pool.push_back(t.a);
    ctx->event_pool.push_back(t.b);
  }
  ctx->timed.clear();
  return NTRU_OK;
}

int ntru_timing_read(ntru_ctx *ctx, int kind, double *total_ms, uint64_t *launches) {
  int rc = check(ctx);
  if (rc) return rc;
  if (kind < 0 || kind >= NTRU_K_COUNT || !total_ms || !launches) return fail(ctx, NTRU_E_PARAM, "bad timing query");
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  double sum = 0;
  uint64_t n = 0;
  for (auto &t : ctx->timed) {
    if (t.kind != kind) continue;
    float ms = 0;
    NTRU_CUDA(ctx, cudaEventElapsedTime(&ms, t.a, t.b));
    sum += ms;
    ++n;
  }
  *total_ms = sum;
  *launches = n;
  return NTRU_OK;
}

int ntru_set_public_key(ntru_ctx *ctx, const uint16_t *h) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!h) return fail(ctx, NTRU_E_PARAM, "h is NULL");
  uint16_t tmp[kMaxN + 32];
  memset(tmp, 0, sizeof tmp);
  for (int i = 0; i < ctx->N; ++i) {
    if (h[i] >= ctx->q) return fail(ctx, NTRU_E_PARAM, "h coefficient outside [0,q)");
    tmp[i] = h[i];
  }
  // on the context's stream, so that calls queued before this one finish under the key they were queued with; a plain
  // cudaMemcpy runs on the legacy stream, which does not wait for a non-blocking one.  tmp lives on this frame.
  NTRU_CUDA(ctx, cudaMemcpyAsync(ctx->d_h.ptr, tmp, (size_t)ctx->P * 2, cudaMemcpyHostToDevice, ctx->stream));
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->has_pub = true;
  ctx->km_h.ready = false;
  if (ctx->tensor_ok) {
    rc = umma_prepare_public(ctx);
    if (rc) return rc;
  }
  return NTRU_OK;
}

int ntru_set_private_key(ntru_ctx *ctx, const int8_t *f, const uint8_t *fp) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!f || !fp) return fail(ctx, NTRU_E_PARAM, "f or fp is NULL");
  int8_t tf[kMaxN + 32];
  uint8_t tp[kMaxN + 32];
  memset(tf, 0, sizeof tf);
  memset(tp, 0, sizeof tp);
  for (int i = 0; i < ctx->N; ++i) {
    if (f[i] < -1 || f[i] > 1) return fail(ctx, NTRU_E_PARAM, "f coefficient outside {-1,0,1}");
    if (fp[i] >= ctx->p) return fail(ctx, NTRU_E_PARAM, "fp coefficient outside [0,p)");
    tf[i] = f[i];
    tp[i] = fp[i];
  }
  // ordered after the queued calls, as in ntru_set_public_key
  NTRU_CUDA(ctx, cudaMemcpyAsync(ctx->d_f.ptr, tf, (size_t)ctx->P, cudaMemcpyHostToDevice, ctx->stream));
  NTRU_CUDA(ctx, cudaMemcpyAsync(ctx->d_fp.ptr, tp, (size_t)ctx->P, cudaMemcpyHostToDevice, ctx->stream));
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->has_priv = true;
  ctx->km_f.ready = ctx->km_fp.ready = false;
  if (ctx->tensor_ok) {
    rc = umma_prepare_private(ctx);
    if (rc) return rc;
  }
  return NTRU_OK;
}

// ---- host-buffer entry points ---------------------------------------------------------------

static int encrypt_host(ntru_ctx *ctx, size_t B, const uint16_t *h, const uint8_t *r, const void *m, int m_wide,
                        uint16_t *value, uint16_t *quo, uint16_t *rem, uint8_t *r_out, bool fe = false) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!m) return fail(ctx, NTRU_E_PARAM, "m is required");
  if (!r) {   // the device draws r (index.js:89): needs dr and an entropy-keyed generator
    if (ctx->opt_dr < 0) return fail(ctx, NTRU_E_PARAM, "r is NULL and NTRU_OPT_DR (the dr of the constructor options) is not set");
    if (!ctx->rng_keyed) return fail(ctx, NTRU_E_UNSUPPORTED, "r is NULL and the device generator has no key (no OS entropy; call ntru_set_rng_key)");
  }
  if (B == 0) return NTRU_OK;
  const size_t N = (size_t)ctx->N;
  HostArr arr[kMaxArr];
  set_in(arr[0], h, 2, N);
  if (r) {
    set_in(arr[1], r, 1, N);
    if (r_out && r_out != r)                             // injected r is echoed (inputs.r, index.js:97)
      memcpy(r_out, r, fe ? B * (size_t)packed_elems(ctx->p - 1, (int)N) * 32 : B * N);
  } else {
    set_out(arr[1], r_out, 1, N);
    arr[1].used = true;                                  // device rows are needed even when r is not returned
  }
  set_in(arr[2], m, m_wide ? 2 : 1, N);
  set_out(arr[3], value, 2, N);
  set_out(arr[4], quo, 2, N + 1);
  set_out(arr[5], rem, 2, N + 1);
  if (fe) {
    set_fe(arr[1], (uint32_t)ctx->p - 1); set_fe(arr[2], (uint32_t)ctx->p - 1);
    for (int a = 3; a <= 5; ++a) set_fe(arr[a], (uint32_t)ctx->q - 1);
  }
  uint64_t next_row = ctx->rng_row;
  if (!r) ctx->rng_row += B;                             // a row number (nonce) is never used twice under one key
  return run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
    if (!r) {
      int rs = launch_sample(ctx, rows, ctx->opt_dr, ctx->opt_dr, 2, next_row, nullptr, (uint8_t *)dev[1]);
      if (rs) return rs;
      next_row += rows;
    }
    return encrypt_dispatch(ctx, rows, (const uint16_t *)dev[0], (const uint8_t *)dev[1], dev[2], m_wide,
                            (uint16_t *)dev[3], (uint16_t *)dev[4], (uint16_t *)dev[5]);
  });
}

int ntru_encrypt_batch(ntru_ctx *ctx, size_t B, const uint8_t *r, const uint8_t *m, uint16_t *value,
                       uint16_t *quotientE, uint16_t *remainderE, uint8_t *r_out) {
  return encrypt_host(ctx, B, nullptr, r, m, 0, value, quotientE, remainderE, r_out);
}

int ntru_encrypt_batch_wide(ntru_ctx *ctx, size_t B, const uint8_t *r, const uint16_t *m, uint16_t *value,
                            uint16_t *quotientE, uint16_t *remainderE, uint8_t *r_out) {
  return encrypt_host(ctx, B, nullptr, r, m, 1, value, quotientE, remainderE, r_out);
}

int ntru_encrypt_batch_keys(ntru_ctx *ctx, size_t B, const uint16_t *h, const uint8_t *r, const uint8_t *m,
                            uint16_t *value, uint16_t *quotientE, uint16_t *remainderE, uint8_t *r_out) {
  if (!h) return fail(ctx, NTRU_E_PARAM, "h is NULL");
  return encrypt_host(ctx, B, h, r, m, 0, value, quotientE, remainderE, r_out);
}

static int decrypt_host(ntru_ctx *ctx, size_t B, const int8_t *f, const uint8_t *fp, const uint16_t *e,
                        uint8_t *value, uint16_t *q1, uint16_t *r1, uint8_t *q2, uint8_t *r2, bool fe = false) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!e) return fail(ctx, NTRU_E_PARAM, "e is required");
  if (B == 0) return NTRU_OK;
  const size_t N = (size_t)ctx->N;
  HostArr arr[kMaxArr];
  set_in(arr[0], f, 1, N);
  set_in(arr[1], fp, 1, N);
  set_in(arr[2], e, 2, N);
  set_out(arr[3], value, 1, N);
  set_out(arr[4], q1, 2, N + 1);
  set_out(arr[5], r1, 2, N + 1);
  set_out(arr[6], q2, 1, N + 1);
  set_out(arr[7], r2, 1, N + 1);
  if (fe) {
    set_fe(arr[2], (uint32_t)ctx->q - 1); set_fe(arr[4], (uint32_t)ctx->q - 1); set_fe(arr[5], (uint32_t)ctx->q - 1);
    set_fe(arr[3], (uint32_t)ctx->p - 1); set_fe(arr[6], (uint32_t)ctx->p - 1); set_fe(arr[7], (uint32_t)ctx->p - 1);
  }
  return run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
    return decrypt_dispatch(ctx, rows, (const int8_t *)dev[0], (const uint8_t *)dev[1], (const uint16_t *)dev[2],
                            (uint8_t *)dev[3], (uint16_t *)dev[4], (uint16_t *)dev[5], (uint8_t *)dev[6],
                            (uint8_t *)dev[7]);
  });
}

int ntru_decrypt_batch(ntru_ctx *ctx, size_t B, const uint16_t *e, uint8_t *value, uint16_t *quotient1,
                       uint16_t *remainder1, uint8_t *quotient2, uint8_t *remainder2) {
  return decrypt_host(ctx, B, nullptr, nullptr, e, value, quotient1, remainder1, quotient2, remainder2);
}

int ntru_decrypt_batch_keys(ntru_ctx *ctx, size_t B, const int8_t *f, const uint8_t *fp, const uint16_t *e,
                            uint8_t *value, uint16_t *quotient1, uint16_t *remainder1, uint8_t *quotient2,
                            uint8_t *remainder2) {
  if (!f || !fp) return fail(ctx, NTRU_E_PARAM, "f or fp is NULL");
  return decrypt_host(ctx, B, f, fp, e, value, quotient1, remainder1, quotient2, remainder2);
}

int ntru_packed_elems(const ntru_ctx *ctx, int mod_q, int width) {
  if (!ctx || width < 0) return 0;
  return packed_elems(mod_q ? (uint32_t)ctx->q - 1 : (uint32_t)ctx->p - 1, width);
}

int ntru_encrypt_batch_packed(ntru_ctx *ctx, size_t B, const void *r, const void *m, void *value, void *quotientE,
                              void *remainderE, void *r_out) {
  return encrypt_host(ctx, B, nullptr, (const uint8_t *)r, m, 0, (uint16_t *)value, (uint16_t *)quotientE, (uint16_t *)remainderE,
                      (uint8_t *)r_out, true);
}

int ntru_decrypt_batch_packed(ntru_ctx *ctx, size_t B, const void *e, void *value, void *quotient1, void *remainder1,
                              void *quotient2, void *remainder2) {
  return decrypt_host(ctx, B, nullptr, nullptr, (const uint16_t *)e, (uint8_t *)value, (uint16_t *)quotient1, (uint16_t *)remainder1,
                      (uint8_t *)quotient2, (uint8_t *)remainder2, true);
}

int ntru_muldiv_dev(ntru_ctx *ctx, size_t B, const int8_t *x, const void *y, int mod_p, void *quotient, void *remainder) {
  int rc = check(ctx);
  if (rc) return rc;
  if (B > 0 && (!x || !y)) return fail(ctx, NTRU_E_PARAM, "x and y are required");
  if (!ctx->tensor_ok) return fail(ctx, NTRU_E_UNSUPPORTED, "multiply + divide needs the sm_100 tensor path");
  return launch_muldiv_imma(ctx, B, x, y, mod_p, quotient, remainder);
}

int ntru_verify_keys_batch(ntru_ctx *ctx, size_t B, const int8_t *f, const uint16_t *fq, const uint8_t *fp, const int8_t *g,
                           uint16_t *quotient_fq, uint16_t *remainder_fq, uint8_t *quotient_fp, uint8_t *remainder_fp,
                           uint16_t *quotient_h, uint16_t *remainder_h) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!f || !fq || !fp || !g) return fail(ctx, NTRU_E_PARAM, "f, fq, fp and g are required");
  if (!ctx->tensor_ok) return fail(ctx, NTRU_E_UNSUPPORTED, "verify_keys needs the sm_100 tensor path");
  if (B == 0) return NTRU_OK;
  const size_t N = (size_t)ctx->N;
  HostArr arr[kMaxArr];
  set_in(arr[0], f, 1, N);
  set_in(arr[1], fq, 2, N);
  set_in(arr[2], fp, 1, N);
  set_in(arr[3], g, 1, N);
  set_out(arr[4], quotient_fq, 2, N + 1);
  set_out(arr[5], remainder_fq, 2, N + 1);
  set_out(arr[6], quotient_fp, 1, N + 1);
  set_out(arr[7], remainder_fp, 1, N + 1);
  set_out(arr[8], quotient_h, 2, N + 1);
  set_out(arr[9], remainder_h, 2, N + 1);
  return run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
    int r2 = NTRU_OK;
    if (dev[4] || dev[5]) r2 = launch_muldiv_imma(ctx, rows, (const int8_t *)dev[0], dev[1], 0, dev[4], dev[5]);
    if (r2) return r2;
    // fp case: x = f (the value p-1 of a -1 is the same residue), y = fp
    if (dev[6] || dev[7]) r2 = launch_muldiv_imma(ctx, rows, (const int8_t *)dev[0], dev[2], 1, dev[6], dev[7]);
    if (r2) return r2;
    if (dev[8] || dev[9])
      r2 = launch_h_product(ctx, rows, (const int8_t *)dev[3], (const uint16_t *)dev[1], (uint16_t *)dev[8], (uint16_t *)dev[9]);
    return r2;
  });
}

int ntru_keygen_batch(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h,
                      uint8_t *valid) {
  int rc = check(ctx);
  if (rc) return rc;
  if (B > 0 && (!f || !g || !fq || !fp || !h || !valid)) return fail(ctx, NTRU_E_PARAM, "f, g, fq, fp, h and valid are required");
  return keygen_batch(ctx, B, f, g, fq, fp, h, valid);
}

int ntru_keygen_dev(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h,
                    uint8_t *valid) {
  int rc = check(ctx);
  if (rc) return rc;
  if (B > 0 && (!f || !g || !fq || !fp || !h || !valid)) return fail(ctx, NTRU_E_PARAM, "f, g, fq, fp, h and valid are required");
  return keygen_dev(ctx, B, f, g, fq, fp, h, valid);
}

int ntru_generate_keys_dev(ntru_ctx *ctx, size_t B, int df, int dg, int8_t *f, int8_t *g, uint16_t *fq, uint8_t *fp,
                           uint16_t *h) {
  int rc = check(ctx);
  if (rc) return rc;
  if (B > 0 && (!f || !g || !fq || !fp || !h)) return fail(ctx, NTRU_E_PARAM, "f, g, fq, fp and h are required");
  // index.js:462-464 (f has df ones and df - 1 minus ones, g dg of each)
  if (df < 1 || 2 * df - 1 > ctx->N || dg < 0 || 2 * dg > ctx->N)
    return fail(ctx, NTRU_E_PARAM, "The total of 1s and -1s cannot exceed the array length.");
  if (!ctx->rng_keyed) return fail(ctx, NTRU_E_UNSUPPORTED, "the device generator has no key (no OS entropy; call ntru_set_rng_key)");
  return generate_keys_dev(ctx, B, df, dg, f, g, fq, fp, h);
}


// ---- witness checks ------------------------------------------------------------------------------------------------

static int check_args(ntru_ctx *ctx, size_t B, bool all_given, size_t key_stride) {
  if (!ctx) return NTRU_E_PARAM;
  if (B > 0 && !all_given) return fail(ctx, NTRU_E_PARAM, "every array of the witness check is required");
  if (key_stride != 0 && key_stride != (size_t)ctx->P) return fail(ctx, NTRU_E_PARAM, "key_stride must be 0 or ntru_pitch(ctx)");
  int rc = check(ctx);
  if (rc) return rc;
  if (!ctx->tensor_ok) return fail(ctx, NTRU_E_UNSUPPORTED, "witness checks need the sm_100 tensor path");
  if (!imma_supported(ctx)) return fail(ctx, NTRU_E_UNSUPPORTED, "witness checks support N <= 832");
  return NTRU_OK;
}

int ntru_check_encrypt_dev(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t key_stride, const uint8_t *r, const uint16_t *m,
                           const uint16_t *quotientE, const uint16_t *remainderE, uint8_t *verdict) {
  int rc = check_args(ctx, B, h && r && m && quotientE && remainderE && verdict, key_stride);
  if (rc) return rc;
  return launch_check_encrypt(ctx, B, h, key_stride, r, m, quotientE, remainderE, verdict);
}

int ntru_check_decrypt_dev(ntru_ctx *ctx, size_t B, const uint16_t *f, const uint8_t *fp, size_t key_stride, const uint16_t *e,
                           const uint16_t *quotient1, const uint16_t *remainder1, const uint8_t *quotient2,
                           const uint8_t *remainder2, uint8_t *verdict) {
  int rc = check_args(ctx, B, f && fp && e && quotient1 && remainder1 && quotient2 && remainder2 && verdict, key_stride);
  if (rc) return rc;
  return launch_check_decrypt(ctx, B, f, fp, key_stride, e, quotient1, remainder1, quotient2, remainder2, verdict);
}

int ntru_check_inverse_dev(ntru_ctx *ctx, size_t B, int mod_p, const uint16_t *x, const void *y, const void *quotientI,
                           const void *remainderI, uint8_t *verdict) {
  int rc = check_args(ctx, B, x && y && quotientI && remainderI && verdict, 0);
  if (rc) return rc;
  return launch_check_inverse(ctx, B, mod_p, x, y, quotientI, remainderI, verdict);
}

// the shared key row of a host-form check: one upload on the context's stream, ahead of the chunks' kernels
static int upload_key_row(ntru_ctx *ctx, int slot, const void *row, size_t elem) {
  const size_t P = (size_t)ctx->P;
  NTRU_CUDA(ctx, ctx->check_key[slot].reserve(P * elem));
  NTRU_CUDA(ctx, cudaMemsetAsync(ctx->check_key[slot].ptr, 0, P * elem, ctx->stream));
  NTRU_CUDA(ctx, cudaMemcpyAsync(ctx->check_key[slot].ptr, row, (size_t)ctx->N * elem, cudaMemcpyHostToDevice, ctx->stream));
  return NTRU_OK;
}

int ntru_check_encrypt_batch(ntru_ctx *ctx, size_t B, const uint16_t *h, int key_shared, const uint8_t *r, const uint16_t *m,
                             const uint16_t *quotientE, const uint16_t *remainderE, uint8_t *verdict) {
  int rc = check_args(ctx, B, h && r && m && quotientE && remainderE && verdict, 0);
  if (rc || B == 0) return rc;
  const size_t N = (size_t)ctx->N;
  HostArr arr[kMaxArr];
  if (key_shared) {
    rc = upload_key_row(ctx, 0, h, 2);
    if (rc) return rc;
  } else {
    set_in(arr[0], h, 2, N);
  }
  set_in(arr[1], r, 1, N);
  set_in(arr[2], m, 2, N);
  set_in(arr[3], quotientE, 2, N + 1);
  set_in(arr[4], remainderE, 2, N + 1);
  set_out(arr[5], verdict, 1, 1);
  arr[5].flat = true;
  return run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
    return launch_check_encrypt(ctx, rows, key_shared ? (const uint16_t *)ctx->check_key[0].ptr : (const uint16_t *)dev[0],
                                key_shared ? 0 : (size_t)ctx->P, (const uint8_t *)dev[1], (const uint16_t *)dev[2],
                                (const uint16_t *)dev[3], (const uint16_t *)dev[4], (uint8_t *)dev[5]);
  });
}

int ntru_check_decrypt_batch(ntru_ctx *ctx, size_t B, const uint16_t *f, const uint8_t *fp, int key_shared, const uint16_t *e,
                             const uint16_t *quotient1, const uint16_t *remainder1, const uint8_t *quotient2,
                             const uint8_t *remainder2, uint8_t *verdict) {
  int rc = check_args(ctx, B, f && fp && e && quotient1 && remainder1 && quotient2 && remainder2 && verdict, 0);
  if (rc || B == 0) return rc;
  const size_t N = (size_t)ctx->N;
  HostArr arr[kMaxArr];
  if (key_shared) {
    rc = upload_key_row(ctx, 0, f, 2);
    if (!rc) rc = upload_key_row(ctx, 1, fp, 1);
    if (rc) return rc;
  } else {
    set_in(arr[0], f, 2, N);
    set_in(arr[1], fp, 1, N);
  }
  set_in(arr[2], e, 2, N);
  set_in(arr[3], quotient1, 2, N + 1);
  set_in(arr[4], remainder1, 2, N + 1);
  set_in(arr[5], quotient2, 1, N + 1);
  set_in(arr[6], remainder2, 1, N + 1);
  set_out(arr[7], verdict, 1, 1);
  arr[7].flat = true;
  return run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
    return launch_check_decrypt(ctx, rows, key_shared ? (const uint16_t *)ctx->check_key[0].ptr : (const uint16_t *)dev[0],
                                key_shared ? (const uint8_t *)ctx->check_key[1].ptr : (const uint8_t *)dev[1],
                                key_shared ? 0 : (size_t)ctx->P, (const uint16_t *)dev[2], (const uint16_t *)dev[3],
                                (const uint16_t *)dev[4], (const uint8_t *)dev[5], (const uint8_t *)dev[6], (uint8_t *)dev[7]);
  });
}

int ntru_check_inverse_batch(ntru_ctx *ctx, size_t B, int mod_p, const uint16_t *x, const void *y, const void *quotientI,
                             const void *remainderI, uint8_t *verdict) {
  int rc = check_args(ctx, B, x && y && quotientI && remainderI && verdict, 0);
  if (rc || B == 0) return rc;
  const size_t N = (size_t)ctx->N, wb = mod_p ? 1 : 2;
  HostArr arr[kMaxArr];
  set_in(arr[0], x, 2, N);
  set_in(arr[1], y, wb, N);
  set_in(arr[2], quotientI, wb, N + 1);
  set_in(arr[3], remainderI, wb, N + 1);
  set_out(arr[4], verdict, 1, 1);
  arr[4].flat = true;
  return run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
    return launch_check_inverse(ctx, rows, mod_p, (const uint16_t *)dev[0], dev[1], dev[2], dev[3], (uint8_t *)dev[4]);
  });
}


int ntru_pack_geometry(uint32_t max_val, int data_len, int *max_input_bits, int *inputs_per_output, int *arr_len,
                       int *output_size) {
  if (max_val == 0 || data_len < 0) return NTRU_E_PARAM;
  const int bits = bit_length(max_val);
  const int n = 252 / bits;
  int arr = ((data_len + n - 1) / n) * n;
  if (arr < 3 * n) arr = 3 * n;
  int outs = (arr + n - 1) / n;
  if (outs < 3) outs = 3;
  if (max_input_bits) *max_input_bits = bits;
  if (inputs_per_output) *inputs_per_output = n;
  if (arr_len) *arr_len = arr;
  if (output_size) *output_size = outs;
  return NTRU_OK;
}

int ntru_pack_output_dev(ntru_ctx *ctx, size_t B, const void *data, int elem_bytes, int data_len, size_t pitch,
                         uint32_t max_val, void *out) {
  int rc = check(ctx);
  if (rc) return rc;
  int bits, n, arr, outs;
  if (ntru_pack_geometry(max_val, data_len, &bits, &n, &arr, &outs) != NTRU_OK || (elem_bytes != 1 && elem_bytes != 2))
    return fail(ctx, NTRU_E_PARAM, "bad maxVal / dataLen / element size");
  if (bits > 8 * elem_bytes + 16) return fail(ctx, NTRU_E_PARAM, "maxVal does not fit the element type");
  if (B > 0 && (!data || !out)) return fail(ctx, NTRU_E_PARAM, "data and out are required");
  return launch_pack_fields(ctx, B, data, elem_bytes, data_len, pitch, bits, n, outs, (uint32_t *)out);
}

int ntru_unpack_input_dev(ntru_ctx *ctx, size_t B, const void *data, int n_elems, uint32_t max_val, int packed_bits,
                          void *out, int elem_bytes, size_t pitch) {
  int rc = check(ctx);
  if (rc) return rc;
  if (max_val == 0 || n_elems < 0 || packed_bits < 1 || packed_bits > 256 || (elem_bytes != 1 && elem_bytes != 2))
    return fail(ctx, NTRU_E_PARAM, "bad maxVal / packedBits / element size");
  const int bits = bit_length(max_val);
  const int n = packed_bits / bits;
  if (n < 1) return fail(ctx, NTRU_E_PARAM, "packedBits is smaller than one coefficient");
  if (bits > 8 * elem_bytes) return fail(ctx, NTRU_E_PARAM, "maxVal does not fit the element type");
  if (B > 0 && (!data || !out)) return fail(ctx, NTRU_E_PARAM, "data and out are required");
  return launch_unpack_fields(ctx, B, (const uint32_t *)data, n_elems, bits, n, pitch, out, elem_bytes);
}

int ntru_sum(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!e || !out) return fail(ctx, NTRU_E_PARAM, "e and out are required");
  NTRU_CUDA(ctx, cudaMemsetAsync(ctx->d_partial.ptr, 0, (size_t)ctx->P * 4, ctx->stream));
  if (B > 0) {
    HostArr arr[kMaxArr];
    set_in(arr[0], e, 2, (size_t)ctx->N);
    // the kernel streams whole pitched rows; pad columns land in partial[k >= N], which finalize ignores
    rc = run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
      return launch_sum_partial(ctx, rows, (const uint16_t *)dev[0], (uint32_t *)ctx->d_partial.ptr);
    });
    if (rc) return rc;
  }
  NTRU_CUDA(ctx, ctx->slot_bufs[0][9].reserve((size_t)ctx->P * 2));
  rc = launch_sum_finalize(ctx, (const uint32_t *)ctx->d_partial.ptr, (uint16_t *)ctx->slot_bufs[0][9].ptr);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaMemcpyAsync(out, ctx->slot_bufs[0][9].ptr, (size_t)ctx->N * 2, cudaMemcpyDeviceToHost,
                                 ctx->stream));
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NTRU_OK;
}

// ---- device-resident entry points -------------------------------------------------------------

int ntru_encrypt_dev(ntru_ctx *ctx, size_t B, const uint16_t *h_rows, const uint8_t *r, const uint8_t *m,
                     uint16_t *value, uint16_t *quotientE, uint16_t *remainderE) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!r || !m) return fail(ctx, NTRU_E_PARAM, "r and m are required");
  return encrypt_dispatch(ctx, B, h_rows, r, m, 0, value, quotientE, remainderE);
}

int ntru_decrypt_dev(ntru_ctx *ctx, size_t B, const int8_t *f_rows, const uint8_t *fp_rows, const uint16_t *e,
                     uint8_t *value, uint16_t *quotient1, uint16_t *remainder1, uint8_t *quotient2,
                     uint8_t *remainder2) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!e) return fail(ctx, NTRU_E_PARAM, "e is required");
  return decrypt_dispatch(ctx, B, f_rows, fp_rows, e, value, quotient1, remainder1, quotient2, remainder2);
}

int ntru_sum_partial_dev(ntru_ctx *ctx, size_t B, const uint16_t *e, uint32_t *partial) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!e || !partial) return fail(ctx, NTRU_E_PARAM, "e and partial are required");
  return launch_sum_partial(ctx, B, e, partial);
}

int ntru_sum_finalize_dev(ntru_ctx *ctx, const uint32_t *partial, uint16_t *out) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!partial || !out) return fail(ctx, NTRU_E_PARAM, "partial and out are required");
  return launch_sum_finalize(ctx, partial, out);
}

static int xchg_release(ntru_ctx *ctx) {
  for (int r = 0; r < ntru_ctx::kMaxRanks; ++r) {
    if (ctx->peer_opened[r] && ctx->peer_window[r]) cudaIpcCloseMemHandle(ctx->peer_window[r]);
    ctx->peer_opened[r] = false;
    ctx->peer_window[r] = nullptr;
  }
  ctx->d_window.release();
  ctx->xchg_connected = false;
  ctx->xchg_world = 1;
  ctx->xchg_rank = 0;
  ctx->xchg_epoch = 0;
  return NTRU_OK;
}

static int xchg_alloc(ntru_ctx *ctx, int world, int rank) {
  xchg_release(ctx);
  const size_t bytes = xchg_window_bytes(ctx, world);
  NTRU_CUDA(ctx, ctx->d_window.reserve(bytes));
  NTRU_CUDA(ctx, cudaMemset(ctx->d_window.ptr, 0, bytes));
  ctx->xchg_world = world;
  ctx->xchg_rank = rank;
  ctx->peer_window[rank] = ctx->d_window.ptr;
  return NTRU_OK;
}

int ntru_xchg_create(ntru_ctx *ctx, int world, int rank, unsigned char handle_out[NTRU_XCHG_HANDLE_BYTES]) {
  int rc = check(ctx);
  if (rc) return rc;
  if (world < 1 || world > ntru_ctx::kMaxRanks || rank < 0 || rank >= world || !handle_out)
    return fail(ctx, NTRU_E_PARAM, "bad world / rank / handle buffer");
  static_assert(sizeof(cudaIpcMemHandle_t) == NTRU_XCHG_HANDLE_BYTES, "IPC handle size");
  rc = xchg_alloc(ctx, world, rank);
  if (rc) return rc;
  cudaIpcMemHandle_t h;
  NTRU_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->d_window.ptr));
  memcpy(handle_out, &h, sizeof h);
  ctx->xchg_connected = world == 1;
  return NTRU_OK;
}

int ntru_xchg_connect(ntru_ctx *ctx, const unsigned char *handles) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!handles) return fail(ctx, NTRU_E_PARAM, "handles is NULL");
  if (!ctx->d_window.ptr) return fail(ctx, NTRU_E_PARAM, "ntru_xchg_create has not been called");
  for (int r = 0; r < ctx->xchg_world; ++r) {
    if (r == ctx->xchg_rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * NTRU_XCHG_HANDLE_BYTES, sizeof h);
    void *p = nullptr;
    NTRU_CUDA(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->peer_window[r] = p;
    ctx->peer_opened[r] = true;
  }
  ctx->xchg_connected = true;
  return NTRU_OK;
}

int ntru_sum_allreduce_dev(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out) {
  int rc = check(ctx);
  if (rc) return rc;
  if ((B > 0 && !e) || !out) return fail(ctx, NTRU_E_PARAM, "e and out are required");
  if (!ctx->d_window.ptr) {                      // no exchange set up: a world of one rank
    rc = xchg_alloc(ctx, 1, 0);
    if (rc) return rc;
    ctx->xchg_connected = true;
  }
  if (!ctx->xchg_connected) return fail(ctx, NTRU_E_PARAM, "ntru_xchg_connect has not been called");
  return launch_sum_allreduce(ctx, B, e, out);
}

int ntru_sum_allreduce(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out) {
  int rc = check(ctx);
  if (rc) return rc;
  if ((B > 0 && !e) || !out) return fail(ctx, NTRU_E_PARAM, "e and out are required");
  if (!ctx->d_window.ptr) {                      // no exchange set up: a world of one rank
    rc = xchg_alloc(ctx, 1, 0);
    if (rc) return rc;
    ctx->xchg_connected = true;
  }
  if (!ctx->xchg_connected) return fail(ctx, NTRU_E_PARAM, "ntru_xchg_connect has not been called");
  // this rank's rows stream through the pipelined chunks into d_partial, then one small kernel runs the exchange
  NTRU_CUDA(ctx, cudaMemsetAsync(ctx->d_partial.ptr, 0, (size_t)ctx->P * 4, ctx->stream));
  if (B > 0) {
    HostArr arr[kMaxArr];
    set_in(arr[0], e, 2, (size_t)ctx->N);
    rc = run_pipeline(ctx, B, arr, [&](size_t rows, void **dev) {
      return launch_sum_partial(ctx, rows, (const uint16_t *)dev[0], (uint32_t *)ctx->d_partial.ptr);
    });
    if (rc) return rc;
  }
  NTRU_CUDA(ctx, ctx->slot_bufs[0][9].reserve((size_t)ctx->P * 2));
  rc = launch_xchg_partial(ctx, (uint32_t *)ctx->d_partial.ptr, (uint16_t *)ctx->slot_bufs[0][9].ptr);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaMemcpyAsync(out, ctx->slot_bufs[0][9].ptr, (size_t)ctx->N * 2, cudaMemcpyDeviceToHost, ctx->stream));
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return xchg_check(ctx);
}

int ntru_pack_output(ntru_ctx *ctx, size_t B, const void *data, int elem_bytes, int data_len, uint32_t max_val, void *out) {
  int rc = check(ctx);
  if (rc) return rc;
  int bits, n, arr, outs;
  if (ntru_pack_geometry(max_val, data_len, &bits, &n, &arr, &outs) != NTRU_OK || (elem_bytes != 1 && elem_bytes != 2))
    return fail(ctx, NTRU_E_PARAM, "bad maxVal / dataLen / element size");
  if (B == 0) return NTRU_OK;
  if (!data || !out) return fail(ctx, NTRU_E_PARAM, "data and out are required");
  const size_t in_bytes = B * (size_t)data_len * elem_bytes, out_bytes = B * (size_t)outs * 32;
  NTRU_CUDA(ctx, ctx->slot_packed[0][8].reserve(in_bytes));
  NTRU_CUDA(ctx, ctx->slot_packed[0][9].reserve(out_bytes));
  NTRU_CUDA(ctx, cudaMemcpyAsync(ctx->slot_packed[0][8].ptr, data, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
  rc = ntru_pack_output_dev(ctx, B, ctx->slot_packed[0][8].ptr, elem_bytes, data_len, (size_t)data_len, max_val, ctx->slot_packed[0][9].ptr);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaMemcpyAsync(out, ctx->slot_packed[0][9].ptr, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NTRU_OK;
}

int ntru_unpack_input(ntru_ctx *ctx, size_t B, const void *data, int n_elems, uint32_t max_val, int packed_bits, void *out,
                      int elem_bytes) {
  int rc = check(ctx);
  if (rc) return rc;
  if (max_val == 0 || n_elems < 0 || packed_bits < 1 || packed_bits > 256 || (elem_bytes != 1 && elem_bytes != 2))
    return fail(ctx, NTRU_E_PARAM, "bad maxVal / packedBits / element size");
  const int bits = bit_length(max_val);
  const int n = packed_bits / bits;
  if (n < 1) return fail(ctx, NTRU_E_PARAM, "packedBits is smaller than one coefficient");
  if (B == 0 || n_elems == 0) return NTRU_OK;
  if (!data || !out) return fail(ctx, NTRU_E_PARAM, "data and out are required");
  const size_t width = (size_t)n * n_elems;
  const size_t in_bytes = B * (size_t)n_elems * 32, out_bytes = B * width * elem_bytes;
  NTRU_CUDA(ctx, ctx->slot_packed[0][8].reserve(in_bytes));
  NTRU_CUDA(ctx, ctx->slot_packed[0][9].reserve(out_bytes));
  NTRU_CUDA(ctx, cudaMemcpyAsync(ctx->slot_packed[0][8].ptr, data, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
  rc = ntru_unpack_input_dev(ctx, B, ctx->slot_packed[0][8].ptr, n_elems, max_val, packed_bits, ctx->slot_packed[0][9].ptr, elem_bytes, width);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaMemcpyAsync(out, ctx->slot_packed[0][9].ptr, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return NTRU_OK;
}

int ntru_get_params(const ntru_ctx *ctx, int *N, int *p, int *q) {
  if (!ctx) return NTRU_E_PARAM;
  if (N) *N = ctx->N;
  if (p) *p = ctx->p;
  if (q) *q = ctx->q;
  return NTRU_OK;
}

int ntru_sample_r_dev(ntru_ctx *ctx, size_t B, int dr, uint64_t row0, uint8_t *r) {
  int rc = check(ctx);
  if (rc) return rc;
  if (!r) return fail(ctx, NTRU_E_PARAM, "r is NULL");
  // index.js:462-464
  if (dr < 0 || 2 * dr > ctx->N) return fail(ctx, NTRU_E_PARAM, "The total of 1s and -1s cannot exceed the array length.");
  if (!ctx->rng_keyed) return fail(ctx, NTRU_E_UNSUPPORTED, "the device generator has no key (no OS entropy; call ntru_set_rng_key)");
  return launch_sample(ctx, B, dr, dr, 2, row0, nullptr, r);
}

int ntru_set_rng_key(ntru_ctx *ctx, const uint8_t key[NTRU_RNG_KEY_BYTES], uint64_t first_row) {
  if (!ctx || !key) return NTRU_E_PARAM;
  for (int i = 0; i < 8; ++i)
    ctx->rng_key[i] = (uint32_t)key[4 * i] | ((uint32_t)key[4 * i + 1] << 8) | ((uint32_t)key[4 * i + 2] << 16) |
                      ((uint32_t)key[4 * i + 3] << 24);
  ctx->rng_row = first_row;
  ctx->rng_keyed = true;
  return NTRU_OK;
}

uint64_t ntru_rng_next_row(const ntru_ctx *ctx) { return ctx ? ctx->rng_row : 0; }

void *ntru_stream(ntru_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int ntru_set_stream(ntru_ctx *ctx, void *stream) {
  int rc = check(ctx);
  if (rc) return rc;
  cudaStream_t next = (cudaStream_t)stream;
  if (ctx->own_stream && ctx->stream) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamDestroy(ctx->stream);
  } else if (ctx->stream != next) {
    // calls queued on the caller's old stream may still use scratch the context owns (the lifted b, the sum tree's rows
    // and tickets, the key-generation buffers, the key matrices): the new stream waits for them
    cudaEvent_t ev = pool_get(ctx);
    if (!ev) return fail(ctx, NTRU_E_CUDA, "CUDA error: cudaEventCreate failed in ntru_set_stream");
    cudaError_t e = cudaEventRecord(ev, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(next, ev, 0);
    ctx->event_pool.push_back(ev);     // the wait holds on to the recorded work; the event can be recorded again
    if (e != cudaSuccess) return cuda_fail(ctx, e, "ordering the new stream after the old one (ntru_set_stream)");
  }
  ctx->stream = next;
  ctx->own_stream = false;
  return NTRU_OK;
}

// error word of this rank's exchange window: set by k_sum_push when a peer's flag never arrived
static int xchg_check(ntru_ctx *ctx) {
  if (!ctx->d_window.ptr) return NTRU_OK;
  uint32_t err = 0;
  const uint32_t *word = (const uint32_t *)ctx->d_window.ptr + (size_t)2 * ctx->xchg_world * ctx->P + ctx->xchg_world;
  NTRU_CUDA(ctx, cudaMemcpy(&err, word, sizeof err, cudaMemcpyDeviceToHost));
  if (err) return fail(ctx, NTRU_E_CUDA, "cross-GPU sum: a peer rank did not arrive within the timeout; the result is invalid");
  return NTRU_OK;
}

int ntru_sync(ntru_ctx *ctx) {
  int rc = check(ctx);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return xchg_check(ctx);
}

int ntru_xchg_destroy(ntru_ctx *ctx) {
  int rc = check(ctx);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  rc = xchg_check(ctx);
  xchg_release(ctx);
  return rc;
}

void *ntru_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
  return p;
}

void ntru_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"
