// Internal declarations shared by the translation units of libntru_b200.so.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/ntru_b200.h"

namespace ntru {

constexpr int kMaxN = 1024;
constexpr int kNumSlots = 2;   // double-buffered host<->device pipeline

// One device allocation that only ever grows.
struct DevBuf {
  void *ptr = nullptr;
  size_t bytes = 0;
  cudaError_t reserve(size_t need) {
    if (need <= bytes) return cudaSuccess;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    bytes = 0;
    cudaError_t e = cudaMalloc(&ptr, need);
    if (e == cudaSuccess) bytes = need;
    return e;
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    bytes = 0;
  }
};

constexpr int kMaxChunks = 8;   // accumulator chunks per product and part (ENC at N = 1024: 8 chunks of 128 outputs)

// Operand matrices of the tcgen05 schedule for one fixed key polynomial (see umma_kernels.cu).
struct KeyMatrix {
  DevBuf mat;            // [3 parts (cyc, hi, lo) * nlimbs * covered columns][klen] bytes, K-major, tile-major per 128-byte K block
  alignas(64) unsigned char tmap_half[2][128];   // CUtensorMaps, box = half the B rows of a chunk of width w[i]
  bool ready = false;
  bool f16 = false;      // DEC1F: 16-bit operands (the first decrypt product on kind::f16 tiles)
  int limbs = 0, nlimbs = 0, klen = 0, nchunks = 0;
  int col0[kMaxChunks + 1] = {};   // chunk c computes output columns [col0[c], col0[c+1])
  int w[2] = {0, 0};               // the (at most two) distinct chunk widths: first chunk's, last chunk's
};

}  // namespace ntru

struct ntru_ctx {
  int N = 0, p = 0, q = 0, logq = 0, device = 0;
  int P = 0;                       // row pitch (elements) of every device array
  cudaStream_t stream = nullptr;   // compute stream
  bool own_stream = false;
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[ntru::kNumSlots] = {}, ev_comp[ntru::kNumSlots] = {}, ev_out[ntru::kNumSlots] = {};
  bool has_pub = false, has_priv = false;
  ntru::DevBuf d_h, d_f, d_fp;     // context keys, P entries each
  ntru::KeyMatrix km_h, km_f, km_fp;
  ntru::DevBuf d_b;                // lifted polynomial b between the two decrypt products (tensor schedule)
  ntru::DevBuf slot_bufs[ntru::kNumSlots][10];     // pitched device arrays of the host pipeline
  ntru::DevBuf slot_packed[ntru::kNumSlots][10];   // packed staging (what the 1-D H2D / D2H copies move)
  ntru::DevBuf d_partial;
  ntru::DevBuf kg_bufs[12];         // key generation: lifting scratch (t, u0, u1, r0, r1), host-form rows, valid, count;
                                    // kg_bufs[0] also holds y = p fq of launch_h_product (ntru_verify_keys_batch too)
  ntru::DevBuf check_key[2];       // witness checks, host form: the shared key row (h, or f and fp)
  ntru::DevBuf d_sum_scratch;      // tree scratch of the ciphertext sum (per-CTA rows, per-group rows, tickets)
  // cross-GPU sum: exchange window (this rank's, cudaMalloc + IPC) and the mapped windows of the peers
  static constexpr int kMaxRanks = 16;
  int xchg_world = 1, xchg_rank = 0;
  bool xchg_connected = false;
  ntru::DevBuf d_window;           // [2 parities][world][P] uint32 slots, then [world] uint32 flags, then the error word
  void *peer_window[kMaxRanks] = {};
  bool peer_opened[kMaxRanks] = {};
  uint32_t xchg_epoch = 0;
  size_t chunk_rows = 32768;
  int opt_path = 0;
  int opt_imma_form = 0;           // NTRU_OPT_IMMA_FORM: 0 auto (compile-time N where instantiated), 1 the bucket's generic kernel
  int opt_epilogue = 0;            // NTRU_OPT_EPILOGUE: 0 auto, 1 two epilogue groups (one per TMEM buffer), 2 one group
  int opt_lohi = 0;                // NTRU_OPT_SCHEDULE: 0 = lo + hi phases (default), 1 = the cyc + hi order of round 1
  int opt_dec1_form = 0;           // NTRU_OPT_DEC1_FORM: 0 auto, 1 byte limbs, 2 fp16 tiles (256 < q <= 2048 only)
  int umma_attr_set = 0;           // bit per kernel mode: dynamic shared memory attribute applied on this device
  bool sampler_attr_set = false;
  // device CSPRNG for r (ChaCha20, generic_kernels.cu): key words (little-endian), next unused row number (= nonce),
  // dr of the reference's constructor options (NTRU_OPT_DR; needed when the device draws r)
  uint32_t rng_key[8] = {};
  bool rng_keyed = false;
  uint64_t rng_row = 0;
  int opt_dr = -1;
  struct ImmaCfg { const void *fn; size_t smem; int per_sm; };
  std::vector<ImmaCfg> imma_cfg;   // launch configuration of the IMMA kernels already prepared on this context's device
  // CUtensorMaps already encoded on this context, keyed by everything cuTensorMapEncodeTiled reads: a steady-state
  // caller (same device buffers, same batch size) pays no driver call per launch
  struct TmapKey {
    const void *base; uint64_t inner, rows, stride; uint32_t box_inner, box_rows; int elem, swz;
    bool operator==(const TmapKey &o) const {
      return base == o.base && inner == o.inner && rows == o.rows && stride == o.stride && box_inner == o.box_inner &&
             box_rows == o.box_rows && elem == o.elem && swz == o.swz;
    }
  };
  struct TmapEntry { TmapKey key; alignas(64) unsigned char map[128]; };
  std::vector<TmapEntry> tmap_cache;
  size_t tmap_next = 0;            // round-robin replacement once the cache holds kTmapCacheMax entries
  static constexpr size_t kTmapCacheMax = 64;
  int last_path = 0;
  int sm_count = 148;
  bool tensor_ok = false;          // device is sm_100 and the tcgen05 schedule initialised
  uint64_t launches = 0;
  std::string err;
  // optional per-launch timing (NTRU_OPT_TIMING)
  bool timing = false;
  struct TimedLaunch { int kind; cudaEvent_t a, b; };
  std::vector<TimedLaunch> timed;
  std::vector<cudaEvent_t> event_pool;
};

namespace ntru {

int fail(ntru_ctx *ctx, int code, const std::string &msg);
int cuda_fail(ntru_ctx *ctx, cudaError_t e, const char *what);

// Brackets one kernel launch with events on ctx->stream when timing is enabled.
struct LaunchTimer {
  ntru_ctx *ctx;
  cudaEvent_t a = nullptr, b = nullptr;
  int kind;
  LaunchTimer(ntru_ctx *c, int k);
  ~LaunchTimer();
};

#define NTRU_CUDA(ctx, expr)                                        \
  do {                                                              \
    cudaError_t _e = (expr);                                        \
    if (_e != cudaSuccess) return ntru::cuda_fail(ctx, _e, #expr);  \
  } while (0)

// ---- CUDA-core schedule (generic_kernels.cu) ----
int launch_encrypt_generic(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t h_stride, const uint8_t *r,
                           const void *m, int m_wide, uint16_t *value, uint16_t *quo, uint16_t *rem);
int launch_decrypt_generic(ntru_ctx *ctx, size_t B, const int8_t *f, const uint8_t *fp, size_t key_stride,
                           const uint16_t *e, uint8_t *value, uint16_t *q1, uint16_t *r1, uint8_t *q2,
                           uint8_t *r2);
int launch_sum_partial(ntru_ctx *ctx, size_t B, const uint16_t *e, uint32_t *partial);
int launch_sum_finalize(ntru_ctx *ctx, const uint32_t *partial, uint16_t *out);
size_t xchg_window_bytes(const ntru_ctx *ctx, int world);
int launch_sum_allreduce(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out);
int launch_xchg_partial(ntru_ctx *ctx, uint32_t *partial, uint16_t *out);   // exchange of already accumulated column sums
// generateCustomArray(N, ones, neg_ones) with -1 stored as neg_code, rows [row0, row0 + B) of the ChaCha20 generator;
// rows with skip[b] != 0 (skip may be NULL) are left untouched
int launch_sample(ntru_ctx *ctx, size_t B, int ones, int neg_ones, uint8_t neg_code, uint64_t row0, const uint8_t *skip,
                  uint8_t *r);
int launch_wire_unpack(ntru_ctx *ctx, size_t B, const uint32_t *data, int in_elems, int bits, int n, int width, void *out,
                       int elem_bytes);
int launch_pack_fields(ntru_ctx *ctx, size_t B, const void *data, int elem_bytes, int data_len, size_t pitch, int bits, int n,
                       int out_elems, uint32_t *out);
int launch_unpack_fields(ntru_ctx *ctx, size_t B, const uint32_t *data, int in_elems, int bits, int n, size_t pitch, void *out,
                         int elem_bytes);
int launch_repitch(ntru_ctx *ctx, const void *src, void *dst, size_t rows, int width, int elem, bool to_pitched);

// ---- register-fragment tensor schedule (imma_kernels.cu): one warp per ciphertext, distinct keys ----
bool imma_supported(const ntru_ctx *ctx);
int launch_encrypt_imma(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t h_stride, const uint8_t *r, const uint8_t *m,
                        uint16_t *value, uint16_t *quo, uint16_t *rem);
int launch_decrypt_imma(ntru_ctx *ctx, size_t B, const int8_t *f, const uint8_t *fp, size_t key_stride, const uint16_t *e,
                        uint8_t *value, uint16_t *q1, uint16_t *r1, uint8_t *q2, uint8_t *r2);

int launch_muldiv_imma(ntru_ctx *ctx, size_t B, const int8_t *x, const void *y, int mod_p, void *quo, void *rem);

// witness checks (VerifyEncrypt / VerifyDecrypt / VerifyInverse) on the same product, one verdict byte per row
int launch_check_encrypt(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t h_stride, const uint8_t *r, const uint16_t *m,
                         const uint16_t *quo, const uint16_t *rem, uint8_t *verdict);
int launch_check_decrypt(ntru_ctx *ctx, size_t B, const uint16_t *f, const uint8_t *fp, size_t key_stride, const uint16_t *e,
                         const uint16_t *q1, const uint16_t *r1, const uint8_t *q2, const uint8_t *r2, uint8_t *verdict);
int launch_check_inverse(ntru_ctx *ctx, size_t B, int mod_p, const uint16_t *x, const void *y, const void *quo, const void *rem,
                         uint8_t *verdict);

// ---- batched key generation (keygen.cu): divstep inversions modulo 2 and 3, IMMA lifting to q and h ----
constexpr int kKeygenRounds = 100;   // draws of f per key before giving up (index.js:52-64)
int keygen_dev(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h,
               uint8_t *valid);
int keygen_batch(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h,
                 uint8_t *valid);
int generate_keys_dev(ntru_ctx *ctx, size_t B, int df, int dg, int8_t *f, int8_t *g, uint16_t *fq, uint8_t *fp,
                      uint16_t *h);
// h = (p fq) * g mod (q, x^N - 1) for B rows on the IMMA schedule: quotient and remainder (h) of the division by
// 1 - x^N, either may be NULL
int launch_h_product(ntru_ctx *ctx, size_t B, const int8_t *g, const uint16_t *fq, uint16_t *quo, uint16_t *rem);

// ---- tcgen05 schedule (umma_kernels.cu) ----
int umma_init(ntru_ctx *ctx);                    // probes the device, sets ctx->tensor_ok
int umma_prepare_public(ntru_ctx *ctx);          // builds km_h from d_h
int umma_prepare_private(ntru_ctx *ctx);         // builds km_f, km_fp from d_f, d_fp
int umma_encrypt(ntru_ctx *ctx, size_t B, const uint8_t *r, const uint8_t *m, uint16_t *value, uint16_t *quo,
                 uint16_t *rem);
int umma_decrypt(ntru_ctx *ctx, size_t B, const uint16_t *e, uint8_t *value, uint16_t *q1, uint16_t *r1,
                 uint8_t *q2, uint8_t *r2);

}  // namespace ntru
