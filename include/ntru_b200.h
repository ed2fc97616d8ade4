/*
 * ntru_b200.h -- C ABI of the B200-native batched NTRU engine (libntru_b200.so).
 *
 * Drop-in boundary for the hot path of numtel/ntru-circom.  The reference has no
 * FFI of its own (it is one ES module, index.js); these entry points are what an
 * N-API / ctypes binding for that path binds.  Each one names the reference
 * interface it replaces (file:line relative to the reference repository).
 *
 * Conventions
 *   - Polynomials are little-endian coefficient arrays, FIXED LENGTH and
 *     un-trimmed: trimPolynomial / expandArray (index.js:218-221, 534-536) live in
 *     the host-language wrapper, never here.
 *   - mod-q coefficients are uint16_t, small coefficients (r, m, f, fp, mod-p
 *     outputs) are one byte.  r carries -1 as p-1 = 2 (index.js:89); f is the raw
 *     ternary key in {-1,0,1} (the witness value q-1 of index.js:112 is a wrapper
 *     concern); fp is in [0,p).
 *   - Host-buffer entry points take PACKED rows: pitch N for r, m, e, value and
 *     N+1 for the witness arrays, exactly the reference's array lengths
 *     (index.js:96-103, 123-131).  Any output pointer may be NULL (not produced).
 *   - Device-buffer entry points (*_dev) take device pointers whose row pitch is
 *     ntru_pitch(ctx) ELEMENTS for every array (a multiple of 16, >= N+1), run
 *     asynchronously on the context's stream and copy nothing.  Columns N..pitch-1
 *     of every INPUT row must be zero; every output row is written with zeros there
 *     (so an output row is the reference's expandArray(., N+1) witness field and can
 *     be fed back as an input).
 *   - Every function returns NTRU_OK (0) or a negative NTRU_E_* code;
 *     ntru_last_error(ctx) gives the message.  There is no CPU fallback: without
 *     a CUDA device every compute entry point fails with NTRU_E_CUDA.
 *   - A context is single-caller (one host thread at a time), one per GPU.
 *   - Ordering.  A context runs on one stream at a time: its own non-blocking stream from ntru_create, or
 *     the caller's after ntru_set_stream.  Key and option setters apply to the calls made after them;
 *     calls already queued keep the key and options they were queued with.  ntru_set_stream orders the
 *     new stream after the work queued on the old one.  Ordering the caller's own input and output
 *     buffers against ntru_stream(ctx) stays the caller's job.
 */
#ifndef NTRU_B200_H
#define NTRU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ntru_ctx ntru_ctx;

enum {
  NTRU_OK = 0,
  NTRU_E_PARAM = -1,       /* bad N/p/q/argument (reference: Error thrown by the constructor's users) */
  NTRU_E_LENGTH = -2,      /* reference: RangeError from expandArray, index.js:98,126 */
  NTRU_E_NOKEY = -3,       /* reference: TypeError on null h / f, index.js:90,112 */
  NTRU_E_CUDA = -4,
  NTRU_E_NCCL = -5,
  NTRU_E_NOMEM = -6,
  NTRU_E_UNSUPPORTED = -7
};

/* ntru_set_option keys */
enum {
  NTRU_OPT_PATH = 1,        /* 0 auto (same key: tcgen05 from 4096 rows up, IMMA below; distinct keys: IMMA), 1 force the fp32 CUDA-core
                               schedule, 2 force the tcgen05 schedule (same-key only), 3 force the register-fragment schedule */
  NTRU_OPT_CHUNK_ROWS = 2,  /* rows per pipelined chunk of the host-buffer entry points (default 32768) */
  NTRU_OPT_TIMING = 3,      /* 1: bracket every kernel launch with CUDA events on its stream (ntru_timing_read) */
  /* 4 was NTRU_OPT_TENSOR_VARIANT (a single-CTA tcgen05 kernel kept as a cross-check in round 1; removed) */
  NTRU_OPT_DR = 5,          /* dr of new NTRU({..., dr}) (index.js:15): weights of the r the device draws when r == NULL */
  NTRU_OPT_DEC1_FORM = 6,   /* tcgen05 schedule, first decrypt product at 256 < q <= 2048: 2 = fp16 tiles (a uint16 coefficient
                               below 2048 is its own fp16 encoding: no operand transform, sixteen epilogue warps), 1 = the
                               two-byte-limb int8 form used at every other q, 0 (default) = the faster one as measured on B200: fp16
                               (DEC1 at N = 677: 1.43 against 1.61 ms; at N = 509: 0.796 against 0.819 ms).  Both forms are exact;
                               each is the other's cross-check in the tests. */
  NTRU_OPT_SCHEDULE = 7,    /* tcgen05 schedule with the quotient witness: 0 (default) = the hi product of a chunk, then the lo
                               product accumulated on top of it in the same TMEM buffer (remainder = lo + hi: N^2 multiply-adds
                               plus the diagonal blocks); 1 = the full cyclic product and the hi product separately (1.5 N^2,
                               the round-1 order).  Same results bit for bit; each is the other's cross-check in the tests. */
  NTRU_OPT_EPILOGUE = 8,    /* tcgen05 schedule: 1 = two groups of epilogue warps, one per TMEM accumulator buffer; 2 = one group,
                               every warp drains every phase (the buffer goes back to the MMAs after half the time); 0 (default)
                               = one group where it measured faster (first and second decrypt product up to N = 512).  Same
                               results bit for bit. */
  NTRU_OPT_IMMA_FORM = 9    /* IMMA schedule (distinct keys, small batches): 0 (default) = the instantiation compiled for this N
                               where there is one (the BASELINE N: exact Toeplitz band, every offset a constant); 1 = always the
                               generic instantiation of the N bucket.  Same results bit for bit; each is the other's cross-check
                               in the tests. */
};

/* kernel kinds reported by ntru_timing_read */
enum {
  NTRU_K_ENC_TENSOR = 0,    /* tcgen05: lin(r,h) + m, fold, quotientE */
  NTRU_K_DEC1_TENSOR = 1,   /* tcgen05: lin(f,e), fold, quotient1, lift to b */
  NTRU_K_DEC2_TENSOR = 2,   /* tcgen05: lin(fp,b) mod 3, fold, quotient2 */
  NTRU_K_ENC_CORE = 3,      /* CUDA-core encrypt */
  NTRU_K_DEC_CORE = 4,      /* CUDA-core decrypt (both products) */
  NTRU_K_SUM = 5,           /* ciphertext column sum */
  NTRU_K_OTHER = 6,         /* sampler, finalize, key-matrix build */
  NTRU_K_ENC_IMMA = 7,      /* mma.sync (IMMA) encrypt, one warp per ciphertext: distinct keys */
  NTRU_K_DEC_IMMA = 8,      /* mma.sync (IMMA) decrypt (both products) */
  NTRU_K_MULDIV = 9,        /* mma.sync (IMMA) multiply + divide by 1 - x^N (verifyKeysInputs products) */
  NTRU_K_PACK = 10,         /* packOutput / unpackInput bit packing */
  NTRU_K_INVERSE = 11,      /* key generation: f^-1 modulo 2 and modulo 3 (divsteps) */
  NTRU_K_CHECK = 12,        /* mma.sync (IMMA) witness checks (ntru_check_*) */
  NTRU_K_COUNT = 13
};

/* new NTRU({N,p,q}) -- index.js:8-28.  p must be 3, q a power of two in [4, 8192], 8 <= N <= 1024
 * (q >= 16384 is refused with NTRU_E_PARAM: no schedule of this library is exact there). */
int ntru_create(ntru_ctx **ctx, int N, int p, int q, int device);
void ntru_destroy(ntru_ctx *ctx);
const char *ntru_last_error(const ntru_ctx *ctx);
const char *ntru_strerror(int code);
int ntru_set_option(ntru_ctx *ctx, int key, long value);
/* the N, p, q the context was created with (any pointer may be NULL) */
int ntru_get_params(const ntru_ctx *ctx, int *N, int *p, int *q);
/* device row pitch, in elements, of every *_dev array: roundup(N+1, 16) */
int ntru_pitch(const ntru_ctx *ctx);
/* number of CUDA kernels this context has launched so far */
uint64_t ntru_launch_count(const ntru_ctx *ctx);
/* which schedule the last batch call used: 1 CUDA-core (fp32 FMA), 2 tcgen05, 3 register-fragment IMMA */
int ntru_last_path(const ntru_ctx *ctx);
/* with NTRU_OPT_TIMING on: synchronises, then returns the summed device time (ms) and launch count of one
 * kernel kind since the last ntru_timing_reset */
int ntru_timing_read(ntru_ctx *ctx, int kind, double *total_ms, uint64_t *launches);
int ntru_timing_reset(ntru_ctx *ctx);

/* this.h = ... (index.js:72-79 result, expanded to N entries in [0,q)).  The key is copied on the context's stream,
 * after the calls queued there, and the stream is synchronised before the function returns (queued calls finish under
 * the key they were queued with; the same holds for ntru_set_private_key). */
int ntru_set_public_key(ntru_ctx *ctx, const uint16_t *h);
/* this.f, this.fp (index.js:30-36): f in {-1,0,1}, fp expanded to N entries in [0,p) */
int ntru_set_private_key(ntru_ctx *ctx, const int8_t *f, const uint8_t *fp);

/* encryptBits, B messages under the context's public key -- index.js:87-110.
 * value = remainderE[0..N); quotientE/remainderE are the VerifyEncrypt witness (N+1 entries per row).
 * r (B x N, entries 0/1/2 with 2 = -1): the blinding polynomials, injected by the caller -- or NULL: the DEVICE draws
 *   them like index.js:89 (generateCustomArray(N, dr, dr), -1 -> p-1) from its keyed ChaCha20 generator; needs
 *   NTRU_OPT_DR.  r_out (B x N or NULL) receives the r that was used (inputs.r, index.js:97) in either case. */
int ntru_encrypt_batch(ntru_ctx *ctx, size_t B, const uint8_t *r, const uint8_t *m,
                       uint16_t *value, uint16_t *quotientE, uint16_t *remainderE, uint8_t *r_out);
/* same with messages whose coefficients do not fit a byte (m already reduced into [0,q)) -- index.js:91 */
int ntru_encrypt_batch_wide(ntru_ctx *ctx, size_t B, const uint8_t *r, const uint16_t *m,
                            uint16_t *value, uint16_t *quotientE, uint16_t *remainderE, uint8_t *r_out);
/* encryptBits with a distinct public key per row: h is B x N */
int ntru_encrypt_batch_keys(ntru_ctx *ctx, size_t B, const uint16_t *h, const uint8_t *r, const uint8_t *m,
                            uint16_t *value, uint16_t *quotientE, uint16_t *remainderE, uint8_t *r_out);

/* The device generator behind r == NULL and ntru_sample_r_dev: ChaCha20 in counter mode (256-bit key, nonce = a
 * 64-bit global row number that the context never reuses under one key, block counter = position in the row's
 * keystream); the draws replace crypto.getRandomValues in the reference's Fisher-Yates shuffle (index.js:476-485)
 * one for one.  ntru_create keys it with 256 bits from the operating system (getrandom(2)).  ntru_set_rng_key
 * replaces the key and sets the next row number: for tests, reproducible benchmarks, or an audit replay of the r of
 * given rows by the key holder.  ntru_rng_next_row: the row number the next device-drawn r will use. */
#define NTRU_RNG_KEY_BYTES 32
int ntru_set_rng_key(ntru_ctx *ctx, const uint8_t key[NTRU_RNG_KEY_BYTES], uint64_t first_row);
uint64_t ntru_rng_next_row(const ntru_ctx *ctx);

/* decryptBits, B ciphertexts under the context's private key -- index.js:111-140.
 * value = remainder2[0..N); quotient1/remainder1 (mod q) and quotient2/remainder2 (mod p) are the
 * VerifyDecrypt witness (N+1 entries per row). */
int ntru_decrypt_batch(ntru_ctx *ctx, size_t B, const uint16_t *e, uint8_t *value,
                       uint16_t *quotient1, uint16_t *remainder1, uint8_t *quotient2, uint8_t *remainder2);
/* decryptBits with a distinct private key per row: f, fp are B x N */
int ntru_decrypt_batch_keys(ntru_ctx *ctx, size_t B, const int8_t *f, const uint8_t *fp, const uint16_t *e,
                            uint8_t *value, uint16_t *quotient1, uint16_t *remainder1,
                            uint8_t *quotient2, uint8_t *remainder2);

/* verifyKeysInputs, B keys at once -- index.js:141-197: the three multiplyPolynomials + dividePolynomials(., I, .)
 * pairs behind the VerifyInverse witness (circuits/ntru.circom:242-256):
 *   fq case: (fq * f) / I mod q      fp case: (fp * f) / I mod p      h case: ((p fq) * g) / I mod q
 * f, g: B x N ternary in {-1,0,1}; fq: B x N in [0,q); fp: B x N in [0,p).  Outputs are N+1 entries per row
 * (quotientI / remainderI of each case); any output may be NULL.  The echoed inputs of the witness (f with -1 as
 * q-1 or p-1, fq, fp, p*fq un-reduced) and the reference's validity checks are the wrapper's concern. */
int ntru_verify_keys_batch(ntru_ctx *ctx, size_t B, const int8_t *f, const uint16_t *fq, const uint8_t *fp, const int8_t *g,
                           uint16_t *quotient_fq, uint16_t *remainder_fq, uint8_t *quotient_fp, uint8_t *remainder_fp,
                           uint16_t *quotient_h, uint16_t *remainder_h);
/* the primitive, device-resident: multiplyPolynomials(x, y, mod) then dividePolynomials(., 1 - x^N, mod) for B
 * independent pairs.  x: int8 in [-1, 2]; mod_p == 0: y uint16 (any value), outputs uint16 mod q;
 * mod_p != 0: y bytes in [0, p), outputs bytes mod p.  Pitch ntru_pitch() elements everywhere. */
int ntru_muldiv_dev(ntru_ctx *ctx, size_t B, const int8_t *x, const void *y, int mod_p, void *quotient, void *remainder);

/* loadPrivateKeyF + generatePublicKeyH for B keys at once -- index.js:30-79, 491-514.  f, g: B x N ternary (the
 * generateCustomArray draws stay with the caller's CSPRNG).  fp = f^-1 mod (p, x^N-1), fq = f^-1 mod (q, x^N-1),
 * h = (p fq) * g mod (q, x^N-1); rows of N entries, un-trimmed.  Everything runs on the GPU: the inversions modulo 2
 * and modulo p (the reference's extended Euclid, index.js:425-459) as constant-time divsteps, one warp per key, then
 * the Newton lifting 2 -> q (index.js:497-509) and h.  Synchronous (host buffers in and out).
 * valid[b] = 1 iff f_b and g_b are in {-1,0,1} and f_b is invertible modulo 2 and modulo p -- then the outputs equal
 * the reference's (the inverse is unique); otherwise the row's outputs are zero and the caller redraws f as
 * generatePrivateKeyF does. */
int ntru_keygen_batch(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h,
                      uint8_t *valid);

/* Witness checks -- the constraint systems of VerifyEncrypt, VerifyDecrypt and VerifyInverse
 * (circuits/ntru.circom:155-256) evaluated for B witnesses at once.  One verdict byte per row:
 *   NTRU_CHECK_SATISFIED  the constraints hold (for decrypt: both divisions), computed on the raw witness values;
 *   NTRU_CHECK_CANONICAL  satisfied, every quotient / remainder entry below its modulus and remainder[N] == 0: the arrays
 *                         are exactly what dividePolynomials returns (expanded to N + 1), i.e. what this library and the
 *                         reference emit.  The constraints alone accept more: adding t to quotient[0] and remainder[N]
 *                         and subtracting it from remainder[0], or raising any entry by a multiple of the modulus;
 *   NTRU_CHECK_DOMAIN     not evaluated (bits 1 and 2 clear): an entry of the small operand (r, f, or the x of
 *                         VerifyInverse), reduced modulo the product's modulus M, is outside {M-1, 0, 1, 2}.
 * Witness forms as the reference's `inputs`: r bytes; f, m, e, h, fq, the inverse's x and y uint16 (-1 as q-1 or p-1;
 * y = fq or the un-reduced p*fq), except y, quotientI and remainderI as bytes when mod_p != 0 (the fp case); quotient2,
 * remainder2 bytes.  h, e, m are taken modulo q and fp modulo 3 at any value; the lift of decrypt reads the raw
 * remainder1.  Columns >= N of the inputs and >= N + 1 of the witness arrays are ignored.  Supports N <= 832
 * (NTRU_E_UNSUPPORTED above).  Every array is required when B > 0 (NTRU_E_PARAM); bad values are not an error, they
 * are what the verdict reports.
 * Device form: rows of pitch ntru_pitch(ctx) elements; key_stride = 0 (one key row for every witness) or ntru_pitch(ctx)
 * (NTRU_E_PARAM otherwise); verdict: B device bytes, exactly B written; asynchronous on the context's stream. */
enum { NTRU_CHECK_SATISFIED = 1, NTRU_CHECK_CANONICAL = 2, NTRU_CHECK_DOMAIN = 4 };
int ntru_check_encrypt_dev(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t key_stride, const uint8_t *r,
                           const uint16_t *m, const uint16_t *quotientE, const uint16_t *remainderE, uint8_t *verdict);
int ntru_check_decrypt_dev(ntru_ctx *ctx, size_t B, const uint16_t *f, const uint8_t *fp, size_t key_stride,
                           const uint16_t *e, const uint16_t *quotient1, const uint16_t *remainder1,
                           const uint8_t *quotient2, const uint8_t *remainder2, uint8_t *verdict);
int ntru_check_inverse_dev(ntru_ctx *ctx, size_t B, int mod_p, const uint16_t *x, const void *y,
                           const void *quotientI, const void *remainderI, uint8_t *verdict);
/* Host form: packed rows (pitch N for the inputs, N + 1 for quotient / remainder), verdict B host bytes; key_shared != 0:
 * h (or f and fp) is one row of N entries for every witness.  Synchronous. */
int ntru_check_encrypt_batch(ntru_ctx *ctx, size_t B, const uint16_t *h, int key_shared, const uint8_t *r, const uint16_t *m,
                             const uint16_t *quotientE, const uint16_t *remainderE, uint8_t *verdict);
int ntru_check_decrypt_batch(ntru_ctx *ctx, size_t B, const uint16_t *f, const uint8_t *fp, int key_shared, const uint16_t *e,
                             const uint16_t *quotient1, const uint16_t *remainder1, const uint8_t *quotient2,
                             const uint8_t *remainder2, uint8_t *verdict);
int ntru_check_inverse_batch(ntru_ctx *ctx, size_t B, int mod_p, const uint16_t *x, const void *y,
                             const void *quotientI, const void *remainderI, uint8_t *verdict);

/* packOutput / unpackInput -- index.js:572-620: coefficients <-> BN254 field elements (CombineArray / UnpackArray,
 * circuits/ntru.circom:259-306).  A field element is 32 bytes, little-endian.
 * ntru_pack_geometry is packOutput's header: maxInputBits = floor(log2(maxVal) + 1), n = floor(252 / maxInputBits),
 * arrLen = max(ceil(dataLen / n) n, 3 n), outputSize = max(ceil(arrLen / n), 3). */
int ntru_pack_geometry(uint32_t max_val, int data_len, int *max_input_bits, int *inputs_per_output, int *arr_len,
                       int *output_size);
/* data: B rows of data_len coefficients (elem_bytes 1 or 2, row pitch `pitch` elements), every value < 2^maxInputBits;
 * out: B x outputSize x 32 bytes.  Device pointers, asynchronous on the context's stream. */
int ntru_pack_output_dev(ntru_ctx *ctx, size_t B, const void *data, int elem_bytes, int data_len, size_t pitch,
                         uint32_t max_val, void *out);
/* data: B x n_elems field elements; out: B rows of floor(packed_bits / maxInputBits) * n_elems coefficients
 * (un-trimmed), row pitch `pitch` elements */
int ntru_unpack_input_dev(ntru_ctx *ctx, size_t B, const void *data, int n_elems, uint32_t max_val, int packed_bits,
                          void *out, int elem_bytes, size_t pitch);

/* host-buffer forms of the two calls above (packed rows in, packed field elements / rows out; synchronous) */
int ntru_pack_output(ntru_ctx *ctx, size_t B, const void *data, int elem_bytes, int data_len, uint32_t max_val, void *out);
int ntru_unpack_input(ntru_ctx *ctx, size_t B, const void *data, int n_elems, uint32_t max_val, int packed_bits, void *out,
                      int elem_bytes);

/* encryptBits / decryptBits with every array crossing the host link as BN254 field elements, the form the circuits'
 * CombineArray / UnpackArray take (circuits/ntru.circom:259-306): row b of an array of `width` coefficients is
 * packOutput(maxVal, width, row).expected (index.js:572-596) -- ntru_packed_elems(ctx, mod_q, width) elements of 32
 * bytes, little-endian -- with maxVal = q - 1 for the arrays modulo q (value / e, quotientE, remainderE, quotient1,
 * remainder1) and maxVal = p - 1 for the small ones (r with 2 = -1, m, decrypt's value, quotient2, remainder2).
 * Widths as in the calls above (N, or N + 1 for the witness arrays).  Inputs must hold zeros beyond `width` (packOutput
 * pads with zeros).  The bits are packed / unpacked on the device: at N = 509, q = 2048 a ciphertext with its full
 * witness crosses the link in 3392 bytes device -> host instead of 5097, 1088 instead of 2036 host -> device.
 * r == NULL, r_out, NULL outputs: as in ntru_encrypt_batch / ntru_decrypt_batch. */
int ntru_packed_elems(const ntru_ctx *ctx, int mod_q, int width);
int ntru_encrypt_batch_packed(ntru_ctx *ctx, size_t B, const void *r, const void *m, void *value, void *quotientE,
                              void *remainderE, void *r_out);
int ntru_decrypt_batch_packed(ntru_ctx *ctx, size_t B, const void *e, void *value, void *quotient1, void *remainder1,
                              void *quotient2, void *remainder2);

/* fold of addPolynomials(.,.,q) over B ciphertexts -- index.js:235-244, test/reference.test.js:58.  out: N entries */
int ntru_sum(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out);
/* the same fold over the rows of EVERY rank of the exchange (ntru_xchg_create / ntru_xchg_connect below; one rank
 * without them): this rank's B packed host rows, the total on every rank.  Every rank must call it the same number
 * of times (B may be 0). */
int ntru_sum_allreduce(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out);

/* ---- device-resident variants (pitch = ntru_pitch(ctx) elements; async on ntru_stream(ctx)) ---- */
/* h_rows == NULL: context key (same-key schedule); else one key per row */
int ntru_encrypt_dev(ntru_ctx *ctx, size_t B, const uint16_t *h_rows, const uint8_t *r, const uint8_t *m,
                     uint16_t *value, uint16_t *quotientE, uint16_t *remainderE);
int ntru_decrypt_dev(ntru_ctx *ctx, size_t B, const int8_t *f_rows, const uint8_t *fp_rows, const uint16_t *e,
                     uint8_t *value, uint16_t *quotient1, uint16_t *remainder1,
                     uint8_t *quotient2, uint8_t *remainder2);
/* adds the column sums of this call's rows into partial (pitch entries): afterwards each partial[k] is congruent to its
 * old value plus sum_b e[b][k] modulo 2^16, so modulo q.  It is not the uint32 sum: only its value modulo q is defined. */
int ntru_sum_partial_dev(ntru_ctx *ctx, size_t B, const uint16_t *e, uint32_t *partial);
/* out[k] = partial[k] mod q for k < N (and 0 up to pitch) */
int ntru_sum_finalize_dev(ntru_ctx *ctx, const uint32_t *partial, uint16_t *out);
/* generateCustomArray(N, dr, dr).map(-1 -> p-1) into device rows, drawn by the context's ChaCha20 generator for the
 * global row numbers [row0, row0+B) -- index.js:89, 461-488.  The caller owns the row numbering here: never sample
 * two different rows with the same number under one key. */
int ntru_sample_r_dev(ntru_ctx *ctx, size_t B, int dr, uint64_t row0, uint8_t *r);
/* ntru_keygen_batch on device rows (pitch ntru_pitch(ctx)), asynchronous on the context's stream; valid: B device bytes.
 * f, g are int8 (-1 as 0xFF); fq, h uint16; fp bytes in [0,p). */
int ntru_keygen_dev(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g,
                    uint16_t *fq, uint8_t *fp, uint16_t *h, uint8_t *valid);
/* generatePrivateKeyF + generateNewPublicKeyGH for B keys, entirely on the device (index.js:51-79): f drawn with
 * weights (df, df - 1), g with (dg, dg) (generateCustomArray, index.js:461-488) by the context's ChaCha20 generator;
 * every f that is not invertible modulo 2 and p is redrawn on the device, for at most 100 rounds in all
 * (index.js:52-64; then NTRU_E_PARAM "Could not find invertible f").  Every returned row is a valid key pair.
 * The context owns the row numbers: with R = ntru_rng_next_row at entry, f of key b comes from row R + b and g from
 * R + B + b; redraw round k >= 1 takes f of key b from row R + (k+1) B + b, and on return the next row is
 * R + (last round + 2) B.  Each round ends with a 4-byte copy to the host and a stream synchronisation (the count of
 * rows still to redraw); the lifting and h run once after the last round, asynchronously. */
int ntru_generate_keys_dev(ntru_ctx *ctx, size_t B, int df, int dg,
                           int8_t *f, int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h);

/* ---- cross-GPU homomorphic sum (one context = one rank = one GPU of the same node) ----
 * The only exchange step of the hot path: every rank reduces its rows to N column sums mod q and all ranks need the
 * total (fold of addPolynomials over the whole batch, test/reference.test.js:58).  The exchange runs inside the
 * library's own kernels over peer memory (NVLink / NVSwitch): the CTA that finishes a rank's column sums stores them
 * straight into every peer's exchange window and raises a flag there; a one-CTA kernel waits for all flags and adds
 * the slots.  No collective library on the data path. */
#define NTRU_XCHG_HANDLE_BYTES 64
/* allocates this rank's exchange window and returns its CUDA IPC handle (to be all-gathered by the caller).
 * Calling it again replaces the window: see ntru_xchg_destroy for the barrier this requires. */
int ntru_xchg_create(ntru_ctx *ctx, int world, int rank, unsigned char handle_out[NTRU_XCHG_HANDLE_BYTES]);
/* handles: world x NTRU_XCHG_HANDLE_BYTES, rank-major, as gathered from ntru_xchg_create on every rank */
int ntru_xchg_connect(ntru_ctx *ctx, const unsigned char *handles);
/* out[k] = (sum over every rank's rows of e[b][k]) mod q for k < N (0 up to pitch), on every rank; asynchronous on
 * the context's stream.  Every rank must call it the same number of times (B may differ per rank and may be 0).
 * Without ntru_xchg_create: world = 1.  If a peer does not arrive within ~4 s the kernel gives up, fills out[] with
 * 0xFFFF (no valid residue) and the next ntru_sync / ntru_xchg_destroy on this context returns NTRU_E_CUDA. */
int ntru_sum_allreduce_dev(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out);
/* Unmaps the peers' windows and frees this rank's.  COLLECTIVE like create / connect: every rank must have finished
 * (ntru_sync) its last ntru_sum_allreduce_dev and the caller must pass a barrier over all ranks BEFORE any rank calls
 * this or ntru_xchg_create again -- peers store into this window until their last call has completed.
 * (ntru_destroy implies it, under the same rule.) */
int ntru_xchg_destroy(ntru_ctx *ctx);

void *ntru_stream(ntru_ctx *ctx);              /* cudaStream_t */
/* The context runs its calls on `stream` from now on (0 = the legacy default stream).  The context's own stream is
 * synchronised and destroyed; a previous caller stream is not waited for on the host, but the new stream waits for
 * the work queued on it (that work may still use the context's scratch). */
int ntru_set_stream(ntru_ctx *ctx, void *stream);
int ntru_sync(ntru_ctx *ctx);

/* pinned host memory for the host-buffer entry points (pageable memory works, but copies then serialise) */
void *ntru_host_alloc(size_t bytes);
void ntru_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* NTRU_B200_H */
