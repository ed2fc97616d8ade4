// Batched key generation (SURVEY.md section 8f-3): loadPrivateKeyF + generatePublicKeyH (index.js:30-79) for B keys,
// and generatePrivateKeyF + generateNewPublicKeyGH (index.js:51-79) with f and g drawn on the device.
//
//   fp = f^-1 mod (p, x^N - 1)        polyInv(f, I, p): extended Euclid over GF(3)              (index.js:510-513)
//   fq = f^-1 mod (q, x^N - 1)        polyInv(f, I, q): extended Euclid over GF(2), then the Newton / Hensel lifting
//                                     inverse <- 2 inverse - f inverse^2 (mod q, x^N - 1)        (index.js:494-509)
//   h  = (p fq) * g mod (q, x^N - 1)                                                             (index.js:72-79)
//
// The inverse of f in Z_m[x]/(x^N - 1) is unique, so any correct algorithm returns the reference's coefficients
// (the reference trims; rows here are fixed length).  Everything runs on the GPU, device-resident (keygen_dev):
//   1. k_inverse_2_3: both inversions of a key in one warp, Bernstein-Yang divsteps (constant time, below);
//   2. the lifting 2 -> q and h, polynomial products through the multiply + divide kernel of imma_kernels.cu.  One
//      lifting step, written for that kernel (small operand int8, wide operand uint16):
//          t = f * inv                      (f ternary)                    u = (2 - t) mod q = u0 + 128 u1  (u0 < 128, u1 < 64)
//          inv <- inv * u = inv * u0 + 128 (inv * u1)     (mod q, x^N - 1)
//      which is the same map inv -> inv (2 - f inv) = 2 inv - f inv^2; precision doubles per step, so ceil(log2 log2 q)
//      steps reach q (the reference runs log2 q - 1 steps of the same map: same fixed point);
//   3. k_zero_invalid: rows whose f is not invertible modulo 2 or modulo p, or whose f or g is not ternary, are flagged
//      in valid[] and their outputs zeroed (the reference's own checks are vacuous there, SURVEY appendix A: it would
//      hand back garbage; callers redraw f like generatePrivateKeyF does, generate_keys_dev does it on the device).
// keygen_batch is the host-buffer form: copy in, keygen_dev, copy out.

#include <cuda_runtime.h>
#include <stdint.h>

#include "ntru_internal.cuh"

namespace ntru {

namespace {

// ---- device: f^-1 modulo (2, x^N - 1) and modulo (3, x^N - 1), Bernstein-Yang divsteps ----------------------------
// The inverse of a in GF(p)[x]/(x^N - 1), p in {2, 3} (D. J. Bernstein, B.-Y. Yang, "Fast constant-time gcd computation
// and modular inversion", 2019), on reversed polynomials:
//   F = 1 - x^N, G = reverse_{N-1}(a), V = 0, R = 1, delta = 1
//   2N - 1 times:  V = x V
//                  if delta > 0 and G[0] != 0: delta = -delta, swap(F, G), swap(V, R)
//                  delta += 1;  c = -G[0] F[0] (mod p);  G += c F;  R += c V;  G = G / x   (G[0] is 0 here)
//   a is invertible iff delta == 0; then inverse[i] = F[0] V[N-1-i] (mod p).
// The step count is fixed and every step does the same work: the swap and the scalar c are masks, never a branch or
// an address, so the time does not depend on the secret f.  For an invertible a no polynomial outgrows N + 1
// coefficients.  For the others V and R can, and their top words then drop bits; that is harmless, because V and R
// never feed delta, F or G, and the outputs of such a row are discarded.
// One warp per key: lane l holds coefficients 32 l ... 32 l + 31 of F, G, V, R in one word per bit plane (N + 1 <= 1024
// for every N the lifting accepts).  GF(2) is one plane per polynomial; GF(3) two one-hot planes, "= 1" and "= 2"
// (c F with c = 2 is F with its planes swapped).  x V and G / x are funnel shifts with the neighbour lane's word;
// delta, F[0] and the swap are warp-uniform.  The two chains are independent and interleaved, so each hides the
// other's shuffle latency.
constexpr int kInvWarps = 4;   // keys (warps) per CTA
constexpr unsigned kFull = 0xFFFFFFFFu;

// a += b in GF(3), one-hot planes
__device__ __forceinline__ void add_gf3(uint32_t &a1, uint32_t &a2, uint32_t b1, uint32_t b2) {
  const uint32_t a0 = ~(a1 | a2), b0 = ~(b1 | b2);
  const uint32_t s1 = (a0 & b1) | (a1 & b0) | (a2 & b2);
  const uint32_t s2 = (a0 & b2) | (a2 & b0) | (a1 & b1);
  a1 = s1;
  a2 = s2;
}

__device__ __forceinline__ void swap_masked(uint32_t &a, uint32_t &b, uint32_t m) {
  const uint32_t t = (a ^ b) & m;
  a ^= t;
  b ^= t;
}

// f, g: B rows of int8 (pitch P).  inv2: f^-1 mod 2 as uint16 rows, fp: f^-1 mod 3 as byte rows (pitch P, zero pads).
// valid[b] = f_b and g_b in {-1, 0, 1} and both inverses exist; rows that are not valid get all-zero inv2 / fp.
// skip_valid: rows whose valid[b] is already 1 are left as they are (redraw rounds).  invalid_count (may be NULL):
// number of rows this launch found invalid.
__global__ void __launch_bounds__(32 * kInvWarps) k_inverse_2_3(int N, int P, size_t B, const int8_t *__restrict__ f,
                                                              const int8_t *__restrict__ g, uint16_t *__restrict__ inv2,
                                                              uint8_t *__restrict__ fp, uint8_t *__restrict__ valid,
                                                              int skip_valid, unsigned *__restrict__ invalid_count) {
  const size_t b = (size_t)blockIdx.x * kInvWarps + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  if (skip_valid && valid[b]) return;                  // warp-uniform
  const int8_t *fb = f + b * (size_t)P, *gb = g + b * (size_t)P;
  // G = reverse_{N-1}(f): word k of a plane is the ballot of coefficients N-1-32k-l over the lanes l
  uint32_t g2 = 0, g31 = 0, g32 = 0;
  bool bad = false;
  for (int k = 0; 32 * k < N; ++k) {
    const int i = 32 * k + lane;
    int a = 0;
    if (i < N) {
      a = fb[N - 1 - i];
      const int c = gb[i];
      bad = bad || a < -1 || a > 1 || c < -1 || c > 1;
    }
    const uint32_t w2 = __ballot_sync(kFull, a != 0), w31 = __ballot_sync(kFull, a == 1), w32 = __ballot_sync(kFull, a == -1);
    if (lane == k) { g2 = w2; g31 = w31; g32 = w32; }
  }
  bad = __any_sync(kFull, bad);
  // F = 1 - x^N: F[0] = 1, F[N] = p - 1;  R = 1, V = 0
  const uint32_t one0 = lane == 0 ? 1u : 0u;
  const uint32_t topN = lane == (N >> 5) ? 1u << (N & 31) : 0u;
  uint32_t f2 = one0 | topN, v2 = 0, r2 = one0;
  uint32_t f31 = one0, f32 = topN, v31 = 0, v32 = 0, r31 = one0, r32 = 0;
  int d2 = 1, d3 = 1;
  uint32_t f0 = 1;                                     // F[0] of the GF(3) chain (1 or 2); F[0] = 1 over GF(2)
  const uint32_t up = lane ? kFull : 0u, down = lane < 31 ? kFull : 0u;
#pragma unroll 2
  for (int step = 0; step < 2 * N - 1; ++step) {
    // G[0] of both chains from lane 0: bit 0 over GF(2), bits 1-2 the GF(3) value
    const uint32_t g0 = __shfl_sync(kFull, (g2 & 1u) | ((g31 & 1u) << 1) | ((g32 & 1u) << 2), 0);
    const uint32_t g02 = g0 & 1u, g03 = g0 >> 1;
    // V = x V
    v2 = __funnelshift_l(__shfl_up_sync(kFull, v2, 1) & up, v2, 1);
    v31 = __funnelshift_l(__shfl_up_sync(kFull, v31, 1) & up, v31, 1);
    v32 = __funnelshift_l(__shfl_up_sync(kFull, v32, 1) & up, v32, 1);
    // GF(2): swap when delta > 0 and G[0] = 1; c = G[0] (the same before and after the swap: F[0] = 1)
    const uint32_t s2 = (uint32_t)(d2 > 0) & g02, m2 = 0u - s2, c2 = 0u - g02;
    swap_masked(f2, g2, m2);
    swap_masked(v2, r2, m2);
    d2 = (d2 ^ -(int)s2) + (int)s2 + 1;
    g2 ^= f2 & c2;
    r2 ^= v2 & c2;
    // GF(3): c = -G[0] F[0] is symmetric in the two, so it is taken before the swap: 2 if G[0] = F[0], else 1 (0 if
    // G[0] = 0)
    const uint32_t nz = (uint32_t)(g03 != 0u), s3 = (uint32_t)(d3 > 0) & nz, m3 = 0u - s3;
    const uint32_t same = nz & (uint32_t)(g03 == f0), c31 = 0u - (nz & (same ^ 1u)), c32 = 0u - same;
    swap_masked(f31, g31, m3);
    swap_masked(f32, g32, m3);
    swap_masked(v31, r31, m3);
    swap_masked(v32, r32, m3);
    f0 ^= (f0 ^ g03) & m3;
    d3 = (d3 ^ -(int)s3) + (int)s3 + 1;
    add_gf3(g31, g32, (f31 & c31) | (f32 & c32), (f32 & c31) | (f31 & c32));
    add_gf3(r31, r32, (v31 & c31) | (v32 & c32), (v32 & c31) | (v31 & c32));
    // G = G / x
    g2 = __funnelshift_r(g2, __shfl_down_sync(kFull, g2, 1) & down, 1);
    g31 = __funnelshift_r(g31, __shfl_down_sync(kFull, g31, 1) & down, 1);
    g32 = __funnelshift_r(g32, __shfl_down_sync(kFull, g32, 1) & down, 1);
  }
  const bool ok = !bad && d2 == 0 && d3 == 0;
  if (f0 == 2u) {                                      // inverse = F[0] V: times 2 swaps the planes
    const uint32_t t = v31; v31 = v32; v32 = t;
  }
  // inverse[i] = V[N-1-i]: coefficient i of the output row comes from bit (N-1-i) & 31 of lane (N-1-i) >> 5
  uint16_t *ib = inv2 + b * (size_t)P;
  uint8_t *pb = fp + b * (size_t)P;
  for (int i = lane; i < ((P + 31) & ~31); i += 32) {
    const int j = N - 1 - i;
    const int src = j >= 0 ? j >> 5 : 0;
    const uint32_t w2 = __shfl_sync(kFull, v2, src), w31 = __shfl_sync(kFull, v31, src), w32 = __shfl_sync(kFull, v32, src);
    if (i < P) {
      const bool in = ok && j >= 0;
      const uint32_t sh = (uint32_t)j & 31u;
      ib[i] = in ? (uint16_t)((w2 >> sh) & 1u) : (uint16_t)0;
      pb[i] = in ? (uint8_t)(((w31 >> sh) & 1u) | (((w32 >> sh) & 1u) << 1)) : (uint8_t)0;
    }
  }
  if (lane == 0) {
    valid[b] = ok ? 1 : 0;
    if (!ok && invalid_count) atomicAdd(invalid_count, 1u);
  }
}

// zeroes fq / fp / h of the rows that are not valid
__global__ void k_zero_invalid(const uint8_t *__restrict__ valid, size_t B, int P, uint16_t *__restrict__ fq,
                               uint8_t *__restrict__ fp, uint16_t *__restrict__ h) {
  const size_t n = B * (size_t)P;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    if (valid[i / P]) continue;
    fq[i] = 0;
    fp[i] = 0;
    h[i] = 0;
  }
}

// ---- device: the element-wise parts of a lifting step ------------------------------------------------------------
__global__ void k_newton_u(const uint16_t *__restrict__ t, size_t n, int P, int N, uint32_t qmask, int8_t *__restrict__ u0,
                           int8_t *__restrict__ u1) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % P);
    uint32_t u = k < N ? (((k == 0 ? 2u : 0u) - (uint32_t)t[i]) & qmask) : 0u;   // (2 - f inv) mod q, the 2 is the constant term
    u0[i] = (int8_t)(u & 127u);
    u1[i] = (int8_t)(u >> 7);
  }
}

__global__ void k_scale16(const uint16_t *__restrict__ src, size_t n, uint32_t mul, uint16_t *__restrict__ dst) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dst[i] = (uint16_t)((uint32_t)src[i] * mul);
}

__global__ void k_newton_combine(const uint16_t *__restrict__ r0, const uint16_t *__restrict__ r1, size_t n, uint32_t qmask,
                                 uint16_t *__restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = (uint16_t)(((uint32_t)r0[i] + 128u * (uint32_t)r1[i]) & qmask);
}

int launch_inverse(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *inv2, uint8_t *fp, uint8_t *valid,
                   bool skip_valid, unsigned *invalid_count) {
  if (B == 0) return NTRU_OK;
  const size_t blocks = (B + kInvWarps - 1) / kInvWarps;
  {
    LaunchTimer timer(ctx, NTRU_K_INVERSE);
    k_inverse_2_3<<<(unsigned)blocks, 32 * kInvWarps, 0, ctx->stream>>>(ctx->N, ctx->P, B, f, g, inv2, fp, valid,
                                                                         skip_valid ? 1 : 0, invalid_count);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

// fq holds f^-1 mod 2 on entry and f^-1 mod q on return; then h = (p fq) * g mod (q, x^N - 1).  Rows with inverse 0 (the
// rows that are not valid) stay 0 through every step.
int keygen_lift(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint16_t *h) {
  const int N = ctx->N, P = ctx->P;
  const uint32_t qmask = (uint32_t)ctx->q - 1;
  const size_t n = B * (size_t)P;
  DevBuf &d_t = ctx->kg_bufs[0], &d_u0 = ctx->kg_bufs[1], &d_u1 = ctx->kg_bufs[2], &d_r0 = ctx->kg_bufs[3],
         &d_r1 = ctx->kg_bufs[4];
  NTRU_CUDA(ctx, d_t.reserve(2 * n));
  NTRU_CUDA(ctx, d_u0.reserve(n)); NTRU_CUDA(ctx, d_u1.reserve(n));
  NTRU_CUDA(ctx, d_r0.reserve(2 * n)); NTRU_CUDA(ctx, d_r1.reserve(2 * n));
  cudaStream_t st = ctx->stream;
  int steps = 0;
  while ((1 << steps) < ctx->logq) ++steps;
  const unsigned grid = (unsigned)ctx->sm_count * 8;
  int rc;
  for (int s = 0; s < steps; ++s) {
    rc = launch_muldiv_imma(ctx, B, f, fq, 0, nullptr, d_t.ptr);                                            // t = f * inv
    if (rc) return rc;
    {
      LaunchTimer timer(ctx, NTRU_K_OTHER);
      k_newton_u<<<grid, 256, 0, st>>>((const uint16_t *)d_t.ptr, n, P, N, qmask, (int8_t *)d_u0.ptr, (int8_t *)d_u1.ptr);
    }
    rc = launch_muldiv_imma(ctx, B, (const int8_t *)d_u0.ptr, fq, 0, nullptr, d_r0.ptr);                    // inv * u0
    if (rc) return rc;
    rc = launch_muldiv_imma(ctx, B, (const int8_t *)d_u1.ptr, fq, 0, nullptr, d_r1.ptr);                    // inv * u1
    if (rc) return rc;
    {
      LaunchTimer timer(ctx, NTRU_K_OTHER);
      k_newton_combine<<<grid, 256, 0, st>>>((const uint16_t *)d_r0.ptr, (const uint16_t *)d_r1.ptr, n, qmask, fq);
    }
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return launch_h_product(ctx, B, g, fq, nullptr, h);
}

int keygen_check(ntru_ctx *ctx) {
  if (!ctx->tensor_ok || !imma_supported(ctx)) return fail(ctx, NTRU_E_UNSUPPORTED, "batched key generation needs the sm_100 tensor path and N <= 832");
  if (ctx->q < 4) return fail(ctx, NTRU_E_PARAM, "q too small");
  return NTRU_OK;
}

}  // namespace

int launch_h_product(ntru_ctx *ctx, size_t B, const int8_t *g, const uint16_t *fq, uint16_t *quo, uint16_t *rem) {
  // y = p fq as uint16, un-reduced (p (q - 1) < 65536; the same product modulo q as the reduced
  // multiplyPolynomialsByScalar(fq, p, q) of index.js:75, and the y of verifyKeysInputs, index.js:155)
  const size_t n = B * (size_t)ctx->P;
  DevBuf &d_y = ctx->kg_bufs[0];
  NTRU_CUDA(ctx, d_y.reserve(2 * n));
  {
    LaunchTimer timer(ctx, NTRU_K_OTHER);
    k_scale16<<<(unsigned)ctx->sm_count * 8, 256, 0, ctx->stream>>>(fq, n, (uint32_t)ctx->p, (uint16_t *)d_y.ptr);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return launch_muldiv_imma(ctx, B, g, d_y.ptr, 0, quo, rem);
}

int keygen_dev(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h,
               uint8_t *valid) {
  int rc = keygen_check(ctx);
  if (rc || B == 0) return rc;
  rc = launch_inverse(ctx, B, f, g, fq, fp, valid, false, nullptr);
  if (rc) return rc;
  rc = keygen_lift(ctx, B, f, g, fq, h);
  if (rc) return rc;
  {
    LaunchTimer timer(ctx, NTRU_K_OTHER);
    k_zero_invalid<<<(unsigned)ctx->sm_count * 8, 256, 0, ctx->stream>>>(valid, B, ctx->P, fq, fp, h);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

int keygen_batch(ntru_ctx *ctx, size_t B, const int8_t *f, const int8_t *g, uint16_t *fq, uint8_t *fp, uint16_t *h,
                 uint8_t *valid) {
  int rc = keygen_check(ctx);
  if (rc || B == 0) return rc;
  const int N = ctx->N, P = ctx->P;
  const size_t n = B * (size_t)P;
  DevBuf &d_f = ctx->kg_bufs[5], &d_g = ctx->kg_bufs[6], &d_fq = ctx->kg_bufs[7], &d_fp = ctx->kg_bufs[8],
         &d_h = ctx->kg_bufs[9], &d_valid = ctx->kg_bufs[10];
  NTRU_CUDA(ctx, d_f.reserve(n)); NTRU_CUDA(ctx, d_g.reserve(n));
  NTRU_CUDA(ctx, d_fq.reserve(2 * n)); NTRU_CUDA(ctx, d_fp.reserve(n)); NTRU_CUDA(ctx, d_h.reserve(2 * n));
  NTRU_CUDA(ctx, d_valid.reserve(B));
  cudaStream_t st = ctx->stream;
  // packed host rows -> pitched device rows with zero pad columns
  NTRU_CUDA(ctx, cudaMemsetAsync(d_f.ptr, 0, n, st));
  NTRU_CUDA(ctx, cudaMemsetAsync(d_g.ptr, 0, n, st));
  NTRU_CUDA(ctx, cudaMemcpy2DAsync(d_f.ptr, (size_t)P, f, (size_t)N, (size_t)N, B, cudaMemcpyHostToDevice, st));
  NTRU_CUDA(ctx, cudaMemcpy2DAsync(d_g.ptr, (size_t)P, g, (size_t)N, (size_t)N, B, cudaMemcpyHostToDevice, st));
  rc = keygen_dev(ctx, B, (const int8_t *)d_f.ptr, (const int8_t *)d_g.ptr, (uint16_t *)d_fq.ptr, (uint8_t *)d_fp.ptr,
                  (uint16_t *)d_h.ptr, (uint8_t *)d_valid.ptr);
  if (rc) return rc;
  NTRU_CUDA(ctx, cudaMemcpy2DAsync(fq, (size_t)N * 2, d_fq.ptr, (size_t)P * 2, (size_t)N * 2, B, cudaMemcpyDeviceToHost, st));
  NTRU_CUDA(ctx, cudaMemcpy2DAsync(fp, (size_t)N, d_fp.ptr, (size_t)P, (size_t)N, B, cudaMemcpyDeviceToHost, st));
  NTRU_CUDA(ctx, cudaMemcpy2DAsync(h, (size_t)N * 2, d_h.ptr, (size_t)P * 2, (size_t)N * 2, B, cudaMemcpyDeviceToHost, st));
  NTRU_CUDA(ctx, cudaMemcpyAsync(valid, d_valid.ptr, B, cudaMemcpyDeviceToHost, st));
  NTRU_CUDA(ctx, cudaStreamSynchronize(st));
  return NTRU_OK;
}

int generate_keys_dev(ntru_ctx *ctx, size_t B, int df, int dg, int8_t *f, int8_t *g, uint16_t *fq, uint8_t *fp,
                      uint16_t *h) {
  int rc = keygen_check(ctx);
  if (rc || B == 0) return rc;
  DevBuf &d_valid = ctx->kg_bufs[10], &d_count = ctx->kg_bufs[11];
  NTRU_CUDA(ctx, d_valid.reserve(B));
  NTRU_CUDA(ctx, d_count.reserve(sizeof(unsigned)));
  cudaStream_t st = ctx->stream;
  unsigned *count = (unsigned *)d_count.ptr;
  uint8_t *valid = (uint8_t *)d_valid.ptr;
  const uint64_t R = ctx->rng_row;
  // generatePrivateKeyF + generateNewPublicKeyGH (index.js:51-79): f with weights (df, df - 1) from rows R + b, g with
  // (dg, dg) from rows R + B + b; -1 is the int8 byte 0xFF
  ctx->rng_row = R + 2 * (uint64_t)B;                  // a row number (nonce) is never used twice under one key
  rc = launch_sample(ctx, B, df, df - 1, 0xFF, R, nullptr, (uint8_t *)f);
  if (rc) return rc;
  rc = launch_sample(ctx, B, dg, dg, 0xFF, R + B, nullptr, (uint8_t *)g);
  if (rc) return rc;
  unsigned invalid = 0;
  for (int round = 0; round < kKeygenRounds; ++round) {
    if (round > 0) {                                   // redraw f of the rows still invalid from rows R + (round+1) B + b
      ctx->rng_row = R + (uint64_t)(round + 2) * B;
      rc = launch_sample(ctx, B, df, df - 1, 0xFF, R + (uint64_t)(round + 1) * B, valid, (uint8_t *)f);
      if (rc) return rc;
    }
    NTRU_CUDA(ctx, cudaMemsetAsync(count, 0, sizeof(unsigned), st));
    rc = launch_inverse(ctx, B, f, g, fq, fp, valid, round > 0, count);
    if (rc) return rc;
    NTRU_CUDA(ctx, cudaMemcpyAsync(&invalid, count, sizeof invalid, cudaMemcpyDeviceToHost, st));
    NTRU_CUDA(ctx, cudaStreamSynchronize(st));
    if (invalid == 0) break;
  }
  if (invalid) return fail(ctx, NTRU_E_PARAM, "Could not find invertible f");   // index.js:63
  return keygen_lift(ctx, B, f, g, fq, h);
}

}  // namespace ntru
