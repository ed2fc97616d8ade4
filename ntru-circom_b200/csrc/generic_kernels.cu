// CUDA-core schedule: one CTA per ciphertext, operands resident in shared memory.
//
// Used for distinct-key batches (every row brings its own h, or f and fp), for wide
// messages, and as the on-GPU cross-check of the tcgen05 schedule.  Also holds the
// HBM-streaming ciphertext sum and the device sampler for r.
//
// What is computed (closed form of the reference, SURVEY.md section 8a):
//   encryptBits  (index.js:87-110):  c = lin(r,h) + m  mod q;  lo[k] = c[k], hi[k] = c[k+N]
//       remainderE[k] = (lo[k] + hi[k]) mod q,  quotientE[k] = (-hi[k]) mod q
//   decryptBits  (index.js:111-140): the same split for a = lin(f,e) mod q, then
//       b[k] = (r1[k] + [r1[k] > q/2]) mod 3  (the reference's lift, index.js:117),
//       and the same split for c = lin(fp,b) mod 3.
//   dividePolynomials(., 1 - x^N, .) (index.js:358-401) is that lo/hi split: the quotient
//       is -hi, the remainder is lo + hi; multiplyPolynomials (index.js:319-355) is the
//       exact integer product (the float64 FFT's rounding margin is < 1e-4).
//
// Arithmetic: fp32 FMA on integer-valued operands.  Every partial sum is an integer of
// magnitude <= N*2*(q-1) < 2^24 (N <= 1024, q <= 8192), so fp32 is exact; it runs on both
// FMA pipes where IMAD has one.  (ntru_create refuses q > 8192 for every schedule.)
//
// Thread mapping: thread c owns outputs k = 8c .. 8c+7.  The i-loop runs over blocks of 8
// multiplier coefficients; the window of 15 multiplicand values slides by 8 per block (two
// LDS.128), the 8 multiplier values are a warp-wide broadcast.  Contributions with i <= k
// belong to lo, with i > k (index k - i + N of the cyclic extension) to hi; the switch
// happens inside block b == c, where the accumulator is snapshotted.

#include <cuda_runtime.h>
#include <stdint.h>

#include "ntru_internal.cuh"

namespace ntru {

namespace {

constexpr int T = 8;   // outputs per thread

// lo[t] = sum_{i<=k} mul[i] * win[k-i],  hi[t] = sum_{i>k} mul[i] * win[k-i+N],  k = 8c+t.
// S[y] = win[(y + 1 - 8NB) mod N] for y in [0,16NB);  mulS[i] = mul[i] (0 for i >= N), i in [0,8NB).
__device__ __forceinline__ void conv8(const float *__restrict__ S, const float *__restrict__ mulS, int NB, int c,
                                      float (&lo)[T], float (&hi)[T]) {
  float acc[T], L[T], H[T], rv[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    acc[t] = 0.f;
    lo[t] = 0.f;
  }
  int y0 = T * (c - 1 + NB);
  {
    const float4 a = *reinterpret_cast<const float4 *>(S + y0 + 8);
    const float4 b = *reinterpret_cast<const float4 *>(S + y0 + 12);
    H[0] = a.x; H[1] = a.y; H[2] = a.z; H[3] = a.w;
    H[4] = b.x; H[5] = b.y; H[6] = b.z; H[7] = b.w;
  }
#pragma unroll 2
  for (int b = 0; b < NB; ++b) {
    {
      const float4 a0 = *reinterpret_cast<const float4 *>(S + y0);
      const float4 a1 = *reinterpret_cast<const float4 *>(S + y0 + 4);
      L[0] = a0.x; L[1] = a0.y; L[2] = a0.z; L[3] = a0.w;
      L[4] = a1.x; L[5] = a1.y; L[6] = a1.z; L[7] = a1.w;
      const float4 r0 = *reinterpret_cast<const float4 *>(mulS + T * b);
      const float4 r1 = *reinterpret_cast<const float4 *>(mulS + T * b + 4);
      rv[0] = r0.x; rv[1] = r0.y; rv[2] = r0.z; rv[3] = r0.w;
      rv[4] = r1.x; rv[5] = r1.y; rv[6] = r1.z; rv[7] = r1.w;
    }
    // window W[w] = w < 8 ? L[w] : H[w-8];  term (t, di) uses W[7 + t - di]
#pragma unroll
    for (int t = 0; t < T; ++t) {
#pragma unroll
      for (int di = 0; di <= t; ++di) {
        const int w = 7 + t - di;                 // 7..14
        acc[t] = fmaf(rv[di], w < 8 ? L[w] : H[w - 8], acc[t]);
      }
    }
    if (b == c) {                                  // i <= k ends here: snapshot lo, restart for hi
#pragma unroll
      for (int t = 0; t < T; ++t) {
        lo[t] = acc[t];
        acc[t] = 0.f;
      }
    }
#pragma unroll
    for (int t = 0; t < T; ++t) {
#pragma unroll
      for (int di = t + 1; di < T; ++di) acc[t] = fmaf(rv[di], L[7 + t - di], acc[t]);   // w in 0..6
    }
#pragma unroll
    for (int t = 0; t < T; ++t) H[t] = L[t];
    y0 -= T;
  }
#pragma unroll
  for (int t = 0; t < T; ++t) hi[t] = acc[t];
}

__device__ __forceinline__ uint32_t mod3_u16(uint32_t v) {   // v < 65536
  return v - 3u * ((v * 0xAAABu) >> 17);
}

__device__ __forceinline__ uint4 pack8_u16(const uint32_t (&v)[T]) {
  return make_uint4(v[0] | (v[1] << 16), v[2] | (v[3] << 16), v[4] | (v[5] << 16), v[6] | (v[7] << 16));
}

__device__ __forceinline__ uint2 pack8_u8(const uint32_t (&v)[T]) {
  return make_uint2(v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24),
                    v[4] | (v[5] << 8) | (v[6] << 16) | (v[7] << 24));
}

struct EncArgs {
  int N, P, NB;
  uint32_t qmask;
  size_t B;
  const uint16_t *h;
  size_t h_stride;
  const uint8_t *r;
  const void *m;
  uint16_t *value, *quo, *rem;
};

template <bool kWideM>
__global__ void __launch_bounds__(160) k_encrypt_generic(const EncArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int N = a.N, P = a.P, NB = a.NB;
  float *S = smem;
  float *mulS = smem + 16 * NB;
  const int c = threadIdx.x;
  const bool active = c < NB && T * c < P;
  for (size_t row = blockIdx.x; row < a.B; row += gridDim.x) {
    const uint16_t *h = a.h + row * a.h_stride;
    const uint8_t *r = a.r + row * (size_t)P;
    for (int y = threadIdx.x; y < 16 * NB; y += blockDim.x) {
      const int j = (y + 1 - 8 * NB + 2 * N) % N;
      S[y] = (float)h[j];
    }
    for (int i = threadIdx.x; i < 8 * NB; i += blockDim.x) mulS[i] = i < N ? (float)r[i] : 0.f;
    __syncthreads();
    if (active) {
      float lo[T], hi[T];
      conv8(S, mulS, NB, c, lo, hi);
      uint32_t mv[T];
      if (kWideM) {
        const uint4 w = *reinterpret_cast<const uint4 *>(reinterpret_cast<const uint16_t *>(a.m) + row * (size_t)P + T * c);
        mv[0] = w.x & 0xffff; mv[1] = w.x >> 16; mv[2] = w.y & 0xffff; mv[3] = w.y >> 16;
        mv[4] = w.z & 0xffff; mv[5] = w.z >> 16; mv[6] = w.w & 0xffff; mv[7] = w.w >> 16;
      } else {
        const uint2 w = *reinterpret_cast<const uint2 *>(reinterpret_cast<const uint8_t *>(a.m) + row * (size_t)P + T * c);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          mv[t] = (w.x >> (8 * t)) & 0xff;
          mv[4 + t] = (w.y >> (8 * t)) & 0xff;
        }
      }
      uint32_t rem[T], quo[T];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int k = T * c + t;
        const int l = __float2int_rn(lo[t]) + (int)mv[t];
        const int hh = __float2int_rn(hi[t]);
        const bool in = k < N;
        rem[t] = in ? ((uint32_t)(l + hh) & a.qmask) : 0u;
        quo[t] = in ? ((uint32_t)(-hh) & a.qmask) : 0u;
      }
      const size_t off = row * (size_t)P + T * c;
      if (a.value) *reinterpret_cast<uint4 *>(a.value + off) = pack8_u16(rem);
      if (a.rem) *reinterpret_cast<uint4 *>(a.rem + off) = pack8_u16(rem);
      if (a.quo) *reinterpret_cast<uint4 *>(a.quo + off) = pack8_u16(quo);
    } else if (T * c < P) {   // pad columns beyond the last 8-coefficient block: zero, like every schedule
      const size_t off = row * (size_t)P + T * c;
      const uint4 z = make_uint4(0, 0, 0, 0);
      if (a.value) *reinterpret_cast<uint4 *>(a.value + off) = z;
      if (a.rem) *reinterpret_cast<uint4 *>(a.rem + off) = z;
      if (a.quo) *reinterpret_cast<uint4 *>(a.quo + off) = z;
    }
    __syncthreads();
  }
}

struct DecArgs {
  int N, P, NB, q;
  uint32_t qmask;
  size_t B;
  const int8_t *f;
  const uint8_t *fp;
  size_t key_stride;
  const uint16_t *e;
  uint8_t *value, *q2, *r2;
  uint16_t *q1, *r1;
};

__global__ void __launch_bounds__(160) k_decrypt_generic(const DecArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int N = a.N, P = a.P, NB = a.NB;
  float *S = smem;
  float *mulS = smem + 16 * NB;
  const int c = threadIdx.x;
  const bool active = c < NB && T * c < P;
  const uint32_t halfq = (uint32_t)a.q >> 1;
  for (size_t row = blockIdx.x; row < a.B; row += gridDim.x) {
    const int8_t *f = a.f + row * a.key_stride;
    const uint8_t *fp = a.fp + row * a.key_stride;
    const uint16_t *e = a.e + row * (size_t)P;
    // product 1: a = lin(f, e) -- window = e, multiplier = f
    for (int y = threadIdx.x; y < 16 * NB; y += blockDim.x) S[y] = (float)e[(y + 1 - 8 * NB + 2 * N) % N];
    for (int i = threadIdx.x; i < 8 * NB; i += blockDim.x) mulS[i] = i < N ? (float)f[i] : 0.f;
    __syncthreads();
    float lo[T], hi[T];
    uint32_t bv[T];
    if (active) {
      conv8(S, mulS, NB, c, lo, hi);
      uint32_t rem[T], quo[T];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int k = T * c + t;
        const int l = __float2int_rn(lo[t]);
        const int hh = __float2int_rn(hi[t]);
        const bool in = k < N;
        rem[t] = in ? ((uint32_t)(l + hh) & a.qmask) : 0u;
        quo[t] = in ? ((uint32_t)(-hh) & a.qmask) : 0u;
        bv[t] = mod3_u16(rem[t] + (rem[t] > halfq ? 1u : 0u));   // index.js:117
      }
      const size_t off = row * (size_t)P + T * c;
      if (a.r1) *reinterpret_cast<uint4 *>(a.r1 + off) = pack8_u16(rem);
      if (a.q1) *reinterpret_cast<uint4 *>(a.q1 + off) = pack8_u16(quo);
    } else if (T * c < P) {
      const size_t off = row * (size_t)P + T * c;
      const uint4 z = make_uint4(0, 0, 0, 0);
      if (a.r1) *reinterpret_cast<uint4 *>(a.r1 + off) = z;
      if (a.q1) *reinterpret_cast<uint4 *>(a.q1 + off) = z;
    }
    __syncthreads();
    // product 2: c = lin(fp, b) -- window = fp, multiplier = b
    for (int y = threadIdx.x; y < 16 * NB; y += blockDim.x) S[y] = (float)fp[(y + 1 - 8 * NB + 2 * N) % N];
    if (active) {
#pragma unroll
      for (int t = 0; t < T; ++t) mulS[T * c + t] = (float)bv[t];
    }
    __syncthreads();
    if (active) {
      conv8(S, mulS, NB, c, lo, hi);
      uint32_t rem[T], quo[T];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int k = T * c + t;
        const uint32_t l3 = mod3_u16((uint32_t)__float2int_rn(lo[t]));
        const uint32_t h3 = mod3_u16((uint32_t)__float2int_rn(hi[t]));
        const bool in = k < N;
        rem[t] = in ? mod3_u16(l3 + h3) : 0u;
        quo[t] = in ? mod3_u16(3u - h3) : 0u;
      }
      const size_t off = row * (size_t)P + T * c;
      if (a.value) *reinterpret_cast<uint2 *>(a.value + off) = pack8_u8(rem);
      if (a.r2) *reinterpret_cast<uint2 *>(a.r2 + off) = pack8_u8(rem);
      if (a.q2) *reinterpret_cast<uint2 *>(a.q2 + off) = pack8_u8(quo);
    } else if (T * c < P) {
      const size_t off = row * (size_t)P + T * c;
      const uint2 z = make_uint2(0, 0);
      if (a.value) *reinterpret_cast<uint2 *>(a.value + off) = z;
      if (a.r2) *reinterpret_cast<uint2 *>(a.r2 + off) = z;
      if (a.q2) *reinterpret_cast<uint2 *>(a.q2 + off) = z;
    }
    __syncthreads();
  }
}

// ---- homomorphic ciphertext sum: column sums of B x N uint16 rows -------------------------------
// Pure HBM streaming (2N bytes per ciphertext).  Thread (vx, ry) owns the 8 columns of 16-byte
// vector vx and rows ry, ry+RY, ...; uint32 accumulation wraps mod 2^32, which is exact mod q | 2^16.
//
// The CTAs' column sums are combined by a two-level tree in global scratch, not by atomics: the first version
// issued P atomicAdds per CTA onto P words = 22 cache lines, ~19 000 same-line reductions per line when 592 CTAs
// finish together, ~60 us of serialised L2 work per call (10 M rows: 1.95 ms, 1.25 M rows: 0.296 ms => 7.4 TB/s
// streaming + 0.06 ms fixed).  Now every CTA stores its P sums as one row of `scratch`; the last CTA of each group
// of kSumGroup CTAs (one ticket per group) adds the group's rows into a group row, and the last group leader adds
// the group rows: two rounds of <= 16 / <= 37 independent 16-byte loads per thread.
constexpr int kSumRows = 4;      // rows per CTA iteration (fewer when a row has > 128 vectors)
constexpr int kSumUnroll = 4;    // independent 16-byte loads in flight per thread
constexpr int kSumGroup = 16;    // CTAs per first-level group of the tree

struct SumScratch {
  uint32_t *rows;      // [gridDim.x][P]  per-CTA column sums
  uint32_t *grows;     // [ngroups][P]    per-group column sums
  uint32_t *tickets;   // [ngroups + 1]   arrival counters (groups, then the group leaders); zero between calls
};

// This CTA's column sums of rows blockIdx.x * RY + ry, stepping by gridDim.x * RY; on return the threads with
// ry == 0 hold the eight sums of columns 8 vx .. 8 vx + 7 in s[].
__device__ __forceinline__ void cta_column_sums(const uint16_t *__restrict__ e, size_t B, int P, uint32_t *red, uint32_t (&s)[8]) {
  const int VX = P / 8;
  const int vx = threadIdx.x, ry = threadIdx.y;
  uint32_t lo[4] = {0, 0, 0, 0}, hi[4] = {0, 0, 0, 0};
  const int RY = blockDim.y;
  const size_t step = (size_t)gridDim.x * RY;
  size_t row = (size_t)blockIdx.x * RY + ry;
  const uint4 *base = reinterpret_cast<const uint4 *>(e) + vx;
  for (; row + (kSumUnroll - 1) * step < B; row += kSumUnroll * step) {
    uint4 v[kSumUnroll];
#pragma unroll
    for (int u = 0; u < kSumUnroll; ++u) v[u] = __ldcs(base + (row + u * step) * (size_t)VX);
#pragma unroll
    for (int u = 0; u < kSumUnroll; ++u) {
      lo[0] += v[u].x; hi[0] += v[u].x >> 16;
      lo[1] += v[u].y; hi[1] += v[u].y >> 16;
      lo[2] += v[u].z; hi[2] += v[u].z >> 16;
      lo[3] += v[u].w; hi[3] += v[u].w >> 16;
    }
  }
  for (; row < B; row += step) {
    const uint4 v = __ldcs(base + row * (size_t)VX);
    lo[0] += v.x; hi[0] += v.x >> 16;
    lo[1] += v.y; hi[1] += v.y >> 16;
    lo[2] += v.z; hi[2] += v.z >> 16;
    lo[3] += v.w; hi[3] += v.w >> 16;
  }
  // low halves: only bits [0,16) of lo[] are meaningful (the high half holds the odd column's sum
  // plus carries); hi[] are clean sums of the odd columns.
  uint32_t *mine = red + ((size_t)ry * VX + vx) * 8;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    mine[2 * j] = lo[j] & 0xffffu;
    mine[2 * j + 1] = hi[j];
  }
  __syncthreads();
  if (ry == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      uint32_t t = 0;
      for (int y = 0; y < RY; ++y) t += red[((size_t)y * VX + vx) * 8 + j];
      s[j] = t;
    }
  }
}

// Tree over the CTAs.  Returns true in exactly one CTA per launch (the last group leader to arrive); there, thread
// tid < P / 4 holds the grand totals of columns 4 tid .. 4 tid + 3 in tot.  The tickets are left at zero.
__device__ __forceinline__ bool grid_column_totals(const SumScratch sc, int P, const uint32_t (&s)[8], bool *flag, uint4 &tot) {
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nvec = P / 4;                                  // 16-byte vectors of uint32 per row (blockDim.x * 2 <= threads)
  const int ngroups = (gridDim.x + kSumGroup - 1) / kSumGroup;
  const int grp = blockIdx.x / kSumGroup;
  const int gsize = min(kSumGroup, (int)gridDim.x - grp * kSumGroup);
  if (threadIdx.y == 0) {
    uint4 *dst = reinterpret_cast<uint4 *>(sc.rows + (size_t)blockIdx.x * P) + 2 * threadIdx.x;
    dst[0] = make_uint4(s[0], s[1], s[2], s[3]);
    dst[1] = make_uint4(s[4], s[5], s[6], s[7]);
    __threadfence();
  }
  __syncthreads();
  if (tid == 0) {
    __threadfence();                                       // release: this CTA's row before its ticket
    *flag = atomicAdd(sc.tickets + grp, 1u) == (uint32_t)gsize - 1;
    __threadfence();                                       // acquire: the last arrival sees every row of the group
  }
  __syncthreads();
  if (!*flag) return false;
  __syncthreads();                                         // everyone has read *flag before thread 0 rewrites it below
  uint4 acc = make_uint4(0, 0, 0, 0);
  if (tid < nvec) {
    const uint4 *src = reinterpret_cast<const uint4 *>(sc.rows + (size_t)grp * kSumGroup * P) + tid;
#pragma unroll
    for (int i = 0; i < kSumGroup; ++i) {
      if (i < gsize) {
        const uint4 v = __ldcg(src + (size_t)i * nvec);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    }
    reinterpret_cast<uint4 *>(sc.grows + (size_t)grp * P)[tid] = acc;
    __threadfence();
  }
  __syncthreads();
  if (tid == 0) {
    sc.tickets[grp] = 0;                                   // ready for the next call
    __threadfence();
    *flag = atomicAdd(sc.tickets + ngroups, 1u) == (uint32_t)ngroups - 1;
    __threadfence();
  }
  __syncthreads();
  if (!*flag) return false;
  tot = make_uint4(0, 0, 0, 0);
  if (tid < nvec) {
    const uint4 *src = reinterpret_cast<const uint4 *>(sc.grows) + tid;
    int g = 0;
    for (; g + 4 <= ngroups; g += 4) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldcg(src + (size_t)(g + u) * nvec);
#pragma unroll
      for (int u = 0; u < 4; ++u) { tot.x += v[u].x; tot.y += v[u].y; tot.z += v[u].z; tot.w += v[u].w; }
    }
    for (; g < ngroups; ++g) {
      const uint4 v = __ldcg(src + (size_t)g * nvec);
      tot.x += v.x; tot.y += v.y; tot.z += v.z; tot.w += v.w;
    }
  }
  if (tid == 0) sc.tickets[ngroups] = 0;
  return true;
}

// partial[k] += column sums of this call's rows (one writer: the CTA that finishes the tree)
__global__ void __launch_bounds__(512) k_sum_partial(const uint16_t *__restrict__ e, size_t B, int P, const SumScratch sc,
                                                      uint32_t *__restrict__ partial) {
  extern __shared__ __align__(16) uint32_t red[];
  __shared__ bool flag;
  uint32_t s[8];
  cta_column_sums(e, B, P, red, s);
  uint4 tot;
  if (!grid_column_totals(sc, P, s, &flag, tot)) return;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  if (tid < P / 4) {
    uint4 *dst = reinterpret_cast<uint4 *>(partial) + tid;
    uint4 v = *dst;
    v.x += tot.x; v.y += tot.y; v.z += tot.z; v.w += tot.w;
    *dst = v;
  }
}

// ---- cross-GPU sum: column sums fused with the exchange over peer memory --------------------------------------
// Window of one rank: slots[2][world][P] uint32 (parity of the call number, sender rank), flags[world], error word.
// k_sum_push   = the column sums above + the CTA that finishes the tree owns the exchange: it masks the N totals,
//                stores them into slot[parity][rank] of EVERY rank's window (plain stores over NVLink for the peers),
//                fences system-wide and raises flag[rank] = epoch in every window.
//                Then the same CTA gathers: it waits until flag[r] has REACHED epoch for every r (acquire loads of its
//                own window; a peer may already be one call ahead and have written epoch + 1 -- its slot of this
//                call's parity is still intact then), adds the world slots per column, masks, writes out[].  A rank
//                cannot run two calls ahead of a peer (it needs the peer's flag of call n to finish call n), so two
//                slot parities are enough.
//                If a peer never arrives (~4 s), the error word of this rank's window is set, out[] is filled with
//                0xFFFF (no valid residue) and the host reports NTRU_E_CUDA at the next ntru_sync / sum call.
// One launch per call: HBM streaming, exchange and final sum.
struct XchgPeers {
  uint32_t *window[ntru_ctx::kMaxRanks];   // only indexed with compile-time-unrolled, bounded loops (stays in the constant bank)
};

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// The exchange itself, run by ONE CTA: thread tid < P / 4 brings the rank's totals of columns 4 tid .. 4 tid + 3.
__device__ __forceinline__ void exchange_totals(const uint4 tot, int P, const XchgPeers &peers, int world, int rank, uint32_t epoch,
                                                uint32_t qmask, int N, uint16_t *__restrict__ out, int *timed_out) {
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  if (tid == 0) *timed_out = 0;
  const size_t slot = ((size_t)(epoch & 1u) * world + rank) * P;
  if (tid < P / 4) {
    const uint4 v = make_uint4(tot.x & qmask, tot.y & qmask, tot.z & qmask, tot.w & qmask);
#pragma unroll
    for (int r = 0; r < ntru_ctx::kMaxRanks; ++r)
      if (r < world) reinterpret_cast<uint4 *>(peers.window[r] + slot)[tid] = v;   // peer stores travel over NVLink
  }
  __syncthreads();
  // release at system scope, cumulative over the stores the barrier above ordered before it
#pragma unroll
  for (int r = 0; r < ntru_ctx::kMaxRanks; ++r)
    if (r == tid && r < world) st_release_sys(peers.window[r] + (size_t)2 * world * P + rank, epoch);
  // ---- gather: wait for every rank's flag in this rank's window, add the slots ----
  uint32_t *window = peers.window[rank];
  const uint32_t *flags = window + (size_t)2 * world * P;
  if (tid < world) {
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys(flags + tid) - epoch) < 0) {
      if (clock64() - t0 > 8000000000ll) {                    // ~4 s: a peer never arrived; do not hang the GPU
        atomicExch(window + (size_t)2 * world * P + world, 1u);
        *timed_out = 1;
        break;
      }
    }
  }
  __syncthreads();
  const int nthr = blockDim.x * blockDim.y;
  if (*timed_out) {
    for (int k = tid; k < P; k += nthr) out[k] = (uint16_t)0xFFFFu;
    return;
  }
  const uint32_t *slots = window + (size_t)(epoch & 1u) * world * P;
  for (int k = tid; k < P; k += nthr) {
    uint32_t t = 0;
    for (int r = 0; r < world; ++r) t += __ldcv(slots + (size_t)r * P + k);
    out[k] = k < N ? (uint16_t)(t & qmask) : (uint16_t)0;
  }
}

__global__ void __launch_bounds__(512) k_sum_push(const uint16_t *__restrict__ e, size_t B, int P, const SumScratch sc,
                                                  const XchgPeers peers, int world, int rank, uint32_t epoch, uint32_t qmask,
                                                  int N, uint16_t *__restrict__ out) {
  extern __shared__ __align__(16) uint32_t red[];
  __shared__ bool flag;
  __shared__ int timed_out;
  uint32_t s[8];
  cta_column_sums(e, B, P, red, s);
  uint4 tot;
  if (!grid_column_totals(sc, P, s, &flag, tot)) return;
  exchange_totals(tot, P, peers, world, rank, epoch, qmask, N, out, &timed_out);   // this CTA owns the exchange
}

// the exchange alone, for column sums that were accumulated over several launches (host-buffer entry point: the
// shard streams through the pipelined chunks into partial[], which is cleared here for the next call)
__global__ void __launch_bounds__(512) k_xchg_partial(uint32_t *__restrict__ partial, int P, const XchgPeers peers, int world, int rank,
                                                      uint32_t epoch, uint32_t qmask, int N, uint16_t *__restrict__ out) {
  __shared__ int timed_out;
  const int tid = threadIdx.x;
  uint4 tot = make_uint4(0, 0, 0, 0);
  if (tid < P / 4) {
    tot = reinterpret_cast<const uint4 *>(partial)[tid];
    reinterpret_cast<uint4 *>(partial)[tid] = make_uint4(0, 0, 0, 0);
  }
  exchange_totals(tot, P, peers, world, rank, epoch, qmask, N, out, &timed_out);
}

__global__ void k_sum_finalize(const uint32_t *__restrict__ partial, int N, int P, uint32_t qmask,
                               uint16_t *__restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < P) out[k] = k < N ? (uint16_t)(partial[k] & qmask) : (uint16_t)0;
}

// ---- device sampler: generateCustomArray(N, ones, neg_ones) ----------------------------------
// Same algorithm as index.js:461-488 (`ones` ones, `neg_ones` "minus ones", Fisher-Yates from the top with
// j = rand32 % (i+1)); a -1 is stored as the byte neg_code: 2 for r (generateCustomArray(N, dr, dr).map(-1 -> 2),
// index.js:89), 0xFF (int8 -1) for the key polynomials f and g (index.js:52-70).  The WebCrypto draw (index.js:481-483)
// is replaced by a keyed counter-mode CSPRNG so that the device can draw r itself (ntru_encrypt_batch with r == NULL) and any row can be replayed by the key holder:
// ChaCha20 (D. J. Bernstein's layout: 256-bit key, 64-bit block counter, 64-bit nonce), nonce = global row number,
// block counter = 0, 1, ... within the row; the draw for position i = N-1, N-2, ..., 1 is keystream word
// w = N-1-i (word w % 16 of block w / 16).  The key comes from the operating system's entropy (ntru_create) or
// from ntru_set_rng_key.  The block function is pinned on the RFC 8439 section 2.3.2 vector through its host copy
// (tests/test_host.py), the device against the host copy (tests/test_gpu_parity.py).
struct ChaChaKey {
  uint32_t k[8];
};

#define NTRU_CHACHA_QR(a, b, c, d)                    \
  a += b; d ^= a; d = __funnelshift_l(d, d, 16);      \
  c += d; b ^= c; b = __funnelshift_l(b, b, 12);      \
  a += b; d ^= a; d = __funnelshift_l(d, d, 8);       \
  c += d; b ^= c; b = __funnelshift_l(b, b, 7);

__device__ __forceinline__ void chacha20_block(const ChaChaKey &key, uint64_t counter, uint64_t nonce, uint32_t (&out)[16]) {
  const uint32_t in[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u,
                           key.k[0], key.k[1], key.k[2], key.k[3], key.k[4], key.k[5], key.k[6], key.k[7],
                           (uint32_t)counter, (uint32_t)(counter >> 32), (uint32_t)nonce, (uint32_t)(nonce >> 32)};
  uint32_t x[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = in[i];
#pragma unroll 2
  for (int round = 0; round < 10; ++round) {
    NTRU_CHACHA_QR(x[0], x[4], x[8], x[12])
    NTRU_CHACHA_QR(x[1], x[5], x[9], x[13])
    NTRU_CHACHA_QR(x[2], x[6], x[10], x[14])
    NTRU_CHACHA_QR(x[3], x[7], x[11], x[15])
    NTRU_CHACHA_QR(x[0], x[5], x[10], x[15])
    NTRU_CHACHA_QR(x[1], x[6], x[11], x[12])
    NTRU_CHACHA_QR(x[2], x[7], x[8], x[13])
    NTRU_CHACHA_QR(x[3], x[4], x[9], x[14])
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) out[i] = x[i] + in[i];
}

constexpr int kSampleRows = 64;   // rows (threads) per CTA

// skip (may be NULL): rows b with skip[b] != 0 are neither drawn nor written
__global__ void __launch_bounds__(kSampleRows) k_sample_ternary(int N, int P, int ones, int neg_ones, uint8_t neg_code,
                                                                const ChaChaKey key, uint64_t row0, size_t B,
                                                                const uint8_t *__restrict__ skip, uint8_t *__restrict__ r) {
  extern __shared__ __align__(16) uint8_t arr[];
  const int stride = P + 4;                       // bytes; (P+4)/4 is odd, so rows start in distinct banks
  const size_t first = (size_t)blockIdx.x * kSampleRows;
  const size_t row = first + threadIdx.x;
  uint8_t *mine = arr + (size_t)threadIdx.x * stride;
  if (row < B && !(skip && skip[row])) {
    for (int i = 0; i < P; ++i) mine[i] = i < ones ? 1 : (i < ones + neg_ones ? neg_code : 0);
    int i = N - 1;
    for (uint64_t blk = 0; i > 0; ++blk) {
      uint32_t ks[16];
      chacha20_block(key, blk, row0 + row, ks);
#pragma unroll
      for (int w = 0; w < 16; ++w) {
        if (i > 0) {
          const uint32_t j = ks[w] % (uint32_t)(i + 1);
          const uint8_t a = mine[i], b = mine[j];
          mine[i] = b;
          mine[j] = a;
          --i;
        }
      }
    }
  }
  __syncthreads();
  // coalesced copy-out: 4-byte words, one row after another
  const int wpr = P / 4;
  const size_t rows_here = (B - first) < (size_t)kSampleRows ? (B - first) : (size_t)kSampleRows;
  for (size_t idx = threadIdx.x; idx < rows_here * wpr; idx += blockDim.x) {
    const size_t rr = idx / wpr;
    const int w = (int)(idx % wpr);
    if (skip && skip[first + rr]) continue;
    reinterpret_cast<uint32_t *>(r + (first + rr) * (size_t)P)[w] =
        *reinterpret_cast<const uint32_t *>(arr + rr * stride + 4 * w);
  }
}

}  // namespace

// ---- packOutput / unpackInput (index.js:572-620): coefficients <-> BN254 field elements ---------------------------
// packOutput puts n = floor(252 / bits) coefficients of `bits` bits each into one field element, little-endian in the
// bit string: element o = sum_j data[o n + j] << (j bits).  A field element is stored as 32 bytes, little-endian
// (eight uint32 words).  One thread per output word: it gathers the (at most 32 / bits + 2) coefficients that
// overlap its 32 bits.  Values must fit `bits` bits (the reference adds BigInts, so larger values would carry).
template <typename T>
__global__ void k_pack_fields(const T *__restrict__ data, size_t B, int data_len, size_t pitch, int bits, int n,
                              int out_elems, uint32_t *__restrict__ out) {
  const size_t total = B * (size_t)out_elems * 8;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int w = (int)(idx & 7);
    const size_t eo = idx >> 3;
    const int o = (int)(eo % out_elems);
    const size_t row = eo / out_elems;
    const int bit0 = 32 * w;                       // first bit of this word inside the element
    uint32_t word = 0;
    if (bit0 < n * bits) {
      const int j0 = bit0 / bits;
      for (int j = j0; j < n && j * bits < bit0 + 32; ++j) {
        const int i = o * n + j;
        const uint32_t v = i < data_len ? (uint32_t)data[row * pitch + i] : 0u;
        const int sh = j * bits - bit0;            // position of the coefficient's bit 0 relative to this word
        word |= sh >= 0 ? (v << sh) : (v >> (-sh));
      }
    }
    out[idx] = word;
  }
}

// unpackInput: coefficient (i, j) = (element i >> (j bits)) & mask, n = floor(packedBits / bits) per element
template <typename T>
__global__ void k_unpack_fields(const uint32_t *__restrict__ data, size_t B, int in_elems, int bits, int n, size_t pitch,
                                T *__restrict__ out) {
  const size_t per_row = (size_t)in_elems * n;
  const size_t total = B * per_row;
  const uint32_t mask = bits >= 32 ? 0xffffffffu : ((1u << bits) - 1u);
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t row = idx / per_row;
    const int k = (int)(idx % per_row);
    const int i = k / n, j = k % n;
    const uint32_t *el = data + (row * in_elems + i) * 8;
    const int bit0 = j * bits, w = bit0 >> 5, sh = bit0 & 31;
    uint64_t two = el[w];
    if (w + 1 < 8) two |= (uint64_t)el[w + 1] << 32;
    out[row * pitch + k] = (T)((uint32_t)(two >> sh) & mask);
  }
}

// Wire form of unpackInput for the *_batch_packed entry points: B x in_elems field elements -> device rows of pitch P
// whose first `width` columns are the coefficients (element i, position j -> column i n + j) and whose other columns
// are zero.  packOutput pads a row to arrLen >= width coefficients (index.js:575-581): the padding must be zero, it is
// not copied.  One thread per device column.
template <typename T>
__global__ void k_wire_unpack(const uint32_t *__restrict__ data, size_t B, int in_elems, int bits, int n, int width, int P,
                              T *__restrict__ out) {
  const size_t total = B * (size_t)P;
  const uint32_t mask = (1u << bits) - 1u;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t row = idx / P;
    const int k = (int)(idx % P);
    uint32_t v = 0;
    if (k < width) {
      const int i = k / n, j = k % n;
      const uint32_t *el = data + (row * in_elems + i) * 8;
      const int bit0 = j * bits, w = bit0 >> 5, sh = bit0 & 31;
      uint64_t two = el[w];
      if (sh + bits > 32) two |= (uint64_t)el[w + 1] << 32;     // w + 1 <= 7: n bits <= 252
      v = (uint32_t)(two >> sh) & mask;
    }
    out[idx] = (T)v;
  }
}

int launch_wire_unpack(ntru_ctx *ctx, size_t B, const uint32_t *data, int in_elems, int bits, int n, int width, void *out,
                       int elem_bytes) {
  if (B == 0) return NTRU_OK;
  const size_t total = B * (size_t)ctx->P;
  size_t blocks = (total + 255) / 256;
  const size_t cap = (size_t)ctx->sm_count * 16;
  if (blocks > cap) blocks = cap;
  {
    LaunchTimer timer(ctx, NTRU_K_PACK);
    if (elem_bytes == 2)
      k_wire_unpack<uint16_t><<<(unsigned)blocks, 256, 0, ctx->stream>>>(data, B, in_elems, bits, n, width, ctx->P, (uint16_t *)out);
    else
      k_wire_unpack<uint8_t><<<(unsigned)blocks, 256, 0, ctx->stream>>>(data, B, in_elems, bits, n, width, ctx->P, (uint8_t *)out);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

// ---- pitch conversion for the host-buffer entry points --------------------------------------------
// Host rows are packed (N or N+1 elements), device rows are pitched (P elements).  A 2-D DMA copy with ~1 KB
// rows runs at a fraction of PCIe speed (measured 12 GB/s D2H), so the pipeline moves packed buffers with
// plain 1-D copies and converts on the device.  kToPitched: packed -> pitched (pad columns zeroed).
template <typename T, bool kToPitched>
__global__ void k_repitch(const T *__restrict__ src, T *__restrict__ dst, size_t rows, int width, int P) {
  const size_t total = rows * (size_t)(kToPitched ? P : width);
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    if (kToPitched) {
      const size_t r = idx / P;
      const int c = (int)(idx % P);
      dst[idx] = c < width ? src[r * width + c] : (T)0;
    } else {
      const size_t r = idx / width;
      const int c = (int)(idx % width);
      dst[idx] = src[r * (size_t)P + c];
    }
  }
}

int launch_repitch(ntru_ctx *ctx, const void *src, void *dst, size_t rows, int width, int elem, bool to_pitched) {
  if (rows == 0) return NTRU_OK;
  const size_t total = rows * (size_t)(to_pitched ? ctx->P : width);
  size_t blocks = (total + 255) / 256;
  const size_t cap = (size_t)ctx->sm_count * 16;
  if (blocks > cap) blocks = cap;
  {
    LaunchTimer timer(ctx, NTRU_K_OTHER);
    if (elem == 2) {
      if (to_pitched) k_repitch<uint16_t, true><<<(unsigned)blocks, 256, 0, ctx->stream>>>((const uint16_t *)src, (uint16_t *)dst, rows, width, ctx->P);
      else k_repitch<uint16_t, false><<<(unsigned)blocks, 256, 0, ctx->stream>>>((const uint16_t *)src, (uint16_t *)dst, rows, width, ctx->P);
    } else {
      if (to_pitched) k_repitch<uint8_t, true><<<(unsigned)blocks, 256, 0, ctx->stream>>>((const uint8_t *)src, (uint8_t *)dst, rows, width, ctx->P);
      else k_repitch<uint8_t, false><<<(unsigned)blocks, 256, 0, ctx->stream>>>((const uint8_t *)src, (uint8_t *)dst, rows, width, ctx->P);
    }
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

int launch_pack_fields(ntru_ctx *ctx, size_t B, const void *data, int elem_bytes, int data_len, size_t pitch, int bits, int n,
                       int out_elems, uint32_t *out) {
  if (B == 0) return NTRU_OK;
  const size_t total = B * (size_t)out_elems * 8;
  size_t blocks = (total + 255) / 256;
  const size_t cap = (size_t)ctx->sm_count * 16;
  if (blocks > cap) blocks = cap;
  {
    LaunchTimer timer(ctx, NTRU_K_PACK);
    if (elem_bytes == 2)
      k_pack_fields<uint16_t><<<(unsigned)blocks, 256, 0, ctx->stream>>>((const uint16_t *)data, B, data_len, pitch, bits, n, out_elems, out);
    else
      k_pack_fields<uint8_t><<<(unsigned)blocks, 256, 0, ctx->stream>>>((const uint8_t *)data, B, data_len, pitch, bits, n, out_elems, out);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

int launch_unpack_fields(ntru_ctx *ctx, size_t B, const uint32_t *data, int in_elems, int bits, int n, size_t pitch, void *out,
                         int elem_bytes) {
  if (B == 0) return NTRU_OK;
  const size_t total = B * (size_t)in_elems * n;
  size_t blocks = (total + 255) / 256;
  const size_t cap = (size_t)ctx->sm_count * 16;
  if (blocks > cap) blocks = cap;
  {
    LaunchTimer timer(ctx, NTRU_K_PACK);
    if (elem_bytes == 2)
      k_unpack_fields<uint16_t><<<(unsigned)blocks, 256, 0, ctx->stream>>>(data, B, in_elems, bits, n, pitch, (uint16_t *)out);
    else
      k_unpack_fields<uint8_t><<<(unsigned)blocks, 256, 0, ctx->stream>>>(data, B, in_elems, bits, n, pitch, (uint8_t *)out);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

static int block_threads(int NB) { return ((NB + 31) / 32) * 32; }

int launch_encrypt_generic(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t h_stride, const uint8_t *r,
                           const void *m, int m_wide, uint16_t *value, uint16_t *quo, uint16_t *rem) {
  if (B == 0) return NTRU_OK;
  EncArgs a;
  a.N = ctx->N; a.P = ctx->P; a.NB = (ctx->N + 1 + T - 1) / T;
  a.qmask = (uint32_t)ctx->q - 1; a.B = B; a.h = h; a.h_stride = h_stride; a.r = r; a.m = m;
  a.value = value; a.quo = quo; a.rem = rem;
  const int threads = block_threads(a.NB);
  const size_t smem = (size_t)24 * a.NB * sizeof(float);
  const size_t cap = (size_t)ctx->sm_count * 16;
  const unsigned grid = (unsigned)(B < cap ? B : cap);
  {
    LaunchTimer timer(ctx, NTRU_K_ENC_CORE);
    if (m_wide)
      k_encrypt_generic<true><<<grid, threads, smem, ctx->stream>>>(a);
    else
      k_encrypt_generic<false><<<grid, threads, smem, ctx->stream>>>(a);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

int launch_decrypt_generic(ntru_ctx *ctx, size_t B, const int8_t *f, const uint8_t *fp, size_t key_stride,
                           const uint16_t *e, uint8_t *value, uint16_t *q1, uint16_t *r1, uint8_t *q2,
                           uint8_t *r2) {
  if (B == 0) return NTRU_OK;
  DecArgs a;
  a.N = ctx->N; a.P = ctx->P; a.NB = (ctx->N + 1 + T - 1) / T; a.q = ctx->q;
  a.qmask = (uint32_t)ctx->q - 1; a.B = B; a.f = f; a.fp = fp; a.key_stride = key_stride; a.e = e;
  a.value = value; a.q1 = q1; a.r1 = r1; a.q2 = q2; a.r2 = r2;
  const int threads = block_threads(a.NB);
  const size_t smem = (size_t)24 * a.NB * sizeof(float);
  const size_t cap = (size_t)ctx->sm_count * 16;
  const unsigned grid = (unsigned)(B < cap ? B : cap);
  {
    LaunchTimer timer(ctx, NTRU_K_DEC_CORE);
    k_decrypt_generic<<<grid, threads, smem, ctx->stream>>>(a);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

// launch geometry of the sum kernels + their tree scratch (rows, group rows, tickets; zeroed once, the kernels leave
// the tickets at zero)
static int sum_geometry(ntru_ctx *ctx, size_t B, dim3 &block, size_t &smem, unsigned &blocks, SumScratch &sc) {
  const int VX = ctx->P / 8;
  const int RY = VX * kSumRows <= 512 ? kSumRows : 512 / VX;
  block = dim3(VX, RY);
  smem = (size_t)VX * RY * 8 * sizeof(uint32_t);
  size_t nb = (B + RY - 1) / RY;
  const size_t cap = (size_t)ctx->sm_count * 4;
  if (nb > cap) nb = cap;
  if (nb == 0) nb = 1;                                           // an empty shard still takes part in the exchange
  blocks = (unsigned)nb;
  const size_t max_groups = (cap + kSumGroup - 1) / kSumGroup;
  const size_t words = (cap + max_groups) * (size_t)ctx->P + max_groups + 1;
  if (ctx->d_sum_scratch.bytes < words * 4) {
    NTRU_CUDA(ctx, ctx->d_sum_scratch.reserve(words * 4));
    NTRU_CUDA(ctx, cudaMemsetAsync(ctx->d_sum_scratch.ptr, 0, words * 4, ctx->stream));
  }
  sc.rows = (uint32_t *)ctx->d_sum_scratch.ptr;
  sc.grows = sc.rows + cap * (size_t)ctx->P;
  sc.tickets = sc.grows + max_groups * (size_t)ctx->P;
  return NTRU_OK;
}

int launch_sum_partial(ntru_ctx *ctx, size_t B, const uint16_t *e, uint32_t *partial) {
  if (B == 0) return NTRU_OK;
  dim3 block;
  size_t smem;
  unsigned blocks;
  SumScratch sc;
  int rc = sum_geometry(ctx, B, block, smem, blocks, sc);
  if (rc) return rc;
  {
    LaunchTimer timer(ctx, NTRU_K_SUM);
    k_sum_partial<<<blocks, block, smem, ctx->stream>>>(e, B, ctx->P, sc, partial);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

// window of one rank: slots[2][world][P], flags[world], error word
size_t xchg_window_bytes(const ntru_ctx *ctx, int world) {
  return ((size_t)2 * world * ctx->P + world + 1) * sizeof(uint32_t);
}

int launch_sum_allreduce(ntru_ctx *ctx, size_t B, const uint16_t *e, uint16_t *out) {
  const int world = ctx->xchg_world, rank = ctx->xchg_rank;
  XchgPeers peers = {};
  for (int r = 0; r < world; ++r) peers.window[r] = (uint32_t *)ctx->peer_window[r];
  const uint32_t epoch = ++ctx->xchg_epoch;
  dim3 block;
  size_t smem;
  unsigned blocks;
  SumScratch sc;
  int rc = sum_geometry(ctx, B, block, smem, blocks, sc);
  if (rc) return rc;
  {
    LaunchTimer timer(ctx, NTRU_K_SUM);
    k_sum_push<<<blocks, block, smem, ctx->stream>>>(e, B, ctx->P, sc, peers, world, rank, epoch, (uint32_t)ctx->q - 1, ctx->N, out);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

int launch_xchg_partial(ntru_ctx *ctx, uint32_t *partial, uint16_t *out) {
  const int world = ctx->xchg_world, rank = ctx->xchg_rank;
  XchgPeers peers = {};
  for (int r = 0; r < world; ++r) peers.window[r] = (uint32_t *)ctx->peer_window[r];
  const uint32_t epoch = ++ctx->xchg_epoch;
  {
    LaunchTimer timer(ctx, NTRU_K_SUM);
    k_xchg_partial<<<1, 512, 0, ctx->stream>>>(partial, ctx->P, peers, world, rank, epoch, (uint32_t)ctx->q - 1, ctx->N, out);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

int launch_sum_finalize(ntru_ctx *ctx, const uint32_t *partial, uint16_t *out) {
  {
    LaunchTimer timer(ctx, NTRU_K_OTHER);
    k_sum_finalize<<<(ctx->P + 255) / 256, 256, 0, ctx->stream>>>(partial, ctx->N, ctx->P, (uint32_t)ctx->q - 1, out);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

int launch_sample(ntru_ctx *ctx, size_t B, int ones, int neg_ones, uint8_t neg_code, uint64_t row0, const uint8_t *skip,
                  uint8_t *r) {
  if (B == 0) return NTRU_OK;
  const size_t smem = (size_t)kSampleRows * (ctx->P + 4);
  if (!ctx->sampler_attr_set) {
    NTRU_CUDA(ctx, cudaFuncSetAttribute(k_sample_ternary, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    ctx->sampler_attr_set = true;
  }
  ChaChaKey key;
  for (int i = 0; i < 8; ++i) key.k[i] = ctx->rng_key[i];
  const size_t blocks = (B + kSampleRows - 1) / kSampleRows;
  {
    LaunchTimer timer(ctx, NTRU_K_OTHER);
    k_sample_ternary<<<(unsigned)blocks, kSampleRows, smem, ctx->stream>>>(ctx->N, ctx->P, ones, neg_ones, neg_code, key, row0,
                                                                            B, skip, r);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

}  // namespace ntru
