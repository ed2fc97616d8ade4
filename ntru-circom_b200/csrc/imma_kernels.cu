// Register-fragment tensor schedule (mma.sync.m16n8k32, SASS IMMA.16832): ONE WARP PER CIPHERTEXT.
//
// Used for distinct-key batches: every row brings its own h (or f and fp), so nothing is shared between
// ciphertexts and the 128-row operand tiles of tcgen05 do not apply.  The per-ciphertext linear product
// c = lin(x, y) (multiplyPolynomials, index.js:319-355), x = the small polynomial (r, f or b; one byte), y = h, e
// (two byte limbs) or fp, is cut into 16 x 16 Toeplitz blocks and evaluated as a small GEMM on the warp-level
// tensor path (measured 570 TMAC/s on B200, scripts/imma_peak.cu; the fp32 FMA schedule it replaces ran at 17):
//
//     k = 16 K1 + k0,  i = 16 i1 + i0,  t = K1 - i1:      c[k] = sum_{t, i0} y[16 t + k0 - i0] * x[16 (K1 - t) + i0]
//     D[k0][K1] = sum_{(t,i0)} A[k0][(t,i0)] * B[(t,i0)][K1]      A = Toeplitz(y) (16 rows),  B = Hankel blocks of x
//
// One mma.sync covers 16 outputs k0 x 8 blocks K1 x 32 positions (two t values).  The A fragment of a K step is
// the same for every column block: 9 consecutive bytes of the REVERSED y limb array per lane (three aligned LDS.32 +
// funnel shifts).  The B fragment is one aligned LDS.64 of the zero-padded x array per (column block, step).  Blocks
// with K1 - t outside [0, ceil(N/16)) are all zero and skipped: 1.2 N^2 executed MACs per limb product (137 IMMAs at N = 677).
// Index maps (chosen so that every shared-memory access is aligned and the accumulator pairs pack into words):
//     row m = g + 8 rh  <->  k0 = 2 g + rh          (g = lane / 4, t' = lane % 4)
//     K slot (hf, t', j) <-> t = 2 s + (t' >> 1),  i0 = 8 (t' & 1) + 4 hf + j
//     column n = g       <->  K1 = 8 jn + g
// The full linear product (2N - 1 coefficients, mod 2^16) goes to a per-warp shared buffer; the output pass reads
// lo[k] = c[k] and hi[k] = c[k + N] and applies the closed form of dividePolynomials(., 1 - x^N, .)
// (index.js:358-401; SURVEY.md section 8a): remainder = lo + hi, quotient = -hi, then the message add (encrypt) or
// the reference's lift (index.js:117) and the second product (decrypt).  All global accesses are 16-byte vectors
// of the packed uint16 / byte rows.
//
// One product routine, conv_band, in two forms.  MERGE (encrypt, decrypt: q <= 8192, small multiplier) accumulates both
// limbs of y in one accumulator set; it is written to the instruction-issue bound described above it.  Without MERGE
// (k_muldiv_imma: verifyKeysInputs and the key generation, where y may be any uint16) each limb has its accumulator set.

#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "ntru_internal.cuh"

namespace ntru {

namespace {

constexpr int kImmaWarps = 4;      // warps (= ciphertexts in flight) per CTA
constexpr int kXPad = 112;         // zero bytes in front of x: block index K1 - t reaches -7

__device__ __forceinline__ void imma_u8s8(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void imma_u8u8(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t mod3_16(uint32_t v) {   // two instructions: floor(v / 3) = umulhi(v, (2^32 + 2) / 3) for v < 2^31
  return v - 3u * __umulhi(v, 0x55555556u);
}

// residue mod 3 of a product coefficient c in (-2N, 4N) (x may hold -1) from its 16-bit word w = c mod 65536:
// 65536 = 1 (mod 3), so the representative c + 65536 of a negative c is 1 too high, and adding 2 removes that
__device__ __forceinline__ uint32_t mod3_prod16(uint32_t w) { return mod3_16(w + (w >> 15) * 2u); }

// Column blocks visited per K step: jn = (s >> 2) + d, d = 0 .. kDMax.  Some K1 - t of block (jn, s) lies in [0, I1)
// iff  s >> 2 <= jn <= (2 s + I1) >> 3; with I1 <= 4 NJ that is d <= (6 + 4 NJ) >> 3.  The few visited blocks outside
// the exact range multiply zero padding (about 10 % extra MMAs) and buy a loop body without branches.
template <int NJ> struct ImmaShape {
  static constexpr int kDMax = (6 + 4 * NJ) >> 3;
  static constexpr int kSGroups = (2 * NJ + 1 + 3) / 4;     // S <= 2 NJ + 1 K steps, four per group
  // resident CTAs (of four warps) per SM the encrypt / decrypt kernels are compiled for.  Two warps per scheduler
  // already reach the issue-bound rate (conv_merged); three leave the compiler 168 registers and nothing spills
  // (at five or six it spills 50 - 150 words and every variant measured slower, profiles/r2_imma_merged.txt).
#ifndef NTRU_IMMA_SGC
#define NTRU_IMMA_SGC 2
#endif
#ifndef NTRU_IMMA_MINB
#define NTRU_IMMA_MINB 3
#endif
  static constexpr int kMinBlocks = NJ <= 3 ? 8 : NTRU_IMMA_MINB;
  static constexpr int kSgChunk = NTRU_IMMA_SGC < kSGroups ? NTRU_IMMA_SGC : kSGroups;
};

// The encrypt / decrypt form of the product (round 2): ONE accumulator set for both limbs of y, every operand fragment
// read from shared memory once, no run-time condition inside the product.
//  * What the kernels are bound by (scripts/imma_pattern_probe.cu, profiles/r2_imma_pattern_probe.txt and the
//    occupancy sweep in profiles/r2_imma_merged.txt): a scheduler spends 8.4 cycles per IMMA.16832 and about one more
//    cycle for every other instruction of its warps -- cycles per ciphertext and scheduler = 8.4 IMMAs + the rest, reached
//    with two warps per scheduler and unchanged by a third or fourth.  The tensor pipe never waits for a free warp, it
//    waits while the issue port handles loads, shifts and address arithmetic.  So every instruction next to the MMAs
//    counts like an eighth of an MMA, and the whole kernel is written to that rule.
//  * y = y0 + 256 y1 with y1 < 64 (q <= 8192, ntru_create).  The staged high limb is 4 y1 and its multiplier 64 x
//    (x in {-1, 0, 1} signed or {0, 1, 2} unsigned: |64 x| fits the byte), so  y0 x + (4 y1)(64 x) = y x  lands in the
//    same int32 accumulator: 4 NJ accumulator registers instead of 8 NJ and half the accumulator traffic afterwards.
//    64 x is a second staged array (x6), not a shift next to the MMAs.
//  * Loop order (s4) -> A fragments of a group of steps -> (d) -> one B fragment per limb -> (sg): the B fragment of
//    (column block sg + d, step 4 sg + s4) does not depend on sg.
//  * I1X = ceil(N / 16) as a template argument for the BASELINE parameter sets: blocks whose K1 - t lies outside [0, I1)
//    -- d > (2 s4 + I1) >> 3 -- and steps beyond S are dropped at compile time (a warp-uniform run-time branch around
//    an mma.sync costs a WARPSYNC and a BRA per instruction).  I1X = 0, any N of the bucket: every (step, block) of the
//    bucket runs; the limb arrays are zero below their first coefficient as far as the last step of the bucket reads
//    (make_layout), the x arrays are zero outside [0, N).
//  * MERGE = false (k_muldiv_imma: y may be any uint16, its high limb does not fit a quarter of a byte): one accumulator
//    set per limb, both limbs multiply the same B fragment, the limbs are recombined when the product is stored.
template <int NJ, int LIMBS, bool MERGE, bool XU8, int I1X>
__device__ __forceinline__ void conv_band(int Z, const uint8_t *y0, const uint8_t *y1, const uint8_t *x0, const uint8_t *x6, int lane,
                                          int (&acc)[NJ][MERGE ? 1 : LIMBS][4]) {
  constexpr int NACC = MERGE ? 1 : LIMBS;
  constexpr int SG = ImmaShape<NJ>::kSGroups, DM = ImmaShape<NJ>::kDMax, SGC = ImmaShape<NJ>::kSgChunk;
  const int g = lane >> 2, tq = lane & 3;
#pragma unroll
  for (int jn = 0; jn < NJ; ++jn)
#pragma unroll
    for (int l = 0; l < NACC; ++l) acc[jn][l][0] = acc[jn][l][1] = acc[jn][l][2] = acc[jn][l][3] = 0;
  // A fragment: bytes z0-1 .. z0+7 of the reversed array, z0 = Z - 32 s - 16 (t'>>1) - 2 g + 8 (t'&1):
  // a1 = [z0-1, z0+3)  a0 = [z0, z0+4)  a3 = [z0+3, z0+7)  a2 = [z0+4, z0+8)
  const int zfirst = Z - 16 * (tq >> 1) - 2 * g + 8 * (tq & 1) - 1;
  const int zb = zfirst & ~3;
  const uint32_t sh0 = 8u * (uint32_t)(zfirst - zb), sh1 = sh0 + 8u;
  const uint8_t *pa0 = y0 + zb, *pa1 = y1 + zb;
  const int boff = 16 * (g - (tq >> 1)) + 8 * (tq & 1);
  const uint8_t *pb0 = x0 + boff, *pb1 = x6 + boff;
#pragma unroll
  for (int s4 = 0; s4 < 4; ++s4) {
    const int dlim = I1X ? (2 * s4 + I1X) >> 3 : DM;
    const int nsg = I1X ? (I1X / 2 + 1 - s4 + 3) >> 2 : SG;      // step groups with 4 sg + s4 < S = I1 / 2 + 1
#pragma unroll
    for (int c0 = 0; c0 < SG; c0 += SGC) {                // SGC step groups at a time: 4 SGC LIMBS A-fragment registers
      if (c0 < nsg) {
        uint32_t a[LIMBS][SGC][4];
#pragma unroll
        for (int l = 0; l < LIMBS; ++l) {
#pragma unroll
          for (int i = 0; i < SGC; ++i) {
            const int sg = c0 + i;
            if (sg < SG && sg < nsg) {
              const uint32_t *w = reinterpret_cast<const uint32_t *>((l ? pa1 : pa0) - 32 * (4 * sg + s4));
              const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
              a[l][i][0] = __funnelshift_rc(w0, w1, sh1);
              a[l][i][1] = __funnelshift_r(w0, w1, sh0);
              a[l][i][2] = __funnelshift_rc(w1, w2, sh1);
              a[l][i][3] = __funnelshift_r(w1, w2, sh0);
            }
          }
        }
#pragma unroll
        for (int d = 0; d <= DM; ++d) {
          if (d <= dlim && c0 + d < NJ) {
            uint2 b[LIMBS];
#pragma unroll
            for (int l = 0; l < LIMBS; ++l)
              b[l] = (l && !MERGE) ? b[0] : *reinterpret_cast<const uint2 *>((l ? pb1 : pb0) + 128 * d - 32 * s4);
#pragma unroll
            for (int i = 0; i < SGC; ++i) {
              const int sg = c0 + i;
              if (sg < SG && sg + d < NJ && sg < nsg) {
#pragma unroll
                for (int l = 0; l < LIMBS; ++l) {
                  if (XU8) imma_u8u8(acc[sg + d][MERGE ? 0 : l], a[l][i], b[l].x, b[l].y);
                  else imma_u8s8(acc[sg + d][MERGE ? 0 : l], a[l][i], b[l].x, b[l].y);
                }
              }
            }
          }
        }
      }
    }
  }
}

// accumulators -> product buffer: cbuf[k] = c[k] mod 2^16, k = 16 (8 jn + 2 t' + {0,1}) + 2 g + {0,1};
// NACC = 2: one accumulator set per limb of y, c = c0 + 256 c1
template <int NJ, int NACC>
__device__ __forceinline__ void store_product(int nj, int lane, const int (&acc)[NJ][NACC][4], uint16_t *cbuf) {
  const int g = lane >> 2, tq = lane & 3;
  uint32_t *dst = reinterpret_cast<uint32_t *>(cbuf) + 16 * tq + g;      // u16 index 32 t' + 2 g
#pragma unroll
  for (int jn = 0; jn < NJ; ++jn) {
    if (jn < nj) {
      uint32_t v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = (uint32_t)acc[jn][0][i] + (NACC == 2 ? (uint32_t)acc[jn][NACC - 1][i] << 8 : 0u);
      dst[64 * jn] = __byte_perm(v[0], v[2], 0x5410);          // (K1 = 8 jn + 2 t'    ; k0 = 2 g, 2 g + 1)
      dst[64 * jn + 8] = __byte_perm(v[1], v[3], 0x5410);      // (K1 = 8 jn + 2 t' + 1; k0 = 2 g, 2 g + 1)
    }
  }
}

// ---- encrypt / decrypt: shared-memory layout of one ciphertext (one warp) --------------------------------------------
// [y0 | y1 | (y2) | x6 | (xb) | cbuf | in[0] | in[1]]
//   y0, y1  reversed limb arrays of h (encrypt) or e (decrypt); y2 reversed fp (decrypt)
//   x6      64 x behind kXPad zero bytes (x = r or f); xb the lifted polynomial b of decrypt, same shape
//   cbuf    the 2N - 1 product coefficients mod 2^16
//   in[2]   the row's inputs as cp.async delivers them, double buffered, in_bytes each; in_bytes = 0: the encrypt / decrypt
//           form [kXPad zeros | x : P | zeros up to Lx] [y : 2P] [m or fp : P], laid out so that the B fragments of the
//           low limb are read from the x part in place
struct ImmaLayout {
  int N, P, I1, S, NJ, Z, Ly, Lx, Lc, Lin;
  int o_y1, o_y2, o_x6, o_xb, o_c, o_in, warp_bytes;
};

__host__ __device__ constexpr ImmaLayout make_layout(int N, int nj_bucket, bool exact, bool dec, int in_bytes) {
  ImmaLayout L{};
  L.N = N;
  L.P = ((N + 1 + 15) / 16) * 16;
  L.I1 = (N + 15) / 16;
  L.S = ((N + 14) / 16) / 2 + 1;
  L.NJ = ((2 * N - 1 + 15) / 16 + 7) / 8;
  // exact: the kernel is instantiated for this N, the limb arrays end at the last step that is run; otherwise they are
  // zero-padded down to the last step of the bucket
  const int s_alloc = exact ? L.S : 4 * ((2 * nj_bucket + 1 + 3) / 4);
  L.Z = 32 * s_alloc + 15;
  L.Ly = 32 * s_alloc + 48;
  // x is read at block indices K1 - t in [-7, 8 kDMax + 7]
  const int dmax = (6 + 4 * nj_bucket) >> 3;
  L.Lx = kXPad + (128 * (dmax + 1) > L.P ? 128 * (dmax + 1) : L.P);
  L.Lc = 2 * (128 * L.NJ + 32);
  L.Lin = in_bytes ? in_bytes : L.Lx + 3 * L.P;
  int o = L.Ly;
  L.o_y1 = o; o += L.Ly;
  L.o_y2 = o; if (dec) o += L.Ly;
  L.o_x6 = o; o += L.Lx;
  L.o_xb = o; if (dec) o += L.Lx;
  L.o_c = o; o += L.Lc;
  L.o_in = o; o += 2 * L.Lin;
  L.warp_bytes = o;
  return L;
}

// u16 coefficients -> reversed byte-limb arrays: y0[Z - j] = y[j] & 255 and, MERGE (the coefficients are reduced mod q
// first): y1[Z - j] = 4 (y[j] >> 8), otherwise y1[Z - j] = y[j] >> 8
template <int LIMBS, bool MERGE>
__device__ __forceinline__ void stage_limbs(int N, int Z, uint32_t Q2, const uint8_t *src, uint8_t *y0, uint8_t *y1, int lane) {
#pragma unroll 4
  for (int j0 = 8 * lane; j0 < N; j0 += 256) {
    uint4 v = *reinterpret_cast<const uint4 *>(src + 2 * j0);
    if (MERGE) v = make_uint4(v.x & Q2, v.y & Q2, v.z & Q2, v.w & Q2);
    const int z = Z - j0 - 7;                                  // multiple of 8
    *reinterpret_cast<uint2 *>(y0 + z) = make_uint2(__byte_perm(v.w, v.z, 0x4602), __byte_perm(v.y, v.x, 0x4602));
    if (LIMBS == 2) {
      uint2 hi = make_uint2(__byte_perm(v.w, v.z, 0x5713), __byte_perm(v.y, v.x, 0x5713));
      if (MERGE) hi = make_uint2(hi.x << 2, hi.y << 2);        // every high byte < 64: the shift carries nothing into the next byte
      *reinterpret_cast<uint2 *>(y1 + z) = hi;
    }
  }
}

// bytes -> reversed array; MOD3: every byte reduced modulo 3 on the way.  The copy is unrolled twice; the mod-3 form,
// four times the instructions per step, is not unrolled (the compiler's choice for it before the two were merged,
// pinned here so that either form keeps its code)
template <bool MOD3>
__device__ __forceinline__ void stage_rev8(int N, int Z, const uint8_t *src, uint8_t *y, int lane) {
#pragma unroll (MOD3 ? 1 : 2)
  for (int j0 = 16 * lane; j0 < N; j0 += 512) {
    const uint4 v = *reinterpret_cast<const uint4 *>(src + j0);
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
    if (MOD3) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint32_t o = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) o |= mod3_16((w[i] >> (8 * b)) & 0xffu) << (8 * b);
        w[i] = o;
      }
    }
    *reinterpret_cast<uint4 *>(y + (Z - j0 - 15)) =
        make_uint4(__byte_perm(w[3], 0u, 0x0123), __byte_perm(w[2], 0u, 0x0123), __byte_perm(w[1], 0u, 0x0123), __byte_perm(w[0], 0u, 0x0123));
  }
}

// x6 = 64 x per byte (x in {0, 1, 2} or {-1, 0, 1}: only the two low bits of a byte matter)
__device__ __forceinline__ void stage_x6(int N, const uint8_t *x, uint8_t *x6, int lane) {
#pragma unroll 2
  for (int j0 = 16 * lane; j0 < N; j0 += 512) {
    const uint4 v = *reinterpret_cast<const uint4 *>(x + j0);
    *reinterpret_cast<uint4 *>(x6 + j0) =
        make_uint4((v.x << 6) & 0xC0C0C0C0u, (v.y << 6) & 0xC0C0C0C0u, (v.z << 6) & 0xC0C0C0C0u, (v.w << 6) & 0xC0C0C0C0u);
  }
}

// lo = c[k0 .. k0+8), hi = c[k0+N .. k0+N+8) as packed uint16 pairs
__device__ __forceinline__ void load_lo_hi2(int N, const uint16_t *cbuf, int k0, uint32_t (&lo)[4], uint32_t (&hi)[4]) {
  const uint4 l = *reinterpret_cast<const uint4 *>(cbuf + k0);
  lo[0] = l.x; lo[1] = l.y; lo[2] = l.z; lo[3] = l.w;
  const int kh = k0 + N;
  const uint32_t *w = reinterpret_cast<const uint32_t *>(cbuf + (kh & ~1));
  if (N & 1) {
    uint32_t x[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) x[i] = w[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) hi[i] = __byte_perm(x[i], x[i + 1], 0x5432);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) hi[i] = w[i];
  }
}

// residues mod 3 of both 16-bit lanes of v (each lane < 2^14), the lanes stay packed: floor(x / 3) = (x * 0x5556) >> 16 below
// 26 000, and the low lane adds less than 2^-4 to the high lane's quotient before the floor.  Five instructions for two
// coefficients.
__device__ __forceinline__ uint32_t mod3_2x16(uint32_t v) {
  const uint32_t qh = __umulhi(v, 0x5556u), ql = __umulhi(v << 16, 0x5556u);
  return v - 3u * (ql + (qh << 16));
}

// keeps the first n (of 4) bytes of a word, n any integer
__device__ __forceinline__ uint32_t keep_bytes(uint32_t v, int n) {
  return n >= 4 ? v : (n <= 0 ? 0u : v & (0xffffffffu >> (32 - 8 * n)));
}

__device__ __forceinline__ void prefetch_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void prefetch_wait() {
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncwarp();
}

// one array of a row by cp.async: `bytes` (multiple of 16), 16 per lane and step; dst and src already point at the lane's
// first 16 bytes.  BX != 0: the byte count as a compile-time constant (no loop, no address arithmetic).
template <int BX>
__device__ __forceinline__ void prefetch_lane(uint32_t dst, const char *src, int bytes, int lane) {
  if (BX) {
#pragma unroll
    for (int o = 0; o < BX; o += 512)
      if (o + 512 <= BX || o + 16 * lane < BX)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + o), "l"(src + o) : "memory");
  } else {
    for (int o = 0; o + 16 * lane < bytes; o += 512)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + o), "l"(src + o) : "memory");
  }
}

// division by 1 - x^N modulo q (Q2 = q - 1 in both lanes) of 8 packed coefficients: remainder lo + hi, quotient -hi
__device__ __forceinline__ void div_xn_q(uint32_t Q2, const uint32_t (&lo)[4], const uint32_t (&hi)[4], uint32_t (&rem)[4],
                                         uint32_t (&quo)[4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    rem[i] = __vadd2(lo[i], hi[i]) & Q2;
    quo[i] = __vsub2(0u, hi[i]) & Q2;
  }
}

// zeroes the packed uint16 lanes k0 + i >= N of an 8-coefficient vector (branch-free)
__device__ __forceinline__ void mask_tail(uint32_t (&v)[4], int nv) {
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] &= (2 * i < nv ? 0xffffu : 0u) | (2 * i + 1 < nv ? 0xffff0000u : 0u);
}

struct ImmaEncArgs {
  ImmaLayout L;
  uint32_t qmask;
  size_t B;
  const uint16_t *h;
  size_t h_stride;
  const uint8_t *r;
  const uint8_t *m;
  uint16_t *value, *quo, *rem;
};

#define NTRU_LF(f) (NX ? LX.f : a.L.f)

template <int NJ, int LIMBS, int NX>
__global__ void __launch_bounds__(kImmaWarps * 32, ImmaShape<NJ>::kMinBlocks) k_encrypt_imma(const ImmaEncArgs a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  constexpr ImmaLayout LX = make_layout(NX ? NX : 16, NJ, true, false, 0);
  constexpr int I1X = NX ? (NX + 15) / 16 : 0;
  const int N = NTRU_LF(N), P = NTRU_LF(P), Z = NTRU_LF(Z), Lx = NTRU_LF(Lx), Lin = NTRU_LF(Lin);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t *base = smem_raw + (size_t)warp * NTRU_LF(warp_bytes);
  uint8_t *y0 = base, *y1 = base + NTRU_LF(o_y1), *x6 = base + NTRU_LF(o_x6);
  uint16_t *cbuf = reinterpret_cast<uint16_t *>(base + NTRU_LF(o_c));
  uint8_t *in0 = base + NTRU_LF(o_in);
  for (int i = lane * 16; i < NTRU_LF(warp_bytes); i += 512) *reinterpret_cast<uint4 *>(base + i) = make_uint4(0, 0, 0, 0);
  __syncwarp();
  const uint32_t Q2 = a.qmask | (a.qmask << 16);
  const size_t nwarps = (size_t)gridDim.x * kImmaWarps;
  constexpr int PX = NX ? LX.P : 0;
  const uint32_t in_lane = (uint32_t)__cvta_generic_to_shared(in0) + 16 * lane;
  auto prefetch = [&](size_t row, int buf) {     // source addresses from the kernel arguments each time: no registers held across the products
    const uint32_t d = in_lane + buf * Lin;
    const size_t o = row * (size_t)P + 16 * lane;
    prefetch_lane<PX>(d + kXPad, reinterpret_cast<const char *>(a.r) + o, P, lane);
    prefetch_lane<2 * PX>(d + Lx, reinterpret_cast<const char *>(a.h) + (row * a.h_stride * 2 + 16 * lane), 2 * P, lane);
    prefetch_lane<PX>(d + Lx + 2 * P, reinterpret_cast<const char *>(a.m) + o, P, lane);
    prefetch_commit();
  };
  size_t row = (size_t)blockIdx.x * kImmaWarps + warp;
  if (row < a.B) prefetch(row, 0);
  int cur = 0;
  for (; row < a.B; row += nwarps, cur ^= 1) {
    uint8_t *in = in0 + cur * Lin;
    uint8_t *xr = in + kXPad, *hr = in + Lx, *mr = in + Lx + 2 * P;
    prefetch_wait();
    if (lane < P - N) {        // the caller's pad columns may hold anything
      xr[N + lane] = 0;
      reinterpret_cast<uint16_t *>(hr)[N + lane] = 0;
    }
    __syncwarp();
    stage_limbs<LIMBS, true>(N, Z, Q2, hr, y0, y1, lane);
    if (LIMBS == 2) stage_x6(N, xr, x6 + kXPad, lane);
    __syncwarp();
    if (row + nwarps < a.B) prefetch(row + nwarps, cur ^ 1);    // in flight during this row's products
    {
      int acc[NJ][1][4];
      conv_band<NJ, LIMBS, true, true, I1X>(Z, y0, y1, xr, x6 + kXPad, lane, acc);      // r in {0, 1, 2}: unsigned multiplier
      store_product<NJ, 1>(NTRU_LF(NJ), lane, acc, cbuf);
    }
    __syncwarp();
    // this lane's 8 coefficients of pass 0, per output array
    const size_t rlane = row * (size_t)P + 8 * lane;
    uint16_t *const vp = a.value ? a.value + rlane : nullptr, *const rp = a.rem ? a.rem + rlane : nullptr, *const qp = a.quo ? a.quo + rlane : nullptr;
#pragma unroll
    for (int kb = 0; kb < (NX ? LX.P : 1024); kb += 256) {
      const int k0 = kb + 8 * lane;
      if (kb < P && (kb + 256 <= P || k0 < P)) {
        uint32_t lo[4], hi[4], rem[4], quo[4];
        load_lo_hi2(N, cbuf, k0, lo, hi);
        const uint2 mm = *reinterpret_cast<const uint2 *>(mr + k0);
        const uint32_t mp[4] = {__byte_perm(mm.x, 0u, 0x4140), __byte_perm(mm.x, 0u, 0x4342), __byte_perm(mm.y, 0u, 0x4140),
                                __byte_perm(mm.y, 0u, 0x4342)};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          rem[i] = __vadd2(__vadd2(lo[i], hi[i]), mp[i]) & Q2;
          quo[i] = __vsub2(0u, hi[i]) & Q2;
        }
        if (kb + 256 > N) {       // only the last pass holds columns beyond N
          mask_tail(rem, N - k0);
          mask_tail(quo, N - k0);
        }
        const uint4 rv = make_uint4(rem[0], rem[1], rem[2], rem[3]);
        if (vp) *reinterpret_cast<uint4 *>(vp + kb) = rv;
        if (rp) *reinterpret_cast<uint4 *>(rp + kb) = rv;
        if (qp) *reinterpret_cast<uint4 *>(qp + kb) = make_uint4(quo[0], quo[1], quo[2], quo[3]);
      }
    }
    __syncwarp();
  }
}

struct ImmaDecArgs {
  ImmaLayout L;
  uint32_t qmask;
  int q, logq;
  size_t B;
  const int8_t *f;
  const uint8_t *fp;
  size_t key_stride;
  const uint16_t *e;
  uint8_t *value, *q2, *r2;
  uint16_t *q1, *r1;
};

template <int NJ, int LIMBS, int NX>
__global__ void __launch_bounds__(kImmaWarps * 32, ImmaShape<NJ>::kMinBlocks) k_decrypt_imma(const ImmaDecArgs a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  constexpr ImmaLayout LX = make_layout(NX ? NX : 16, NJ, true, true, 0);
  constexpr int I1X = NX ? (NX + 15) / 16 : 0;
  const int N = NTRU_LF(N), P = NTRU_LF(P), Z = NTRU_LF(Z), Lx = NTRU_LF(Lx), Lin = NTRU_LF(Lin);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t *base = smem_raw + (size_t)warp * NTRU_LF(warp_bytes);
  uint8_t *y0 = base, *y1 = base + NTRU_LF(o_y1), *y2 = base + NTRU_LF(o_y2), *x6 = base + NTRU_LF(o_x6), *xb = base + NTRU_LF(o_xb);
  uint16_t *cbuf = reinterpret_cast<uint16_t *>(base + NTRU_LF(o_c));
  uint8_t *in0 = base + NTRU_LF(o_in);
  for (int i = lane * 16; i < NTRU_LF(warp_bytes); i += 512) *reinterpret_cast<uint4 *>(base + i) = make_uint4(0, 0, 0, 0);
  __syncwarp();
  const uint32_t Q2 = a.qmask | (a.qmask << 16);
  const uint32_t LA2 = (((uint32_t)a.q >> 1) - 1u) * 0x00010001u;       // x > q/2  <=>  bit logq of x + q/2 - 1
  const size_t nwarps = (size_t)gridDim.x * kImmaWarps;
  constexpr int PX = NX ? LX.P : 0;
  const uint32_t in_lane = (uint32_t)__cvta_generic_to_shared(in0) + 16 * lane;
  auto prefetch = [&](size_t row, int buf) {     // source addresses from the kernel arguments each time: no registers held across the products
    const uint32_t d = in_lane + buf * Lin;
    const size_t ok = row * a.key_stride + 16 * lane;
    prefetch_lane<PX>(d + kXPad, reinterpret_cast<const char *>(a.f) + ok, P, lane);
    prefetch_lane<2 * PX>(d + Lx, reinterpret_cast<const char *>(a.e) + (row * (size_t)(2 * P) + 16 * lane), 2 * P, lane);
    prefetch_lane<PX>(d + Lx + 2 * P, reinterpret_cast<const char *>(a.fp) + ok, P, lane);
    prefetch_commit();
  };
  size_t row = (size_t)blockIdx.x * kImmaWarps + warp;
  if (row < a.B) prefetch(row, 0);
  int cur = 0;
  for (; row < a.B; row += nwarps, cur ^= 1) {
    const size_t rlane = row * (size_t)P + 8 * lane;     // this lane's 8 coefficients of pass 0
    uint8_t *in = in0 + cur * Lin;
    uint8_t *fr = in + kXPad, *er = in + Lx, *fpr = in + Lx + 2 * P;
    prefetch_wait();
    if (lane < P - N) {        // the caller's pad columns may hold anything
      fr[N + lane] = 0;
      reinterpret_cast<uint16_t *>(er)[N + lane] = 0;
      fpr[N + lane] = 0;
    }
    __syncwarp();
    stage_limbs<LIMBS, true>(N, Z, Q2, er, y0, y1, lane);
    if (LIMBS == 2) stage_x6(N, fr, x6 + kXPad, lane);
    stage_rev8<false>(N, Z, fpr, y2, lane);
    __syncwarp();
    if (row + nwarps < a.B) prefetch(row + nwarps, cur ^ 1);    // in flight during this row's products
    {   // product 1: a = lin(f, e) mod q  (f in {-1, 0, 1}: signed multiplier)
      int acc[NJ][1][4];
      conv_band<NJ, LIMBS, true, false, I1X>(Z, y0, y1, fr, x6 + kXPad, lane, acc);
      store_product<NJ, 1>(NTRU_LF(NJ), lane, acc, cbuf);
    }
    __syncwarp();
    {
      uint16_t *const r1p = a.r1 ? a.r1 + rlane : nullptr, *const q1p = a.q1 ? a.q1 + rlane : nullptr;
#pragma unroll
      for (int kb = 0; kb < (NX ? LX.P : 1024); kb += 256) {
        const int k0 = kb + 8 * lane;
        if (kb < P && (kb + 256 <= P || k0 < P)) {
          uint32_t lo[4], hi[4], rem[4], quo[4];
          load_lo_hi2(N, cbuf, k0, lo, hi);
          div_xn_q(Q2, lo, hi, rem, quo);
          if (kb + 256 > N) {       // only the last pass holds columns beyond N
            mask_tail(rem, N - k0);
            mask_tail(quo, N - k0);
          }
          if (r1p) *reinterpret_cast<uint4 *>(r1p + kb) = make_uint4(rem[0], rem[1], rem[2], rem[3]);
          if (q1p) *reinterpret_cast<uint4 *>(q1p + kb) = make_uint4(quo[0], quo[1], quo[2], quo[3]);
          // b = (remainder1 + [remainder1 > q/2]) mod 3  (index.js:117), the multiplier of product 2; a masked
          // column gives 0
          uint32_t b2[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) b2[i] = mod3_2x16(rem[i] + (((rem[i] + LA2) >> a.logq) & 0x00010001u));
          *reinterpret_cast<uint2 *>(xb + kXPad + k0) = make_uint2(__byte_perm(b2[0], b2[1], 0x6420), __byte_perm(b2[2], b2[3], 0x6420));
        }
      }
    }
    __syncwarp();
    {   // product 2: c = lin(fp, b) mod 3
      int acc[NJ][1][4];
      conv_band<NJ, 1, true, false, I1X>(Z, y2, y2, xb + kXPad, xb + kXPad, lane, acc);
      store_product<NJ, 1>(NTRU_LF(NJ), lane, acc, cbuf);
    }
    __syncwarp();
    {
      uint8_t *const vp = a.value ? a.value + rlane : nullptr, *const r2p = a.r2 ? a.r2 + rlane : nullptr, *const q2p = a.q2 ? a.q2 + rlane : nullptr;
#pragma unroll
      for (int kb = 0; kb < (NX ? LX.P : 1024); kb += 256) {
        const int k0 = kb + 8 * lane;
        if (kb < P && (kb + 256 <= P || k0 < P)) {
          uint32_t lo[4], hi[4];
          load_lo_hi2(N, cbuf, k0, lo, hi);
          // remainder2 = (lo + hi) mod 3, quotient2 = -hi = 2 hi (mod 3): lo, hi <= 4 N, every sum stays below 2^14 and
          // the 16-bit lanes never carry into each other
          uint32_t r3[4], q3[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            r3[i] = mod3_2x16(lo[i] + hi[i]);
            q3[i] = mod3_2x16(hi[i] << 1);
          }
          uint2 rv = make_uint2(__byte_perm(r3[0], r3[1], 0x6420), __byte_perm(r3[2], r3[3], 0x6420));
          uint2 qv = make_uint2(__byte_perm(q3[0], q3[1], 0x6420), __byte_perm(q3[2], q3[3], 0x6420));
          if (kb + 256 > N) {       // only the last pass holds columns beyond N
            rv = make_uint2(keep_bytes(rv.x, N - k0), keep_bytes(rv.y, N - k0 - 4));
            qv = make_uint2(keep_bytes(qv.x, N - k0), keep_bytes(qv.y, N - k0 - 4));
          }
          if (vp) *reinterpret_cast<uint2 *>(vp + kb) = rv;
          if (r2p) *reinterpret_cast<uint2 *>(r2p + kb) = rv;
          if (q2p) *reinterpret_cast<uint2 *>(q2p + kb) = qv;
        }
      }
    }
    __syncwarp();
  }
}

// ---- multiplyPolynomials(a, b, mod) + dividePolynomials(., 1 - x^N, mod) for B independent pairs -----------------
// The primitive under verifyKeysInputs (index.js:141-197): (f, fq) and (g, p * fq) modulo q, (f mod p, fp) modulo p.
// x is the small operand (int8 in [-1, 2]; the witness value q-1 or p-1 of a -1 is the wrapper's concern: the
// product is the same modulo q or p), y the wide one: uint16 (any value: p * fq is NOT reduced mod q, index.js:155)
// in mod-q mode, one byte in mod-p mode.
struct ImmaMulDivArgs {
  ImmaLayout L;
  uint32_t qmask;
  size_t B;
  const int8_t *x;
  const void *y;
  void *quo, *rem;      // uint16 (mod q) or uint8 (mod p), pitch P
};

template <int NJ, bool kModP>
__global__ void __launch_bounds__(kImmaWarps * 32) k_muldiv_imma(const ImmaMulDivArgs a) {
  constexpr int LIMBS = kModP ? 1 : 2;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const ImmaLayout &L = a.L;
  const int N = L.N, P = L.P, Z = L.Z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t *base = smem_raw + (size_t)warp * L.warp_bytes;
  uint8_t *y0 = base, *y1 = base + L.o_y1;
  uint16_t *cbuf = reinterpret_cast<uint16_t *>(base + L.o_c);
  uint8_t *in0 = base + L.o_in;           // per buffer: [kXPad zeros | x : P | zeros up to Lx] [y : 2P or P]
  for (int i = lane * 16; i < L.warp_bytes; i += 512) *reinterpret_cast<uint4 *>(base + i) = make_uint4(0, 0, 0, 0);
  __syncwarp();
  const uint32_t Q2 = a.qmask | (a.qmask << 16);
  const int ybytes = kModP ? P : 2 * P;
  const size_t nwarps = (size_t)gridDim.x * kImmaWarps;
  const uint32_t in_lane = (uint32_t)__cvta_generic_to_shared(in0) + 16 * lane;
  auto prefetch = [&](size_t row, int buf) {
    const uint32_t d = in_lane + buf * L.Lin;
    prefetch_lane<0>(d + kXPad, reinterpret_cast<const char *>(a.x) + (row * (size_t)P + 16 * lane), P, lane);
    prefetch_lane<0>(d + L.Lx, reinterpret_cast<const char *>(a.y) + (row * (size_t)ybytes + 16 * lane), ybytes, lane);
    prefetch_commit();
  };
  size_t row = (size_t)blockIdx.x * kImmaWarps + warp;
  if (row < a.B) prefetch(row, 0);
  int cur = 0;
  for (; row < a.B; row += nwarps, cur ^= 1) {
    uint8_t *in = in0 + cur * L.Lin;
    uint8_t *xr = in + kXPad, *yr = in + L.Lx;
    prefetch_wait();
    if (lane < P - N) {        // the caller's pad columns may hold anything
      xr[N + lane] = 0;
      if (kModP) yr[N + lane] = 0;
      else reinterpret_cast<uint16_t *>(yr)[N + lane] = 0;
    }
    __syncwarp();
    if (kModP) stage_rev8<false>(N, Z, yr, y0, lane);
    else stage_limbs<2, false>(N, Z, Q2, yr, y0, y1, lane);
    __syncwarp();
    if (row + nwarps < a.B) prefetch(row + nwarps, cur ^ 1);
    {
      int acc[NJ][LIMBS][4];
      conv_band<NJ, LIMBS, false, false, 0>(Z, y0, y1, xr, xr, lane, acc);       // x in [-1, 2]: signed multiplier
      store_product<NJ, LIMBS>(L.NJ, lane, acc, cbuf);
    }
    __syncwarp();
    const size_t rbase = row * (size_t)P;
    for (int k0 = 8 * lane; k0 < P; k0 += 256) {
      uint32_t lo[4], hi[4];
      load_lo_hi2(N, cbuf, k0, lo, hi);
      if (kModP) {
        uint32_t rem[2] = {0, 0}, quo[2] = {0, 0};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          // x may hold -1: the 16-bit product is then c mod 65536 with c in (-2N, 4N); 65536 = 1 (mod 3), so the
          // representative c + 65536 keeps the residue up to that 1, which is removed again for negative c
          const uint32_t lw = (lo[i >> 1] >> (16 * (i & 1))) & 0xffffu, hw = (hi[i >> 1] >> (16 * (i & 1))) & 0xffffu;
          const uint32_t l3 = mod3_16(lw + (lw >> 15) * 2u);
          const uint32_t h3 = mod3_16(hw + (hw >> 15) * 2u);
          const bool valid = k0 + i < N;
          rem[i >> 2] |= (valid ? mod3_16(l3 + h3) : 0u) << (8 * (i & 3));
          quo[i >> 2] |= (valid ? mod3_16(3u - h3) : 0u) << (8 * (i & 3));
        }
        if (a.rem) *reinterpret_cast<uint2 *>(reinterpret_cast<uint8_t *>(a.rem) + rbase + k0) = make_uint2(rem[0], rem[1]);
        if (a.quo) *reinterpret_cast<uint2 *>(reinterpret_cast<uint8_t *>(a.quo) + rbase + k0) = make_uint2(quo[0], quo[1]);
      } else {
        uint32_t rem[4], quo[4];
        div_xn_q(Q2, lo, hi, rem, quo);
        mask_tail(rem, N - k0);
        mask_tail(quo, N - k0);
        if (a.rem) *reinterpret_cast<uint4 *>(reinterpret_cast<uint16_t *>(a.rem) + rbase + k0) = make_uint4(rem[0], rem[1], rem[2], rem[3]);
        if (a.quo) *reinterpret_cast<uint4 *>(reinterpret_cast<uint16_t *>(a.quo) + rbase + k0) = make_uint4(quo[0], quo[1], quo[2], quo[3]);
      }
    }
    __syncwarp();
  }
}

// ---- witness checks: VerifyEncrypt / VerifyDecrypt / VerifyInverse (circuits/ntru.circom:155-256) ------------------
// One warp per witness row, the product of k_muldiv_imma (x signed in [-1, 2], y any uint16, one accumulator set per
// limb), and an epilogue that compares instead of storing.  With a = the 2N - 1 coefficients of lin(x, y) (+ m on the
// first N for encrypt) and Q, R the N + 1 entries of the witness, the division by I = 1 - x^N modulo M holds iff
//     k < N:  Q[k] + R[k] = a[k]      k = N:  Q[N] - Q[0] + R[N] = a[N]      1 <= k <= N:  Q[k] + a[k + N] = 0
// (a[k] = 0 for k >= 2N - 1: the last two rows are Q[N-1] = Q[N] = 0).  Every operand is read as the raw witness value,
// reduced modulo M only where the constraint reduces it.  The witness is canonical -- the arrays dividePolynomials
// returns -- iff it also has every entry below M and R[N] = 0.
struct CheckArgs {
  ImmaLayout L;
  uint32_t M;               // modulus of the (first) division: q, or p for the mod-p inverse
  size_t B;
  const void *x;            // small operand in its witness form: r (bytes), f or x (uint16)
  const void *y;            // h, e (uint16), or the inverse's y (uint16; bytes modulo p)
  size_t x_stride, y_stride;   // elements between rows (0: one row for every witness)
  const uint16_t *m;        // encrypt
  const uint8_t *fp;        // decrypt (row stride x_stride)
  const void *quo, *rem;    // the (first) division's witness, uint16 (bytes for the mod-p inverse)
  const uint8_t *quo2, *rem2;   // decrypt: the second division's witness
  uint8_t *verdict;
};

// x operand, witness form -> the signed bytes the product takes: v mod M, with M - 1 as -1.  Columns >= N become 0.
// Returns false when an entry of this lane lies outside {M - 1, 0, 1, 2} (the row is not evaluated then).
template <bool U16>
__device__ __forceinline__ bool stage_small(int N, int P, uint32_t M, const uint8_t *src, uint8_t *xs, int lane) {
  bool ok = true;
  for (int j0 = 8 * lane; j0 < P; j0 += 256) {
    uint32_t w[2] = {0u, 0u};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint32_t v = U16 ? reinterpret_cast<const uint16_t *>(src)[j0 + i] : src[j0 + i];
      const uint32_t r = M == 3 ? mod3_16(v) : v & (M - 1);
      const bool valid = j0 + i < N;
      ok = ok && (!valid || r <= 2u || r == M - 1);
      const uint32_t s = r == M - 1 ? 0xffu : (r <= 2u ? r : 0u);
      w[i >> 2] |= (valid ? s : 0u) << (8 * (i & 3));
    }
    *reinterpret_cast<uint2 *>(xs + j0) = make_uint2(w[0], w[1]);
  }
  return ok;
}

// packed uint16 lanes of the 8 coefficients k0 .. k0+7 with lo_k <= k <= hi_k
__device__ __forceinline__ uint32_t lane_mask2(int k0, int i, int lo_k, int hi_k) {
  const int k = k0 + 2 * i;
  return (k >= lo_k && k <= hi_k ? 0xffffu : 0u) | (k + 1 >= lo_k && k + 1 <= hi_k ? 0xffff0000u : 0u);
}

// One pass of a division modulo M = 2^logq (uint16 witness): this lane's coefficients k0 .. k0+7.  lo, hi = product
// coefficients k and k + N; mv = m (encrypt) or 0; q0 = Q[0].  Mismatches go to bad, canonical-form violations to nonc.
__device__ __forceinline__ void check_pass_q(int N, int k0, uint32_t Q2, const uint32_t (&lo)[4], const uint32_t (&hi)[4],
                                             const uint32_t (&mv)[4], const uint32_t (&qv)[4], const uint32_t (&rv)[4],
                                             uint32_t q0, uint32_t &bad, uint32_t &nonc) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t le_n = lane_mask2(k0, i, 0, N), at_n = lane_mask2(k0, i, N, N);
    const uint32_t e1 = __vsub2(__vsub2(__vadd2(qv[i], rv[i]), __vadd2(lo[i], mv[i])), (q0 | (q0 << 16)) & at_n);
    const uint32_t e2 = __vadd2(qv[i], hi[i]) & lane_mask2(k0, i, 1, N);
    bad |= (e1 & le_n | e2) & Q2;
    nonc |= ((qv[i] | rv[i]) & ~Q2 & le_n) | (rv[i] & at_n);
  }
}

// The same modulo 3 with byte witness arrays (qb, rb: 8 bytes).  The product coefficients are 16-bit residues of
// c in (-2N, 4N), as in k_muldiv_imma.
__device__ __forceinline__ void check_pass_3(int N, int k0, const uint32_t (&lo)[4], const uint32_t (&hi)[4], uint2 qb, uint2 rb,
                                             uint32_t q0, uint32_t &bad, uint32_t &nonc) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = k0 + i;
    const uint32_t lw = (lo[i >> 1] >> (16 * (i & 1))) & 0xffffu, hw = (hi[i >> 1] >> (16 * (i & 1))) & 0xffffu;
    const uint32_t l3 = mod3_prod16(lw), h3 = mod3_prod16(hw);
    const uint32_t qk = ((i < 4 ? qb.x : qb.y) >> (8 * (i & 3))) & 0xffu, rk = ((i < 4 ? rb.x : rb.y) >> (8 * (i & 3))) & 0xffu;
    // -v = 2 v (mod 3): every term stays non-negative
    const bool e1 = mod3_16(qk + rk + 2u * l3 + (k == N ? 2u * q0 : 0u)) != 0u;
    const bool e2 = mod3_16(qk + h3) != 0u;
    bad |= (k <= N && e1) || (k >= 1 && k <= N && e2);
    nonc |= (k <= N && (qk >= 3u || rk >= 3u)) || (k == N && rk != 0u);
  }
}

__device__ __forceinline__ void load_u16x8(const void *base, size_t off, bool act, uint32_t (&v)[4]) {
  const uint4 t = act ? *reinterpret_cast<const uint4 *>(reinterpret_cast<const uint16_t *>(base) + off) : make_uint4(0, 0, 0, 0);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}

__device__ __forceinline__ uint2 load_u8x8(const void *base, size_t off, bool act) {
  return act ? *reinterpret_cast<const uint2 *>(reinterpret_cast<const uint8_t *>(base) + off) : make_uint2(0, 0);
}

// Division modulo q of the product in cbuf against the uint16 witness (quo, rem) of `row`; m (encrypt) or nullptr.
// Returns nonzero in bit 0 for a mismatch, bit 1 for a canonical-form violation (this lane's part).
// R1 (decrypt): the lift b = (R1 + [R1 > q/2]) mod 3 of the raw witness remainder1 goes to xb.
template <bool LIFT>
__device__ __forceinline__ uint32_t check_div_q(int N, int P, uint32_t qmask, const uint16_t *cbuf, const void *quo, const void *rem,
                                                const uint16_t *m, size_t row, int lane, uint8_t *xb) {
  const uint32_t Q2 = qmask | (qmask << 16);
  uint32_t bad = 0, nonc = 0, q0 = 0;
  for (int kb = 0; kb < P; kb += 256) {
    const int k0 = kb + 8 * lane;
    const bool act = k0 < P;
    const size_t off = row * (size_t)P + k0;
    uint32_t lo[4] = {0, 0, 0, 0}, hi[4] = {0, 0, 0, 0}, qv[4], rv[4], mv[4] = {0, 0, 0, 0};
    if (act) load_lo_hi2(N, cbuf, k0, lo, hi);
    load_u16x8(quo, off, act, qv);
    load_u16x8(rem, off, act, rv);
    if (m) {
      load_u16x8(m, off, act, mv);
      mask_tail(mv, N - k0);          // m's pad columns are not part of the witness
    }
    if (kb == 0) q0 = __shfl_sync(0xffffffffu, qv[0], 0) & 0xffffu;
    check_pass_q(N, k0, Q2, lo, hi, mv, qv, rv, q0, bad, nonc);
    if (LIFT && act) {
      const uint32_t half = (qmask + 1) >> 1;
      uint32_t b[2] = {0u, 0u};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t r = (rv[i >> 1] >> (16 * (i & 1))) & 0xffffu;
        b[i >> 2] |= (k0 + i < N ? mod3_16(r + (r > half ? 1u : 0u)) : 0u) << (8 * (i & 3));
      }
      *reinterpret_cast<uint2 *>(xb + k0) = make_uint2(b[0], b[1]);
    }
  }
  return (bad ? 1u : 0u) | (nonc ? 2u : 0u);
}

__device__ __forceinline__ uint32_t check_div_3(int N, int P, const uint16_t *cbuf, const void *quo, const void *rem, size_t row, int lane) {
  uint32_t bad = 0, nonc = 0, q0 = 0;
  for (int kb = 0; kb < P; kb += 256) {
    const int k0 = kb + 8 * lane;
    const bool act = k0 < P;
    const size_t off = row * (size_t)P + k0;
    uint32_t lo[4] = {0, 0, 0, 0}, hi[4] = {0, 0, 0, 0};
    if (act) load_lo_hi2(N, cbuf, k0, lo, hi);
    const uint2 qb = load_u8x8(quo, off, act), rb = load_u8x8(rem, off, act);
    if (kb == 0) q0 = __shfl_sync(0xffffffffu, qb.x, 0) & 0xffu;
    if (act) check_pass_3(N, k0, lo, hi, qb, rb, q0, bad, nonc);
  }
  return (bad ? 1u : 0u) | (nonc ? 2u : 0u);
}

// the warp's verdict byte from every lane's domain flag and check bits
__device__ __forceinline__ uint8_t check_verdict(bool domain_ok, uint32_t bits) {
  const bool in_domain = __all_sync(0xffffffffu, domain_ok);
  const bool sat = !__any_sync(0xffffffffu, bits & 1u);
  const bool canon = sat && !__any_sync(0xffffffffu, bits & 2u);
  return in_domain ? (uint8_t)((sat ? NTRU_CHECK_SATISFIED : 0) | (canon ? NTRU_CHECK_CANONICAL : 0)) : (uint8_t)NTRU_CHECK_DOMAIN;
}

// per-warp shared memory: the layout of the IMMA kernels (y0 | y1 | (y2) | xs | (xb) | cbuf), then the double-buffered
// inputs [x : x_bytes][y : y_bytes][fp : P]; xs is the re-staged x behind kXPad zero bytes (the x6 slot)
#define NTRU_CHECK_PROLOGUE                                                                                               \
  extern __shared__ __align__(16) uint8_t smem_raw[];                                                                    \
  const ImmaLayout &L = a.L;                                                                                             \
  const int N = L.N, P = L.P, Z = L.Z;                                                                                   \
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;                                                            \
  uint8_t *base = smem_raw + (size_t)warp * L.warp_bytes;                                                                \
  uint8_t *y0 = base, *y1 = base + L.o_y1, *y2 = base + L.o_y2, *xs = base + L.o_x6 + kXPad, *xb = base + L.o_xb + kXPad; \
  uint16_t *cbuf = reinterpret_cast<uint16_t *>(base + L.o_c);                                                           \
  uint8_t *in0 = base + L.o_in;                                                                                          \
  for (int i = lane * 16; i < L.warp_bytes; i += 512) *reinterpret_cast<uint4 *>(base + i) = make_uint4(0, 0, 0, 0);     \
  __syncwarp();                                                                                                          \
  const size_t nwarps = (size_t)gridDim.x * kImmaWarps;                                                                  \
  const uint32_t in_lane = (uint32_t)__cvta_generic_to_shared(in0) + 16 * lane;                                          \
  (void)y2; (void)xb

template <int NJ>
__global__ void __launch_bounds__(kImmaWarps * 32) k_check_encrypt(const CheckArgs a) {
  NTRU_CHECK_PROLOGUE;
  auto prefetch = [&](size_t row, int buf) {
    const uint32_t d = in_lane + buf * L.Lin;
    prefetch_lane<0>(d, reinterpret_cast<const char *>(a.x) + (row * a.x_stride + 16 * lane), P, lane);
    prefetch_lane<0>(d + P, reinterpret_cast<const char *>(a.y) + (row * a.y_stride * 2 + 16 * lane), 2 * P, lane);
    prefetch_commit();
  };
  size_t row = (size_t)blockIdx.x * kImmaWarps + warp;
  if (row < a.B) prefetch(row, 0);
  int cur = 0;
  for (; row < a.B; row += nwarps, cur ^= 1) {
    uint8_t *in = in0 + cur * L.Lin;
    uint8_t *xr = in, *yr = in + P;
    prefetch_wait();
    if (lane < P - N) reinterpret_cast<uint16_t *>(yr)[N + lane] = 0;      // the caller's pad columns may hold anything
    __syncwarp();
    stage_limbs<2, false>(N, Z, 0u, yr, y0, y1, lane);
    const bool ok = stage_small<false>(N, P, a.M, xr, xs, lane);
    __syncwarp();
    if (row + nwarps < a.B) prefetch(row + nwarps, cur ^ 1);
    {
      int acc[NJ][2][4];
      conv_band<NJ, 2, false, false, 0>(Z, y0, y1, xs, xs, lane, acc);
      store_product<NJ, 2>(L.NJ, lane, acc, cbuf);
    }
    __syncwarp();
    const uint32_t bits = check_div_q<false>(N, P, a.M - 1, cbuf, a.quo, a.rem, a.m, row, lane, nullptr);
    const uint8_t v = check_verdict(ok, bits);
    if (lane == 0) a.verdict[row] = v;
    __syncwarp();
  }
}

template <int NJ>
__global__ void __launch_bounds__(kImmaWarps * 32) k_check_decrypt(const CheckArgs a) {
  NTRU_CHECK_PROLOGUE;
  auto prefetch = [&](size_t row, int buf) {
    const uint32_t d = in_lane + buf * L.Lin;
    prefetch_lane<0>(d, reinterpret_cast<const char *>(a.x) + (row * a.x_stride * 2 + 16 * lane), 2 * P, lane);
    prefetch_lane<0>(d + 2 * P, reinterpret_cast<const char *>(a.y) + (row * a.y_stride * 2 + 16 * lane), 2 * P, lane);
    prefetch_lane<0>(d + 4 * P, reinterpret_cast<const char *>(a.fp) + (row * a.x_stride + 16 * lane), P, lane);
    prefetch_commit();
  };
  size_t row = (size_t)blockIdx.x * kImmaWarps + warp;
  if (row < a.B) prefetch(row, 0);
  int cur = 0;
  for (; row < a.B; row += nwarps, cur ^= 1) {
    uint8_t *in = in0 + cur * L.Lin;
    uint8_t *fr = in, *er = in + 2 * P, *fpr = in + 4 * P;
    prefetch_wait();
    if (lane < P - N) {
      reinterpret_cast<uint16_t *>(er)[N + lane] = 0;
      fpr[N + lane] = 0;
    }
    __syncwarp();
    stage_limbs<2, false>(N, Z, 0u, er, y0, y1, lane);
    stage_rev8<true>(N, Z, fpr, y2, lane);
    const bool ok = stage_small<true>(N, P, a.M, fr, xs, lane);
    __syncwarp();
    if (row + nwarps < a.B) prefetch(row + nwarps, cur ^ 1);
    {   // product 1: lin(f, e) mod q
      int acc[NJ][2][4];
      conv_band<NJ, 2, false, false, 0>(Z, y0, y1, xs, xs, lane, acc);
      store_product<NJ, 2>(L.NJ, lane, acc, cbuf);
    }
    __syncwarp();
    uint32_t bits = check_div_q<true>(N, P, a.M - 1, cbuf, a.quo, a.rem, nullptr, row, lane, xb);
    __syncwarp();
    {   // product 2: lin(fp mod 3, b), b in {0, 1, 2}: every coefficient in [0, 4N]
      int acc[NJ][1][4];
      conv_band<NJ, 1, false, false, 0>(Z, y2, y2, xb, xb, lane, acc);
      store_product<NJ, 1>(L.NJ, lane, acc, cbuf);
    }
    __syncwarp();
    bits |= check_div_3(N, P, cbuf, a.quo2, a.rem2, row, lane);
    const uint8_t v = check_verdict(ok, bits);
    if (lane == 0) a.verdict[row] = v;
    __syncwarp();
  }
}

template <int NJ, bool kModP>
__global__ void __launch_bounds__(kImmaWarps * 32) k_check_inverse(const CheckArgs a) {
  constexpr int LIMBS = kModP ? 1 : 2;
  NTRU_CHECK_PROLOGUE;
  const int ybytes = kModP ? P : 2 * P;
  auto prefetch = [&](size_t row, int buf) {
    const uint32_t d = in_lane + buf * L.Lin;
    prefetch_lane<0>(d, reinterpret_cast<const char *>(a.x) + (row * (size_t)(2 * P) + 16 * lane), 2 * P, lane);
    prefetch_lane<0>(d + 2 * P, reinterpret_cast<const char *>(a.y) + (row * (size_t)ybytes + 16 * lane), ybytes, lane);
    prefetch_commit();
  };
  size_t row = (size_t)blockIdx.x * kImmaWarps + warp;
  if (row < a.B) prefetch(row, 0);
  int cur = 0;
  for (; row < a.B; row += nwarps, cur ^= 1) {
    uint8_t *in = in0 + cur * L.Lin;
    uint8_t *xr = in, *yr = in + 2 * P;
    prefetch_wait();
    if (lane < P - N) {
      if (kModP) yr[N + lane] = 0;
      else reinterpret_cast<uint16_t *>(yr)[N + lane] = 0;
    }
    __syncwarp();
    if (kModP) stage_rev8<true>(N, Z, yr, y0, lane);
    else stage_limbs<2, false>(N, Z, 0u, yr, y0, y1, lane);
    const bool ok = stage_small<true>(N, P, a.M, xr, xs, lane);
    __syncwarp();
    if (row + nwarps < a.B) prefetch(row + nwarps, cur ^ 1);
    {
      int acc[NJ][LIMBS][4];
      conv_band<NJ, LIMBS, false, false, 0>(Z, y0, y1, xs, xs, lane, acc);
      store_product<NJ, LIMBS>(L.NJ, lane, acc, cbuf);
    }
    __syncwarp();
    const uint32_t bits = kModP ? check_div_3(N, P, cbuf, a.quo, a.rem, row, lane)
                                : check_div_q<false>(N, P, a.M - 1, cbuf, a.quo, a.rem, nullptr, row, lane, nullptr);
    const uint8_t v = check_verdict(ok, bits);
    if (lane == 0) a.verdict[row] = v;
    __syncwarp();
  }
}

// every launch of this file: nothing to do for B = 0, an error for N or q beyond the schedule
template <class K, class A>
int launch_imma(ntru_ctx *ctx, K kernel, const A &args, int kind) {
  const size_t B = args.B;
  if (B == 0) return NTRU_OK;
  if (!imma_supported(ctx)) return fail(ctx, NTRU_E_UNSUPPORTED, "register-fragment tensor schedule supports N <= 832");
  const size_t smem = (size_t)kImmaWarps * args.L.warp_bytes;
  // occupancy: once per (context, kernel, footprint), not per launch
  int per_sm = 0;
  for (const auto &c : ctx->imma_cfg)
    if (c.fn == (const void *)kernel && c.smem == smem) per_sm = c.per_sm;
  if (per_sm == 0) {
    // The opt-in is per function and device, shared by every context: always the same value (the largest footprint of
    // any instantiation, decrypt at N = 832), so contexts cannot undercut each other.
    constexpr int kMaxSmem = 72 * 1024;
    if (smem > kMaxSmem) return fail(ctx, NTRU_E_UNSUPPORTED, "IMMA schedule: shared-memory footprint above 72 KB");
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaFuncSetAttribute(imma, MaxDynamicSharedMemorySize)");
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kImmaWarps * 32, smem);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaOccupancyMaxActiveBlocksPerMultiprocessor(imma)");
    if (per_sm < 1) per_sm = 1;
    ctx->imma_cfg.push_back({(const void *)kernel, smem, per_sm});
  }
  const size_t want = (B + kImmaWarps - 1) / kImmaWarps;
#ifdef NTRU_IMMA_CTA_CAP      // occupancy experiments only
  if (per_sm > NTRU_IMMA_CTA_CAP) per_sm = NTRU_IMMA_CTA_CAP;
#endif
  const size_t cap = (size_t)ctx->sm_count * per_sm;
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  {
    LaunchTimer timer(ctx, kind);
    kernel<<<grid, kImmaWarps * 32, smem, ctx->stream>>>(args);
  }
  NTRU_CUDA(ctx, cudaGetLastError());
  return NTRU_OK;
}

}  // namespace

static int imma_bucket(const ntru_ctx *ctx) {
  const int nj = ((2 * ctx->N - 1 + 15) / 16 + 7) / 8;
  return nj <= 3 ? 3 : (nj <= 8 ? 8 : (nj <= 11 ? 11 : 13));
}

bool imma_supported(const ntru_ctx *ctx) {
  // 13 column blocks of accumulators (104 registers for two limbs) is the largest instantiation: N <= 832
  return ((2 * ctx->N - 1 + 15) / 16 + 7) / 8 <= 13 && ctx->q <= 65536;
}

// N of the instantiations with compile-time geometry (the BASELINE parameter sets), 0 = the bucket's generic one
static int imma_exact_n(const ntru_ctx *ctx) {
  if (ctx->opt_imma_form == 1) return 0;
  const bool two = ctx->q > 256;
  switch (ctx->N) {
    case 167: return two ? 0 : 167;
    case 509: case 677: case 701: case 821: return two ? ctx->N : 0;
    default: return 0;
  }
}

template <int V> using Int = std::integral_constant<int, V>;

// launch(Int<NJ>{}) for the N bucket of ctx: the generic instantiation of NJ column blocks
template <class F>
static int for_bucket(const ntru_ctx *ctx, F launch) {
  switch (imma_bucket(ctx)) {
    case 3: return launch(Int<3>{});
    case 8: return launch(Int<8>{});
    case 11: return launch(Int<11>{});
    default: return launch(Int<13>{});
  }
}

// encrypt / decrypt: launch(Int<NJ>{}, Int<LIMBS>{}, Int<NX>{}) for the instantiation that serves ctx
template <class F>
static int for_enc_dec_form(const ntru_ctx *ctx, F launch) {
  switch (imma_exact_n(ctx)) {
    case 167: return launch(Int<3>{}, Int<1>{}, Int<167>{});
    case 509: return launch(Int<8>{}, Int<2>{}, Int<509>{});
    case 677: return launch(Int<11>{}, Int<2>{}, Int<677>{});
    case 701: return launch(Int<11>{}, Int<2>{}, Int<701>{});
    case 821: return launch(Int<13>{}, Int<2>{}, Int<821>{});
    default: break;
  }
  const bool two = ctx->q > 256;
  return for_bucket(ctx, [&](auto nj) { return two ? launch(nj, Int<2>{}, Int<0>{}) : launch(nj, Int<1>{}, Int<0>{}); });
}

int launch_muldiv_imma(ntru_ctx *ctx, size_t B, const int8_t *x, const void *y, int mod_p, void *quo, void *rem) {
  ImmaMulDivArgs a;
  a.L = make_layout(ctx->N, imma_bucket(ctx), false, false, 0);
  a.qmask = (uint32_t)ctx->q - 1;
  a.B = B; a.x = x; a.y = y; a.quo = quo; a.rem = rem;
  return for_bucket(ctx, [&](auto nj) {
    return mod_p ? launch_imma(ctx, k_muldiv_imma<nj, true>, a, NTRU_K_MULDIV) : launch_imma(ctx, k_muldiv_imma<nj, false>, a, NTRU_K_MULDIV);
  });
}

int launch_encrypt_imma(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t h_stride, const uint8_t *r, const uint8_t *m,
                        uint16_t *value, uint16_t *quo, uint16_t *rem) {
  ImmaEncArgs a;
  a.L = make_layout(ctx->N, imma_bucket(ctx), imma_exact_n(ctx) != 0, false, 0);
  a.qmask = (uint32_t)ctx->q - 1;
  a.B = B; a.h = h; a.h_stride = h_stride; a.r = r; a.m = m; a.value = value; a.quo = quo; a.rem = rem;
  return for_enc_dec_form(ctx, [&](auto nj, auto limbs, auto nx) {
    return launch_imma(ctx, k_encrypt_imma<nj, limbs, nx>, a, NTRU_K_ENC_IMMA);
  });
}

int launch_decrypt_imma(ntru_ctx *ctx, size_t B, const int8_t *f, const uint8_t *fp, size_t key_stride, const uint16_t *e,
                        uint8_t *value, uint16_t *q1, uint16_t *r1, uint8_t *q2, uint8_t *r2) {
  ImmaDecArgs a;
  a.L = make_layout(ctx->N, imma_bucket(ctx), imma_exact_n(ctx) != 0, true, 0);
  a.qmask = (uint32_t)ctx->q - 1; a.q = ctx->q; a.logq = ctx->logq;
  a.B = B; a.f = f; a.fp = fp; a.key_stride = key_stride; a.e = e;
  a.value = value; a.q1 = q1; a.r1 = r1; a.q2 = q2; a.r2 = r2;
  return for_enc_dec_form(ctx, [&](auto nj, auto limbs, auto nx) {
    return launch_imma(ctx, k_decrypt_imma<nj, limbs, nx>, a, NTRU_K_DEC_IMMA);
  });
}

// ---- witness checks: the generic instantiation of each N bucket ------------------------------------------------------
static CheckArgs check_launch_args(const ntru_ctx *ctx, size_t B, bool dec, int in_bytes, uint8_t *verdict) {
  CheckArgs a{};
  a.L = make_layout(ctx->N, imma_bucket(ctx), false, dec, in_bytes);
  a.M = (uint32_t)ctx->q;
  a.B = B;
  a.verdict = verdict;
  return a;
}

int launch_check_encrypt(ntru_ctx *ctx, size_t B, const uint16_t *h, size_t h_stride, const uint8_t *r, const uint16_t *m,
                         const uint16_t *quo, const uint16_t *rem, uint8_t *verdict) {
  CheckArgs a = check_launch_args(ctx, B, false, 3 * ctx->P, verdict);
  a.x = r; a.x_stride = (size_t)ctx->P; a.y = h; a.y_stride = h_stride; a.m = m; a.quo = quo; a.rem = rem;
  return for_bucket(ctx, [&](auto nj) { return launch_imma(ctx, k_check_encrypt<nj>, a, NTRU_K_CHECK); });
}

int launch_check_decrypt(ntru_ctx *ctx, size_t B, const uint16_t *f, const uint8_t *fp, size_t key_stride, const uint16_t *e,
                         const uint16_t *q1, const uint16_t *r1, const uint8_t *q2, const uint8_t *r2, uint8_t *verdict) {
  CheckArgs a = check_launch_args(ctx, B, true, 5 * ctx->P, verdict);
  a.x = f; a.fp = fp; a.x_stride = key_stride; a.y = e; a.y_stride = (size_t)ctx->P;
  a.quo = q1; a.rem = r1; a.quo2 = q2; a.rem2 = r2;
  return for_bucket(ctx, [&](auto nj) { return launch_imma(ctx, k_check_decrypt<nj>, a, NTRU_K_CHECK); });
}

int launch_check_inverse(ntru_ctx *ctx, size_t B, int mod_p, const uint16_t *x, const void *y, const void *quo, const void *rem,
                         uint8_t *verdict) {
  CheckArgs a = check_launch_args(ctx, B, false, (mod_p ? 3 : 4) * ctx->P, verdict);
  if (mod_p) a.M = (uint32_t)ctx->p;
  a.x = x; a.y = y; a.quo = quo; a.rem = rem;
  return for_bucket(ctx, [&](auto nj) {
    return mod_p ? launch_imma(ctx, k_check_inverse<nj, true>, a, NTRU_K_CHECK) : launch_imma(ctx, k_check_inverse<nj, false>, a, NTRU_K_CHECK);
  });
}

}  // namespace ntru
