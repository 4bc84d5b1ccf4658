// lgmi_dense.cuh -- the deep-unit path: contingency counts as a dense int8
// contraction on the 5th-generation tensor cores (tcgen05 / TMEM / TMA).
//
// For a unit with many reads the cells of every pair's 3x3 table are blocks of a Gram matrix
//        G[a][b][i][j] = sum_r X[a][i][r] * X[b][j][r]
// of 0/1 indicator rows X (one byte per read, K-contiguous, K_pad = 32*W columns); integer and
// exact (s32 accumulators, counts <= R < 2^31).  The indicator sets are nested -- C covered,
// P = covered with the site's major or minor allele, M = major -- and the table follows by
// inclusion-exclusion (gram_table in lgmi_kernels.cuh).  Two forms, chosen on the device per unit and run:
//
//   four blocks   reads labelled "other" (covered, neither major nor minor) are rare: only P.P, P.M, M.P, M.M
//   (mode 0)      go through the tensor cores (2.25 x fewer multiply-accumulates); the five cells that
//                 involve an "other" label come from the listed (site, read) entries: k_dense_prep lists them
//                 and writes the label planes transposed (one bit row per read), k_other_fix
//                 adds, for every listed read of a site, that read's bit rows into per-partner counters
//   nine blocks   some site lists more than R/64 "other" reads: all of C, P, M against C, P, M
//   (mode != 0)
//
//   k_dense_prep      four blocks: per site the reads with label "other" (more than the list holds -> mode 1)
//                     and the transposed label planes O, m, M
//   k_dense_x         bit-planes [M | m | C] -> X row groups P, M (and C for nine blocks)
//   k_other_fix       the "other" cells of every pair from the lists and the transposed planes
//   k_gram_i8         one 128 x 256 output tile per CTA iteration:
//                       warp 0  TMA producer (cp.async.bulk.tensor, 128B swizzle)
//                       warp 1  single-thread tcgen05.mma.kind::i8 issuer, M=128 N=256 K=32
//                       warp 2  TMEM allocation (256 columns of s32 accumulators)
//                       warps 4-7  epilogue: tcgen05.ld -> global scratch
//                     4-stage smem ring (48 KB per stage) with full/empty mbarriers.
//                     Only tiles that contain some pair i < j are computed.
// k_count / k_pairs_generic then read the tables from the scratch instead of
// popcounting (DevUnit::gram_off).
//
// Het-anchored form (HetDensePlan, HET_ONLY | SKIP_NONHET): k_dense_x also packs the het sites' rows into X_het,
// k_gram_i8 takes its A operand from there and writes row h of a tile into row het[h], and k_other_fix writes the
// "other" cells of the het rows on both sides of the diagonal; the readers take a pair whose first site is not het
// from its second site's row, transposed.
//
// Reference semantics: the counts of /root/reference/src/giremi/mutual_information.py:15-40
// (labels over the common reads), bit-exact.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "lgmi_plan.h"  // the tile shape kDenseBM x kDenseBN x kDenseBK and DenseTile

namespace lgmi {

constexpr int kDenseStages = 4;
constexpr int kDenseThreads = 256;
constexpr uint32_t kDenseStageBytes = (kDenseBM + kDenseBN) * kDenseBK;  // 48 KB
constexpr uint32_t kDenseSmemBytes = kDenseStages * kDenseStageBytes + 1024 /*align*/ + 256 /*barriers*/;
constexpr uint32_t kDenseTmemCols = 256;

struct DenseParams {
  const DenseTile* tiles;
  uint32_t n_tiles;
  uint32_t k_blocks;  // K_pad / 128
  uint32_t S_pad;     // multiple of 256
  uint32_t* gram;     // [9][S_pad][S_pad]
  uint32_t* error;    // set to 1 if a barrier wait ran out (never in a correct run)
  const uint32_t* mode;  // the unit's form this run (0 four blocks, else nine): a launch whose list is of the
  uint32_t nine;         // other form (nine != 0 vs *mode != 0) returns at once
  uint32_t a_rows;       // rows per group of the A operand: S_pad (X), or H_pad (X_het, the het-anchored form)
  const uint32_t* rows;  // het-anchored form: the count-matrix row of each A row (~0: a pad row); NULL: the same row
};

// ------------------------------------------------------------------ expansion
// 4 bits -> 4 bytes of 0/1
__device__ __forceinline__ uint32_t spread4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }

// 32 x 32 bit transpose across a warp: lane p ends up with bit q = bit p of lane q's word
__device__ __forceinline__ uint32_t transpose32(uint32_t x, uint32_t lane) {
#pragma unroll
  for (uint32_t j = 16u, m = 0x0000ffffu; j; j >>= 1, m ^= m << j) {
    const uint32_t y = __shfl_xor_sync(0xffffffffu, x, j);
    x = (lane & j) ? ((x & ~m) | ((y & ~m) >> j)) : ((x & m) | ((y & m) << j));
  }
  return x;
}

// Four-block form, first pass over the planes.  CTA = 256 sites (a warp per group of 32, a lane per site) x 256
// reads (8 words): every lane reads whole 32-byte sectors of its site's rows, lists the site's reads with label
// "other" (any order; a list that overflows sets *mode: nine blocks) and transposes the label words O, m, M in
// registers (5 shuffle steps per 32 x 32 block); those leave through a shared-memory tile as whole sectors of
// xt[label][read][site word].  Returns at once when the run was told "nine blocks" up front (*mode != 0).
__global__ void __launch_bounds__(256) k_dense_prep(const uint32_t* __restrict__ planes, uint32_t S, uint32_t W,
                                                    uint32_t S_pad, uint32_t* __restrict__ xt, uint32_t* __restrict__ cnt,
                                                    uint32_t* __restrict__ list, uint32_t cap, uint32_t* __restrict__ mode) {
  __shared__ __align__(16) uint32_t tile[3][256][8];  // [label][read of the block][site group of the block]
  __shared__ uint32_t s_nine;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  // one read per CTA: another CTA of this launch may set the flag meanwhile (the four-block outputs are not used then)
  if (tid == 0) s_nine = *reinterpret_cast<volatile uint32_t*>(mode);
  __syncthreads();
  if (s_nine) return;
  const uint32_t w0 = blockIdx.x * 8u, sg0 = blockIdx.y * 8u;
  const uint32_t s = (sg0 + warp) * 32u + lane;
  const uint64_t K_pad = 32ull * W;
  const uint32_t Sw = S_pad >> 5;
  const bool second = w0 + 4u < W;  // W is a multiple of 4: the block's second four words may lie past the row
  uint32_t Mw[8], mw[8], Cw[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) Mw[k] = mw[k] = Cw[k] = 0u;
  if (s < S) {
    const uint32_t* row = planes + (size_t)s * 3u * W + w0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !second) break;
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(row) + h);
      const uint4 b = __ldg(reinterpret_cast<const uint4*>(row + W) + h);
      const uint4 c = __ldg(reinterpret_cast<const uint4*>(row + 2u * W) + h);
      Mw[4 * h] = a.x; Mw[4 * h + 1] = a.y; Mw[4 * h + 2] = a.z; Mw[4 * h + 3] = a.w;
      mw[4 * h] = b.x; mw[4 * h + 1] = b.y; mw[4 * h + 2] = b.z; mw[4 * h + 3] = b.w;
      Cw[4 * h] = c.x; Cw[4 * h + 1] = c.y; Cw[4 * h + 2] = c.z; Cw[4 * h + 3] = c.w;
    }
  }
  {  // the site's "other" reads of these eight words, one reservation in its list
    uint32_t n = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) n += (uint32_t)__popc(Cw[k] & ~Mw[k] & ~mw[k]);
    if (n) {
      uint32_t idx = atomicAdd(cnt + s, n);
      if (idx + n > cap) {
        *mode = 1u;
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          uint32_t O = Cw[k] & ~Mw[k] & ~mw[k];
          while (O) {
            const uint32_t bit = (uint32_t)__ffs((int)O) - 1u;
            O &= O - 1u;
            list[(size_t)s * cap + idx++] = (w0 + (uint32_t)k) * 32u + bit;
          }
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint32_t L2 = Mw[k] & Cw[k], L1 = mw[k] & Cw[k] & ~Mw[k], L0 = Cw[k] & ~Mw[k] & ~mw[k];
    tile[0][k * 32 + lane][warp] = transpose32(L0, lane);
    tile[1][k * 32 + lane][warp] = transpose32(L1, lane);
    tile[2][k * 32 + lane][warp] = transpose32(L2, lane);
  }
  __syncthreads();
  const uint32_t n_reads = second ? 256u : 128u;
  for (uint32_t e = tid; e < 3u * n_reads * 2u; e += 256u) {
    const uint32_t half = e & 1u, r = (e >> 1) % n_reads, b = (e >> 1) / n_reads;
    const uint4 v = *reinterpret_cast<const uint4*>(&tile[b][r][4u * half]);
    *reinterpret_cast<uint4*>(xt + ((size_t)b * K_pad + (size_t)w0 * 32u + r) * Sw + sg0 + 4u * half) = v;
  }
}

// Second pass: the X row groups the unit's form needs -- 1 (major or minor) and 2 (major), plus 0 (covered) for
// nine blocks -- X[g][s][r], one byte per read.  A warp takes 256 reads (8 words) of one site at a time: a lane
// reads the word its 8 reads live in (one sector per plane and warp) and stores 8 bytes per group, so that every
// warp-wide store is 256 contiguous bytes.  Independent of the lists and the transposed planes: in the
// four-block form k_other_fix runs beside it on a second stream.  With `sites` (the het-anchored form) it writes
// X_het instead: row s of each group holds site sites[s], and a row whose entry is ~0 (padding) is zeroed; S is
// then the number of rows and S_pad the group stride.
__global__ void __launch_bounds__(256) k_dense_x(const uint32_t* __restrict__ planes, uint32_t S, uint32_t W, uint32_t S_pad,
                                                 uint8_t* __restrict__ X, const uint32_t* __restrict__ mode,
                                                 const uint32_t* __restrict__ sites) {
  const uint32_t nine = *mode;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t k = lane >> 2, q4 = lane & 3u;
  const uint64_t K_pad = 32ull * W;
  const uint32_t octets = (W + 7u) >> 3;
  const uint64_t total = (uint64_t)S * octets;
  const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  for (uint64_t e = warp0; e < total; e += n_warps) {
    const uint32_t s = (uint32_t)(e / octets), w = (uint32_t)(e - (uint64_t)s * octets) * 8u + k;
    if (w >= W) continue;
    const uint32_t site = sites ? __ldg(sites + s) : s;
    uint32_t Cw = 0u, Mw = 0u, Pw = 0u;
    if (site != ~0u) {
      const uint32_t* row = planes + (size_t)site * 3u * W + w;
      Cw = __ldg(row + 2u * W), Mw = __ldg(row) & Cw, Pw = (Mw | __ldg(row + W)) & Cw;
    }
    uint8_t* x = X + (size_t)s * K_pad + (size_t)w * 32u + q4 * 8u;
    const uint32_t sh = 8u * q4;
    if (nine) {
      const uint32_t bits = (Cw >> sh) & 0xffu;
      *reinterpret_cast<uint2*>(x) = make_uint2(spread4(bits & 15u), spread4(bits >> 4));
    }
    {
      const uint32_t bits = (Pw >> sh) & 0xffu;
      *reinterpret_cast<uint2*>(x + (size_t)S_pad * K_pad) = make_uint2(spread4(bits & 15u), spread4(bits >> 4));
    }
    {
      const uint32_t bits = (Mw >> sh) & 0xffu;
      *reinterpret_cast<uint2*>(x + 2ull * S_pad * K_pad) = make_uint2(spread4(bits & 15u), spread4(bits >> 4));
    }
  }
}

// The table cells with an "other" label, four-block form.  One CTA per site s: for every listed read r of s and
// every partner t, xt[b][r] says whether t carries label b at r.  A warp owns one label, one half of a pass of
// 64 site words and every other listed read; the bit rows of seven reads are requested together (L2 hits), folded
// by a carry-save tree into three words (ones, twos, fours), added into packed 4-bit counters (two such groups),
// those into packed bytes (252 reads), those into shared memory.  Written where gram_table reads them: slot
// 0 / 1 / 2 of pair (s, t), t > s, = reads "other" at s and other / minor / major at t; slot 3 / 6 of pair
// (t, s), t < s, = reads minor / major at t and "other" at s.  rows: the row limit of a piece of a split unit
// (S otherwise, a multiple of 128 below S): only pairs with a first site below it are read, so a site at or past
// it counts its partners below the limit and nothing else.  het (the unit's flag bytes, het-anchored form; else
// NULL): only the rows of het sites are read, but on both sides of the diagonal -- row s gets slots 0 / 1 / 2 of
// every partner t when s is het, and row t gets slots 3 / 6 of partner s when t is het.
constexpr int kFixThreads = 384;  // 12 warps = 3 labels x 2 word halves x 2 read halves
constexpr uint32_t kFixStride = 65u;  // words of shared memory per partner bit: (bit, word) and (word, bit) walks both hit 32 banks

__device__ __forceinline__ uint32_t fix_spread(uint32_t x, uint32_t q) { return (x >> q) & 0x11111111u; }

__global__ void __launch_bounds__(kFixThreads, 3) k_other_fix(const uint32_t* __restrict__ xt, uint64_t K_pad, uint32_t S,
                                                           uint32_t S_pad, uint32_t rows, const uint32_t* __restrict__ cnt,
                                                           const uint32_t* __restrict__ list, uint32_t cap,
                                                           uint32_t* __restrict__ gram, const uint32_t* __restrict__ mode,
                                                           const uint8_t* __restrict__ het) {
  if (*mode) return;
  __shared__ uint32_t acc[3][32u * kFixStride];  // [label][partner bit * 65 + site word of the pass]
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t label = warp % 3u, half = (warp / 3u) & 1u, parity = warp / 6u;
  const uint32_t s = blockIdx.x, Sw = S_pad >> 5;
  const uint32_t Sw_s = s < rows ? Sw : rows >> 5;  // words of the partners this site needs
  const uint32_t n = min(cnt[s], cap);
  const uint32_t* __restrict__ mine = list + (size_t)s * cap;
  const size_t plane = (size_t)S_pad * S_pad;
  const uint32_t n_mine = n > parity ? (n - parity + 1u) / 2u : 0u;  // this warp's listed reads: k = parity + 2 m
  for (uint32_t w0 = 0; w0 < Sw_s; w0 += 64u) {
    for (uint32_t e = tid; e < 3u * 32u * kFixStride; e += kFixThreads) (&acc[0][0])[e] = 0u;
    __syncthreads();
    const uint32_t wl = half * 32u + lane, word = w0 + wl;
    const bool valid = word < Sw_s;
    const uint32_t* __restrict__ col = xt + (size_t)label * K_pad * Sw + (valid ? word : 0u);  // (an invalid lane's sums go nowhere)
    uint32_t nb[4] = {0u, 0u, 0u, 0u}, by[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    auto bytes_to_smem = [&]() {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t v = (by[c] >> (8 * k)) & 0xffu;
          if (v) atomicAdd(&acc[label][(8u * k + c) * kFixStride + wl], v);
        }
        by[c] = 0u;
      }
    };
    uint32_t groups = 0;
    for (uint32_t m0 = 0; m0 < n_mine; m0 += 28u) {
      const uint32_t have = min(28u, n_mine - m0);
      // the next 28 reads, one per lane, as word offsets of their bit rows (K_pad * Sw < 2^32: checked by the host)
      const uint32_t my = lane < have ? __ldg(mine + parity + 2u * (m0 + lane)) * Sw : 0u;
      for (uint32_t q0 = 0; q0 < have; q0 += 14u) {
        uint32_t x[14];  // two groups of seven: fourteen bit rows requested before the first is used
#pragma unroll
        for (int u = 0; u < 14; ++u) {  // (rows past the warp's last listed read: row 0, masked out below)
          const uint32_t off = __shfl_sync(0xffffffffu, my, (q0 + (uint32_t)u) & 31u);
          x[u] = __ldg(col + off);
        }
        if (q0 + 14u > have) {  // (warp-uniform) the last, partial round
#pragma unroll
          for (int u = 0; u < 14; ++u)
            if (q0 + (uint32_t)u >= have) x[u] = 0u;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t* y = x + 7 * h;
          // seven one-bit rows -> ones + 2 twos + 4 fours
          const uint32_t a1 = y[0] ^ y[1] ^ y[2], c1 = (y[0] & y[1]) | (y[2] & (y[0] ^ y[1]));
          const uint32_t a2 = y[3] ^ y[4] ^ y[5], c2 = (y[3] & y[4]) | (y[5] & (y[3] ^ y[4]));
          const uint32_t ones = a1 ^ a2 ^ y[6], c3 = (a1 & a2) | (y[6] & (a1 ^ a2));
          const uint32_t twos = c1 ^ c2 ^ c3, fours = (c1 & c2) | (c3 & (c1 ^ c2));
#pragma unroll
          for (uint32_t q = 0; q < 4u; ++q)
            nb[q] += fix_spread(ones, q) + 2u * fix_spread(twos, q) + 4u * fix_spread(fours, q);  // <= 7 per group
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {           // two groups: a nibble holds at most 14
          by[q] += nb[q] & 0x0f0f0f0fu;         // byte k <- partner bit 8 k + q
          by[4 + q] += (nb[q] >> 4) & 0x0f0f0f0fu;  // byte k <- partner bit 8 k + 4 + q
          nb[q] = 0u;
        }
        if (++groups == 18u) {  // 18 x 14 = 252 per byte
          bytes_to_smem();
          groups = 0;
        }
      }
    }
    bytes_to_smem();
    __syncthreads();
    for (uint32_t tl = tid; tl < 2048u; tl += kFixThreads) {
      const uint32_t t = w0 * 32u + tl;
      if (t >= S || (s >= rows && t >= rows)) break;
      const uint32_t at = (tl & 31u) * kFixStride + (tl >> 5);
      const bool fwd = het ? t != s && (het[s] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP : t > s, bwd = het ? t != s && (het[t] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP : t < s;
      if (fwd) {
        uint32_t* out = gram + (size_t)s * S_pad + t;
        out[0] = acc[0][at];
        out[plane] = acc[1][at];
        out[2u * plane] = acc[2][at];
      }
      if (bwd) {
        uint32_t* out = gram + (size_t)t * S_pad + s;
        out[3u * plane] = acc[1][at];
        out[6u * plane] = acc[2][at];
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded wait: a protocol bug becomes an error flag + trap instead of a hung GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, uint32_t* error) {
  const uint32_t addr = smem_u32(bar);
  const long long t0 = clock64();
  for (uint32_t spin = 0;; ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
    if ((spin & 1023u) == 1023u && clock64() - t0 > 4000000000LL) {  // ~2 s: no tile takes milliseconds
      if (error) atomicExch(error, 1u);
      __trap();
    }
  }
}

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, 128B-swizzled operand tile whose rows are 128 bytes: 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3fffu) | (1ull << 16) /* LBO = 16 B (unused with swizzle) */ |
         (64ull << 32) /* SBO = 1024 B */ | (1ull << 46) /* descriptor version: Blackwell */ |
         (2ull << 61) /* SWIZZLE_128B */;
}

// kind::i8 instruction descriptor: D = s32, A = B = unsigned 8 bit, both K-major
__device__ __forceinline__ uint32_t umma_idesc_u8(uint32_t M, uint32_t N) {
  return (2u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
// arrives on the mbarrier when every previously issued MMA of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void tmem_load_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// zero the 128 x 256 output tiles that several work items add into (one CTA per listed item; an item whose
// kb0 is 0 zeroes its tile, the others skip)
__global__ void __launch_bounds__(256) k_zero_partial_tiles(const DenseTile* __restrict__ tiles, uint32_t n_tiles,
                                                            uint32_t S_pad, uint32_t* __restrict__ gram,
                                                            const uint32_t* __restrict__ mode, uint32_t nine,
                                                            const uint32_t* __restrict__ rows) {
  if ((*mode != 0u) != (nine != 0u)) return;  // the list of the unit's other form
  const DenseTile tile = tiles[blockIdx.x];
  if (blockIdx.x >= n_tiles || !tile.partial || tile.kb0 != 0) return;
  uint32_t* base = gram + (size_t)(tile.a * 3u + tile.b) * S_pad * S_pad + (size_t)tile.J * kDenseBN;
  for (uint32_t e = threadIdx.x; e < (uint32_t)kDenseBM * (kDenseBN / 4); e += blockDim.x) {
    const uint32_t r = tile.I * kDenseBM + e / (kDenseBN / 4), q = e % (kDenseBN / 4);
    const uint32_t row = rows ? rows[r] : r;  // (het-anchored form: the tile's rows are the het sites' rows)
    if (row != ~0u) reinterpret_cast<uint4*>(base + (size_t)row * S_pad)[q] = make_uint4(0u, 0u, 0u, 0u);
  }
}

// ------------------------------------------------------------------ the GEMM
// tmap_a: the A operand's rows (X, or X_het in the het-anchored form), tmap: X, the B operand's
__global__ void __launch_bounds__(kDenseThreads, 1) k_gram_i8(const __grid_constant__ CUtensorMap tmap_a,
                                                              const __grid_constant__ CUtensorMap tmap,
                                                              const DenseParams P) {
  if ((*P.mode != 0u) != (P.nine != 0u)) return;  // the list of the unit's other form (CTA-uniform, before any barrier)
  extern __shared__ uint8_t dense_smem_raw[];
  // 128B swizzle needs 1024-byte aligned tiles
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(dense_smem_raw) + 1023u) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kDenseStages * kDenseStageBytes);
  uint64_t* full = bars;                       // [stages]  TMA -> MMA
  uint64_t* empty = bars + kDenseStages;       // [stages]  MMA -> TMA
  uint64_t* acc_full = bars + 2 * kDenseStages;   // MMA -> epilogue
  uint64_t* acc_empty = acc_full + 1;             // epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    for (int s = 0; s < kDenseStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 128);  // the four epilogue warps
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kDenseTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ---------------- TMA producer
      uint32_t stage = 0, phase = 0;
      for (uint32_t t = blockIdx.x; t < P.n_tiles; t += gridDim.x) {
        const DenseTile tile = P.tiles[t];
        const int32_t row_a = (int32_t)(tile.a * P.a_rows + tile.I * kDenseBM);
        const int32_t row_b = (int32_t)(tile.b * P.S_pad + tile.J * kDenseBN);
        for (uint32_t kb = tile.kb0; kb < tile.kb1; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1u, P.error);
          uint8_t* sa = smem + stage * kDenseStageBytes;
          uint8_t* sb = sa + kDenseBM * kDenseBK;
          mbar_expect_tx(&full[stage], kDenseStageBytes);
          const int32_t k0 = (int32_t)(kb * kDenseBK);
          tma_load_2d(sa, &tmap_a, &full[stage], k0, row_a);
          tma_load_2d(sb, &tmap, &full[stage], k0, row_b);
          tma_load_2d(sb + 128 * kDenseBK, &tmap, &full[stage], k0, row_b + 128);
          if (++stage == kDenseStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ---------------- MMA issuer
      const uint32_t idesc = umma_idesc_u8(kDenseBM, kDenseBN);
      uint32_t stage = 0, phase = 0, acc_phase = 0;
      for (uint32_t t = blockIdx.x; t < P.n_tiles; t += gridDim.x) {
        const DenseTile tile = P.tiles[t];
        mbar_wait(acc_empty, acc_phase ^ 1u, P.error);  // epilogue has drained the accumulator
        tc_fence_after();
        for (uint32_t kb = tile.kb0; kb < tile.kb1; ++kb) {
          mbar_wait(&full[stage], phase, P.error);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kDenseStageBytes);
          const uint32_t sb = sa + kDenseBM * kDenseBK;
          const uint64_t da = umma_desc_sw128(sa), db = umma_desc_sw128(sb);
#pragma unroll
          for (uint32_t k = 0; k < kDenseBK / 32; ++k)  // K = 32 bytes per instruction: +32 B on both operands
            umma_i8(tmem_base, da + 2ull * k, db + 2ull * k, idesc, ((kb - tile.kb0) | k) != 0u);
          umma_commit(&empty[stage]);  // smem slot free once these MMAs have read it
          if (++stage == kDenseStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit(acc_full);  // accumulator complete
        acc_phase ^= 1u;
      }
    }
  } else if (warp >= 4) {  // ---------------- epilogue: TMEM -> registers -> global
    const uint32_t q = warp - 4u;  // TMEM lane quarter of this warp
    uint32_t acc_phase = 0;
    for (uint32_t t = blockIdx.x; t < P.n_tiles; t += gridDim.x) {
      const DenseTile tile = P.tiles[t];
      mbar_wait(acc_full, acc_phase, P.error);
      tc_fence_after();
      const uint32_t a_row = tile.I * kDenseBM + q * 32u + lane;
      const uint32_t row = P.rows ? __ldg(P.rows + a_row) : a_row;  // (~0: a pad row of X_het, not stored)
      const bool store = row != ~0u;
      uint32_t* out = P.gram + ((size_t)(tile.a * 3u + tile.b) * P.S_pad + (store ? row : 0u)) * P.S_pad + (size_t)tile.J * kDenseBN;
#pragma unroll 1
      for (uint32_t c = 0; c < kDenseBN / 32; ++c) {
        uint32_t r[32];
        tmem_load_32x32(tmem_base + ((q * 32u) << 16) + c * 32u, r);
        if (store && tile.partial) {
#pragma unroll
          for (int v = 0; v < 32; ++v) atomicAdd(out + c * 32u + v, r[v]);  // (RED: no return value is used)
        } else if (store) {
#pragma unroll
          for (int v = 0; v < 8; ++v)
            reinterpret_cast<uint4*>(out + c * 32u)[v] = make_uint4(r[4 * v], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(acc_empty);
      acc_phase ^= 1u;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kDenseTmemCols)
                 : "memory");
  }
}

}  // namespace lgmi
