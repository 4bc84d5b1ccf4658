// lgmi_fast.cuh -- the small-unit path of the pair kernel: units with S <= 64
// sites and R <= 256 reads, one unit per CTA iteration, everything staged in
// shared memory.  Persistent CTAs stride over the fast items; the next unit's
// planes are prefetched with cp.async while the current one is processed.
//
// Per unit:
//   land     raw plane rows [M | m | C] arrive by cp.async (LDGSTS) into rows of
//            28 words (112 B stride: LDS.128 by 8 consecutive lanes hits 32
//            distinct banks); transformed in place to M&C and P = (M|m)&C; reads
//            labelled "other" (C & ~P, rare) go to a short per-site list
//   fixup    the five table cells that involve an "other" label, from the lists
//   counts   |Pi&Pj|, |Mi&Pj|, |Pi&Mj|, |Mi&Mj| per pair: AND + carry-save adder
//            tree + 3 POPC per set (7 words); min-common filter; the warp ballot
//            of each 32-pair chunk is its emit mask; surviving pairs are listed
//            as "2x2" or "3x3" (an "other" label among the common reads)
//   mi       branch-free fp64 epilogues over warp-sized chunks of the two lists
//   emit     ordered 16-byte records at the offset fixed by k_count + scan
//   mean     per-site mean over het-kept pairs (CPython's compensated sum)
// The arithmetic is the one in lgmi_math.cuh (same operation order, same
// roundings); only its evaluation is reorganised:
//   * n/N is computed as Markstein's correctly rounded quotient from a table of
//     RN(1/N):  q0 = n*y; r = fma(-q0, N, n); q = fma(r, y, q0)  ==  RN(n/N)
//   * (double)n, ln n (hi, lo) and 1/n come from one shared-memory table
//   * a zero cell contributes an exact 0.0 (q = 0), so no branch is needed
//
// Reference semantics: /root/reference/src/giremi/mutual_information.py:6-60,
// sklearn/metrics/cluster/_supervised.py:920-935.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lgmi_math.cuh"
#include "lgmi_plan.h"  // kFastMaxS, kFastMaxR and FastItem

namespace lgmi {

constexpr int kFastThreads = 256;
constexpr int kFastWarps = kFastThreads / 32;
constexpr int kFastMaxPairs = 2048;  // >= 64*63/2 = 2016, whole 32-pair chunks
constexpr int kFastChunks = kFastMaxPairs / 32;
constexpr int kRowStride = 28;       // words per landed site row: M[8] | P[8] | C[8] | pad[4]
constexpr int kOthCap = 7;           // "other" reads kept per site (3-bit cells); more -> generic kernel
constexpr uint32_t kFastMathMaxCount = (1u << 21) - 1u;  // the reorganised epilogues below are host-tested bit for bit
                                     // against lgmi_math.cuh for table counts up to here (tests/test_fast_host.py);
                                     // units with more reads keep the straightforward arithmetic

// ln k as hi + lo (hi = RN(ln k)); entry 0 is {0, 0}
struct __align__(16) FastLn {
  double hi, lo;
};
struct FastTab {
  FastLn ln[kFastMaxR + 1];   // 4112 B
  double inv[kFastMaxR + 1];  // RN(1/k), inv[0] = 0
  __device__ __forceinline__ const FastLn& ln_at(uint32_t k) const { return ln[k]; }
  __device__ __forceinline__ double inv_at(uint32_t k) const { return inv[k]; }
};
// the same two look-ups for counts of any size: ln k from the context's global table, 1/k by the correctly
// rounded reciprocal (what the shared-memory table holds for k <= 256)
struct GlobalTab {
  const lg_dd* ln;
  __device__ __forceinline__ FastLn ln_at(uint32_t k) const {
    const double2 v = __ldg(reinterpret_cast<const double2*>(ln) + k);
    FastLn r;
    r.hi = v.x;
    r.lo = v.y;
    return r;
  }
  __device__ __forceinline__ double inv_at(uint32_t k) const { return k ? __drcp_rn((double)k) : 0.0; }
};

struct FastSmem {
  FastTab tab;                                           // 6176 B
  uint32_t rows[2][kFastMaxS * kRowStride];              // 14336 B, double-buffered
  unsigned long long val[kFastMaxPairs];                 // 16 KB: packed counts, then MI bits
  uint16_t list[kFastMaxPairs];                          // 4 KB: pairs with a 2x2 table from the front,
                                                         //       pairs with "other" cells from the back
  uint32_t emit_mask[kFastChunks];                       // ballot of each 32-pair chunk
  uint32_t chunk_off[kFastChunks];
  uint32_t m2_mask[kFastChunks], m3_mask[kFastChunks];   // ... of its pairs with a 2x2 / a 3x3 table (all-pairs kernel)
  uint32_t ocell[kFastMaxPairs / 2];                     // 4 KB: per pair, 15 bits: the five 3-bit "other" cells
  uint16_t oth_flat[kFastMaxS * kOthCap];                // every (site << 8 | word) holding reads with label "other", any order
  uint32_t n_oth[kFastMaxS];
  uint32_t n_oth_total;
  uint8_t flags[kFastMaxS];
  uint8_t info[kFastMaxS];                               // bit 0 het_snp, bits 1-4 number of "other" reads
  uint8_t het_list[kFastMaxS];                           // het sites ascending, then ...
  uint8_t nonhet_list[kFastMaxS];                        // ... the other sites ascending
  unsigned long long het_mask;
  uint32_t n_list2, n_list3, next_chunk, total;
  __device__ __forceinline__ uint32_t oth_count(uint32_t s) const {
    return n_oth[s] < (uint32_t)kOthCap ? n_oth[s] : (uint32_t)kOthCap;
  }
};

__device__ __forceinline__ double mi_nan() { return __longlong_as_double(0x7ff8000000000000LL); }

// ---------------------------------------------------------------------------
// popcount of the AND of two NW-word rows through a carry-save adder tree
__device__ __forceinline__ void csa(uint32_t& h, uint32_t& l, uint32_t a, uint32_t b, uint32_t c) {
  const uint32_t u = a ^ b;
  h = (a & b) | (u & c);
  l = u ^ c;
}

template <int NW>
__device__ __forceinline__ uint32_t and_popc(const uint32_t* __restrict__ x, const uint32_t* __restrict__ y) {
  if constexpr (NW <= 4) {
    uint32_t n = 0;
#pragma unroll
    for (int k = 0; k < NW; ++k) n += __popc(x[k] & y[k]);
    return n;
  } else {
    uint32_t w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = (k < NW) ? (x[k] & y[k]) : 0u;
    uint32_t h0, l0, h1, l1, h2, ones, fours, twos;
    csa(h0, l0, w[0], w[1], w[2]);
    csa(h1, l1, w[3], w[4], w[5]);
    csa(h2, ones, l0, l1, w[6]);
    csa(fours, twos, h0, h1, h2);
    uint32_t n = __popc(ones) + 2u * __popc(twos) + 4u * __popc(fours);
    if constexpr (NW == 8) n += __popc(w[7]);
    return n;
  }
}

// packed per-pair value between the counts phase and the MI phase (R <= 256, so a
// count needs 9 bits):  bits 0-8 |Pi&Pj|, 9-17 |Mi&Pj|, 18-26 |Pi&Mj|, 27-35 |Mi&Mj|,
// 36-50 the five 3-bit "other" cells T[0][0], T[0][1], T[0][2], T[1][0], T[2][0].
// A candidate without MI holds the NaN pattern 0x7ff8000000000000 instead.
constexpr unsigned long long kNoMi = 0x7ff8000000000000ull;

// the four counts of a pair.  ri / rj point at landed rows: M at word 0, P at word 8.
// |Pi&Pj| comes first: with the "other" cells it is the number of common reads, and a pair below
// the min-common threshold (most pairs of sparsely covered units) skips the other three sets.
template <int NW>
__device__ __forceinline__ void load_row(uint32_t (&w)[8], const uint32_t* __restrict__ r) {
#pragma unroll
  for (int k = 0; k < (NW + 3) / 4; ++k) {
    const uint4 a = *reinterpret_cast<const uint4*>(r + 4 * k);
    w[4 * k] = a.x; w[4 * k + 1] = a.y; w[4 * k + 2] = a.z; w[4 * k + 3] = a.w;
  }
}

// returns false (and leaves `packed` alone) when nPP + n_other < min_common
template <int NW>
__device__ __forceinline__ bool pair_counts(const uint32_t* __restrict__ ri, const uint32_t* __restrict__ rj,
                                            uint32_t n_other, int min_common, unsigned long long& packed) {
  uint32_t Pi[8], Pj[8];
  load_row<NW>(Pi, ri + 8);
  load_row<NW>(Pj, rj + 8);
  const uint32_t nPP = and_popc<NW>(Pi, Pj);
  if ((int)(nPP + n_other) < min_common) return false;  // strict '<' drops (mutual_information.py:19)
  uint32_t Mi[8], Mj[8];
  load_row<NW>(Mi, ri);
  load_row<NW>(Mj, rj);
  const uint32_t nMP = and_popc<NW>(Mi, Pj);
  const uint32_t nPM = and_popc<NW>(Pi, Mj);
  const uint32_t nMM = and_popc<NW>(Mi, Mj);
  packed = (unsigned long long)(nPP | (nMP << 9) | (nPM << 18)) | ((unsigned long long)nMM << 27);
  return true;
}

// ---------------------------------------------------------------------------
// fp64 epilogue pieces (operation order of lgmi_math.cuh / sklearn)
struct CellCtx {
  double dN, invN, lnN;
};

// RN(ln(a*b)) from the double-double logs of a and b (lg_ln_product)
__device__ __forceinline__ double ln_prod(const FastLn& a, const FastLn& b) {
  const double s = __dadd_rn(a.hi, b.hi);
  const double bb = __dsub_rn(s, a.hi);
  double e = __dadd_rn(__dsub_rn(a.hi, __dsub_rn(s, bb)), __dsub_rn(b.hi, bb));
  e = __dadd_rn(e, __dadd_rn(a.lo, b.lo));
  return __dadd_rn(s, e);
}

// (double)n for 0 <= n < 2^32 without a conversion instruction: 2^52 + n is exact
__device__ __forceinline__ double u32_to_double(uint32_t n) {
  return __dsub_rn(__hiloint2double(0x43300000, (int)n), 4503599627370496.0);
}

// one cell's term; n == 0 yields exactly 0.0
__device__ __forceinline__ double cell_term(double ln_n, double dn, const CellCtx& c, double ln_ab) {
  const double q0 = __dmul_rn(dn, c.invN);
  const double r = __fma_rn(-q0, c.dN, dn);
  const double q = __fma_rn(r, c.invN, q0);                    // == RN(n / N)
  const double lo = __dadd_rn(__dadd_rn(-ln_ab, c.lnN), c.lnN);
  const double t = __dadd_rn(__dmul_rn(q, __dsub_rn(ln_n, c.lnN)), __dmul_rn(q, lo));
  return (fabs(t) < LG_EPS) ? 0.0 : t;
}

template <class Tab>
__device__ __forceinline__ double cell_of(const Tab& tab, uint32_t n, const CellCtx& cx, const FastLn& er,
                                          const FastLn& ec) {
  return cell_term(tab.ln_at(n).hi, u32_to_double(n), cx, ln_prod(er, ec));
}

// 2x2 table (no "other" label among the common reads).  Cell order mm, mM, Mm, MM.
template <class Tab>
__device__ __forceinline__ double mi_2x2(const Tab& tab, uint32_t n_mm, uint32_t n_mM, uint32_t n_Mm,
                                         uint32_t n_MM) {
  const uint32_t r_m = n_mm + n_mM, r_M = n_Mm + n_MM;
  const uint32_t c_m = n_mm + n_Mm, c_M = n_mM + n_MM;
  const uint32_t N = r_m + r_M;
  const CellCtx cx{u32_to_double(N), tab.inv_at(N), tab.ln_at(N).hi};
  const FastLn ecm = tab.ln_at(c_m), ecM = tab.ln_at(c_M);
  double s = 0.0;
  {
    const FastLn erm = tab.ln_at(r_m);
    s = __dadd_rn(s, cell_of(tab, n_mm, cx, erm, ecm));
    s = __dadd_rn(s, cell_of(tab, n_mM, cx, erm, ecM));
  }
  {
    const FastLn erM = tab.ln_at(r_M);
    s = __dadd_rn(s, cell_of(tab, n_Mm, cx, erM, ecm));
    s = __dadd_rn(s, cell_of(tab, n_MM, cx, erM, ecM));
  }
  const bool degenerate = (r_m == 0u) | (r_M == 0u) | (c_m == 0u) | (c_M == 0u);  // :920 one class
  return (degenerate || !(s > 0.0)) ? 0.0 : s;
}

// 3x3 table T[a*3+b] (label order other, minor, major)
template <class Tab>
__device__ __forceinline__ double mi_3x3(const Tab& tab, const uint32_t T[9]) {
  uint32_t r[3], c[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) r[a] = T[3 * a] + T[3 * a + 1] + T[3 * a + 2];
#pragma unroll
  for (int b = 0; b < 3; ++b) c[b] = T[b] + T[3 + b] + T[6 + b];
  const uint32_t N = r[0] + r[1] + r[2];
  const int nrow = (r[0] != 0u) + (r[1] != 0u) + (r[2] != 0u);
  const int ncol = (c[0] != 0u) + (c[1] != 0u) + (c[2] != 0u);
  int nnz = 0;
#pragma unroll
  for (int k = 0; k < 9; ++k) nnz += (T[k] != 0u);
  const CellCtx cx{u32_to_double(N), tab.inv_at(N), tab.ln_at(N).hi};
  FastLn ec[3];
#pragma unroll
  for (int b = 0; b < 3; ++b) ec[b] = tab.ln_at(c[b]);
  double s;
  if (nnz < 8) {  // ndarray.sum(): plain loop below 8 elements; absent cells add an exact 0.0
    s = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const FastLn er = tab.ln_at(r[a]);
#pragma unroll
      for (int b = 0; b < 3; ++b) s = __dadd_rn(s, cell_of(tab, T[3 * a + b], cx, er, ec[b]));
    }
  } else {        // numpy pairwise_sum over the 8 or 9 present cells (z = the absent one, if any); rare
    double t[9];
    int z = 9;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const FastLn er = tab.ln_at(r[a]);
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        t[3 * a + b] = cell_of(tab, T[3 * a + b], cx, er, ec[b]);
        if (T[3 * a + b] == 0u) z = 3 * a + b;
      }
    }
    double u[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) u[k] = (k < z) ? t[k] : t[k + 1];
    s = __dadd_rn(__dadd_rn(__dadd_rn(u[0], u[1]), __dadd_rn(u[2], u[3])),
                  __dadd_rn(__dadd_rn(u[4], u[5]), __dadd_rn(u[6], u[7])));
    if (nnz == 9) s = __dadd_rn(s, t[8]);
  }
  return (nrow <= 1 || ncol <= 1 || !(s > 0.0)) ? 0.0 : s;
}

// triangular pair tables: for every S in [2, 64] the (i, j) of its S(S-1)/2 pairs in
// lexicographic order, i * 64 + j as u16; table of S starts at C(S, 3) entries.
constexpr uint32_t kIjTabEntries = 64u * 63u * 62u / 6u + 64u * 63u / 2u;  // C(64,3) + C(64,2)
LG_HD uint32_t lg_ij_tab_off(uint32_t S) { return S * (S - 1u) * (S - 2u) / 6u; }

}  // namespace lgmi
