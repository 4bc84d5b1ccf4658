// lgmi_kernels.cuh -- sm_100a kernels of the MI step.
//
//   k_count, k_count_fast  K0: emitted pairs per work item; an exclusive scan of
//                      these fixes every item's place in the ordered output.
//   k_pairs_generic    K1+K2: per-pair contingency counts over the common reads
//                      (AND+popcount, or read from what k_tile_mi, k_tile_gram_ws
//                      or k_gram_i8 computed), fp64 MI, min-common and het
//                      filters, emission at the item's offset and, for units of
//                      one item, the per-site mean MI.  The small units take
//                      k_pairs_fast (lgmi_fast_kernel.cuh).
//   k_tile_mi          counts + MI of the mid-depth units per 16 x 16 site block.
//   k_site_mean_dense  per-site mean MI for units spanning several items.
//   k_site_mean_csr    mean of caller-supplied rows (drop-in for
//                      mean_mismatch_pair_mutual_info).
//   k_ecdf_*           K4: het-SNP mean collection, searchsorted-left, mip, call.
//
// Reference semantics: /root/reference/src/giremi/mutual_information.py:6-60,
// mismatch.py:393-396, stat.py:7-29, script/giremi.py:97-114,415-429.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/lgmi.h"
#include "lgmi_math.cuh"
#include "lgmi_plan.h"
#include "lgmi_fast_kernel.cuh"
#include "lgmi_dense.cuh"

namespace lgmi {

constexpr int kThreads = 256;   // CTA size of k_pairs_generic, k_count, k_count_fast, k_tile_mi and k_tile_finish

struct Header {
  unsigned long long n_records;
  unsigned long long pad;
};

struct RunParams {
  const DevUnit* units;
  const Item* items;
  uint32_t n_items;
  uint32_t n_units;
  const uint32_t* planes;
  const uint8_t* site_flags;
  const lg_dd* lntab;
  uint32_t ln_cap;
  int min_common;
  uint32_t mode;
  unsigned long long* item_cnt;        // per item: emitted pairs (k_count)
  const unsigned long long* item_off;  // exclusive scan of item_cnt, n_items + 1 entries
  uint8_t* item_dense;                 // k_count: fast-eligible item with > kOthCap "other" reads at a site
  uint32_t* n_generic;                 // items k_pairs_generic has to process (host count + dense ones)
  const uint32_t* gram;                // count matrices of the tensor-core path (DevUnit::gram_off)
  const uint32_t* unit_mode;           // per unit, tensor-core path: 0 four Gram blocks + "other" cells, else nine blocks
  const uint8_t* unit_het;             // per unit, tensor-core path: 1 het-anchored count matrices (HetDensePlan); NULL:
                                       // none this run
  uint32_t* tile_counts;               // EMIT_COUNTS: 3x3 tables of the k_tile_mi units, 9 per dense slot
  uint32_t unit_base;                  // added to the unit field of every record
  const TiledDesc* tiled_desc;         // k_pairs_generic<1>: its items, in item order
  uint32_t n_tiled_desc;
  Header* header;
  lgmi_pair_rec* records;
  uint32_t* counts;
  double* site_mean;
  uint32_t* site_cnt;
  double* dense;
  unsigned long long* unit_rec_off;
};

struct LnGlobal {
  const lg_dd* tab;
  __device__ __forceinline__ lg_dd operator()(uint32_t k) const {
    const double2 v = __ldg(reinterpret_cast<const double2*>(tab) + k);
    lg_dd r;
    r.hi = v.x;
    r.lo = v.y;
    return r;
  }
};

__device__ __forceinline__ uint32_t popc4(uint4 a, uint4 b) {
  return __popc(a.x & b.x) + __popc(a.y & b.y) + __popc(a.z & b.z) + __popc(a.w & b.w);
}

__device__ __forceinline__ double lg_nan() { return __longlong_as_double(0x7ff8000000000000LL); }

// Common reads of sites i and j: |C_i & C_j|  (mutual_information.py:17-19).
__device__ __forceinline__ uint32_t pair_common(const uint4* __restrict__ ri,
                                                const uint4* __restrict__ rj, uint32_t W4) {
  uint32_t n = 0;
  for (uint32_t k = 0; k < W4; ++k) n += popc4(__ldg(ri + 2 * W4 + k), __ldg(rj + 2 * W4 + k));
  return n;
}

// Fills the 3x3 table (label order other/minor/major) of a pair whose common
// read count is already known.  Returns true when no "other" label occurs
// among the common reads (the table is then 2x2 in the minor/major block).
__device__ __forceinline__ bool pair_table(const uint4* __restrict__ ri, const uint4* __restrict__ rj,
                                           uint32_t W4, uint32_t n_common, uint32_t T[9]) {
  uint32_t MM = 0, Mm = 0, mM = 0, mm = 0;
  for (uint32_t k = 0; k < W4; ++k) {
    const uint4 Mi = __ldg(ri + k), mi = __ldg(ri + W4 + k);
    const uint4 Mj = __ldg(rj + k), mj = __ldg(rj + W4 + k);
    MM += popc4(Mi, Mj);
    Mm += popc4(Mi, mj);
    mM += popc4(mi, Mj);
    mm += popc4(mi, mj);
  }
  T[8] = MM;
  T[7] = Mm;
  T[5] = mM;
  T[4] = mm;
  if (MM + Mm + mM + mm == n_common) {
    T[0] = T[1] = T[2] = T[3] = T[6] = 0;
    return true;
  }
  uint32_t aM = 0, am = 0, bM = 0, bm = 0;  // marginals against the partner's coverage
  for (uint32_t k = 0; k < W4; ++k) {
    const uint4 Mi = __ldg(ri + k), mi = __ldg(ri + W4 + k), Ci = __ldg(ri + 2 * W4 + k);
    const uint4 Mj = __ldg(rj + k), mj = __ldg(rj + W4 + k), Cj = __ldg(rj + 2 * W4 + k);
    aM += popc4(Mi, Cj);
    am += popc4(mi, Cj);
    bM += popc4(Ci, Mj);
    bm += popc4(Ci, mj);
  }
  T[6] = aM - MM - Mm;  // site1 major, site2 other
  T[3] = am - mM - mm;  // site1 minor, site2 other
  T[2] = bM - MM - mM;  // site1 other, site2 major
  T[1] = bm - Mm - mm;  // site1 other, site2 minor
  T[0] = n_common - (MM + Mm + mM + mm) - T[6] - T[3] - T[2] - T[1];
  return false;
}

// 3x3 table of pair (i, j) from the count matrices of the tensor-core path (lgmi_dense.cuh); returns N.
// Slot a * 3 + b of the scratch holds, for row group a of site i and b of site j (0 covered, 1 major or
// minor, 2 major), |X_a,i & X_b,j|; the sets are nested, so the labels follow by inclusion-exclusion.
// nine == 0 (four-block form): only slots 4, 5, 7, 8 are Gram blocks; slots 0, 1, 2, 3, 6 hold the cells
// with an "other" label as k_other_fix counted them.  tr (het-anchored form, i not het): the pair is read from row
// j, slot a * 3 + b from slot b * 3 + a.
__device__ __forceinline__ uint32_t gram_table(const uint32_t* __restrict__ g, uint32_t S_pad, uint32_t i, uint32_t j,
                                               uint32_t nine, uint32_t T[9], bool tr = false) {
  const size_t plane = (size_t)S_pad * S_pad;
  const uint32_t* p = g + (tr ? (size_t)j * S_pad + i : (size_t)i * S_pad + j);
  uint32_t G[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) G[k] = __ldg(p + (size_t)k * plane);
  if (tr) {
    const uint32_t g1 = G[1], g2 = G[2], g5 = G[5];
    G[1] = G[3], G[3] = g1;
    G[2] = G[6], G[6] = g2;
    G[5] = G[7], G[7] = g5;
  }
  const uint32_t PP = G[4], PM = G[5], MP = G[7], MM = G[8];
  T[8] = MM;
  T[7] = MP - MM;            // i major, j minor
  T[5] = PM - MM;            // i minor, j major
  T[4] = PP - MP - PM + MM;
  if (nine) {
    const uint32_t CC = G[0], CP = G[1], CM = G[2], PC = G[3], MC = G[6];
    T[6] = MC - MP;                  // i major, j other
    T[3] = (PC - MC) - (PP - MP);    // i minor, j other
    T[2] = CM - PM;                  // i other, j major
    T[1] = (CP - CM) - (PP - PM);    // i other, j minor
    T[0] = CC - CP - PC + PP;
  } else {
    T[0] = G[0];
    T[1] = G[1];
    T[2] = G[2];
    T[3] = G[3];
    T[6] = G[6];
  }
  uint32_t n = 0;
#pragma unroll
  for (int k = 0; k < 9; ++k) n += T[k];
  return n;
}

// ---------------------------------------------------------------------------
// K1 + K2, generic path: up to 2048 consecutive pairs of any unit per work item,
// one thread per pair, planes read through L1/L2.  Handles everything the
// small-unit kernel (lgmi_fast_kernel.cuh) does not: units with more than 64
// sites or 256 reads, pair-less units, and small units with dense third alleles.
// The output offset of every item is known before the kernel starts (k_count +
// exclusive scan), so no CTA ever waits on another.
// kKind 1: only the items whose MI k_tile_mi / k_tile_finish has already computed (pure ordering and
// emission: few registers, four CTAs per SM to hide the loads); kKind 2: the items of the deep units,
// tables from the count matrices of the tensor-core path -- classified first, then the branch-free
// epilogues of lgmi_fast.cuh over full warps of each class; kKind 0: everything else.
// 2x2 block of a deep unit's table alone (the pairs without an "other" label need nothing else)
__device__ __forceinline__ void gram_table_2x2(const uint32_t* __restrict__ g, uint32_t S_pad, uint32_t i, uint32_t j,
                                               uint32_t& mm, uint32_t& mM, uint32_t& Mm, uint32_t& MM, bool tr = false) {
  const size_t plane = (size_t)S_pad * S_pad;
  const uint32_t* p = g + (tr ? (size_t)j * S_pad + i : (size_t)i * S_pad + j);
  const uint32_t PP = __ldg(p + 4u * plane), G5 = __ldg(p + 5u * plane), G7 = __ldg(p + 7u * plane);
  const uint32_t PM = tr ? G7 : G5, MP = tr ? G5 : G7;
  MM = __ldg(p + 8u * plane);
  Mm = MP - MM;
  mM = PM - MM;
  mm = PP - MP - PM + MM;
}

// a deep unit's pair (i, j), i < j, is read transposed from row j when the unit's count matrices are het-anchored
// (anchored: only the het sites' rows were written) and i is not het
__device__ __forceinline__ bool gram_tr(bool anchored, const uint8_t* flags, uint32_t i) {
  return anchored && (flags[i] & LGMI_SITE_TYPE_MASK) != LGMI_SITE_HET_SNP;
}

template <int kKind>
__global__ void __launch_bounds__(kThreads, kKind == 1 ? 4 : (kKind == 2 ? 3 : 2)) k_pairs_generic(const RunParams P) {
  constexpr bool kTiled = kKind == 1;
  __shared__ double s_mi_all[(kKind == 1 ? 2 : 1) * kPairsMax];  // MI of each pair of the item, NaN = no MI (kKind 1: and of the next item)
  __shared__ uint32_t s_ij[kPairsMax];  // (i << 16) | j
  __shared__ uint32_t s_warp[kThreads / 32];
  __shared__ uint16_t s_list[kKind == 2 ? kPairsMax : 1];  // kKind 2: pairs with a 2x2 table from the front, the others from the back
  __shared__ uint32_t s_tr[kKind == 2 ? kPairsMax / 32 : 1];  // kKind 2: bit pl: pair pl's table is read transposed (gram_tr)
  __shared__ uint32_t s_n2, s_n3;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const LnGlobal ln{P.lntab};
  const bool het_only = (P.mode & LGMI_MODE_HET_ONLY) != 0u;
  const bool skip_nonhet = het_only && (P.mode & LGMI_MODE_SKIP_NONHET) != 0u;
  if (kKind == 0 && *P.n_generic == 0u) return;  // every item was a small unit taken by k_pairs_fast

  // kTiled: the kernel walks its own list of item records (TiledDesc) and requests, a whole item ahead, the record
  // after the next and the MI values of the next item (k_tile_finish's output, 8 bytes per pair) by cp.async:
  // nothing of an item's input is waited for at its head.
  __shared__ TiledDesc s_desc[kTiled ? 3 : 1];
  const uint32_t n_loop = kTiled ? P.n_tiled_desc : P.n_items;
  uint32_t n_it = 0u;  // items this CTA has started
  auto request_desc = [&](uint32_t slot, uint32_t q) {
    if (tid < 3u && q < n_loop)
      cp_async16(reinterpret_cast<char*>(&s_desc[slot]) + 16u * tid, reinterpret_cast<const char*>(P.tiled_desc + q) + 16u * tid, true);
  };
  auto request_mi = [&](uint32_t slot, uint32_t half) {  // (the record in `slot` has landed)
    const TiledDesc& d = s_desc[slot];
    const double* src = P.dense + d.dense_off + d.pair_begin;
    double* dst = s_mi_all + half * kPairsMax;
    for (uint32_t pl = tid; pl < d.pair_cnt; pl += kThreads) cp_async8(dst + pl, src + pl);
  };
  if constexpr (kTiled) {
    request_desc(0u, blockIdx.x);
    request_desc(1u, blockIdx.x + gridDim.x);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    if (blockIdx.x < n_loop) request_mi(0u, 0u);
    cp_async_commit();
  }
  for (uint32_t q = blockIdx.x; q < n_loop; q += gridDim.x, ++n_it) {
    uint32_t item_idx = q;
    Item it;
    DevUnit u;
    double* const s_mi = s_mi_all + (kTiled ? (n_it & 1u) * kPairsMax : 0u);
    if constexpr (kTiled) {
      cp_async_wait<0>();
      __syncthreads();  // this item's record and MI values and the next record have landed; previous item fully consumed
      const TiledDesc d = s_desc[n_it % 3u];
      item_idx = d.item_idx;
      it.unit = d.unit, it.pair_begin = d.pair_begin, it.pair_cnt = d.pair_cnt, it.flags = d.flags;
      u = DevUnit{};
      u.S = d.S, u.site_off = d.site_off, u.dense_off = d.dense_off, u.tiled = 1u;
      // (the buffers written now were last read an item ago, before the barrier above)
      if (q + gridDim.x < n_loop) request_mi((n_it + 1u) % 3u, (n_it + 1u) & 1u);
      request_desc((n_it + 2u) % 3u, q + 2u * gridDim.x);
      cp_async_commit();
    } else {
      it = P.items[item_idx];
      if (it.flags & ITEM_TILED) continue;                              // another instantiation's
      if ((kKind == 2) != ((it.flags & ITEM_GRAM) != 0u)) continue;
      if ((it.flags & ITEM_FAST) && !P.item_dense[item_idx]) continue;  // k_pairs_fast's
      u = P.units[it.unit];
      __syncthreads();  // previous item fully consumed
    }
    unsigned long long item_out = 0ull;
    if constexpr (kTiled) item_out = P.item_off[item_idx];  // (needed after the counting pass: requested here)
    const uint32_t W4 = u.W >> 2;
    const uint4* __restrict__ base = reinterpret_cast<const uint4*>(P.planes + u.plane_off);
    const uint8_t* __restrict__ flags = P.site_flags + u.site_off;

    // ---- counts + MI for every candidate pair of the item
    uint32_t i = 0, j = 0;
    if (tid < it.pair_cnt) lg_pair_ij(it.pair_begin + tid, u.S, i, j);  // one square root per thread, then steps
    if constexpr (kTiled) {
      // k_tile_mi / k_tile_finish have been here (NaN: dropped / not evaluated) and the values are in s_mi already
      for (uint32_t pl = tid; pl < it.pair_cnt; pl += kThreads) {
        if (pl != tid) lg_pair_advance(i, j, u.S, kThreads);
        s_ij[pl] = (i << 16) | j;
      }
    } else if constexpr (kKind == 2) {
      const uint32_t nine = P.unit_mode[it.unit];
      const uint32_t* __restrict__ g = P.gram + u.gram_off;
      const uint32_t lt = (1u << lane) - 1u;
      if (tid == 0) {
        s_n2 = 0u;
        s_n3 = 0u;
      }
      __syncthreads();
      // pass 1: the tables -> min-common filter, class of every pair (NaN for those without MI)
      const uint32_t n_slots = (it.pair_cnt + 31u) & ~31u;
      for (uint32_t pl = tid; pl < n_slots; pl += kThreads) {
        uint32_t cls = 0u;  // 0 no MI, 2 -> 2x2 list, 3 -> 3x3 list
        bool tr = false;
        if (pl < it.pair_cnt) {
          if (pl != tid) lg_pair_advance(i, j, u.S, kThreads);
          s_ij[pl] = (i << 16) | j;
          bool evaluate = true;
          if (skip_nonhet)
            evaluate = ((flags[i] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP) ||
                       ((flags[j] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
          if (evaluate) {
            uint32_t T[9];
            tr = gram_tr(P.unit_het && P.unit_het[it.unit], flags, i);
            const uint32_t n_common = gram_table(g, u.S_pad, i, j, nine, T, tr);
            if ((int)n_common >= P.min_common)  // strict '<' drops (mutual_information.py:19)
              cls = (T[0] | T[1] | T[2] | T[3] | T[6]) ? 3u : 2u;
          }
          if (!cls) s_mi[pl] = lg_nan();
        }
        const uint32_t m2 = __ballot_sync(0xffffffffu, cls == 2u);
        const uint32_t m3 = __ballot_sync(0xffffffffu, cls == 3u);
        const uint32_t mt = __ballot_sync(0xffffffffu, tr);
        if (lane == 0) s_tr[pl >> 5] = mt;  // (a warp's 32 slots are consecutive pairs)
        uint32_t b2 = 0u, b3 = 0u;
        if (lane == 0) {
          if (m2) b2 = atomicAdd(&s_n2, (uint32_t)__popc(m2));
          if (m3) b3 = atomicAdd(&s_n3, (uint32_t)__popc(m3));
        }
        b2 = __shfl_sync(0xffffffffu, b2, 0);
        b3 = __shfl_sync(0xffffffffu, b3, 0);
        if (cls == 2u) s_list[b2 + __popc(m2 & lt)] = (uint16_t)pl;
        if (cls == 3u) s_list[kPairsMax - 1u - (b3 + __popc(m3 & lt))] = (uint16_t)pl;
      }
      __syncthreads();
      // pass 2: MI over warp-sized chunks of each class (the tables again: L2 hits)
      const uint32_t n2 = s_n2, n3 = s_n3;
      const uint32_t nc2 = (n2 + 31u) >> 5, nc3 = (n3 + 31u) >> 5;
      const GlobalTab tab{P.lntab};
      const bool small_counts = u.R <= kFastMathMaxCount;  // (else the straightforward arithmetic of lgmi_math.cuh)
      for (uint32_t c = warp; c < nc2 + nc3; c += kThreads / 32) {
        if (c < nc2) {
          const uint32_t q = c * 32u + lane;
          if (q < n2) {
            const uint32_t pl = s_list[q], ij = s_ij[pl];
            uint32_t mm, mM, Mm, MM;
            gram_table_2x2(g, u.S_pad, ij >> 16, ij & 0xffffu, mm, mM, Mm, MM, (s_tr[pl >> 5] >> (pl & 31u)) & 1u);
            s_mi[pl] = small_counts ? mi_2x2(tab, mm, mM, Mm, MM) : lg_mi_from_2x2(mm, mM, Mm, MM, ln);
          }
        } else {
          const uint32_t q = (c - nc2) * 32u + lane;
          if (q < n3) {
            const uint32_t pl = s_list[kPairsMax - 1u - q], ij = s_ij[pl];
            uint32_t T[9];
            gram_table(g, u.S_pad, ij >> 16, ij & 0xffffu, nine, T, (s_tr[pl >> 5] >> (pl & 31u)) & 1u);
            s_mi[pl] = small_counts ? mi_3x3(tab, T) : lg_mi_from_table(T, ln);
          }
        }
      }
    } else {
      for (uint32_t pl = tid; pl < it.pair_cnt; pl += kThreads) {
        if (pl != tid) lg_pair_advance(i, j, u.S, kThreads);
        s_ij[pl] = (i << 16) | j;
        double mi = lg_nan();
        bool evaluate = true;
        if (skip_nonhet)
          evaluate = ((flags[i] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP) ||
                     ((flags[j] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
        if (evaluate) {
          const uint4* ri = base + (size_t)i * 3u * W4;
          const uint4* rj = base + (size_t)j * 3u * W4;
          const uint32_t n_common = pair_common(ri, rj, W4);
          if ((int)n_common >= P.min_common) {  // strict '<' drops (mutual_information.py:19)
            uint32_t T[9];
            if (pair_table(ri, rj, W4, n_common, T))
              mi = lg_mi_from_2x2(T[4], T[5], T[7], T[8], ln);
            else
              mi = lg_mi_from_table(T, ln);
          }
        }
        s_mi[pl] = mi;
      }
    }
    __syncthreads();

    // ---- ordered write: each warp owns a contiguous, 32-aligned range of pairs
    const uint32_t per_warp = ((it.pair_cnt + kThreads - 1) / kThreads) * 32u;
    const uint32_t p_begin = warp * per_warp;
    const uint32_t p_end = min(p_begin + per_warp, it.pair_cnt);
    auto emitted = [&](uint32_t pl, double& mi, uint32_t& ij) -> bool {
      if (pl >= p_end) return false;
      mi = s_mi[pl];
      if (isnan(mi)) return false;
      ij = s_ij[pl];
      if (het_only)
        return ((flags[ij >> 16] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP) ||
               ((flags[ij & 0xffffu] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
      return true;
    };
    uint32_t mine = 0;
    for (uint32_t pl = p_begin + lane; pl < p_begin + per_warp; pl += 32) {
      double mi;
      uint32_t ij;
      mine += __popc(__ballot_sync(0xffffffffu, emitted(pl, mi, ij)));
    }
    if (lane == 0) s_warp[warp] = mine;
    __syncthreads();
    unsigned long long out = kTiled ? item_out : P.item_off[item_idx];
    if (tid == 0 && (it.flags & ITEM_FIRST)) P.unit_rec_off[it.unit] = out;
    for (uint32_t w = 0; w < warp; ++w) out += s_warp[w];
    for (uint32_t pl = p_begin + lane; pl < p_begin + per_warp; pl += 32) {
      double mi = 0.0;
      uint32_t ij = 0;
      const bool e = emitted(pl, mi, ij);
      const uint32_t bal = __ballot_sync(0xffffffffu, e);
      if (e) {
        const unsigned long long slot = out + __popc(bal & ((1u << lane) - 1u));
        uint4 rec;  // {unit, i | j << 16, mi}
        rec.x = it.unit + P.unit_base;
        rec.y = (ij >> 16) | (ij << 16);
        rec.z = (uint32_t)__double2loint(mi);
        rec.w = (uint32_t)__double2hiint(mi);
        reinterpret_cast<uint4*>(P.records)[slot] = rec;
        if (P.mode & LGMI_MODE_EMIT_COUNTS) {
          uint32_t T[9];
          if (u.tiled) {
            const uint32_t* src = P.tile_counts + (u.dense_off + it.pair_begin + pl) * 9ull;
#pragma unroll
            for (int k = 0; k < 9; ++k) T[k] = src[k];
          } else if (u.gram_off != kNoGram) {
            gram_table(P.gram + u.gram_off, u.S_pad, ij >> 16, ij & 0xffffu, P.unit_mode[it.unit], T,
                       kKind == 2 && ((s_tr[pl >> 5] >> (pl & 31u)) & 1u));
          } else {
            const uint4* ri = base + (size_t)(ij >> 16) * 3u * W4;
            const uint4* rj = base + (size_t)(ij & 0xffffu) * 3u * W4;
            pair_table(ri, rj, W4, pair_common(ri, rj, W4), T);
          }
#pragma unroll
          for (int k = 0; k < 9; ++k) P.counts[slot * 9ull + k] = T[k];
        }
      }
      out += __popc(bal);
    }

    // ---- per-site mean over the het-kept pairs (mutual_information.py:48-60)
    if (it.flags & ITEM_SINGLE) {
      for (uint32_t s = tid; s < u.S; s += kThreads) {
        const bool s_het = (flags[s] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP;
        lg_neumaier acc;
        lg_neumaier_init(acc);
        for (uint32_t t = 0; t < u.S; ++t) {
          if (t == s) continue;
          if (!s_het && (flags[t] & LGMI_SITE_TYPE_MASK) != LGMI_SITE_HET_SNP) continue;
          const uint32_t p = (t < s) ? (uint32_t)lg_row_off(t, u.S) + (s - t - 1u)
                                     : (uint32_t)lg_row_off(s, u.S) + (t - s - 1u);
          const double v = s_mi[p];
          if (!isnan(v)) lg_neumaier_add(acc, v);
        }
        P.site_mean[u.site_off + s] = lg_neumaier_mean(acc);
        P.site_cnt[u.site_off + s] = (uint32_t)acc.n;
      }
    } else if (!u.tiled) {
      for (uint32_t pl = tid; pl < it.pair_cnt; pl += kThreads) P.dense[u.dense_off + it.pair_begin + pl] = s_mi[pl];
    }
  }
}

// ---------------------------------------------------------------------------
// K1 + K2, tiled path: units too large for k_pairs_fast and too shallow for the
// tensor cores.  One CTA per 16 x 16 block of site pairs (upper block triangle),
// one pair per thread: the three planes of both site blocks are staged in shared
// memory 1 024 reads at a time; the nine AND+popcount sums of the pair run
// through a carry-save adder tree (Harley-Seal: 8 words -> 14 LOP3 + ONE POPC,
// the popcount pipe is a quarter-rate unit), and the fp64 epilogue writes the
// pair's MI (NaN: dropped by min-common / not evaluated) to the unit's dense
// scratch in pair order.  k_count / k_pairs_generic then only compact and order
// what is already there.
constexpr int kTileKC = 32;      // words of each plane per staged chunk
constexpr int kTileStride = 36;  // words per staged row: 16-byte aligned; 8 consecutive rows cover all 32 banks

// running bit-sliced count of one AND+popcount set
struct CsaAcc {
  uint32_t ones, twos, fours, eights;  // eights: already popcounted, in units of 8
  __device__ __forceinline__ void init() { ones = twos = fours = eights = 0u; }
  __device__ __forceinline__ static void csa(uint32_t& carry, uint32_t& sum, uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t s = a ^ b ^ c;
    carry = (a & b) | (c & (a ^ b));
    sum = s;
  }
  // eight words of x & y
  __device__ __forceinline__ void add8(const uint4& x0, const uint4& x1, const uint4& y0, const uint4& y1) {
    uint32_t ta, tb, fa, fb, e;
    csa(ta, ones, ones, x0.x & y0.x, x0.y & y0.y);
    csa(tb, ones, ones, x0.z & y0.z, x0.w & y0.w);
    csa(fa, twos, twos, ta, tb);
    csa(ta, ones, ones, x1.x & y1.x, x1.y & y1.y);
    csa(tb, ones, ones, x1.z & y1.z, x1.w & y1.w);
    csa(fb, twos, twos, ta, tb);
    csa(e, fours, fours, fa, fb);
    eights += (uint32_t)__popc(e);
  }
  __device__ __forceinline__ uint32_t total() const {
    return 8u * eights + 4u * (uint32_t)__popc(fours) + 2u * (uint32_t)__popc(twos) + (uint32_t)__popc(ones);
  }
};

// fp64 epilogue of one pair, straight from the registers
__device__ __forceinline__ void tile_epilogue(const RunParams& P, const TileItem& tile, const DevUnit& u,
                                              const CsaAcc (&acc)[9], uint32_t ty, uint32_t tx) {
  const uint32_t i = tile.I * (uint32_t)kTileSites + ty, j = tile.J * (uint32_t)kTileSites + tx;
  if (i >= j || j >= u.S) return;
  const LnGlobal ln{P.lntab};
  const uint8_t* __restrict__ flags = P.site_flags + u.site_off;
  const bool skip_nonhet = (P.mode & LGMI_MODE_HET_ONLY) && (P.mode & LGMI_MODE_SKIP_NONHET);
  const uint32_t N = acc[0].total();
  const uint32_t MM = acc[1].total(), Mm = acc[2].total(), mM = acc[3].total(), mm = acc[4].total();
  uint32_t T[9];
  T[8] = MM;
  T[7] = Mm;
  T[5] = mM;
  T[4] = mm;
  T[6] = acc[5].total() - MM - Mm;  // site1 major, site2 other
  T[3] = acc[6].total() - mM - mm;  // site1 minor, site2 other
  T[2] = acc[7].total() - MM - mM;  // site1 other, site2 major
  T[1] = acc[8].total() - Mm - mm;  // site1 other, site2 minor
  T[0] = N - (MM + Mm + mM + mm) - T[6] - T[3] - T[2] - T[1];
  double v = lg_nan();
  bool evaluate = true;
  if (skip_nonhet)
    evaluate = ((flags[i] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP) ||
               ((flags[j] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
  if (evaluate && (int)N >= P.min_common) {  // strict '<' drops (mutual_information.py:19)
    if ((T[0] | T[1] | T[2] | T[3] | T[6]) == 0u) v = lg_mi_from_2x2(mm, mM, Mm, MM, ln);
    else v = lg_mi_from_table(T, ln);
  }
  const uint64_t slot = u.dense_off + lg_row_off(i, u.S) + (j - i - 1u);
  P.dense[slot] = v;
  if (P.mode & LGMI_MODE_EMIT_COUNTS) {
#pragma unroll
    for (int k = 0; k < 9; ++k) P.tile_counts[slot * 9ull + k] = T[k];
  }
}

// stage one 1 024-read chunk of both site blocks of a tile: [block (i / j)][plane M, m, C][site][word]
typedef uint32_t TileRows[2][3][kTileSites][kTileStride];
__device__ __forceinline__ void tile_prefetch(TileRows& rows, const RunParams& P, const TileItem& tile, const DevUnit& u,
                                              uint32_t k0) {
  const uint32_t* __restrict__ planes = P.planes + u.plane_off;
  const uint32_t W = u.W;
  for (uint32_t e = threadIdx.x; e < 2u * 3u * kTileSites * (kTileKC / 4); e += kThreads) {
    const uint32_t q = e & 7u, row = e >> 3;  // row = (blk * 3 + plane) * 16 + site
    const uint32_t site = row & 15u, bp = row >> 4, plane = bp % 3u, blk = bp / 3u;
    const uint32_t s = (blk ? tile.J : tile.I) * (uint32_t)kTileSites + site;
    const bool have = s < u.S && k0 + 4u * q < W;  // absent words are zero-filled
    cp_async16(&rows[blk][plane][site][4u * q],
               planes + ((size_t)(have ? s : 0u) * 3u + plane) * W + (have ? k0 + 4u * q : 0u), have);
  }
}

// persistent: CTA c takes tiles c, c + grid, ...; the next chunk (of this tile or of the
// CTA's next tile) is in flight while the current one is counted
__global__ void __launch_bounds__(kThreads, 3) k_tile_mi(const RunParams P, const TileItem* __restrict__ tiles,
                                                         uint32_t n_tiles) {
  __shared__ __align__(16) TileRows s_rows[2];
  const uint32_t tid = threadIdx.x;
  const uint32_t ty = tid >> 4, tx = tid & 15u;  // pair (site0[0] + ty, site0[1] + tx)
  uint32_t t = blockIdx.x;
  if (t >= n_tiles) return;
  TileItem tile = tiles[t];
  DevUnit u = P.units[tile.unit];
  uint32_t buf = 0;
  tile_prefetch(s_rows[0], P, tile, u, 0u);
  cp_async_commit();

  while (true) {
    const uint32_t t_next = t + gridDim.x;
    TileItem tile_next = tile;
    DevUnit u_next = u;
    if (t_next < n_tiles) {
      tile_next = tiles[t_next];
      u_next = P.units[tile_next.unit];
    }
    const uint32_t W = u.W;
    CsaAcc acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k].init();

    for (uint32_t k0 = 0; k0 < W; k0 += (uint32_t)kTileKC) {
      // request what comes next into the other buffer (its last readers passed the barrier below)
      if (k0 + (uint32_t)kTileKC < W) tile_prefetch(s_rows[buf ^ 1u], P, tile, u, k0 + (uint32_t)kTileKC);
      else if (t_next < n_tiles) tile_prefetch(s_rows[buf ^ 1u], P, tile_next, u_next, 0u);
      cp_async_commit();
      cp_async_wait<1>();
      __syncthreads();
      const TileRows& rows = s_rows[buf];
      const uint32_t kw = min((uint32_t)kTileKC, (W - k0 + 7u) & ~7u);  // whole groups of 8 words (the tail is zeros)
      for (uint32_t k8 = 0; k8 < kw; k8 += 8u) {
        const uint4 Mi0 = *reinterpret_cast<const uint4*>(&rows[0][0][ty][k8]);
        const uint4 Mi1 = *reinterpret_cast<const uint4*>(&rows[0][0][ty][k8 + 4]);
        const uint4 mi0 = *reinterpret_cast<const uint4*>(&rows[0][1][ty][k8]);
        const uint4 mi1 = *reinterpret_cast<const uint4*>(&rows[0][1][ty][k8 + 4]);
        const uint4 Ci0 = *reinterpret_cast<const uint4*>(&rows[0][2][ty][k8]);
        const uint4 Ci1 = *reinterpret_cast<const uint4*>(&rows[0][2][ty][k8 + 4]);
        const uint4 Mj0 = *reinterpret_cast<const uint4*>(&rows[1][0][tx][k8]);
        const uint4 Mj1 = *reinterpret_cast<const uint4*>(&rows[1][0][tx][k8 + 4]);
        const uint4 mj0 = *reinterpret_cast<const uint4*>(&rows[1][1][tx][k8]);
        const uint4 mj1 = *reinterpret_cast<const uint4*>(&rows[1][1][tx][k8 + 4]);
        const uint4 Cj0 = *reinterpret_cast<const uint4*>(&rows[1][2][tx][k8]);
        const uint4 Cj1 = *reinterpret_cast<const uint4*>(&rows[1][2][tx][k8 + 4]);
        acc[0].add8(Ci0, Ci1, Cj0, Cj1);  // N
        acc[1].add8(Mi0, Mi1, Mj0, Mj1);
        acc[2].add8(Mi0, Mi1, mj0, mj1);
        acc[3].add8(mi0, mi1, Mj0, Mj1);
        acc[4].add8(mi0, mi1, mj0, mj1);
        acc[5].add8(Mi0, Mi1, Cj0, Cj1);
        acc[6].add8(mi0, mi1, Cj0, Cj1);
        acc[7].add8(Ci0, Ci1, Mj0, Mj1);
        acc[8].add8(Ci0, Ci1, mj0, mj1);
      }
      __syncthreads();  // this buffer may be refilled by the prefetch of the next iteration
      buf ^= 1u;
    }
    tile_epilogue(P, tile, u, acc, ty, tx);
    if (t_next >= n_tiles) break;
    t = t_next;
    tile = tile_next;
    u = u_next;
  }
  cp_async_wait<0>();
}

// ---------------------------------------------------------------------------
// K0: number of pairs each item will emit -- |Ci & Cj| >= min_common (and the
// het filter of the mode).  Its exclusive scan gives every item its place in
// the ordered output, so k_pairs needs no inter-CTA communication.
constexpr int kCountStride = 12;  // words per staged C row (48 B: conflict-free LDS.128)

// pairs a small unit will emit: |Ci & Cj| >= min_common (and the het filter of the mode) over the
// unit's C planes only.  Persistent CTAs over the fast items, the next unit's C rows in flight
// (cp.async) while the current one is counted; (i, j) from the per-S pair table.
struct CountFastParams {
  const FastItem* items;
  uint32_t n_items;
  const uint32_t* planes;
  const uint8_t* site_flags;
  const uint16_t* ij_tab;
  int min_common;
  uint32_t mode;
  unsigned long long* item_cnt;
  uint8_t* fast_empty;  // per fast item (same index as `items`): 1 when the unit emits nothing -> k_pairs_fast skips it
};

template <int NW>
__device__ __forceinline__ uint32_t count_fast_item(const uint32_t* __restrict__ s_c, unsigned long long het_mask,
                                                    const uint16_t* __restrict__ ijt, uint32_t n_pairs, int min_common,
                                                    bool need_het) {
  uint32_t mine = 0;
  for (uint32_t p = threadIdx.x; p < n_pairs; p += kThreads) {
    const uint32_t ij = __ldg(ijt + p);
    const uint32_t i = ij >> 6, j = ij & 63u;
    uint32_t a[8], b[8];
#pragma unroll
    for (int q = 0; q < (NW + 3) / 4; ++q) {
      const uint4 x = *reinterpret_cast<const uint4*>(s_c + i * kCountStride + 4 * q);
      const uint4 y = *reinterpret_cast<const uint4*>(s_c + j * kCountStride + 4 * q);
      a[4 * q] = x.x; a[4 * q + 1] = x.y; a[4 * q + 2] = x.z; a[4 * q + 3] = x.w;
      b[4 * q] = y.x; b[4 * q + 1] = y.y; b[4 * q + 2] = y.z; b[4 * q + 3] = y.w;
    }
    const uint32_t n = and_popc<NW>(a, b);
    const bool het = (((het_mask >> i) | (het_mask >> j)) & 1ull) != 0ull;
    mine += ((int)n >= min_common && (het || !need_het)) ? 1u : 0u;
  }
  return mine;
}

__global__ void __launch_bounds__(kThreads) k_count_fast(const CountFastParams P) {
  __shared__ __align__(16) uint32_t s_c[2][kFastMaxS * kCountStride];
  __shared__ uint32_t s_het[2][2];
  __shared__ uint32_t s_warp[kThreads / 32];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const bool need_het = (P.mode & LGMI_MODE_HET_ONLY) != 0u;  // (SKIP_NONHET implies HET_ONLY)

  auto request_rows = [&](uint32_t b, const FastItem& it) {  // C rows of a unit by cp.async
    const uint32_t W = it.W, W4 = W >> 2;
    const uint32_t* __restrict__ src = P.planes + it.plane_off + 2u * W;
    for (uint32_t e = tid; e < (uint32_t)it.S * 2u; e += kThreads) {
      const uint32_t s = e >> 1, half = e & 1u;
      const bool have = half < W4;
      cp_async16(&s_c[b][s * kCountStride + half * 4u], src + (size_t)s * 3u * W + (have ? half * 4u : 0u), have);
    }
  };
  auto load_flag = [&](const FastItem& it) -> uint32_t {  // one site's flag byte per thread of the first two warps
    return (tid < it.S) ? (uint32_t)P.site_flags[it.site_off + tid] : 0u;
  };
  auto store_het = [&](uint32_t b, uint32_t f) {
    if (warp < 2u) {
      const uint32_t m = __ballot_sync(0xffffffffu, (f & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
      if (lane == 0) s_het[b][warp] = m;
    }
  };

  uint32_t idx = blockIdx.x, buf = 0;
  FastItem it;
  if (idx < P.n_items) {
    it = P.items[idx];
    request_rows(0, it);
    store_het(0, load_flag(it) | (tid < it.S ? 0u : 3u));
  }
  cp_async_commit();
  while (idx < P.n_items) {
    const uint32_t idx_next = idx + gridDim.x;
    FastItem it_next = it;
    uint32_t f_next = 3u;  // not a site type: never het
    if (idx_next < P.n_items) {
      it_next = P.items[idx_next];
      request_rows(buf ^ 1u, it_next);
      if (tid < it_next.S) f_next = load_flag(it_next);  // consumed after this unit's pairs: the latency is hidden
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const uint32_t S = it.S, n_pairs = S * (S - 1u) / 2u;
    const uint16_t* __restrict__ ijt = P.ij_tab + lg_ij_tab_off(S);
    const unsigned long long het_mask = (unsigned long long)s_het[buf][0] | ((unsigned long long)s_het[buf][1] << 32);
    const uint32_t nw = ((uint32_t)it.R + 31u) >> 5;
    uint32_t mine;
    if (nw <= 2u) mine = count_fast_item<2>(s_c[buf], het_mask, ijt, n_pairs, P.min_common, need_het);
    else if (nw <= 4u) mine = count_fast_item<4>(s_c[buf], het_mask, ijt, n_pairs, P.min_common, need_het);
    else if (nw <= 7u) mine = count_fast_item<7>(s_c[buf], het_mask, ijt, n_pairs, P.min_common, need_het);
    else mine = count_fast_item<8>(s_c[buf], het_mask, ijt, n_pairs, P.min_common, need_het);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if (lane == 0) s_warp[warp] = mine;
    store_het(buf ^ 1u, f_next);
    __syncthreads();  // also: this unit's rows are consumed, the buffer may be refilled two iterations on
    if (tid == 0) {
      uint32_t tot = 0;
#pragma unroll
      for (int w = 0; w < kThreads / 32; ++w) tot += s_warp[w];
      P.item_cnt[it.item] = tot;
      P.fast_empty[idx] = tot == 0u ? 1 : 0;
    }
    it = it_next;
    idx = idx_next;
    buf ^= 1u;
  }
  cp_async_wait<0>();
}

__global__ void __launch_bounds__(kThreads) k_count(const RunParams P) {
  __shared__ uint32_t s_warp[kThreads / 32];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const bool het_only = (P.mode & LGMI_MODE_HET_ONLY) != 0u;
  const bool skip_nonhet = het_only && (P.mode & LGMI_MODE_SKIP_NONHET) != 0u;
  for (uint32_t item_idx = blockIdx.x; item_idx < P.n_items; item_idx += gridDim.x) {
    const Item it = P.items[item_idx];
    if (it.flags & (ITEM_FAST | ITEM_TILED_GRAM)) continue;  // counted by k_count_fast / k_tile_finish
    const DevUnit u = P.units[it.unit];
    const uint8_t* __restrict__ flags = P.site_flags + u.site_off;
    uint32_t mine = 0;
    __syncthreads();
    {
      const uint32_t W4 = u.W >> 2;
      const uint4* __restrict__ base = reinterpret_cast<const uint4*>(P.planes + u.plane_off);
      const bool need_ij = het_only || skip_nonhet || !u.tiled;
      uint32_t i = 0, j = 0;
      if (need_ij && tid < it.pair_cnt) lg_pair_ij(it.pair_begin + tid, u.S, i, j);
      for (uint32_t pl = tid; pl < it.pair_cnt; pl += kThreads) {
        if (need_ij && pl != tid) lg_pair_advance(i, j, u.S, kThreads);
        if (het_only || skip_nonhet) {
          const bool het = ((flags[i] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP) ||
                           ((flags[j] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
          if (!het) continue;
        }
        if (u.tiled) {  // survivors are the pairs k_tile_mi gave an MI
          mine += isnan(P.dense[u.dense_off + it.pair_begin + pl]) ? 0u : 1u;
          continue;
        }
        uint32_t n;
        if (u.gram_off != kNoGram) {
          const bool anchored = P.unit_het && P.unit_het[it.unit];
          uint32_t T[9];
          n = gram_table(P.gram + u.gram_off, u.S_pad, i, j, P.unit_mode[it.unit], T, gram_tr(anchored, flags, i));
        } else {
          n = pair_common(base + (size_t)i * 3u * W4, base + (size_t)j * 3u * W4, W4);
        }
        mine += ((int)n >= P.min_common) ? 1u : 0u;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if (lane == 0) s_warp[warp] = mine;
    __syncthreads();
    if (tid == 0) {
      uint32_t tot = 0;
#pragma unroll
      for (int w = 0; w < kThreads / 32; ++w) tot += s_warp[w];
      P.item_cnt[item_idx] = tot;
    }
  }
}

// Per-site mean for units whose pairs span several work items; reads the dense per-unit MI
// scratch (pair order = upper triangle of the symmetric site x site matrix).  One CTA per 32
// consecutive sites: 32 x 32 tiles of the matrix are staged in shared memory with coalesced
// cp.async loads -- partners below the site block come from the partners' rows, partners above from
// the sites' rows, stored transposed -- four tiles in flight, and warp 0 runs the 32 compensated sums
// side by side, one site per lane, partners ascending.  The order of the additions is part of
// the result (mutual_information.py:56-58 is a left-to-right float sum), so each site's sum is
// serial; the 32 sites of a block are not.
constexpr int kMeanThreads = 256;
constexpr int kMeanBufs = 5;      // tile buffers: one being summed, one being masked, three in flight
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src, bool copy) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int n = copy ? 8 : 0;  // src-size 0: the 8 destination bytes are zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(gmem_src), "r"(n) : "memory");
}

__global__ void __launch_bounds__(kMeanThreads) k_site_mean_dense(const DevUnit* __restrict__ units,
                                                                 const MeanItem* __restrict__ items,
                                                                 const uint8_t* __restrict__ site_flags,
                                                                 const double* __restrict__ dense,
                                                                 double* __restrict__ site_mean,
                                                                 uint32_t* __restrict__ site_cnt) {
  __shared__ double s_tile[kMeanBufs][32][33];  // [buffer][partner][site]
  __shared__ uint32_t s_phet[kMeanBufs];        // bit tl: partner t0 + tl is a het_snp
  const MeanItem mi = items[blockIdx.x];
  const DevUnit u = units[mi.unit];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t S = u.S, s0 = mi.site_begin;
  const uint8_t* __restrict__ flags = site_flags + u.site_off;
  const double* __restrict__ d = dense + u.dense_off;
  const uint32_t n_blocks = (S + 31u) >> 5;

  // a tile by cp.async (nobody waits on its own loads): partners t0 .. t0 + 31 against sites s0 .. s0 + 31
  auto request_tile = [&](uint32_t tb) {
    if (tb < n_blocks && warp != 0u) {  // (warps 1-7: warp 0 only sums)
      const uint32_t t0 = tb << 5, b = tb % kMeanBufs;
      if (t0 + 32u <= s0) {
        // partners below the site block: a warp copies 32 consecutive entries of one partner's row per step
        const uint32_t s_ = s0 + lane;
        for (uint32_t tl = warp - 1u; tl < 32u; tl += 7u) {
          const uint32_t t = t0 + tl;  // (t < s0 <= s_: a pair, t a real site)
          const bool ok = s_ < S;
          cp_async8(&s_tile[b][tl][lane], d + (ok ? lg_row_off(t, S) + (s_ - t - 1u) : 0ull), ok);
        }
      } else if (t0 >= s0 + 32u) {
        // partners above it: 32 consecutive entries of one site's row per step
        const uint32_t t = t0 + lane;
        for (uint32_t sl = warp - 1u; sl < 32u; sl += 7u) {
          const uint32_t s_ = s0 + sl;  // (s_ < t)
          const bool ok = t < S && s_ < S;
          cp_async8(&s_tile[b][lane][sl], d + (ok ? lg_row_off(s_, S) + (t - s_ - 1u) : 0ull), ok);
        }
      } else {
        // the diagonal block: either side of each site
        for (uint32_t e = tid - 32u; e < 1024u; e += kMeanThreads - 32u) {
          const uint32_t tl = e >> 5, sl = e & 31u;
          const uint32_t t = t0 + tl, s_ = s0 + sl;
          const bool ok = t < S && s_ < S && t != s_;
          const uint64_t idx = ok ? ((t < s_) ? lg_row_off(t, S) + (s_ - t - 1u) : lg_row_off(s_, S) + (t - s_ - 1u)) : 0ull;
          cp_async8(&s_tile[b][tl][sl], d + idx, ok);
        }
      }
      if (warp == 1u) {
        const uint32_t t = t0 + lane;
        const uint32_t m = __ballot_sync(0xffffffffu, t < S && (flags[t < S ? t : 0u] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
        if (lane == 0) s_phet[b] = m;
      }
    }
    cp_async_commit();  // (an empty group keeps the count of groups per tile at one)
  };

  const uint32_t s = s0 + lane;  // (a thread's entries of a tile all belong to site s0 + lane)
  const bool s_ok = s < S;
  const bool s_het = s_ok && (flags[s_ok ? s : 0u] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP;
  // all MI values are >= +0.0: CPython's compensated sum (mutual_information.py:56-58) without branches;
  // an absent value adds +0.0, which leaves sum and compensation as they are.  Per tile: every thread first
  // replaces the entries that do not count (no MI, the site itself, neither site a het_snp) by +0.0 and counts
  // the others; warp 0 then runs the 32 serial sums over plain values -- two dependent fp64 additions per step
  // (sum, compensation); the rounding error of each addition comes from the branch-free two_sum_err.
  double acc_s = 0.0, acc_c = 0.0;
  uint32_t my_n = 0;
  __shared__ uint32_t s_n[32];
  if (tid < 32u) s_n[tid] = 0u;
  auto mask_tile = [&](uint32_t tb) {  // warps 1-7: entries (partner warp - 1 + 7 q, site s0 + lane) of tile tb
    if (tb >= n_blocks || warp == 0u) return;
    const uint32_t b = tb % kMeanBufs, t0 = tb << 5;
    const uint32_t partners = s_het ? 0xffffffffu : s_phet[b];  // a non-het site sums over its het partners only
#pragma unroll
    for (uint32_t q = 0; q < 5u; ++q) {
      const uint32_t tl = warp - 1u + 7u * q, t = t0 + tl;
      if (tl >= 32u) break;
      const double v = s_tile[b][tl][lane];
      const bool have = s_ok && t < S && t != s && ((partners >> tl) & 1u) && __double2hiint(v) < 0x7ff00000;  // NaN: no MI
      s_tile[b][tl][lane] = have ? v : 0.0;
      my_n += have ? 1u : 0u;
    }
  };
  // one barrier per tile: while warp 0 sums tile tb, warps 1-7 mask tile tb + 1 and request
  // tile tb + kMeanBufs - 1 into the buffer of tile tb - 1
#pragma unroll
  for (uint32_t tb = 0; tb + 1u < (uint32_t)kMeanBufs; ++tb) request_tile(tb);
  cp_async_wait<kMeanBufs - 2>();  // tile 0 has landed (this thread's part; the barrier covers the rest)
  __syncthreads();
  mask_tile(0u);
  for (uint32_t tb = 0; tb < n_blocks; ++tb) {
    cp_async_wait<kMeanBufs - 3>();  // tile tb + 1
    __syncthreads();                 // ... everybody's part of it; tile tb is masked; tile tb - 1 is summed
    request_tile(tb + kMeanBufs - 1u);
    mask_tile(tb + 1u);
    if (warp == 0) {                 // one site per lane, partners ascending
      const uint32_t b = tb % kMeanBufs;
#pragma unroll 8
      for (uint32_t tl = 0; tl < 32u; ++tl) {
        const double x = s_tile[b][tl][lane];
        const double tt = __dadd_rn(acc_s, x);
        acc_c = __dadd_rn(acc_c, two_sum_err(acc_s, x, tt));
        acc_s = tt;
      }
    }
  }
  cp_async_wait<0>();
  if (my_n) atomicAdd(&s_n[lane], my_n);
  __syncthreads();
  if (warp == 0 && s_ok) {
    const uint32_t acc_n = s_n[lane];
    double mean = lg_nan();
    if (acc_n) {
      double tot = acc_s;
      if (acc_c != 0.0) tot = __dadd_rn(tot, acc_c);
      mean = __ddiv_rn(tot, (double)acc_n);
    }
    site_mean[u.site_off + s] = mean;
    site_cnt[u.site_off + s] = acc_n;
  }
}

// Input in the packed two-plane form (2 bits per site and read: 00 not covered, 01 major,
// 10 minor, 11 other; row of site s = [b0 | b1]): a third fewer bytes over PCIe than [M | m | C].
// Expanded on the device into the [M | m | C] rows every kernel reads.  One CTA per unit.
// tight_off == NULL: plane rows keep their padded width W (unit k starts at 2/3 of its plane_off);
// else the rows are ceil(R/32) words wide and unit k starts at word tight_off[k] (LGMI_MODE_TIGHT_INPUT:
// no 128-read padding on the wire -- 56 instead of 64 bytes per site at 200 reads).
__global__ void __launch_bounds__(256) k_unpack2(const DevUnit* __restrict__ units, uint32_t n_units,
                                                 const uint32_t* __restrict__ packed, uint32_t* __restrict__ planes,
                                                 const unsigned long long* __restrict__ tight_off) {
  for (uint32_t k = blockIdx.x; k < n_units; k += gridDim.x) {
    const DevUnit u = units[k];
    if (tight_off) {
      const uint32_t W = u.W, Wt = (u.R + 31u) >> 5;
      const uint32_t* __restrict__ src = packed + tight_off[k];
      uint32_t* __restrict__ dst = planes + u.plane_off;
      for (uint32_t e = threadIdx.x; e < u.S * W; e += blockDim.x) {
        const uint32_t s = e / W, q = e - s * W;
        const uint32_t b0 = q < Wt ? __ldg(src + (size_t)s * 2u * Wt + q) : 0u;
        const uint32_t b1 = q < Wt ? __ldg(src + (size_t)s * 2u * Wt + Wt + q) : 0u;
        uint32_t* row = dst + (size_t)s * 3u * W + q;
        row[0] = b0 & ~b1;
        row[W] = b1 & ~b0;
        row[2u * W] = b0 | b1;
      }
      continue;
    }
    const uint32_t W4 = u.W >> 2;
    const uint4* __restrict__ src = reinterpret_cast<const uint4*>(packed + u.plane_off / 3u * 2u);
    uint4* __restrict__ dst = reinterpret_cast<uint4*>(planes + u.plane_off);
    for (uint32_t e = threadIdx.x; e < u.S * W4; e += blockDim.x) {
      const uint32_t s = e / W4, q = e - s * W4;
      const uint4 b0 = __ldg(src + (size_t)s * 2u * W4 + q), b1 = __ldg(src + (size_t)s * 2u * W4 + W4 + q);
      uint4* row = dst + (size_t)s * 3u * W4 + q;
      row[0] = make_uint4(b0.x & ~b1.x, b0.y & ~b1.y, b0.z & ~b1.z, b0.w & ~b1.w);       // major
      row[W4] = make_uint4(b1.x & ~b0.x, b1.y & ~b0.y, b1.z & ~b0.z, b1.w & ~b0.w);      // minor
      row[2u * W4] = make_uint4(b0.x | b1.x, b0.y | b1.y, b0.z | b1.z, b0.w | b1.w);     // covered
    }
  }
}

// Output in split form: MI values and the site indices of the emitted pairs as two arrays (12 bytes
// per row over PCIe instead of 16; the unit of a row follows from unit_rec_off).  rec_ij: i | j << 16;
// rec_ij16 (units of at most 256 sites): i | j << 8 -- 10 bytes per row.
__global__ void __launch_bounds__(256) k_split_records(const Header* __restrict__ header,
                                                       const lgmi_pair_rec* __restrict__ records,
                                                       double* __restrict__ rec_mi, uint32_t* __restrict__ rec_ij,
                                                       uint16_t* __restrict__ rec_ij16) {
  const unsigned long long n = header->n_records;
  for (unsigned long long r = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; r < n;
       r += (unsigned long long)gridDim.x * blockDim.x) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(records) + r);  // {unit, i | j << 16, mi}
    if (rec_ij16) rec_ij16[r] = (uint16_t)((v.y & 0xffu) | ((v.y >> 16) << 8));
    else rec_ij[r] = v.y;
    rec_mi[r] = __hiloint2double((int)v.w, (int)v.z);
  }
}

// start of a run: header and offsets zeroed, no item flagged, the count of items for
// k_pairs_generic seeded, every site's mean = NaN / cnt = 0 (sites of units without a
// pair, S < 2, keep that; everything else is overwritten)
__global__ void k_run_init(Header* __restrict__ header, Header* __restrict__ host_header,
                           unsigned long long* __restrict__ unit_rec_off, uint32_t n_off,
                           uint8_t* __restrict__ item_dense, uint32_t n_items, uint32_t* __restrict__ n_generic,
                           uint32_t n_generic0, double* __restrict__ mean, uint32_t* __restrict__ cnt, uint64_t n_sites) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0) {
    header->n_records = 0ull;
    header->pad = 0ull;
    *n_generic = n_generic0;
    if (host_header) {  // pinned host memory (unified addressing): the pipelined step reads the count from there
      host_header->n_records = 0ull;
      host_header->pad = 0ull;
    }
  }
  if (k < n_off) unit_rec_off[k] = 0ull;
  if (k < n_items) item_dense[k] = 0;
  if (k < n_sites) {
    mean[k] = lg_nan();
    cnt[k] = 0u;
  }
}

// after the scan: the total goes to the header and closes the per-unit offsets
__global__ void k_scan_finish(const unsigned long long* __restrict__ total, Header* __restrict__ header,
                              Header* __restrict__ host_header, unsigned long long* __restrict__ unit_rec_off_end) {
  if (threadIdx.x == 0) {
    header->n_records = *total;
    *unit_rec_off_end = *total;
    if (host_header) {
      host_header->n_records = *total;
      __threadfence_system();
    }
  }
}

// mean_mismatch_pair_mutual_info on caller-supplied rows (CSR by site)
__global__ void k_site_mean_csr(const unsigned long long* __restrict__ off,
                                const double* __restrict__ val, uint64_t n, double* __restrict__ out) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  lg_neumaier acc;
  lg_neumaier_init(acc);
  for (unsigned long long k = off[s]; k < off[s + 1]; ++k) lg_neumaier_add(acc, val[k]);
  out[s] = lg_neumaier_mean(acc);
}

// ---------------------------------------------------------------------------
// K4: ecdf / mip / call
__global__ void k_ecdf_keys(const double* __restrict__ mean, const uint8_t* __restrict__ flags,
                            uint64_t n, double* __restrict__ keys, unsigned long long* __restrict__ n_het) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool het = false;
  if (k < n) {
    const double v = mean[k];
    het = !isnan(v) && ((flags[k] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP);
    keys[k] = het ? v : __longlong_as_double(0x7ff0000000000000LL);  // +inf sorts last
  }
  const uint32_t bal = __ballot_sync(0xffffffffu, het);
  if ((threadIdx.x & 31u) == 0 && bal) atomicAdd(n_het, (unsigned long long)__popc(bal));
}

__device__ __forceinline__ uint64_t lower_bound(const double* __restrict__ x, uint64_t n, double v) {
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if (x[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void k_ecdf_mip(const double* __restrict__ mean, const uint8_t* __restrict__ flags,
                           uint64_t n, const double* __restrict__ sorted_keys,
                           const unsigned long long* __restrict__ n_het_p, double threshold,
                           double* __restrict__ mip, uint8_t* __restrict__ call) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint64_t n_het = *n_het_p;
  const double v = mean[k];
  double p = lg_nan();
  uint8_t c = 0;
  if (!isnan(v) && n_het > 0) {
    p = lg_ecdf_y(lower_bound(sorted_keys, n_het, v), n_het);
    const bool is_mm = (flags[k] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_MISMATCH;
    if (p <= threshold && is_mm) c = 1;
    else if (p > threshold && !is_mm) c = 2;
  }
  mip[k] = p;
  if (call) call[k] = c;
}

// numpy.sort puts every NaN last whatever its sign or payload; the radix sort orders by bit pattern,
// so NaNs become the canonical quiet NaN (sorts after +inf) first.  Counts them.
__global__ void k_canon_nan(double* __restrict__ x, uint64_t n, unsigned long long* __restrict__ n_nan) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool nan = false;
  if (k < n) {
    nan = isnan(x[k]);
    if (nan) x[k] = lg_nan();
  }
  const uint32_t bal = __ballot_sync(0xffffffffu, nan);
  if ((threadIdx.x & 31u) == 0 && bal) atomicAdd(n_nan, (unsigned long long)__popc(bal));
}

// ecdf(x)(samples) with x already sorted on the device (NaNs, if any, at the end)
__global__ void k_ecdf_eval(const double* __restrict__ sorted_x, uint64_t n, const unsigned long long* __restrict__ n_nan,
                            const double* __restrict__ samples, uint64_t m, double* __restrict__ out) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m) return;
  const double v = samples[k];
  // np.searchsorted orders NaN after everything: a NaN sample lands on the first NaN of x (or at the end)
  const uint64_t n_num = n - *n_nan;
  const uint64_t idx = isnan(v) ? n_num : lower_bound(sorted_x, n_num, v);
  out[k] = lg_ecdf_y(idx, n);
}

// the ECDF ordinates y = [0] ++ linspace(1/n, 1, n) of stat.py:19, all n + 1 of them
__global__ void k_ecdf_ordinates(uint64_t n, double* __restrict__ y) {
  const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k <= n) y[k] = lg_ecdf_y(k, n);
}

}  // namespace lgmi

#include "lgmi_tilegram.cuh"
