// lgmi_sitesplice.cuh -- sm_100a kernels of the site x splice-site MI (lgmi_site_splice_mi), the reference's
// second mutual_info_score call site: giremi/script/calculate_site_splice_mi.py:106-125.
//
// For a requested triple (site, allele X, splice Y), over the N list entries of the site (a read listed twice counts
// twice): x entries whose read is in X's list at the site, y whose read is in Y's list, xy both.  The 2x2 table
// [[N-x-y+xy, y-xy], [x-xy, xy]] (rows "with seq", columns "with splice") goes through the epilogue of the main step.
//
//   k_ss_keys    key site << read_bits | read and the allele index of every entry, for the CUB radix sort that
//                groups the entries by (site, read).
//   k_ss_count   one work item = (site, tile of up to kSsTileCols requested splice sites, chunk of up to kSsChunk
//                sorted entries).  The head of each (site, read) run takes the run's length and allele bit mask,
//                intersects the read's sorted splice ids with the tile's sorted columns, and accumulates x[a], y[c]
//                and xy[a][c] as integers in shared memory; the tile's triples then add theirs to global counts.
//                Integer atomics only: the result does not depend on the order, and no CTA waits for another.
//   k_ss_mi      one thread per triple: the table and its MI (mi_2x2 up to kFastMathMaxCount entries, above that
//                lg_mi_from_2x2, as k_pairs_generic selects them), written in triple order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lgmi_kernels.cuh"  // GlobalTab, LnGlobal, mi_2x2, lg_mi_from_2x2, kFastMathMaxCount

namespace lgmi {

constexpr int kSsThreads = 256;
constexpr uint32_t kSsMaxAlleles = 64;    // one bit per allele in a run's mask
constexpr uint32_t kSsTileCols = 128;     // requested splice sites per work item: 32 KB of xy counts for 64 alleles
constexpr uint32_t kSsChunk = 4096;       // sorted entries per work item

struct SsItem {
  unsigned long long e0;  // first sorted entry of the chunk
  uint32_t n_e;           // entries in the chunk (>= 1)
  uint32_t site;
  uint32_t slot0;         // first column (requested splice site of the site) of the tile
  uint32_t n_cols;        // columns in the tile (>= 1)
  uint32_t n_rows;        // alleles counted: 1 + the largest allele index requested at the site
  uint32_t pad;
};

// the site of sorted-or-unsorted entry p: the last s with entry_off[s] <= p (empty sites are never it)
__global__ void k_ss_keys(const unsigned long long* __restrict__ entry_off, uint32_t n_sites,
                          const uint32_t* __restrict__ entry_read, const uint32_t* __restrict__ entry_allele,
                          unsigned long long n, uint32_t read_bits, unsigned long long* __restrict__ keys,
                          uint8_t* __restrict__ alleles) {
  for (unsigned long long p = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; p < n;
       p += (unsigned long long)gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = n_sites;  // entry_off[lo] <= p < entry_off[hi]
    while (hi - lo > 1u) {
      const uint32_t mid = (lo + hi) >> 1;
      if (entry_off[mid] <= p) lo = mid; else hi = mid;
    }
    keys[p] = ((unsigned long long)lo << read_bits) | entry_read[p];
    alleles[p] = (uint8_t)entry_allele[p];
  }
}

__global__ void __launch_bounds__(kSsThreads) k_ss_count(
    const SsItem* __restrict__ items, const unsigned long long* __restrict__ keys, const uint8_t* __restrict__ alleles,
    const unsigned long long* __restrict__ entry_off, unsigned long long read_mask,
    const unsigned long long* __restrict__ splice_off, const uint32_t* __restrict__ splice_id,
    const uint32_t* __restrict__ slot_splice, const uint32_t* __restrict__ slot_tri_off,
    const uint32_t* __restrict__ tri_order, const uint8_t* __restrict__ tri_allele, uint32_t* __restrict__ counts) {
  __shared__ uint32_t s_xy[kSsMaxAlleles * kSsTileCols];  // [allele][column]
  __shared__ uint32_t s_y[kSsTileCols], s_cols[kSsTileCols], s_x[kSsMaxAlleles];
  const SsItem it = items[blockIdx.x];
  const uint32_t tid = threadIdx.x;
  for (uint32_t k = tid; k < it.n_rows * kSsTileCols; k += kSsThreads) s_xy[k] = 0u;
  for (uint32_t k = tid; k < it.n_cols; k += kSsThreads) {
    s_y[k] = 0u;
    s_cols[k] = slot_splice[it.slot0 + k];
  }
  if (tid < kSsMaxAlleles) s_x[tid] = 0u;
  __syncthreads();
  const unsigned long long site_lo = entry_off[it.site], site_hi = entry_off[it.site + 1];
  const unsigned long long rows = it.n_rows >= 64u ? ~0ull : (1ull << it.n_rows) - 1ull;
  const uint32_t first = s_cols[0], last = s_cols[it.n_cols - 1];
  for (uint32_t q = tid; q < it.n_e; q += kSsThreads) {
    const unsigned long long p = it.e0 + q;
    const unsigned long long key = keys[p];
    if (p > site_lo && keys[p - 1] == key) continue;  // not the head of its (site, read) run
    unsigned long long mask = 1ull << alleles[p];      // the run: its read's alleles at the site, and its length
    uint32_t len = 1u;
    for (unsigned long long r = p + 1; r < site_hi && keys[r] == key; ++r, ++len) mask |= 1ull << alleles[r];
    mask &= rows;
    for (unsigned long long m = mask; m; m &= m - 1ull) atomicAdd(&s_x[__ffsll((long long)m) - 1], len);
    const unsigned long long read = key & read_mask;
    const unsigned long long b = splice_off[read], e = splice_off[read + 1];
    for (unsigned long long k = b; k < e; ++k) {
      const uint32_t sid = splice_id[k];
      if (sid < first) continue;
      if (sid > last) break;
      uint32_t lo = 0, hi = it.n_cols;
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (s_cols[mid] < sid) lo = mid + 1u; else hi = mid;
      }
      if (s_cols[lo] != sid) continue;  // lo < n_cols: sid <= last
      atomicAdd(&s_y[lo], len);
      for (unsigned long long m = mask; m; m &= m - 1ull)
        atomicAdd(&s_xy[(uint32_t)(__ffsll((long long)m) - 1) * kSsTileCols + lo], len);
    }
  }
  __syncthreads();
  for (uint32_t c = tid; c < it.n_cols; c += kSsThreads) {
    const uint32_t slot = it.slot0 + c, y = s_y[c];
    for (uint32_t k = slot_tri_off[slot]; k < slot_tri_off[slot + 1]; ++k) {
      const uint32_t t = tri_order[k], a = tri_allele[t];
      const uint32_t x = s_x[a], xy = s_xy[a * kSsTileCols + c];
      if (x) atomicAdd(&counts[3ull * t], x);
      if (y) atomicAdd(&counts[3ull * t + 1], y);
      if (xy) atomicAdd(&counts[3ull * t + 2], xy);
    }
  }
}

__global__ void k_ss_mi(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ tri_site,
                        const unsigned long long* __restrict__ entry_off, unsigned long long n_tri,
                        const lg_dd* __restrict__ lntab, double* __restrict__ mi, uint32_t* __restrict__ table) {
  const unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  if (t >= n_tri) return;
  const uint32_t s = tri_site[t];
  const uint32_t N = (uint32_t)(entry_off[s + 1] - entry_off[s]);
  const uint32_t x = counts[3 * t], y = counts[3 * t + 1], xy = counts[3 * t + 2];
  const uint32_t mm = N - x - y + xy, mM = y - xy, Mm = x - xy, MM = xy;  // rows with seq, columns with splice
  const GlobalTab tab{lntab};
  mi[t] = N <= kFastMathMaxCount ? mi_2x2(tab, mm, mM, Mm, MM) : lg_mi_from_2x2(mm, mM, Mm, MM, LnGlobal{lntab});
  if (table) {
    table[4 * t] = mm;
    table[4 * t + 1] = mM;
    table[4 * t + 2] = Mm;
    table[4 * t + 3] = MM;
  }
}

}  // namespace lgmi
