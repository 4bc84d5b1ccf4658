// lgmi_tilegram.cuh -- the mid-depth path: units too large for k_pairs_fast (more than
// 64 sites or 256 reads) and too shallow for k_gram_i8's one-GEMM-per-unit form, counted
// on the tensor cores in ONE batched launch over all of them.
//
//   k_tile_gram_ws work item = (unit, block I of 128 sites, block J of 48 sites) with some pair
//                 i < j.  Per 128-read k-block the CTA expands the unit's bit-planes IN THE
//                 KERNEL (no indicator matrix in HBM, no TMA) straight into the K-major
//                 128-byte-swizzled shared-memory layout tcgen05 reads:
//                     A_a  128 rows (site i, label a), a = other / minor / major   3 x 16 KB
//                     B    144 rows (label b major: row = 48 b + j)                    18 KB
//                 and one thread issues, per K = 32 step, three
//                 tcgen05.mma.cta_group::1.kind::i8 M=128 N=144 -- one per label a, each into
//                 its own 144 TMEM columns.  A TMEM lane is then a SITE: the thread that owns
//                 lane i reads the nine cells of pair (i, j) from its own lane
//                 (D_a[i][48 b + j]) without a shuffle.  Expansion, MMAs and readout run in
//                 their own warps over two smem stages (mbarriers, bounded waits); the readout
//                 (tcgen05.ld 32x32b.x8) writes nine u16 counts + flag bits per pair (24 B)
//                 into a scratch in pair order.
//   k_tile_finish one thread per pair: min-common filter + fp64 MI from the nine counts ->
//                 the unit's dense MI scratch (NaN: dropped / not evaluated) and the number of
//                 emitted pairs per work item (what k_count does for the other paths).
// k_pairs_generic<1> / k_site_mean_dense then order, emit and average as for k_tile_mi,
// which stays as the popcount form of this path (lgmi_set_tile_path(ctx, 0); units deeper
// than 65 535 reads, whose counts do not fit 16 bits, always take it).
//
// Reference semantics: the counts of /root/reference/src/giremi/mutual_information.py:15-40
// (labels over the common reads, strict '<' drop at :19), bit-exact; MI as lgmi_math.cuh.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// (included at the end of lgmi_kernels.cuh: RunParams and LnGlobal are defined there; the tile shape
// kTgSitesI x kTgSitesJ, kTgMaxReads and TgTile in lgmi_plan.h)

namespace lgmi {

constexpr int kTgSites = kTgSitesI + kTgSitesJ;       // plane rows a tile reads per k-block
constexpr int kTgN = 3 * kTgSitesJ;                   // 144 columns per accumulator (label-major)
constexpr uint32_t kTgATile = 128u * 128u;            // one label tile of A: 128 rows x 128 reads, 16 KB
constexpr uint32_t kTgABytes = 3u * kTgATile;         // 48 KB
constexpr uint32_t kTgBBytes = (uint32_t)kTgN * 128u; // 18 KB
constexpr uint32_t kTgStageBytes = kTgABytes + kTgBBytes;
constexpr int kTgStages = 2;                          // expanded operand stages
constexpr int kTgAhead = 2;                           // k-blocks of raw planes requested ahead (cp.async)
constexpr int kTgRawStages = kTgAhead + 1;
constexpr uint32_t kTgLutBytes = 256u * 8u;           // 8 bits -> 8 bytes
constexpr uint32_t kTgTmemCols = 512;                 // 3 x 144 used

// flag bits of a pair's 24-byte count record
constexpr uint32_t kTgNotEvaluated = 1u;  // SKIP_NONHET and no het_snp partner
constexpr uint32_t kTgHetPair = 2u;       // one of the two sites is a het_snp

__device__ __forceinline__ void tmem_load_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// 8 bits -> 8 bytes of 0/1 from a 256-entry shared-memory table (2 KB): two look-ups replace the sixteen
// shift / multiply / mask operations of four spread4 calls
__device__ __forceinline__ void tg_lut_init(uint2* __restrict__ lut, uint32_t tid, uint32_t n_threads) {
  for (uint32_t k = tid; k < 256u; k += n_threads) lut[k] = make_uint2(spread4(k & 15u), spread4(k >> 4));
}
__device__ __forceinline__ uint4 tg_spread16(const uint2* __restrict__ lut, uint32_t bits) {
  const uint2 lo = lut[bits & 0xffu], hi = lut[(bits >> 8) & 0xffu];
  return make_uint4(lo.x, lo.y, hi.x, hi.y);
}

__device__ __forceinline__ void tg_store(uint8_t* __restrict__ Xkb, uint32_t row, uint32_t chunk, uint4 v) {
  // K-major SWIZZLE_128B: 8-row groups of 1024 B, 16-byte chunk index XOR row-in-group
  *reinterpret_cast<uint4*>(Xkb + (row >> 3) * 1024u + (row & 7u) * 128u + ((chunk ^ (row & 7u)) << 4)) = v;
}

// tcgen05.wait::ld with the loaded registers as in/out operands: nothing that reads them can be
// scheduled above the wait
__device__ __forceinline__ void tmem_wait_x8(uint32_t (&r)[8]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])
               :
               : "memory");
}

struct TileGramParams {
  const uint32_t* planes;
  const uint8_t* site_flags;
  uint32_t mode;
  const TgTile* tiles;
  uint32_t n_tiles;
  uint2* cnt;              // three 8-byte words per pair slot (DevUnit::dense_off + pair index)
  uint32_t* error;
};

// One warp's share of a tile's readout: lane = site i of TMEM lane quarter lq, `n_chunks` groups of eight partner
// columns starting at column jl0.  The het_snp flags of the warp's rows and columns come from two coalesced loads
// per tile (a ballot each), not from a dependent global load per pair.
__device__ __forceinline__ void tg_readout(const TileGramParams& P, uint32_t tmem_base, uint32_t lq, uint32_t jl0,
                                           uint32_t n_chunks, uint32_t i0, uint32_t j0, uint32_t S, uint32_t site_off,
                                           uint64_t dense_off, bool skip_nonhet) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t i = i0 + lq * 32u + lane;
  const uint8_t* __restrict__ flags = P.site_flags + site_off;
  const bool i_ok = i < S;
  const uint32_t jc = j0 + jl0 + lane;  // this lane's partner column (lanes below 8 * n_chunks)
  const uint32_t fi = i_ok ? (uint32_t)__ldg(flags + i) : 0u;
  const uint32_t fj = (lane < 8u * n_chunks && jc < S) ? (uint32_t)__ldg(flags + jc) : 0u;
  const bool het_i = i_ok && (fi & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP;
  const uint32_t het_cols = __ballot_sync(0xffffffffu, (fj & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP && jc < S);
  const uint64_t row = dense_off + lg_row_off(i_ok ? i : 0u, S);
#pragma unroll 1
  for (uint32_t c = 0; c < n_chunks; ++c) {
    const uint32_t jl = jl0 + c * 8u;  // first of eight partner columns
    // (warp-uniform) no pair i < j among these rows and columns: skip the loads
    if (j0 + jl >= S || i0 + lq * 32u >= j0 + jl + 7u) continue;
    uint32_t r[3][3][8];
#pragma unroll
    for (uint32_t a = 0; a < 3; ++a)
#pragma unroll
      for (uint32_t b = 0; b < 3; ++b)
        tmem_load_x8(tmem_base + ((lq * 32u) << 16) + a * (uint32_t)kTgN + b * (uint32_t)kTgSitesJ + jl, r[a][b]);
#pragma unroll
    for (uint32_t a = 0; a < 3; ++a)
#pragma unroll
      for (uint32_t b = 0; b < 3; ++b) tmem_wait_x8(r[a][b]);
#pragma unroll
    for (uint32_t q = 0; q < 8; ++q) {
      const uint32_t j = j0 + jl + q;
      if (!i_ok || j >= S || i >= j) continue;
      const bool het = het_i || ((het_cols >> (c * 8u + q)) & 1u) != 0u;
      const uint32_t fl = (het ? kTgHetPair : 0u) | ((skip_nonhet && !het) ? kTgNotEvaluated : 0u);
      uint2 w0, w1, w2;
      w0.x = r[0][0][q] | (r[0][1][q] << 16);
      w0.y = r[0][2][q] | (r[1][0][q] << 16);
      w1.x = r[1][1][q] | (r[1][2][q] << 16);
      w1.y = r[2][0][q] | (r[2][1][q] << 16);
      w2.x = r[2][2][q] | (fl << 16);
      w2.y = 0u;
      uint2* out = P.cnt + (row + (j - i - 1u)) * 3ull;
      out[0] = w0;
      out[1] = w1;
      out[2] = w2;
    }
  }
}

// ---------------------------------------------------------------------------
// k_tile_gram_ws, warp-specialised: with tiles of three or four k-blocks, a CTA whose warps all ran the phases
// one after the other (request, expand, barrier, MMAs, wait, read out) would leave the SM idle most of the
// time.  Here three groups of warps run their own loops over the CTA's tiles (static stride:
// tile = blockIdx.x + n * gridDim.x, deepest first) and meet only through mbarriers:
//   warps 0-7   expanders   each thread requests ITS OWN raw plane words by cp.async (4 bytes per
//                           (site, plane, word): what it reads back is what it asked for, so no
//                           barrier separates landing from expansion) two k-blocks ahead, waits for the
//                           operand stage to be free (x_empty), expands, fences and arrives on x_full
//   warp 8      MMA issuer  one lane: x_full -> (first k-block of a tile: tmem_free) -> 12 tcgen05.mma ->
//                           commit to x_empty; after the tile's last k-block also commit to acc_full
//   warps 9-16  readout     acc_full -> tcgen05.ld -> 24-byte count records -> arrive on tmem_free; two
//                           warps per TMEM lane quarter, 24 partner columns each
// The readout of tile t overlaps the expansion of the first two k-blocks of tile t+1; only its MMAs wait.
constexpr int kTwExpWarps = 8, kTwExpThreads = kTwExpWarps * 32;
constexpr int kTwMmaWarp = kTwExpWarps;
constexpr int kTwOutWarp0 = kTwExpWarps + 1, kTwOutWarps = 8;
constexpr int kTwThreads = (kTwOutWarp0 + kTwOutWarps) * 32;  // 544
constexpr uint32_t kTwRawWords = (uint32_t)kTgSites * 4u * 3u;  // [site][word][plane] = 2112 words per k-block
constexpr uint32_t kTwSmemBytes = kTgStages * kTgStageBytes + kTgRawStages * kTwRawWords * 4u + kTgLutBytes + 1024u /*align*/ + 256u /*barriers*/;

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gmem_src) : "memory");
}

// a role's position in the CTA's tile sequence
struct TwCursor {
  uint32_t t, kb, nkb;  // nkb == 0: past the end
  uint32_t i0, j0, S, W, site_off;
  const uint32_t* planes;
  uint64_t dense_off;
  __device__ __forceinline__ bool valid() const { return nkb != 0u; }
  __device__ __forceinline__ void load(const TileGramParams& P) {
    nkb = 0u;
    kb = 0u;
    if (t >= P.n_tiles) return;
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(P.tiles + t)), b = __ldg(reinterpret_cast<const uint4*>(P.tiles + t) + 1);
    planes = P.planes + (((unsigned long long)a.y << 32) | a.x);
    dense_off = ((unsigned long long)a.w << 32) | a.z;
    S = b.x;
    W = b.y;
    site_off = b.z;
    i0 = (b.w & 0xffffu) * (uint32_t)kTgSitesI;
    j0 = (b.w >> 16) * (uint32_t)kTgSitesJ;
    nkb = W >> 2;
  }
  __device__ __forceinline__ void next_tile(const TileGramParams& P) {
    t += gridDim.x;
    load(P);
  }
  __device__ __forceinline__ void advance(const TileGramParams& P) {
    if (!valid()) return;
    if (++kb < nkb) return;
    next_tile(P);
  }
};

// expander thread et: its items are (site, word) = et, et + 256, et + 512 of the 176 x 4 of a k-block
__device__ __forceinline__ void tw_request(uint32_t* __restrict__ raw, const TwCursor& c, uint32_t et) {
  if (!c.valid()) return;
#pragma unroll
  for (uint32_t e = et; e < (uint32_t)kTgSites * 4u; e += kTwExpThreads) {
    const uint32_t sl = e >> 2, w = e & 3u;
    const uint32_t s = (sl < (uint32_t)kTgSitesI) ? c.i0 + sl : c.j0 + (sl - (uint32_t)kTgSitesI);
    if (s < c.S) {
      const uint32_t* __restrict__ src = c.planes + (size_t)s * 3u * c.W + c.kb * 4u + w;
      cp_async4(raw + e * 3u, src);
      cp_async4(raw + e * 3u + 1u, src + c.W);
      cp_async4(raw + e * 3u + 2u, src + 2u * c.W);
    }
  }
}

__device__ __forceinline__ void tw_expand(uint8_t* __restrict__ stage, const uint32_t* __restrict__ raw, const TwCursor& c,
                                          uint32_t et, const uint2* __restrict__ lut) {
  constexpr uint32_t kItemsA = (uint32_t)kTgSitesI * 4u;
#pragma unroll
  for (uint32_t e = et; e < (uint32_t)kTgSites * 4u; e += kTwExpThreads) {
    const bool is_a = e < kItemsA;
    const uint32_t sl_all = e >> 2, w = e & 3u;
    const uint32_t sl = is_a ? sl_all : sl_all - (uint32_t)kTgSitesI;
    const uint32_t s = (is_a ? c.i0 : c.j0) + sl;
    if (s >= c.S) continue;
    const uint32_t M = raw[e * 3u], m = raw[e * 3u + 1u], C = raw[e * 3u + 2u];
    const uint32_t L2 = M & C, L1 = m & C & ~M, L0 = C & ~M & ~m;
    uint8_t* t0 = is_a ? stage : stage + kTgABytes;
    uint8_t* t1 = is_a ? stage + kTgATile : t0;
    uint8_t* t2 = is_a ? stage + 2u * kTgATile : t0;
    const uint32_t r0 = sl, r1 = is_a ? sl : (uint32_t)kTgSitesJ + sl, r2 = is_a ? sl : 2u * (uint32_t)kTgSitesJ + sl;
    tg_store(t0, r0, 2u * w, tg_spread16(lut, L0));
    tg_store(t0, r0, 2u * w + 1u, tg_spread16(lut, L0 >> 16));
    tg_store(t1, r1, 2u * w, tg_spread16(lut, L1));
    tg_store(t1, r1, 2u * w + 1u, tg_spread16(lut, L1 >> 16));
    tg_store(t2, r2, 2u * w, tg_spread16(lut, L2));
    tg_store(t2, r2, 2u * w + 1u, tg_spread16(lut, L2 >> 16));
  }
}

__global__ void __launch_bounds__(kTwThreads, 1) k_tile_gram_ws(const TileGramParams P) {
  extern __shared__ uint8_t tw_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tw_raw) + 1023u) & ~uintptr_t(1023));
  uint32_t* raw0 = reinterpret_cast<uint32_t*>(smem + kTgStages * kTgStageBytes);
  uint2* lut = reinterpret_cast<uint2*>(raw0 + kTgRawStages * kTwRawWords);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(lut) + kTgLutBytes);
  uint64_t* x_full = bars;                    // [stages] expanders -> MMA issuer (256 arrivals)
  uint64_t* x_empty = bars + kTgStages;       // [stages] MMA commit -> expanders
  uint64_t* acc_full = bars + 2 * kTgStages;  // MMA commit -> readout
  uint64_t* tmem_free = acc_full + 1;         // readout (256 arrivals) -> MMA issuer
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_free + 1);
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;

  if (tid == 0) {
    for (int s = 0; s < kTgStages; ++s) {
      mbar_init(&x_full[s], kTwExpThreads);
      mbar_init(&x_empty[s], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(tmem_free, kTwOutWarps * 32);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tg_lut_init(lut, tid, kTwThreads);
  __syncwarp();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kTgTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  TwCursor cur;
  cur.t = blockIdx.x;
  cur.load(P);

  if (warp < (uint32_t)kTwExpWarps) {
    // ---------------- expanders
    const uint32_t et = tid;
    TwCursor pre = cur;
#pragma unroll
    for (int d = 0; d < kTgAhead; ++d) {
      tw_request(raw0 + (uint32_t)d * kTwRawWords, pre, et);
      cp_async_commit();
      pre.advance(P);
    }
    uint32_t stage = 0, phase = 0;  // x_empty[stage] has completed `phase` ... parity of its next completion to wait for
    for (uint32_t step = 0; cur.valid(); ++step) {
      tw_request(raw0 + ((step + (uint32_t)kTgAhead) % (uint32_t)kTgRawStages) * kTwRawWords, pre, et);
      cp_async_commit();          // (possibly empty: exactly one group per step)
      pre.advance(P);
      cp_async_wait<kTgAhead>();  // this thread's words of step `step` have landed; nobody else reads them
      if (step >= (uint32_t)kTgStages) mbar_wait(&x_empty[stage], phase ^ 1u, P.error);  // the MMAs that read this stage
      tw_expand(smem + stage * kTgStageBytes, raw0 + (step % (uint32_t)kTgRawStages) * kTwRawWords, cur, et, lut);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the tensor core
      mbar_arrive(&x_full[stage]);
      if (++stage == (uint32_t)kTgStages) {
        stage = 0;
        phase ^= 1u;
      }
      cur.advance(P);
    }
    cp_async_wait<0>();
  } else if (warp == (uint32_t)kTwMmaWarp) {
    // ---------------- MMA issuer
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_u8(128u, (uint32_t)kTgN);
      uint32_t stage = 0, phase = 0, n_tile = 0;
      while (cur.valid()) {
        mbar_wait(&x_full[stage], phase, P.error);
        tc_fence_after();
        if (cur.kb == 0u && n_tile > 0u) {  // the previous tile's accumulators have been read out
          mbar_wait(tmem_free, (n_tile - 1u) & 1u, P.error);
          tc_fence_after();
        }
        const uint32_t sa = smem_u32(smem + stage * kTgStageBytes), sb = sa + kTgABytes;
        const uint64_t db = umma_desc_sw128(sb);
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
#pragma unroll
          for (uint32_t a = 0; a < 3; ++a)
            umma_i8(tmem_base + a * (uint32_t)kTgN, umma_desc_sw128(sa + a * kTgATile) + 2ull * k, db + 2ull * k, idesc,
                    (cur.kb | k) != 0u);
        }
        umma_commit(&x_empty[stage]);  // the stage is free once these MMAs have read it
        if (cur.kb + 1u == cur.nkb) {
          umma_commit(acc_full);       // ... and the tile's accumulators are complete
          ++n_tile;
        }
        if (++stage == (uint32_t)kTgStages) {
          stage = 0;
          phase ^= 1u;
        }
        cur.advance(P);
      }
    }
  } else {
    // ---------------- readout: lane = site i; lane quarter lq, partner columns [24 h, 24 h + 24)
    const uint32_t ow = warp - (uint32_t)kTwOutWarp0;
    const uint32_t lq = warp & 3u, h = ow >> 2;  // (warps 9..16: warp & 3 runs 1,2,3,0,1,2,3,0 -- both halves see all four quarters)
    const bool skip_nonhet = (P.mode & LGMI_MODE_HET_ONLY) && (P.mode & LGMI_MODE_SKIP_NONHET);
    uint32_t n_tile = 0;
    while (cur.valid()) {
      mbar_wait(acc_full, n_tile & 1u, P.error);
      tc_fence_after();
      tg_readout(P, tmem_base, lq, h * 24u, 3u, cur.i0, cur.j0, cur.S, cur.site_off, cur.dense_off, skip_nonhet);
      tc_fence_before();
      mbar_arrive(tmem_free);  // this thread is done with the accumulators
      ++n_tile;
      cur.next_tile(P);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTgTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------------------
// MI of the pairs k_tile_gram_ws counted: one CTA per work item (<= 2048 consecutive pairs of a unit).
// Pass 1 (one thread per pair): min-common filter, emitted-pair count of the item (what k_count computes for
// the other paths), NaN into the dense MI scratch for the pairs without MI, and the others listed as "2x2"
// (no "other" label among the common reads) or "3x3".  Pass 2: the branch-free fp64 epilogues of lgmi_fast.cuh
// (same operations and roundings as lgmi_math.cuh: Markstein quotient from the correctly rounded reciprocal,
// double-double logs from the context's table) over warp-sized chunks of each list -- full warps, no divergence.
__device__ __forceinline__ uint32_t tile_cnt_load(const uint2* __restrict__ cnt, uint64_t slot, uint32_t T[9]) {
  const uint2 w0 = __ldg(cnt + slot * 3ull), w1 = __ldg(cnt + slot * 3ull + 1), w2 = __ldg(cnt + slot * 3ull + 2);
  T[0] = w0.x & 0xffffu; T[1] = w0.x >> 16; T[2] = w0.y & 0xffffu; T[3] = w0.y >> 16;
  T[4] = w1.x & 0xffffu; T[5] = w1.x >> 16; T[6] = w1.y & 0xffffu; T[7] = w1.y >> 16;
  T[8] = w2.x & 0xffffu;
  return w2.x >> 16;  // flag bits
}

#ifndef LGMI_FINISH_CTAS
#define LGMI_FINISH_CTAS 4  // resident CTAs per SM the register budget is set for (tools/build_variant.py -DLGMI_FINISH_CTAS=3)
#endif
__global__ void __launch_bounds__(kThreads, LGMI_FINISH_CTAS) k_tile_finish(const RunParams P, const uint2* __restrict__ cnt) {
  __shared__ uint16_t s_list[kPairsMax];  // pairs with a 2x2 table from the front, with "other" cells from the back
  __shared__ uint32_t s_n2, s_n3, s_emit;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  const GlobalTab tab{P.lntab};
  const bool het_only = (P.mode & LGMI_MODE_HET_ONLY) != 0u;
  for (uint32_t item_idx = blockIdx.x; item_idx < P.n_items; item_idx += gridDim.x) {
    const Item it = P.items[item_idx];
    if (!(it.flags & ITEM_TILED_GRAM)) continue;
    const DevUnit u = P.units[it.unit];
    const uint64_t slot0 = u.dense_off + it.pair_begin;
    __syncthreads();  // the previous item's lists have been consumed
    if (tid == 0) {
      s_n2 = 0u;
      s_n3 = 0u;
      s_emit = 0u;
    }
    __syncthreads();
    uint32_t mine = 0;
    const uint32_t n_slots = (it.pair_cnt + 31u) & ~31u;
    // the 24 bytes of the next pair of this thread are requested before the current pair is classified
    uint2 nx0 = make_uint2(0u, 0u), nx1 = nx0, nx2 = nx0;
    if (tid < it.pair_cnt) {
      nx0 = __ldg(cnt + (slot0 + tid) * 3ull);
      nx1 = __ldg(cnt + (slot0 + tid) * 3ull + 1);
      nx2 = __ldg(cnt + (slot0 + tid) * 3ull + 2);
    }
    for (uint32_t pl = tid; pl < n_slots; pl += kThreads) {
      uint32_t cls = 0u;  // 0 no MI, 2 -> 2x2 list, 3 -> 3x3 list
      const uint2 w0 = nx0, w1 = nx1, w2 = nx2;
      if (pl + kThreads < it.pair_cnt) {
        nx0 = __ldg(cnt + (slot0 + pl + kThreads) * 3ull);
        nx1 = __ldg(cnt + (slot0 + pl + kThreads) * 3ull + 1);
        nx2 = __ldg(cnt + (slot0 + pl + kThreads) * 3ull + 2);
      }
      if (pl < it.pair_cnt) {
        uint32_t T[9];
        T[0] = w0.x & 0xffffu; T[1] = w0.x >> 16; T[2] = w0.y & 0xffffu; T[3] = w0.y >> 16;
        T[4] = w1.x & 0xffffu; T[5] = w1.x >> 16; T[6] = w1.y & 0xffffu; T[7] = w1.y >> 16;
        T[8] = w2.x & 0xffffu;
        const uint32_t fl = w2.x >> 16;
        uint32_t N = 0;
#pragma unroll
        for (int k = 0; k < 9; ++k) N += T[k];
        if (!(fl & kTgNotEvaluated) && (int)N >= P.min_common) {  // strict '<' drops (mutual_information.py:19)
          cls = (T[0] | T[1] | T[2] | T[3] | T[6]) ? 3u : 2u;
          mine += ((fl & kTgHetPair) || !het_only) ? 1u : 0u;
        } else {
          P.dense[slot0 + pl] = lg_nan();
        }
        if (P.mode & LGMI_MODE_EMIT_COUNTS) {
#pragma unroll
          for (int k = 0; k < 9; ++k) P.tile_counts[(slot0 + pl) * 9ull + k] = T[k];
        }
      }
      const uint32_t m2 = __ballot_sync(0xffffffffu, cls == 2u);
      const uint32_t m3 = __ballot_sync(0xffffffffu, cls == 3u);
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
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if (lane == 0 && mine) atomicAdd(&s_emit, mine);
    __syncthreads();
    if (tid == 0) P.item_cnt[item_idx] = s_emit;
    const uint32_t n2 = s_n2, n3 = s_n3;
    const uint32_t nc2 = (n2 + 31u) >> 5, nc3 = (n3 + 31u) >> 5;
    for (uint32_t c = warp; c < nc2 + nc3; c += kThreads / 32) {
      if (c < nc2) {
        const uint32_t q = c * 32u + lane;
        if (q < n2) {
          const uint32_t pl = s_list[q];
          uint32_t T[9];
          tile_cnt_load(cnt, slot0 + pl, T);
          P.dense[slot0 + pl] = mi_2x2(tab, T[4], T[5], T[7], T[8]);
        }
      } else {
        const uint32_t q = (c - nc2) * 32u + lane;
        if (q < n3) {
          const uint32_t pl = s_list[kPairsMax - 1u - q];
          uint32_t T[9];
          tile_cnt_load(cnt, slot0 + pl, T);
          P.dense[slot0 + pl] = mi_3x3(tab, T);
        }
      }
    }
  }
}

}  // namespace lgmi
