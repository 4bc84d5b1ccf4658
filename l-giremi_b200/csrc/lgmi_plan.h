// lgmi_plan.h -- the host-side plan of a batch: which kernel path each unit takes and the work tables the
// kernels read; and the groups of a pipelined step.  Plain C++17 (no CUDA types or calls): lgmi.cu uploads what
// plan_batch() builds and sets up the groups plan_pipeline() cuts, and the CPU tests (tests/csrc/plan_host.cpp)
// check the same plans without a device.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/lgmi.h"
#include "lgmi_math.cuh"

namespace lgmi {

constexpr int kPairsMax = 2048;  // pairs per work item (>= 64*63/2: a 64-site unit is one item)
constexpr uint64_t kNoGram = ~0ull;
constexpr int kFastMaxS = 64;    // sites per unit on the fast path
constexpr int kFastMaxR = 256;   // reads per unit on the fast path
constexpr int kTileSites = 16;   // k_tile_mi: sites per block
constexpr int kTgSitesI = 128;   // k_tile_gram_ws: sites per row block (one per TMEM lane)
constexpr int kTgSitesJ = 48;    // ... partner sites per column block
constexpr uint32_t kTgMaxReads = 65535;  // ... counts are stored as u16
constexpr int kDenseBM = 128;    // k_gram_i8: tile rows    (sites i of plane a)
constexpr int kDenseBN = 256;    // ... tile columns (sites j of plane b)
constexpr int kDenseBK = 128;    // ... bytes of K per stage == one 128B swizzle row
constexpr uint32_t kDenseOthDiv = 64u;  // a site lists up to max(256, R / 64) reads with label "other"
constexpr uint32_t kDenseOthMin = 256u;
constexpr int kMeanSites = 32;   // k_site_mean_dense: sites per CTA (= lanes of the consuming warp)
static_assert(kFastMaxS * (kFastMaxS - 1) / 2 <= kPairsMax, "a small unit is one work item");

// ------------------------------------------------------------------ tables read by the kernels (uploaded as bytes)
struct DevUnit {
  uint64_t plane_off;  // words
  uint64_t dense_off;  // first slot in the dense MI scratch (multi-item units), else ~0
  uint64_t gram_off;   // first word of the unit's nine count matrices (tensor-core path), else ~0
  uint32_t S, R, W, site_off;
  uint32_t first_item, n_items;
  uint32_t S_pad;
  uint32_t tiled;      // MI of every pair is precomputed into the dense scratch: 1 by k_tile_mi, 2 by k_tile_gram_ws + k_tile_finish
};
static_assert(sizeof(DevUnit) == 56, "DevUnit layout");

enum : uint32_t {
  ITEM_FIRST = 1u, ITEM_SINGLE = 2u, ITEM_FAST = 4u,
  ITEM_TILED = 16u /* MI precomputed by k_tile_mi or k_tile_gram_ws + k_tile_finish */,
  ITEM_TILED_GRAM = 32u /* ... by the latter, which also counts the item's emitted pairs */,
  ITEM_GRAM = 64u /* deep unit: tables from the count matrices of the tensor-core path (k_pairs_generic<2>) */
};

struct Item {
  uint32_t unit;
  uint32_t pair_begin;
  uint32_t pair_cnt;
  uint32_t flags;
};
static_assert(sizeof(Item) == 16, "Item layout");

// Everything k_pairs_generic<1> needs of a work item of a mid-depth (tiled) unit, in one 48-byte record built on
// the host: the kernel requests the next record (cp.async) while it works on the current item, instead of the
// chain items[] -> units[] at the head of every item.
struct alignas(16) TiledDesc {
  uint32_t item_idx, unit, pair_begin, pair_cnt;
  uint32_t flags, S, site_off, pad;
  uint64_t dense_off, pad2;
};
static_assert(sizeof(TiledDesc) == 48, "three 16-byte copies per record");

// one work item of the fast kernel == one whole unit
struct alignas(16) FastItem {
  unsigned long long plane_off;  // words
  uint32_t site_off;
  uint32_t unit;
  uint32_t item;                 // index into item_off / item_cnt
  uint16_t S, R;
  uint32_t W;                    // row words of the input planes (4 or 8)
  uint32_t pad;
};
static_assert(sizeof(FastItem) == 32, "FastItem layout");

struct TileItem {
  uint32_t unit;
  uint16_t I, J;  // site blocks of 16 sites, I <= J
};
static_assert(sizeof(TileItem) == 8, "TileItem layout");

// one work item of k_tile_gram_ws, self-contained (no dependent look-up of the unit table in the kernel)
struct alignas(16) TgTile {
  unsigned long long plane_off;  // first word of the unit's planes
  unsigned long long dense_off;  // first pair slot of the unit
  uint32_t S, W, site_off;
  uint16_t I, J;                 // row block of 128 sites, column block of 48 sites
};
static_assert(sizeof(TgTile) == 32, "TgTile layout");

struct DenseTile {
  uint8_t a, b;       // row groups of X (0 covered, 1 major or minor, 2 major)
  uint16_t I, J;      // site blocks: rows [128 I, +128), columns [256 J, +256)
  uint16_t partial;   // 1: the tile's K range is shared by several items (last wave): results are added atomically
                      //    into a zeroed tile
  uint32_t kb0, kb1;  // k-blocks [kb0, kb1) of this work item (32 bits: a unit may have millions of reads)
};
static_assert(sizeof(DenseTile) == 16, "DenseTile layout");

struct MeanItem {
  uint32_t unit;
  uint32_t site_begin;
};
static_assert(sizeof(MeanItem) == 8, "MeanItem layout");

// ------------------------------------------------------------------ the plan
// what the plan reads from the context
struct PlanConfig {
  uint32_t num_sms;
  int dense_path;  // 4: the deep units' four-block form may be chosen, 9: always nine blocks
  int tile_path;   // mid-depth units: 0 popcount (k_tile_mi), else tensor cores (k_tile_gram_ws)
  uint32_t dense_min_sites, dense_min_reads;  // deep units are at least this large
};

enum class UnitPath : uint32_t {
  kNoPairs = 0,  // S < 2 (or a piece without pairs): only the bookkeeping of k_pairs_generic<0>
  kSmall,        // k_pairs_fast, one item
  kTilePopc,     // mid-depth, MI precomputed by k_tile_mi
  kTileGram,     // mid-depth, counted by k_tile_gram_ws, MI by k_tile_finish
  kDeep,         // k_gram_i8's count matrices, tables read by k_pairs_generic<2>
};

// one unit of the tensor-core path
struct DenseTileList {
  uint64_t off = 0, macs = 0;
  uint32_t n = 0;
  uint32_t n_whole = 0;  // the first n_whole work items are whole tiles; the rest share tiles (last wave, split in K)
};
struct DensePlan {
  uint32_t unit = 0, S = 0, W = 0, S_pad = 0, k_blocks = 0;
  uint32_t rows = 0;          // pairs (i, j) with i < rows are read: S, or the row limit of a piece
  uint32_t oth_cap = 0;       // listed "other" reads per site (four-block form)
  bool four = false;          // the four-block form may be chosen (else the run is told "nine" up front)
  DenseTileList list4, list9; // P, M x P, M  /  C, P, M x C, P, M
  uint64_t plane_off = 0, gram_off = 0;
};

struct BatchPlan {
  std::vector<DevUnit> units;
  std::vector<Item> items;
  std::vector<FastItem> fast_items;    // k_pairs_fast's, one per small unit
  std::vector<TiledDesc> tiled_desc;   // k_pairs_generic<1>'s, one per item of a mid-depth unit
  std::vector<TileItem> tile_items;    // k_tile_mi's, deepest unit first
  std::vector<TgTile> gram_tiles;      // k_tile_gram_ws's, deepest unit first
  std::vector<DenseTile> dense_tiles;  // k_gram_i8's: the lists of dense_plans
  std::vector<MeanItem> mean_items;    // k_site_mean_dense's, largest unit first
  std::vector<DensePlan> dense_plans;  // the deep units
  uint64_t n_dense = 0;                // dense MI slots
  uint64_t gram_words = 0;             // count matrices of all deep units
  uint64_t x_bytes = 0, xt_words = 0, oth_words = 0;  // scratch of the deep unit being contracted (the largest)
  uint32_t oth_sites = 0;
  uint64_t n_candidates = 0;
  uint32_t max_reads = 0;
  uint32_t n_tiled_work_items = 0;     // items of the mid-depth and deep units: k_pairs_generic<1>'s and <2>'s
};

// pairs (i, j), i < j < S, with i < rows: the first rows rows of the pair order (lg_row_off(rows, S))
inline uint64_t piece_pairs(uint32_t rows, uint32_t S) { return rows ? lg_row_off(rows, S) : 0ull; }

// the pairs a unit evaluates: all of them, or a piece's (row limit != 0)
inline uint64_t unit_pairs(uint32_t S, uint32_t limit) {
  return limit ? piece_pairs(limit, S) : S >= 2 ? (uint64_t)S * (S - 1) / 2 : 0;
}

// The one place a unit's kernel path is decided.  A unit sent to the tensor-core path by a lowered threshold is
// not also k_pairs_fast's; a piece is never k_pairs_fast's (its pairs go to a dense slot).
inline UnitPath route_unit(const lgmi_unit_desc& u, uint32_t limit, const PlanConfig& cfg) {
  if (!unit_pairs(u.n_sites, limit)) return UnitPath::kNoPairs;
  if (u.n_sites >= cfg.dense_min_sites && u.n_reads >= cfg.dense_min_reads) return UnitPath::kDeep;
  if (!limit && u.n_sites <= (uint32_t)kFastMaxS && u.n_reads <= (uint32_t)kFastMaxR) return UnitPath::kSmall;
  // units deeper than kTgMaxReads, whose counts do not fit 16 bits, always take k_tile_mi
  return cfg.tile_path && u.n_reads >= 1u && u.n_reads <= kTgMaxReads ? UnitPath::kTileGram : UnitPath::kTilePopc;
}

// candidate pairs next to a het_snp site, from the host copy of the flag bytes (a piece: its own pairs only)
inline uint64_t het_candidates(const std::vector<lgmi_unit_desc>& units, const std::vector<uint32_t>& row_limit,
                               const uint8_t* site_flags) {
  uint64_t tot = 0;
  for (size_t k = 0; k < units.size(); ++k) {
    const lgmi_unit_desc& u = units[k];
    const uint8_t* f = site_flags + u.site_off;
    auto het = [&](uint32_t s) { return (f[s] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP; };
    const uint32_t rows = row_limit.empty() ? 0u : row_limit[k];
    if (rows) {
      // pairs of the piece minus those whose sites are both non-het: walk the rows from the last, counting the
      // non-het sites after each
      uint64_t o_after = 0, both = 0;
      for (uint32_t s = u.n_sites; s-- > 0;) {
        if (s < rows && !het(s)) both += o_after;
        o_after += het(s) ? 0u : 1u;
      }
      tot += piece_pairs(rows, u.n_sites) - both;
      continue;
    }
    uint64_t h = 0;
    for (uint32_t s = 0; s < u.n_sites; ++s) h += het(s) ? 1u : 0u;
    const uint64_t S = u.n_sites, o = S - h;
    tot += (S >= 2 ? S * (S - 1) / 2 : 0) - (o >= 2 ? o * (o - 1) / 2 : 0);
  }
  return tot;
}

// One CTA per SM walks a tile list with stride #SMs: a last, partly filled wave leaves SMs idle for a whole tile
// time, so its tiles (those listed from L.off on) are cut along K into as many parts as fill it (added atomically
// into zeroed tiles); then the list's length and multiply-accumulates.
inline void finish_dense_list(uint32_t k_blocks, uint32_t num_sms, std::vector<DenseTile>& tiles, DenseTileList& L) {
  const uint32_t n = (uint32_t)(tiles.size() - L.off), grid = num_sms;
  const uint32_t rem = n % grid;
  uint32_t parts = rem ? std::min<uint32_t>(8u, grid / rem) : 1u;
  while (parts > 1u && k_blocks < 8u * parts) --parts;  // at least 8 k-blocks (1 024 reads) per part
  L.n_whole = n;
  if (parts >= 2u) {
    L.n_whole = n - rem;
    std::vector<DenseTile> tail(tiles.end() - rem, tiles.end());
    tiles.resize(tiles.size() - rem);
    for (uint32_t q = 0; q < parts; ++q)
      for (DenseTile t : tail) {
        t.kb0 = (uint32_t)((uint64_t)k_blocks * q / parts);
        t.kb1 = (uint32_t)((uint64_t)k_blocks * (q + 1) / parts);
        t.partial = 1;
        tiles.push_back(t);
      }
  }
  L.n = (uint32_t)(tiles.size() - L.off);
  L.macs = 0;
  for (uint32_t t = 0; t < L.n; ++t) {
    const DenseTile& dt = tiles[L.off + t];
    L.macs += (uint64_t)kDenseBM * kDenseBN * (dt.kb1 - dt.kb0) * kDenseBK;
  }
}

// k_gram_i8's work items for row groups g0 .. 2 of X against each other: the tiles holding a pair i < j with
// i < pl.rows, both real sites
inline void plan_dense_list(const DensePlan& pl, uint32_t g0, uint32_t num_sms, std::vector<DenseTile>& tiles,
                            DenseTileList& L) {
  L.off = tiles.size();
  for (uint32_t a = g0; a < 3; ++a)
    for (uint32_t bb = g0; bb < 3; ++bb)
      for (uint32_t J = 0; J < pl.S_pad / (uint32_t)kDenseBN; ++J)
        for (uint32_t I = 0; I < (pl.rows + (uint32_t)kDenseBM - 1u) / (uint32_t)kDenseBM; ++I) {
          const uint32_t i_min = I * (uint32_t)kDenseBM;
          const uint32_t j_max = std::min(J * (uint32_t)kDenseBN + (uint32_t)kDenseBN, pl.S) - 1u;
          if (J * (uint32_t)kDenseBN >= pl.S || i_min >= j_max) continue;
          tiles.push_back(DenseTile{(uint8_t)a, (uint8_t)bb, (uint16_t)I, (uint16_t)J, 0, 0u, pl.k_blocks});
        }
  finish_dense_list(pl.k_blocks, num_sms, tiles, L);
}

// The het-anchored form of a deep unit.  Under HET_ONLY | SKIP_NONHET only the pairs with a het_snp site are
// evaluated, and the counts those need are the Gram blocks of the het sites' rows against all sites: k_gram_i8 takes
// the A operand from X_het, the het sites' X rows packed into H_pad rows per group (pad rows zero), and writes row h
// of a tile into row het[h] of the unit's count matrices.  A pair (i, j), i < j, is read from row i when i is het and
// from row j, block index transposed, when only j is.
struct HetDensePlan {
  std::vector<uint32_t> het;   // the unit's het sites, ascending
  uint32_t H = 0, H_pad = 0;   // their number, and that rounded up to a whole row block of 128
  DenseTileList list4, list9;  // het row blocks x column blocks of groups P, M  /  C, P, M (offsets into `tiles`)
  bool fewer = false;          // not a piece, and the het lists cost at most half the triangle's multiply-accumulates
};

// The het plan of deep unit pl from its flag bytes (unit_flags[0 .. S)); piece: the unit is a piece of a split unit
// (row limit != 0), which keeps the all-pairs form.  Appends the tile lists to `tiles`.
inline void plan_het_dense(const DensePlan& pl, const uint8_t* unit_flags, bool piece, uint32_t num_sms,
                           std::vector<DenseTile>& tiles, HetDensePlan* out) {
  HetDensePlan& h = *out;
  h = HetDensePlan();
  for (uint32_t s = 0; s < pl.S; ++s)
    if ((unit_flags[s] & LGMI_SITE_TYPE_MASK) == LGMI_SITE_HET_SNP) h.het.push_back(s);
  h.H = (uint32_t)h.het.size();
  h.H_pad = (h.H + (uint32_t)kDenseBM - 1u) / (uint32_t)kDenseBM * (uint32_t)kDenseBM;
  for (uint32_t g0 = 0; g0 < 2u; ++g0) {
    if (g0 == 1u && !pl.four) continue;
    DenseTileList& L = g0 ? h.list4 : h.list9;
    L.off = tiles.size();
    for (uint32_t a = g0; a < 3; ++a)
      for (uint32_t bb = g0; bb < 3; ++bb)
        for (uint32_t J = 0; J < pl.S_pad / (uint32_t)kDenseBN; ++J)
          for (uint32_t I = 0; I < h.H_pad / (uint32_t)kDenseBM; ++I) {
            // some pair (het[r], s), s != het[r], with r in row block I and s in column block J
            const uint32_t s0 = J * (uint32_t)kDenseBN, r0 = I * (uint32_t)kDenseBM;
            if (s0 >= pl.S) continue;
            const uint32_t n_cols = std::min(pl.S - s0, (uint32_t)kDenseBN), n_rows = std::min(h.H - r0, (uint32_t)kDenseBM);
            if (n_cols == 1u && n_rows == 1u && h.het[r0] == s0) continue;
            tiles.push_back(DenseTile{(uint8_t)a, (uint8_t)bb, (uint16_t)I, (uint16_t)J, 0, 0u, pl.k_blocks});
          }
    finish_dense_list(pl.k_blocks, num_sms, tiles, L);
  }
  // (at most half: the form adds a pass over the het rows and transposed table reads; on cfg3 it was faster at 0.44
  // of the triangle's work and slower at 0.89 -- profiles/r4_dense_het_n1_fewer_macs_rule.json)
  h.fewer = !piece && 2u * h.list9.macs <= pl.list9.macs && (!pl.four || 2u * h.list4.macs <= pl.list4.macs);
}

// whether a run takes the het form of a unit: only HET_ONLY | SKIP_NONHET evaluates the het pairs alone, and the
// plan needs the flag bytes on the host (a caller that fills the device buffers itself keeps the all-pairs form)
inline bool take_het_form(const HetDensePlan& h, uint32_t mode, bool host_flags) {
  const uint32_t het_modes = LGMI_MODE_HET_ONLY | LGMI_MODE_SKIP_NONHET;
  return host_flags && (mode & het_modes) == het_modes && h.fewer;
}

// a deep unit: its nine count matrices come from k_gram_i8
inline void plan_deep_unit(uint32_t k, const lgmi_unit_desc& u, uint32_t rows, const PlanConfig& cfg, BatchPlan& P) {
  DensePlan pl;
  pl.unit = k;
  pl.S = u.n_sites;
  pl.W = u.row_words;
  pl.S_pad = (u.n_sites + (uint32_t)kDenseBN - 1u) / (uint32_t)kDenseBN * (uint32_t)kDenseBN;
  pl.rows = rows;
  pl.k_blocks = u.row_words * 32u / (uint32_t)kDenseBK;  // W is a multiple of 4: whole 128-read blocks
  pl.plane_off = u.plane_off;
  pl.gram_off = P.gram_words;
  // (k_other_fix addresses a label's transposed plane with 32-bit word offsets)
  pl.four = cfg.dense_path == 4 && (uint64_t)pl.k_blocks * kDenseBK * (pl.S_pad / 32u) < (1ull << 32);
  pl.oth_cap = std::max<uint32_t>(kDenseOthMin, u.n_reads / kDenseOthDiv);
  if (pl.four) plan_dense_list(pl, 1u, cfg.num_sms, P.dense_tiles, pl.list4);
  plan_dense_list(pl, 0u, cfg.num_sms, P.dense_tiles, pl.list9);
  if (pl.four) {
    P.xt_words = std::max<uint64_t>(P.xt_words, 3ull * pl.k_blocks * kDenseBK * (pl.S_pad / 32u));
    P.oth_words = std::max<uint64_t>(P.oth_words, (uint64_t)pl.S * pl.oth_cap);
    P.oth_sites = std::max<uint32_t>(P.oth_sites, pl.S);
  }
  P.gram_words += 9ull * pl.S_pad * pl.S_pad;
  P.x_bytes = std::max<uint64_t>(P.x_bytes, 3ull * pl.S_pad * pl.k_blocks * kDenseBK);
  P.dense_plans.push_back(pl);
}

inline int plan_error(std::string* err, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (err) *err = buf;
  return code;
}

// The plan of a batch (row_limit NULL: no unit is a piece).  A unit k with row_limit[k] != 0 is a piece of a split
// unit: only its pairs (i, j) with i < row_limit[k] are evaluated and emitted, always through a dense MI slot, and it
// has no per-site means.  Returns LGMI_OK, or LGMI_ERR_ARG / LGMI_ERR_UNSUPPORTED with *err set.
inline int plan_batch(const lgmi_unit_desc* units, uint32_t n_units, const uint32_t* row_limit, uint64_t plane_words,
                      uint64_t n_sites, const PlanConfig& cfg, BatchPlan* plan, std::string* err) {
  BatchPlan& P = *plan;
  P = BatchPlan();
  P.units.resize(n_units);
  for (uint32_t k = 0; k < n_units; ++k) {
    const lgmi_unit_desc& u = units[k];
    if (u.n_sites > 65535u) return plan_error(err, LGMI_ERR_UNSUPPORTED, "unit %u: %u sites > 65535", k, u.n_sites);
    if (u.row_words != 4u * ((u.n_reads + 127u) / 128u) || (u.plane_off & 3ull) ||
        u.plane_off + 3ull * u.n_sites * u.row_words > plane_words || (uint64_t)u.site_off + u.n_sites > n_sites)
      return plan_error(err, LGMI_ERR_ARG,
                        "unit %u: inconsistent descriptor (S=%u R=%u W=%u plane_off=%llu site_off=%u)", k,
                        u.n_sites, u.n_reads, u.row_words, (unsigned long long)u.plane_off, u.site_off);
    const uint32_t limit = row_limit ? row_limit[k] : 0u;
    const bool piece = limit != 0u;
    if (piece && (limit > u.n_sites || (limit % 128u && limit != u.n_sites)))
      return plan_error(err, LGMI_ERR_ARG, "unit %u: row limit %u is neither a multiple of 128 below S nor S = %u", k,
                        limit, u.n_sites);
    const uint32_t rows = piece ? limit : u.n_sites;  // row blocks at or past it hold no pair of the unit
    const uint64_t np = unit_pairs(u.n_sites, limit);
    const uint32_t nit = np ? (uint32_t)((np + kPairsMax - 1) / kPairsMax) : 1u;
    const UnitPath path = route_unit(u, limit, cfg);
    const bool tiled = path == UnitPath::kTilePopc || path == UnitPath::kTileGram;
    P.n_candidates += np;
    P.max_reads = std::max(P.max_reads, u.n_reads);

    DevUnit& d = P.units[k];
    d.plane_off = u.plane_off;
    d.S = u.n_sites;
    d.R = u.n_reads;
    d.W = u.row_words;
    d.site_off = u.site_off;
    d.first_item = (uint32_t)P.items.size();
    d.n_items = nit;
    d.dense_off = ~0ull;
    d.gram_off = kNoGram;
    d.S_pad = 0;
    d.tiled = path == UnitPath::kTileGram ? 2u : tiled ? 1u : 0u;
    // a dense MI slot: mid-depth units (their MI is precomputed there), units of several items and pieces
    if (tiled || nit > 1 || piece) {
      d.dense_off = P.n_dense;
      P.n_dense += np;
    }
    if (nit > 1 && !piece)  // (a piece's means would be partial: lgmi_split_means computes them over all pieces)
      for (uint32_t s0 = 0; s0 < u.n_sites; s0 += (uint32_t)kMeanSites) P.mean_items.push_back(MeanItem{k, s0});

    if (path == UnitPath::kDeep) {
      plan_deep_unit(k, u, rows, cfg, P);
      d.gram_off = P.dense_plans.back().gram_off;
      d.S_pad = P.dense_plans.back().S_pad;
    } else if (path == UnitPath::kTileGram) {
      const uint32_t nI = (rows + (uint32_t)kTgSitesI - 1u) / (uint32_t)kTgSitesI;
      const uint32_t nJ = (u.n_sites + (uint32_t)kTgSitesJ - 1u) / (uint32_t)kTgSitesJ;
      for (uint32_t I = 0; I < nI; ++I)
        for (uint32_t J = 0; J < nJ; ++J) {
          // some pair i < j with i in row block I and j in column block J
          const uint32_t j_max = std::min((J + 1u) * (uint32_t)kTgSitesJ, u.n_sites) - 1u;
          if (I * (uint32_t)kTgSitesI >= j_max) continue;
          P.gram_tiles.push_back(TgTile{u.plane_off, d.dense_off, u.n_sites, u.row_words, u.site_off, (uint16_t)I, (uint16_t)J});
        }
    } else if (path == UnitPath::kTilePopc) {
      const uint32_t nb = (u.n_sites + (uint32_t)kTileSites - 1u) / (uint32_t)kTileSites;
      for (uint32_t I = 0; I < (rows + (uint32_t)kTileSites - 1u) / (uint32_t)kTileSites; ++I)
        for (uint32_t J = I; J < nb; ++J) P.tile_items.push_back(TileItem{k, (uint16_t)I, (uint16_t)J});
    } else if (path == UnitPath::kSmall) {
      P.fast_items.push_back(FastItem{u.plane_off, u.site_off, k, d.first_item, (uint16_t)u.n_sites, (uint16_t)u.n_reads,
                                      u.row_words, 0u});
    }

    const uint32_t flags = (nit == 1 && !piece ? ITEM_SINGLE : 0u) | (tiled ? ITEM_TILED : 0u) |
                           (path == UnitPath::kTileGram ? ITEM_TILED_GRAM : 0u) |
                           (path == UnitPath::kDeep ? ITEM_GRAM : 0u) | (path == UnitPath::kSmall ? ITEM_FAST : 0u);
    for (uint32_t t = 0; t < nit; ++t) {
      Item it;
      it.unit = k;
      it.pair_begin = t * (uint32_t)kPairsMax;
      it.pair_cnt = (uint32_t)std::min<uint64_t>(kPairsMax, np - (uint64_t)t * kPairsMax);
      it.flags = flags | (t == 0 ? ITEM_FIRST : 0u);
      if (tiled || path == UnitPath::kDeep) ++P.n_tiled_work_items;  // (not k_pairs_generic<0>'s)
      if (tiled) {
        TiledDesc td{};
        td.item_idx = (uint32_t)P.items.size();
        td.unit = k, td.pair_begin = it.pair_begin, td.pair_cnt = it.pair_cnt, td.flags = it.flags;
        td.S = u.n_sites, td.site_off = u.site_off, td.dense_off = d.dense_off;
        P.tiled_desc.push_back(td);
      }
      P.items.push_back(it);
    }
  }
  // the deepest tiles first: CTAs are handed out in order, so the long ones do not end up in the tail
  std::stable_sort(P.tile_items.begin(), P.tile_items.end(), [&](const TileItem& x, const TileItem& y) {
    return units[x.unit].row_words > units[y.unit].row_words;
  });
  std::stable_sort(P.gram_tiles.begin(), P.gram_tiles.end(), [](const TgTile& x, const TgTile& y) { return x.W > y.W; });
  // per-site sums: a CTA's time grows with its unit's number of sites (one serial chain of S steps per site), so the
  // CTAs of the largest units go first and the short ones fill the tail
  std::stable_sort(P.mean_items.begin(), P.mean_items.end(), [&](const MeanItem& x, const MeanItem& y) {
    return units[x.unit].n_sites > units[y.unit].n_sites;
  });
  return LGMI_OK;
}

// ------------------------------------------------------------------ the plan of a pipelined step
// one group: a batch of its own over the units [unit0, unit0 + n_units) of the whole batch
struct GroupPlan {
  uint32_t unit0 = 0, n_units = 0;
  uint64_t plane0 = 0, site0 = 0;             // the group's first plane word and site in the whole batch
  uint64_t tight0 = 0, tight_words = 0;       // its slice of the tight two-plane input (LGMI_MODE_TIGHT_INPUT)
  std::vector<lgmi_unit_desc> units;          // its descriptors, rebased to plane0 / site0
  uint64_t plane_words = 0, n_sites = 0;      // ... and the sizes of its batch
  std::vector<unsigned long long> tight_off;  // first word of each unit in the tight input, relative to tight0
};

struct PipelinePlan {
  std::vector<GroupPlan> groups;
  uint64_t n_candidates = 0;
  uint32_t max_sites = 0;
};

// The groups of a pipelined step: the units cut into at most n_chunks consecutive groups of about equal cost.  A
// group's input is a slice of the whole batch's, so the units must lie back to back, in order.  Returns LGMI_OK, or
// LGMI_ERR_ARG / LGMI_ERR_UNSUPPORTED with *err set.
inline int plan_pipeline(const lgmi_unit_desc* units, uint32_t n_units, uint32_t n_chunks, PipelinePlan* plan,
                         std::string* err) {
  PipelinePlan& P = *plan;
  P = PipelinePlan();
  if (n_chunks == 0) return plan_error(err, LGMI_ERR_ARG, "lgmi_pipeline_create: n_chunks must be >= 1");
  std::vector<uint64_t> tight_off((size_t)n_units + 1, 0), cost(n_units);
  uint64_t cost_total = 0;
  for (uint32_t k = 0; k < n_units; ++k) {
    const lgmi_unit_desc& u = units[k];
    const uint64_t want_plane = k ? units[k - 1].plane_off + 3ull * units[k - 1].n_sites * units[k - 1].row_words : u.plane_off;
    const uint64_t want_site = k ? (uint64_t)units[k - 1].site_off + units[k - 1].n_sites : u.site_off;
    if (u.plane_off != want_plane || u.site_off != want_site)
      return plan_error(err, LGMI_ERR_UNSUPPORTED, "lgmi_pipeline_create: unit %u is not laid out right after unit %u",
                        k, k - 1);
    const uint64_t np = unit_pairs(u.n_sites, 0u);
    P.n_candidates += np;
    P.max_sites = std::max(P.max_sites, u.n_sites);
    // the tight two-plane form: rows of ceil(R/32) words, units back to back
    tight_off[k + 1] = tight_off[k] + 2ull * u.n_sites * ((u.n_reads + 31u) / 32u);
    // equal shares of the work: candidate pairs plus a term for the bytes to move
    cost[k] = np + (uint64_t)u.n_sites * u.row_words / 4 + 1;
    cost_total += cost[k];
  }
  n_chunks = std::min<uint32_t>(n_chunks, std::max<uint32_t>(1, n_units));
  uint32_t k = 0;
  uint64_t done_cost = 0;
  for (uint32_t c = 0; c < n_chunks && (k < n_units || c == 0); ++c) {
    const uint32_t unit0 = k;
    const uint64_t target = cost_total * (c + 1) / n_chunks;
    while (k < n_units && (done_cost < target || c + 1 == n_chunks)) done_cost += cost[k++];
    if (k == unit0 && n_units) continue;  // one unit outweighs a whole share
    GroupPlan g;
    g.unit0 = unit0;
    g.n_units = k - unit0;
    g.plane0 = g.n_units ? units[unit0].plane_off : 0;
    g.site0 = g.n_units ? units[unit0].site_off : 0;
    g.tight0 = tight_off[unit0];
    g.tight_words = tight_off[k] - g.tight0;
    g.units.assign(units + unit0, units + k);
    for (uint32_t q = 0; q < g.n_units; ++q) {
      lgmi_unit_desc& u = g.units[q];
      u.plane_off -= g.plane0;
      u.site_off -= (uint32_t)g.site0;
      g.plane_words = u.plane_off + 3ull * u.n_sites * u.row_words;
      g.n_sites = (uint64_t)u.site_off + u.n_sites;
      g.tight_off.push_back(tight_off[unit0 + q] - g.tight0);
    }
    P.groups.push_back(std::move(g));
  }
  return LGMI_OK;
}

}  // namespace lgmi
