// Host build of l-giremi_b200/csrc/lgmi_plan.h for the CPU tests of the batch plan (tests/test_plan_host.py):
// the same plan_batch() lgmi_batch_create runs and plan_pipeline() lgmi_pipeline_create runs, their tables copied
// out for ctypes.  Test infrastructure; not part of the product library.
#include <cstdint>
#include <cstring>
#include "../../l-giremi_b200/csrc/lgmi_plan.h"

using namespace lgmi;

// cfg: num_sms, dense_path, tile_path, dense_min_sites, dense_min_reads
static PlanConfig config(const uint32_t* cfg) { return PlanConfig{cfg[0], (int)cfg[1], (int)cfg[2], cfg[3], cfg[4]}; }

template <class T>
static uint64_t copy_out(const std::vector<T>& v, void* out) {
  if (out) memcpy(out, v.data(), v.size() * sizeof(T));
  return v.size();
}

extern "C" {
// the plan of a batch (row_limit may be NULL): a handle, or NULL with *rc and err[0 .. err_cap) set
void* p_plan(const lgmi_unit_desc* units, uint32_t n_units, const uint32_t* row_limit, uint64_t plane_words,
             uint64_t n_sites, const uint32_t* cfg, int* rc, char* err, uint32_t err_cap) {
  BatchPlan* p = new BatchPlan();
  std::string msg;
  *rc = plan_batch(units, n_units, row_limit, plane_words, n_sites, config(cfg), p, &msg);
  if (*rc == LGMI_OK) return p;
  snprintf(err, err_cap, "%s", msg.c_str());
  delete p;
  return nullptr;
}
void p_free(void* h) { delete static_cast<BatchPlan*>(h); }

// table t: 0 units, 1 items, 2 fast items, 3 tiled descs, 4 tile items, 5 gram tiles, 6 dense tiles, 7 mean items.
// Returns its length; copies its bytes to out unless out is NULL.
uint64_t p_table(void* h, int t, void* out) {
  const BatchPlan& p = *static_cast<BatchPlan*>(h);
  switch (t) {
    case 0: return copy_out(p.units, out);
    case 1: return copy_out(p.items, out);
    case 2: return copy_out(p.fast_items, out);
    case 3: return copy_out(p.tiled_desc, out);
    case 4: return copy_out(p.tile_items, out);
    case 5: return copy_out(p.gram_tiles, out);
    case 6: return copy_out(p.dense_tiles, out);
    case 7: return copy_out(p.mean_items, out);
  }
  return 0;
}
uint32_t p_table_elem(int t) {
  const uint32_t size[8] = {sizeof(DevUnit), sizeof(Item),     sizeof(FastItem),  sizeof(TiledDesc),
                            sizeof(TileItem), sizeof(TgTile), sizeof(DenseTile), sizeof(MeanItem)};
  return size[t];
}

// n_dense, gram_words, x_bytes, xt_words, oth_words, oth_sites, n_candidates, max_reads, n_tiled_work_items
void p_sizes(void* h, uint64_t* out) {
  const BatchPlan& p = *static_cast<BatchPlan*>(h);
  const uint64_t v[9] = {p.n_dense,   p.gram_words, p.x_bytes,      p.xt_words,          p.oth_words,
                         p.oth_sites, p.n_candidates, p.max_reads, p.n_tiled_work_items};
  memcpy(out, v, sizeof v);
}

// the deep units' plans, 18 words each: unit, S, W, S_pad, k_blocks, rows, oth_cap, four, plane_off, gram_off, then
// off, n, n_whole, macs of list4 and of list9.  Returns their number; copies them to out unless out is NULL.
uint64_t p_dense_plans(void* h, uint64_t* out) {
  const BatchPlan& p = *static_cast<BatchPlan*>(h);
  if (out)
    for (const DensePlan& d : p.dense_plans) {
      const uint64_t v[18] = {d.unit,         d.S,           d.W,          d.S_pad,       d.k_blocks,    d.rows,
                              d.oth_cap,      d.four,        d.plane_off,  d.gram_off,    d.list4.off,   d.list4.n,
                              d.list4.n_whole, d.list4.macs, d.list9.off,  d.list9.n,     d.list9.n_whole, d.list9.macs};
      memcpy(out, v, sizeof v);
      out += 18;
    }
  return p.dense_plans.size();
}

uint32_t p_route(const lgmi_unit_desc* u, uint32_t limit, const uint32_t* cfg) {
  return (uint32_t)route_unit(*u, limit, config(cfg));
}

uint64_t p_het_candidates(const lgmi_unit_desc* units, uint32_t n_units, const uint32_t* row_limit,
                          const uint8_t* site_flags) {
  std::vector<lgmi_unit_desc> u(units, units + n_units);
  std::vector<uint32_t> rl;
  if (row_limit) rl.assign(row_limit, row_limit + n_units);
  return het_candidates(u, rl, site_flags);
}

// the plan of a pipelined step: a handle, or NULL with *rc and err[0 .. err_cap) set
void* p_pipeline(const lgmi_unit_desc* units, uint32_t n_units, uint32_t n_chunks, int* rc, char* err,
                 uint32_t err_cap) {
  PipelinePlan* p = new PipelinePlan();
  std::string msg;
  *rc = plan_pipeline(units, n_units, n_chunks, p, &msg);
  if (*rc == LGMI_OK) return p;
  snprintf(err, err_cap, "%s", msg.c_str());
  delete p;
  return nullptr;
}
void p_pipeline_free(void* h) { delete static_cast<PipelinePlan*>(h); }

// n_candidates, max_sites.  Returns the number of groups.
uint64_t p_pipeline_sizes(void* h, uint64_t* out) {
  const PipelinePlan& p = *static_cast<PipelinePlan*>(h);
  out[0] = p.n_candidates;
  out[1] = p.max_sites;
  return p.groups.size();
}

// group g: 8 words unit0, n_units, plane0, site0, tight0, tight_words, plane_words, n_sites; its rebased descriptors
// and relative tight offsets (n_units of each) are copied to units / tight_off unless NULL
void p_group(void* h, uint32_t g, uint64_t* out, void* units, void* tight_off) {
  const GroupPlan& q = static_cast<PipelinePlan*>(h)->groups[g];
  const uint64_t v[8] = {q.unit0, q.n_units, q.plane0, q.site0, q.tight0, q.tight_words, q.plane_words, q.n_sites};
  memcpy(out, v, sizeof v);
  copy_out(q.units, units);
  copy_out(q.tight_off, tight_off);
}
}
