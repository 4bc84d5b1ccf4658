// Host build of the het-anchored plan of a deep unit (plan_het_dense in l-giremi_b200/csrc/lgmi_plan.h) for the
// CPU tests in tests/test_dense_het_plan.py: one unit planned by plan_batch, then its het plan from the flag
// bytes, copied out for ctypes.  Test infrastructure; not part of the product library.
#include <cstdint>
#include <cstring>
#include "../../l-giremi_b200/csrc/lgmi_plan.h"

using namespace lgmi;

struct HetCase {
  BatchPlan batch;
  std::vector<DenseTile> tiles;
  HetDensePlan het;
};

extern "C" {
// unit u (site_off 0, flags[0 .. S)), row_limit 0 or a piece's; cfg: num_sms, dense_path, tile_path,
// dense_min_sites, dense_min_reads.  NULL (with *rc set) when the plan fails or the unit is not deep.
void* hp_plan(const lgmi_unit_desc* u, uint32_t row_limit, const uint32_t* cfg, const uint8_t* flags, int* rc) {
  HetCase* c = new HetCase();
  const PlanConfig pc{cfg[0], (int)cfg[1], (int)cfg[2], cfg[3], cfg[4]};
  const uint64_t words = u->plane_off + 3ull * u->n_sites * u->row_words;
  *rc = plan_batch(u, 1, row_limit ? &row_limit : nullptr, words, u->n_sites, pc, &c->batch, nullptr);
  if (*rc != LGMI_OK || c->batch.dense_plans.size() != 1) {
    delete c;
    return nullptr;
  }
  plan_het_dense(c->batch.dense_plans[0], flags, row_limit != 0u, cfg[0], c->tiles, &c->het);
  return c;
}
void hp_free(void* h) { delete static_cast<HetCase*>(h); }

// H, H_pad, fewer, four, k_blocks, S_pad, triangle macs4, macs9, het list4 off / n / n_whole / macs, list9 the same
void hp_scalars(void* h, uint64_t* out) {
  const HetCase& c = *static_cast<HetCase*>(h);
  const DensePlan& pl = c.batch.dense_plans[0];
  const HetDensePlan& p = c.het;
  const uint64_t v[16] = {p.H,         p.H_pad,    p.fewer,          pl.four,   pl.k_blocks, pl.S_pad,
                          pl.list4.macs, pl.list9.macs, p.list4.off, p.list4.n, p.list4.n_whole, p.list4.macs,
                          p.list9.off, p.list9.n, p.list9.n_whole, p.list9.macs};
  memcpy(out, v, sizeof v);
}
uint64_t hp_het(void* h, uint32_t* out) {
  const HetCase& c = *static_cast<HetCase*>(h);
  if (out) memcpy(out, c.het.het.data(), c.het.het.size() * sizeof(uint32_t));
  return c.het.het.size();
}
uint64_t hp_tiles(void* h, void* out) {
  const HetCase& c = *static_cast<HetCase*>(h);
  if (out) memcpy(out, c.tiles.data(), c.tiles.size() * sizeof(DenseTile));
  return c.tiles.size();
}
int hp_take(void* h, uint32_t mode, int host_flags) {
  return take_het_form(static_cast<HetCase*>(h)->het, mode, host_flags != 0) ? 1 : 0;
}
}
