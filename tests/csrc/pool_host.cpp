// Host build of l-giremi_b200/csrc/lgmi_pool.h for the CPU tests of the block cache (tests/test_pool_host.py): a
// MemPool over a counting fake allocator, and a PoolBuf<uint32_t> from it, driven through ctypes.  Test
// infrastructure; not part of the product library.
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <unordered_map>
#include <utility>
#include "../../l-giremi_b200/csrc/lgmi_pool.h"

using namespace lgmi;

namespace {
constexpr int kOutOfMemory = 2;

// malloc'd blocks, at most `limit` bytes outstanding; every call counted
struct Fake {
  uint64_t allocs = 0, frees = 0, ooms = 0, bad_frees = 0;  // allocs counts the failed calls too
  uint64_t limit = UINT64_MAX, outstanding = 0;
  std::unordered_map<void*, size_t> blocks;
} g;

int fake_alloc(void** out, size_t n) {
  ++g.allocs;
  if (g.outstanding + n > g.limit) {
    ++g.ooms;
    return kOutOfMemory;
  }
  *out = malloc(n);
  g.blocks[*out] = n;
  g.outstanding += n;
  return 0;
}

void fake_free(void* p) {
  ++g.frees;
  auto it = g.blocks.find(p);
  if (it == g.blocks.end()) {  // freed twice, or never allocated here
    ++g.bad_frees;
    return;
  }
  g.outstanding -= it->second;
  g.blocks.erase(it);
  free(p);
}

typedef PoolBuf<uint32_t> Buf;
}  // namespace

extern "C" {
// counters back to zero (the blocks outstanding stay), and the byte limit
void fake_reset(uint64_t limit) {
  g.allocs = g.frees = g.ooms = g.bad_frees = 0;
  g.limit = limit;
}
// allocs, frees, ooms, bad_frees, outstanding bytes, outstanding blocks
void fake_counts(uint64_t* out) {
  const uint64_t v[6] = {g.allocs, g.frees, g.ooms, g.bad_frees, g.outstanding, g.blocks.size()};
  memcpy(out, v, sizeof v);
}
// a block the pool has not handed out
void* fake_raw(uint64_t n) {
  void* p = nullptr;
  return fake_alloc(&p, n) ? nullptr : p;
}

void* pool_new(uint64_t cap_bytes) {
  MemPool* p = new MemPool(RawAllocator{fake_alloc, fake_free, kOutOfMemory});
  p->cap_bytes = cap_bytes;
  return p;
}
void pool_delete(void* p) { delete static_cast<MemPool*>(p); }
uint64_t pool_bucket(uint64_t n) { return MemPool::bucket(n); }
int pool_alloc(void* p, uint64_t bytes, void** out) { return static_cast<MemPool*>(p)->alloc(out, bytes); }
void pool_release(void* p, void* block) { static_cast<MemPool*>(p)->release(block); }
void pool_destroy(void* p) { static_cast<MemPool*>(p)->destroy(); }
// cached bytes, hits, misses, cached blocks, live blocks
void pool_stats(void* h, uint64_t* out) {
  const MemPool& p = *static_cast<MemPool*>(h);
  const uint64_t v[5] = {p.cached_bytes, p.hits, p.misses, p.free_blocks.size(), p.live.size()};
  memcpy(out, v, sizeof v);
}

void* buf_new() { return new Buf(); }
void* buf_moved(void* src) { return new Buf(std::move(*static_cast<Buf*>(src))); }
void buf_assign(void* dst, void* src) { *static_cast<Buf*>(dst) = std::move(*static_cast<Buf*>(src)); }
void buf_delete(void* b) { delete static_cast<Buf*>(b); }
int buf_alloc(void* b, void* pool, uint64_t n, uint64_t keep) {
  return static_cast<Buf*>(b)->alloc(*static_cast<MemPool*>(pool), n, keep);
}
void* buf_ptr(void* b) { return static_cast<Buf*>(b)->get(); }
uint64_t buf_size(void* b) { return static_cast<Buf*>(b)->size(); }
}
