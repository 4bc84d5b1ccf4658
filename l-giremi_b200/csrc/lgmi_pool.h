// lgmi_pool.h -- the size-bucketed cache of device and pinned-host blocks a context owns (MemPool), and the owner of
// one block from it (PoolBuf).
//
// Plain C++17, no CUDA types or calls: the raw allocate and free are injected (lgmi.cu: cudaMalloc / cudaHostAlloc,
// cudaFree / cudaFreeHost), so tests/test_pool_host.py drives the pool with a fake allocator on the host.
#pragma once

#include <cstddef>
#include <cstdint>
#include <cstring>
#include <map>
#include <unordered_map>

namespace lgmi {

struct RawAllocator {
  int (*alloc)(void** out, size_t bytes);  // 0 on success, else an error code
  void (*free)(void* p);
  int out_of_memory;                       // alloc's code for exhausted memory: give the cache back and retry once
};

// Batches and pipelines are created and destroyed per submit by the drop-in seam (one chunk of footprints = one
// submit); cudaMalloc / cudaHostAlloc / cudaFree cost tens of microseconds to milliseconds each and cudaFree
// synchronises the device, so their buffers are recycled instead.  A block may only be released once nothing in
// flight can still touch it: its owner synchronises first (~lgmi_batch, ~lgmi_pipeline).
struct MemPool {
  explicit MemPool(RawAllocator r) : raw(r) {}
  MemPool(const MemPool&) = delete;
  MemPool& operator=(const MemPool&) = delete;
  ~MemPool() { destroy(); }

  RawAllocator raw;
  std::multimap<size_t, void*> free_blocks;
  std::unordered_map<void*, size_t> live;
  size_t cached_bytes = 0, cap_bytes = 0;
  uint64_t hits = 0, misses = 0;

  static size_t bucket(size_t n) {  // sixteenth-of-an-octave steps: at most 1/8 over-allocation
    if (n <= 4096) return 4096;
    size_t p = 1;
    while (p < n) p <<= 1;
    const size_t step = p >> 4;
    return (n + step - 1) / step * step;
  }
  void trim() {
    for (auto& kv : free_blocks) raw.free(kv.second);
    free_blocks.clear();
    cached_bytes = 0;
  }
  int alloc(void** out, size_t bytes) {
    const size_t sz = bucket(bytes ? bytes : 1);
    auto it = free_blocks.lower_bound(sz);
    if (it != free_blocks.end() && it->first <= sz + sz / 4) {
      *out = it->second;
      live[*out] = it->first;
      cached_bytes -= it->first;
      free_blocks.erase(it);
      ++hits;
      return 0;
    }
    ++misses;
    int e = raw.alloc(out, sz);
    if (e == raw.out_of_memory) {  // give the cache back and try once more
      trim();
      e = raw.alloc(out, sz);
    }
    if (e == 0) live[*out] = sz;
    return e;
  }
  void release(void* p) {
    if (!p) return;
    auto it = live.find(p);
    if (it == live.end()) {  // not ours (never happens): hand it to the runtime
      raw.free(p);
      return;
    }
    const size_t sz = it->second;
    live.erase(it);
    if (cached_bytes + sz > cap_bytes) {
      raw.free(p);
      return;
    }
    free_blocks.emplace(sz, p);
    cached_bytes += sz;
  }
  void destroy() {
    trim();
    for (auto& kv : live) raw.free(kv.first);
    live.clear();
  }
};

// One block of n elements of T from a MemPool, released to it exactly once: when the owner is destroyed, assigned
// over or re-allocated.  Converts to T* so that kernel parameters and copies read as with a plain pointer.
template <class T>
class PoolBuf {
 public:
  PoolBuf() = default;
  PoolBuf(const PoolBuf&) = delete;
  PoolBuf& operator=(const PoolBuf&) = delete;
  PoolBuf(PoolBuf&& o) noexcept : pool_(o.pool_), p_(o.p_), n_(o.n_) { o.forget(); }
  PoolBuf& operator=(PoolBuf&& o) noexcept {
    if (this != &o) {
      reset();
      pool_ = o.pool_, p_ = o.p_, n_ = o.n_;
      o.forget();
    }
    return *this;
  }
  ~PoolBuf() { reset(); }

  // A block of n elements from pool in place of the one held.  That one goes back first; with keep > 0 (host
  // blocks only, keep <= min(n, size())) it goes back after its first keep elements have been copied to the new
  // block, and a failed allocation leaves it in place.
  int alloc(MemPool& pool, size_t n, size_t keep = 0) {
    if (!keep) reset();
    void* fresh = nullptr;
    if (const int e = pool.alloc(&fresh, n * sizeof(T))) return e;
    if (keep) memcpy(fresh, p_, keep * sizeof(T));
    reset();
    pool_ = &pool, p_ = static_cast<T*>(fresh), n_ = n;
    return 0;
  }
  void reset() {
    if (p_) pool_->release(p_);
    forget();
  }

  T* get() const { return p_; }
  operator T*() const { return p_; }
  T* operator->() const { return p_; }
  size_t size() const { return n_; }  // elements asked for (the block may be larger: MemPool::bucket)

 private:
  void forget() { pool_ = nullptr, p_ = nullptr, n_ = 0; }
  MemPool* pool_ = nullptr;
  T* p_ = nullptr;
  size_t n_ = 0;
};

}  // namespace lgmi
