// lgmi.cu -- host side of liblgmi.so: the C ABI declared in include/lgmi.h.
//
// Owns the CUDA context state (stream, ln table, pinned staging), builds the
// per-batch work tables and launches the kernels in lgmi_kernels.cuh.  There is
// no CPU implementation of the MI step in this library: every entry point that
// computes does so on the device, and lgmi_create() fails without one.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <queue>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include <unistd.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "../../include/lgmi.h"
#include "lgmi_kernels.cuh"
#include "lgmi_sitesplice.cuh"
#include "lgmi_plan.h"
#include "lgmi_pool.h"

extern "C" void lgmi_build_lntab(double* hi_lo_pairs, uint64_t k_begin, uint64_t k_end);

using namespace lgmi;

static thread_local std::string g_create_error;

// Owners of CUDA handles and of the context's plain cudaMalloc blocks: the deleter is the runtime's destroy call.
template <auto Destroy>
struct CudaDeleter {
  template <class P>
  void operator()(P p) const { Destroy(p); }
};
using Stream = std::unique_ptr<CUstream_st, CudaDeleter<cudaStreamDestroy>>;
using Event = std::unique_ptr<CUevent_st, CudaDeleter<cudaEventDestroy>>;
using GraphExec = std::unique_ptr<CUgraphExec_st, CudaDeleter<cudaGraphExecDestroy>>;
template <class T>
using DevPtr = std::unique_ptr<T, CudaDeleter<cudaFree>>;

static cudaError_t create(Stream& s) {
  cudaStream_t h = nullptr;
  const cudaError_t e = cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking);
  s.reset(h);
  return e;
}
static cudaError_t create(Event& ev, unsigned flags) {
  cudaEvent_t h = nullptr;
  const cudaError_t e = cudaEventCreateWithFlags(&h, flags);
  ev.reset(h);
  return e;
}
// the block held before is freed first
template <class T>
static cudaError_t dev_alloc(DevPtr<T>& p, size_t bytes) {
  p.reset();
  T* h = nullptr;
  const cudaError_t e = cudaMalloc(&h, bytes);
  p.reset(h);
  return e;
}

// Blocks and events of other processes' batches (lgmi_piece_ipc), opened here.  Each handle is opened once per owner:
// a second cudaIpcOpenMemHandle of the same handle fails.  Released when the owner goes: mappings closed on the
// device they were opened on, events destroyed.  Whatever was queued on them must have finished by then.
static_assert(sizeof(cudaIpcMemHandle_t) == sizeof(lgmi_piece_ipc{}.plane_mem) &&
                  sizeof(cudaIpcEventHandle_t) == sizeof(lgmi_piece_ipc{}.event),
              "lgmi_piece_ipc carries the runtime's IPC handles as plain bytes");
struct IpcImports {
  struct Mem {
    cudaIpcMemHandle_t handle;
    int device;
    void* ptr;
  };
  struct Ev {
    cudaIpcEventHandle_t handle;
    cudaEvent_t ev;
  };
  std::vector<Mem> mems;
  std::vector<Ev> events;
  IpcImports() = default;
  IpcImports(const IpcImports&) = delete;
  IpcImports& operator=(const IpcImports&) = delete;
  ~IpcImports() {
    int current = 0;
    cudaGetDevice(&current);  // (the owner's own members are released on its device after this)
    for (const Mem& m : mems) {
      cudaSetDevice(m.device);
      cudaIpcCloseMemHandle(m.ptr);
    }
    for (const Ev& e : events) cudaEventDestroy(e.ev);
    cudaSetDevice(current);
  }
  // the block of `bytes` (a cudaIpcMemHandle_t) mapped into `device`'s address space
  cudaError_t open_mem(const uint8_t* bytes, int device, void** out) {
    for (const Mem& m : mems)
      if (m.device == device && !memcmp(&m.handle, bytes, sizeof m.handle)) return *out = m.ptr, cudaSuccess;
    Mem m{{}, device, nullptr};
    memcpy(&m.handle, bytes, sizeof m.handle);
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaIpcOpenMemHandle(&m.ptr, m.handle, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return e;
    mems.push_back(m);
    *out = m.ptr;
    return cudaSuccess;
  }
  // the event of `bytes` (a cudaIpcEventHandle_t), opened with the current device
  cudaError_t open_event(const uint8_t* bytes, cudaEvent_t* out) {
    for (const Ev& e : events)
      if (!memcmp(&e.handle, bytes, sizeof e.handle)) return *out = e.ev, cudaSuccess;
    Ev v{{}, nullptr};
    memcpy(&v.handle, bytes, sizeof v.handle);
    const cudaError_t e = cudaIpcOpenEventHandle(&v.ev, v.handle);
    if (e != cudaSuccess) return e;
    events.push_back(v);
    *out = v.ev;
    return cudaSuccess;
  }
};

// The raw allocations behind the context's pools.  An exhausted device or host returns cudaErrorMemoryAllocation,
// which CU reports as LGMI_ERR_NOMEM; the runtime also keeps it as the thread's last error, cleared here so that a
// later cudaGetLastError() check does not report it again.
static int no_sticky_oom(cudaError_t e) {
  if (e == cudaErrorMemoryAllocation) cudaGetLastError();
  return e;
}
static const RawAllocator kDeviceBlocks{[](void** out, size_t n) { return no_sticky_oom(cudaMalloc(out, n)); },
                                        [](void* p) { cudaFree(p); }, cudaErrorMemoryAllocation};
static const RawAllocator kPinnedBlocks{
    [](void** out, size_t n) { return no_sticky_oom(cudaHostAlloc(out, n, cudaHostAllocDefault)); },
    [](void* p) { cudaFreeHost(p); }, cudaErrorMemoryAllocation};

struct lgmi_ctx {
  ~lgmi_ctx();
  int device = 0;
  Stream own_stream;  // (declared first: destroyed after everything below)
  cudaStream_t stream = nullptr;
  std::string err;
  uint64_t launches = 0;
  // ln table
  DevPtr<lg_dd> d_lntab;
  uint64_t ln_cap = 0;  // entries 0..ln_cap-1 valid
  // one-shot submit state
  lgmi_batch* oneshot = nullptr;
  // scratch for ecdf / csr
  DevPtr<char> d_scratch;
  size_t scratch_cap = 0;
  DevPtr<uint16_t> d_ij_tab;  // triangular pair tables for S <= 64 (lg_ij_tab_off)
  // persistent launch shape of k_pairs
  int num_sms = 0;
  int pairs_ctas_per_sm = 0;
  int dense_path = 4;  // deep units: 4 = four Gram blocks + sparse "other" cells where the "other" reads are rare (decided on
                       // the device per unit and run), 9 = always nine blocks
  int tile_path = 1;   // mid-depth units: 0 popcount (k_tile_mi), else tensor cores (k_tile_gram_ws, default)
  // tensor-core path: units at least this large build their tables with k_gram_i8
  uint32_t dense_min_sites = 48, dense_min_reads = 8192;
  void* encode_tiled = nullptr;  // cuTensorMapEncodeTiled, resolved through the runtime (no libcuda link)
  MemPool dev_pool{kDeviceBlocks}, host_pool{kPinnedBlocks};  // recycled buffers of batches / pipelines
  uint64_t lntab_gen = 0;        // bumped when the ln table moves: captured graphs hold its address
  int pipeline_graphs = 1;       // groups of a pipelined step replay their launch chain as a CUDA graph (LGMI_GRAPHS=0: off)
};

struct lgmi_batch {
  explicit lgmi_batch(lgmi_ctx* c) : ctx(c) {}
  ~lgmi_batch();
  lgmi_ctx* const ctx;
  Stream own_stream;                  // pipeline chunks run on their own stream; otherwise the context's
  uint32_t unit_base = 0;             // added to the unit field of every record (pipeline chunks)
  Event ev[8];                        // 0-1 whole run, 2-3 k_pairs_fast, 4-5 tensor-core path, 6-7 last k_gram_i8
  uint32_t n_units = 0, n_items = 0, n_mean_items = 0, n_fast = 0;
  uint64_t plane_words = 0, n_sites = 0, n_candidates = 0, n_dense = 0;
  uint32_t max_reads = 0;
  std::vector<lgmi_unit_desc> h_units;
  // device
  PoolBuf<DevUnit> d_units;
  PoolBuf<Item> d_items;
  PoolBuf<FastItem> d_fast_items;
  PoolBuf<uint8_t> d_fast_empty;           // per fast item: the pre-pass counted no emitted pair
  PoolBuf<uint8_t> d_item_dense;
  PoolBuf<uint32_t> d_n_generic;
  PoolBuf<MeanItem> d_mean_items;     // 32-site blocks of the multi-item units
  PoolBuf<uint32_t> d_planes;
  PoolBuf<uint8_t> d_flags;
  PoolBuf<unsigned long long> d_item_cnt;  // n_items + 1 (last stays 0)
  PoolBuf<unsigned long long> d_item_off;  // n_items + 1
  PoolBuf<char> d_scan_tmp;
  size_t scan_tmp_bytes = 0;
  PoolBuf<Header> d_header;
  PoolBuf<lgmi_pair_rec> d_records;
  uint64_t rec_cap = 0;
  PoolBuf<uint32_t> d_counts;  // EMIT_COUNTS only, 9 per record slot, allocated on first use
  PoolBuf<double> d_site_mean;
  PoolBuf<uint32_t> d_site_cnt;
  PoolBuf<double> d_dense;
  PoolBuf<unsigned long long> d_unit_rec_off;
  // tensor-core path
  std::vector<DensePlan> dense_plans;
  std::vector<CUtensorMap> tmaps;  // per deep unit, parallel to dense_plans: its X for k_gram_i8's TMA loads
  PoolBuf<uint8_t> d_x;       // indicator matrix of the unit being contracted (reused unit after unit)
  PoolBuf<uint32_t> d_gram;   // nine count matrices per dense unit
  PoolBuf<uint32_t> d_xt;     // four-block form: transposed label planes of the unit being contracted
  PoolBuf<uint32_t> d_oth_cnt, d_oth_list;  // ... and its listed "other" reads per site
  PoolBuf<uint32_t> d_unit_mode;  // per unit: the form of this run (0 four blocks, else nine)
  // graph replays / pipeline groups: the small units' kernels (k_count_fast before the scan, k_pairs_fast after it) run on
  // a second stream beside the kernels of the larger units (forked and joined by events inside the captured chain)
  Stream side_stream;
  Event side_ev[4];
  Stream fix_stream;           // k_other_fix runs beside k_dense_x (forked after k_dense_prep,
  Event fix_fork, fix_join;    // joined before the tables are read)
  PoolBuf<DenseTile> d_tiles;
  uint64_t dense_macs = 0;      // multiply-accumulates the tile lists amount to
  // the het-anchored form of the deep units (HET_ONLY | SKIP_NONHET), planned from the host flag bytes at upload;
  // parallel to dense_plans (empty until flags have been seen)
  std::vector<HetDensePlan> het_plans;
  std::vector<DenseTile> h_het_tiles; // their tile lists
  std::vector<uint32_t> h_het_rows;   // per deep unit H_pad entries from het_rows_off: its het sites, ~0 for padding
  std::vector<uint64_t> het_rows_off;
  std::vector<uint8_t> h_unit_het;    // per unit: 1 if the het form is taken when the run allows it
  std::vector<CUtensorMap> het_tmaps; // per deep unit: its X_het for k_gram_i8's A operand
  PoolBuf<DenseTile> d_het_tiles;
  PoolBuf<uint32_t> d_het_rows;
  PoolBuf<uint8_t> d_unit_het;
  PoolBuf<uint8_t> d_x_het;           // the het sites' X rows of the unit being contracted, H_pad rows per group
  std::vector<std::pair<uint64_t, uint64_t>> run_macs;  // per deep unit, the last run's four- and nine-block lists' MACs
  // tiled popcount path
  PoolBuf<TileItem> d_tile_items;
  uint32_t n_tile_items = 0;
  PoolBuf<TgTile> d_gram_tiles;      // k_tile_gram_ws's work items (128 x 48 site blocks)
  uint32_t n_gram_tiles = 0;
  PoolBuf<uint2> d_tile_cnt;         // its output: 24 bytes of counts per pair slot
  uint32_t n_tiled_work_items = 0;     // work items (Item) of the tiled and of the deep units: k_pairs_generic<1>'s and <2>'s
  PoolBuf<TiledDesc> d_tiled_desc;   // k_pairs_generic<1>'s items, one self-contained record each
  uint32_t n_tiled_desc = 0;
  PoolBuf<uint32_t> d_tile_counts;  // EMIT_COUNTS only, allocated on first use
  // host (pinned) mirrors
  PoolBuf<Header> h_header;
  PoolBuf<lgmi_pair_rec> h_records;
  PoolBuf<uint32_t> h_counts;
  PoolBuf<double> h_site_mean;
  PoolBuf<uint32_t> h_site_cnt;
  PoolBuf<unsigned long long> h_unit_rec_off;
  // launch chains captured as CUDA graphs, one per (min_common, mode).  A graph holds the addresses it was captured
  // with: declared after the buffers, so destroyed before them.
  struct Graph {
    int min_common;
    uint32_t mode;
    uint64_t lntab_gen;
    uint64_t launches;  // kernels in the chain
    GraphExec exec;
  };
  std::vector<Graph> graphs;
  // run state
  bool uploaded = false, ran = false, last_timed = false;
  uint32_t last_mode = 0;
  // candidates with a het_snp partner (what SKIP_NONHET evaluates); known once host flags have been seen
  uint64_t n_het_candidates = 0;
  bool het_known = false;
  // lgmi_batch_create_rows: per unit its row limit (0: an ordinary unit) and first dense slot; empty otherwise
  std::vector<uint32_t> h_row_limit;
  std::vector<uint64_t> h_dense_off;
  Event copy_ev;  // lgmi_batch_copy_planes from this batch: what its stream has queued so far
  // lgmi_piece_export: the interprocess event other processes' copies wait on, and the batch's id in this process
  // (0: never exported)
  Event ipc_ev;
  uint64_t export_id = 0;
  IpcImports imports;  // lgmi_batch_copy_planes_ipc into this batch: the other processes' blocks and events it opened
};

// Batches that have exported a piece, by id: lgmi_split_means_ipc finds a piece of this process here.  Guarded by a
// mutex because batches on different contexts may be created and destroyed from different threads (DevicePool).
static std::mutex g_export_mu;
static std::unordered_map<uint64_t, lgmi_batch*> g_exported;
static uint64_t g_export_ids = 0;

// --------------------------------------------------------------------------- helpers
static inline cudaStream_t bstream(const lgmi_batch* b) { return b->own_stream ? b->own_stream.get() : b->ctx->stream; }

static int fail(lgmi_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_create_error = buf;
  return code;
}

#define CU(ctx, call)                                                                      \
  do {                                                                                     \
    const cudaError_t e__ = static_cast<cudaError_t>(call);                                \
    if (e__ != cudaSuccess)                                                                \
      return fail((ctx), (e__ == cudaErrorMemoryAllocation) ? LGMI_ERR_NOMEM : LGMI_ERR_CUDA, \
                  "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

static int ensure_lntab(lgmi_ctx* ctx, uint64_t k_max) {
  if (k_max + 1 <= ctx->ln_cap) return LGMI_OK;
  uint64_t cap = std::max<uint64_t>(4096, ctx->ln_cap);
  while (cap < k_max + 1) cap *= 2;
  std::vector<double> host(2 * cap);
  lgmi_build_lntab(host.data(), 0, cap);
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->ln_cap = 0;
  CU(ctx, dev_alloc(ctx->d_lntab, cap * sizeof(lg_dd)));
  CU(ctx, cudaMemcpy(ctx->d_lntab.get(), host.data(), cap * sizeof(lg_dd), cudaMemcpyHostToDevice));
  ctx->ln_cap = cap;
  ++ctx->lntab_gen;
  return LGMI_OK;
}

static int ensure_scratch(lgmi_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->scratch_cap) return LGMI_OK;
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->scratch_cap = 0;
  size_t cap = std::max<size_t>(bytes, 1 << 20);
  CU(ctx, dev_alloc(ctx->d_scratch, cap));
  ctx->scratch_cap = cap;
  return LGMI_OK;
}

// --------------------------------------------------------------------------- context
extern "C" int lgmi_version(void) { return LGMI_VERSION; }

extern "C" int lgmi_create(int device, lgmi_t** out) {
  if (!out) return fail(nullptr, LGMI_ERR_ARG, "lgmi_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, LGMI_ERR_NODEVICE,
                "lgmi_create: no CUDA device (%s); this library has no CPU path",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= ndev)
    return fail(nullptr, LGMI_ERR_ARG, "lgmi_create: device %d out of range [0,%d)", device, ndev);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10)
    return fail(nullptr, LGMI_ERR_NODEVICE,
                "lgmi_create: device %d is sm_%d%d; this build contains sm_100a code only", device,
                prop.major, prop.minor);
  // every failure from here on releases what the context holds so far
  std::unique_ptr<lgmi_ctx> ctx(new (std::nothrow) lgmi_ctx());
  if (!ctx) return fail(nullptr, LGMI_ERR_NOMEM, "lgmi_create: out of host memory");
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess || create(ctx->own_stream) != cudaSuccess)
    return fail(nullptr, LGMI_ERR_CUDA, "lgmi_create: %s", cudaGetErrorString(cudaGetLastError()));
  ctx->stream = ctx->own_stream.get();
  ctx->num_sms = prop.multiProcessorCount;
  ctx->dev_pool.cap_bytes = 16ull << 30;   // cached (idle) bytes kept at most; LGMI_POOL_MB overrides both
  ctx->host_pool.cap_bytes = 4ull << 30;
  if (const char* e = getenv("LGMI_POOL_MB")) ctx->dev_pool.cap_bytes = ctx->host_pool.cap_bytes = (size_t)atoll(e) << 20;
  if (cudaFuncSetAttribute(k_pairs_fast, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FastSmem)) !=
          cudaSuccess ||
      cudaFuncSetAttribute(k_pairs_fast_het, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FastSmem)) !=
          cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->pairs_ctas_per_sm, k_pairs_fast, kFastThreads,
                                                    sizeof(FastSmem)) != cudaSuccess ||
      ctx->pairs_ctas_per_sm < 1)
    return fail(nullptr, LGMI_ERR_CUDA, "lgmi_create: k_pairs_fast cannot be resident (%s)",
                cudaGetErrorString(cudaGetLastError()));
  if (const char* e = getenv("LGMI_DENSE_PATH")) ctx->dense_path = atoi(e) == 9 ? 9 : 4;
  if (const char* e = getenv("LGMI_TILE_PATH")) ctx->tile_path = atoi(e) ? 1 : 0;
  if (const char* e = getenv("LGMI_GRAPHS")) ctx->pipeline_graphs = atoi(e) ? 1 : 0;
  if (cudaFuncSetAttribute(k_tile_gram_ws, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTwSmemBytes) != cudaSuccess)
    return fail(nullptr, LGMI_ERR_CUDA, "lgmi_create: k_tile_gram_ws cannot be resident (%s)",
                cudaGetErrorString(cudaGetLastError()));
  {
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ctx->encode_tiled, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess || !ctx->encode_tiled ||
        cudaFuncSetAttribute(k_gram_i8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmemBytes) !=
            cudaSuccess)
      return fail(nullptr, LGMI_ERR_CUDA, "lgmi_create: tensor-core path unavailable (%s)",
                  cudaGetErrorString(cudaGetLastError()));
  }
  {
    std::vector<uint16_t> tab(kIjTabEntries);
    for (uint32_t S = 2; S <= (uint32_t)kFastMaxS; ++S) {
      uint32_t p = lg_ij_tab_off(S);
      for (uint32_t i = 0; i + 1 < S; ++i)
        for (uint32_t j = i + 1; j < S; ++j) tab[p++] = (uint16_t)(i * 64u + j);
    }
    if (dev_alloc(ctx->d_ij_tab, tab.size() * sizeof(uint16_t)) != cudaSuccess ||
        cudaMemcpy(ctx->d_ij_tab.get(), tab.data(), tab.size() * sizeof(uint16_t), cudaMemcpyHostToDevice) != cudaSuccess)
      return fail(nullptr, LGMI_ERR_CUDA, "lgmi_create: pair table upload failed (%s)",
                  cudaGetErrorString(cudaGetLastError()));
  }
  *out = ctx.release();
  return LGMI_OK;
}

// Runtime calls act on the current device, and DevicePool threads hold contexts on different GPUs: every destructor
// that releases device resources selects its context's device first.
lgmi_ctx::~lgmi_ctx() {
  cudaSetDevice(device);
  delete oneshot;  // its blocks go back to the pools below
  if (stream) cudaStreamSynchronize(stream);
}

extern "C" void lgmi_destroy(lgmi_t* ctx) { delete ctx; }

extern "C" const char* lgmi_last_error(const lgmi_t* ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" int lgmi_set_stream(lgmi_t* ctx, void* cuda_stream) {
  if (!ctx) return LGMI_ERR_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : ctx->own_stream.get();
  return LGMI_OK;
}

extern "C" int lgmi_pinned_alloc(lgmi_t* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return LGMI_ERR_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  return LGMI_OK;
}

extern "C" int lgmi_pinned_free(lgmi_t* ctx, void* ptr) {
  if (!ctx) return LGMI_ERR_ARG;
  if (ptr) CU(ctx, cudaFreeHost(ptr));
  return LGMI_OK;
}

extern "C" uint64_t lgmi_launch_count(const lgmi_t* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int lgmi_set_dense_path(lgmi_t* ctx, int blocks) {
  if (!ctx) return LGMI_ERR_ARG;
  if (blocks != 4 && blocks != 9) return fail(ctx, LGMI_ERR_ARG, "lgmi_set_dense_path: blocks must be 4 or 9");
  ctx->dense_path = blocks;
  return LGMI_OK;
}

extern "C" int lgmi_set_tile_path(lgmi_t* ctx, int tensor_cores) {
  if (!ctx) return LGMI_ERR_ARG;
  ctx->tile_path = tensor_cores ? 1 : 0;
  return LGMI_OK;
}

extern "C" int lgmi_set_dense_threshold(lgmi_t* ctx, uint32_t min_sites, uint32_t min_reads) {
  if (!ctx) return LGMI_ERR_ARG;
  if (min_sites < 2) return fail(ctx, LGMI_ERR_ARG, "lgmi_set_dense_threshold: min_sites must be >= 2");
  ctx->dense_min_sites = min_sites;
  ctx->dense_min_reads = min_reads;
  return LGMI_OK;
}

// --------------------------------------------------------------------------- batch
lgmi_batch::~lgmi_batch() {
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(bstream(this));  // nothing in flight touches a block when it goes back to the cache
  if (export_id) {
    std::lock_guard<std::mutex> lock(g_export_mu);
    g_exported.erase(export_id);
  }
}

extern "C" void lgmi_batch_destroy(lgmi_batch_t* b) {
  if (!b) return;
  if (b->ctx->oneshot == b) b->ctx->oneshot = nullptr;
  delete b;
}

// k_gram_i8's tensor map of an X of pl's unit at x: [3 * rows][K_pad bytes], K contiguous; box = 128 rows x 128 bytes,
// 128B swizzle
static int encode_x_map(lgmi_ctx* ctx, CUtensorMap* map, void* x, const DensePlan& pl, uint32_t rows) {
  typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  EncodeTiled encode = reinterpret_cast<EncodeTiled>(ctx->encode_tiled);
  const cuuint64_t dims[2] = {(cuuint64_t)pl.k_blocks * kDenseBK, 3ull * rows};
  const cuuint64_t strides[1] = {(cuuint64_t)pl.k_blocks * kDenseBK};
  const cuuint32_t box[2] = {(cuuint32_t)kDenseBK, 128u};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, x, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ctx, LGMI_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for unit %u", (int)r, pl.unit);
  return LGMI_OK;
}

// The het-anchored plans of the batch's deep units from the host flag bytes (site_flags: the batch's), and their
// tables on the device, copied on stream st.  What a captured launch chain holds of them -- which units take the form,
// their H_pad, the lengths of their tile lists and the buffers' addresses -- is the layout: when it changes, the
// stream is drained, buffers are sized and tensor maps encoded again, and the graphs are dropped.  With the same
// layout, new het sites only replace the tables' contents, in stream order.
static int plan_het(lgmi_batch* b, const uint8_t* site_flags, cudaStream_t st) {
  if (b->dense_plans.empty()) return LGMI_OK;
  lgmi_ctx* ctx = b->ctx;
  const size_t n = b->dense_plans.size();
  std::vector<HetDensePlan> plans(n);
  std::vector<DenseTile> tiles;
  std::vector<uint32_t> rows;
  std::vector<uint64_t> rows_off(n);
  std::vector<uint8_t> unit_het(b->n_units, 0);
  uint64_t x_bytes = 0;
  for (size_t d = 0; d < n; ++d) {
    const DensePlan& pl = b->dense_plans[d];
    const bool piece = !b->h_row_limit.empty() && b->h_row_limit[pl.unit] != 0u;
    HetDensePlan& h = plans[d];
    plan_het_dense(pl, site_flags + b->h_units[pl.unit].site_off, piece, (uint32_t)ctx->num_sms, tiles, &h);
    rows_off[d] = rows.size();
    rows.insert(rows.end(), h.het.begin(), h.het.end());
    rows.resize(rows.size() + (h.H_pad - h.H), ~0u);
    if (h.fewer) {
      unit_het[pl.unit] = 1;
      x_bytes = std::max<uint64_t>(x_bytes, 3ull * h.H_pad * pl.k_blocks * kDenseBK);
    }
  }
  auto layout = [](const HetDensePlan& h) {
    return std::vector<uint64_t>{h.fewer, h.H_pad, h.H != 0u, h.list4.n, h.list4.n_whole, h.list9.n, h.list9.n_whole};
  };
  bool same = b->het_plans.size() == n && b->h_unit_het == unit_het && b->d_het_tiles.size() >= std::max<size_t>(1, tiles.size()) &&
              b->d_het_rows.size() >= std::max<size_t>(1, rows.size()) && b->d_x_het.size() >= std::max<uint64_t>(1, x_bytes);
  for (size_t d = 0; same && d < n; ++d)
    same = layout(b->het_plans[d]) == layout(plans[d]) && b->het_rows_off[d] == rows_off[d];
  if (!same) {
    CU(ctx, cudaStreamSynchronize(st));
    CU(ctx, cudaStreamSynchronize(bstream(b)));  // (runs read the tables there; graphs hold their addresses)
    b->graphs.clear();
    b->het_plans.clear();  // (nothing is taken while the tables are being replaced)
    if (b->d_het_tiles.size() < std::max<size_t>(1, tiles.size())) CU(ctx, b->d_het_tiles.alloc(ctx->dev_pool, std::max<size_t>(1, tiles.size())));
    if (b->d_het_rows.size() < std::max<size_t>(1, rows.size())) CU(ctx, b->d_het_rows.alloc(ctx->dev_pool, std::max<size_t>(1, rows.size())));
    if (!b->d_unit_het) CU(ctx, b->d_unit_het.alloc(ctx->dev_pool, std::max<uint32_t>(1, b->n_units)));
    if (b->d_x_het.size() < std::max<uint64_t>(1, x_bytes)) CU(ctx, b->d_x_het.alloc(ctx->dev_pool, std::max<uint64_t>(1, x_bytes)));
    b->het_tmaps.assign(n, CUtensorMap{});
    for (size_t d = 0; d < n; ++d)
      if (plans[d].fewer && plans[d].H)
        if (const int rc = encode_x_map(ctx, &b->het_tmaps[d], b->d_x_het, b->dense_plans[d], plans[d].H_pad)) return rc;
  }
  b->h_het_tiles = std::move(tiles);
  b->h_het_rows = std::move(rows);
  b->het_rows_off = std::move(rows_off);
  b->h_unit_het = std::move(unit_het);
  if (!b->h_het_tiles.empty())
    CU(ctx, cudaMemcpyAsync(b->d_het_tiles, b->h_het_tiles.data(), b->h_het_tiles.size() * sizeof(DenseTile),
                            cudaMemcpyHostToDevice, st));
  if (!b->h_het_rows.empty())
    CU(ctx, cudaMemcpyAsync(b->d_het_rows, b->h_het_rows.data(), b->h_het_rows.size() * sizeof(uint32_t),
                            cudaMemcpyHostToDevice, st));
  if (b->n_units)
    CU(ctx, cudaMemcpyAsync(b->d_unit_het, b->h_unit_het.data(), b->n_units, cudaMemcpyHostToDevice, st));
  b->het_plans = std::move(plans);
  return LGMI_OK;
}

// lgmi_batch_create, and with row_limit (non-NULL) lgmi_batch_create_rows (a unit k with row_limit[k] != 0 is a piece
// of a split unit, plan_batch): the batch's plan, then its buffers and tables on the device and the tensor maps of
// its deep units.  Nothing is allocated for a batch whose plan fails.
static int batch_create(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units, const uint32_t* row_limit,
                        uint64_t plane_words, uint64_t n_sites, lgmi_batch_t** out) {
  if (!ctx || !out || (!units && n_units)) return fail(ctx, LGMI_ERR_ARG, "lgmi_batch_create: NULL argument");
  *out = nullptr;
  CU(ctx, cudaSetDevice(ctx->device));
  const PlanConfig cfg{(uint32_t)ctx->num_sms, ctx->dense_path, ctx->tile_path, ctx->dense_min_sites, ctx->dense_min_reads};
  BatchPlan plan;
  std::string err;
  if (const int rc = plan_batch(units, n_units, row_limit, plane_words, n_sites, cfg, &plan, &err))
    return fail(ctx, rc, "%s", err.c_str());

  // every failure from here on releases what the batch holds so far
  std::unique_ptr<lgmi_batch> b(new (std::nothrow) lgmi_batch(ctx));
  if (!b) return fail(ctx, LGMI_ERR_NOMEM, "lgmi_batch_create: out of host memory");
  b->n_units = n_units;
  b->plane_words = plane_words;
  b->n_sites = n_sites;
  b->h_units.assign(units, units + n_units);
  if (row_limit) {
    b->h_row_limit.assign(row_limit, row_limit + n_units);
    b->h_dense_off.resize(n_units);
    for (uint32_t k = 0; k < n_units; ++k) b->h_dense_off[k] = plan.units[k].dense_off;
  }
  b->n_items = (uint32_t)plan.items.size();
  b->n_fast = (uint32_t)plan.fast_items.size();
  b->n_mean_items = (uint32_t)plan.mean_items.size();
  b->n_tile_items = (uint32_t)plan.tile_items.size();
  b->n_gram_tiles = (uint32_t)plan.gram_tiles.size();
  b->n_tiled_desc = (uint32_t)plan.tiled_desc.size();
  b->n_tiled_work_items = plan.n_tiled_work_items;
  b->n_dense = plan.n_dense;
  b->n_candidates = plan.n_candidates;
  b->max_reads = plan.max_reads;
  b->dense_plans = std::move(plan.dense_plans);
  const cudaStream_t st = bstream(b.get());
  // a table of the plan on the device: at least min_n entries, the plan's uploaded
  auto upload = [&](auto& dst, const auto& v, size_t min_n) {
    auto e = static_cast<cudaError_t>(dst.alloc(ctx->dev_pool, std::max(min_n, v.size())));
    if (e == cudaSuccess && !v.empty())
      e = cudaMemcpyAsync(dst, v.data(), v.size() * sizeof(v[0]), cudaMemcpyHostToDevice, st);
    return e;
  };

  for (Event& e : b->ev) CU(ctx, create(e, cudaEventDefault));
  if (b->n_fast && (!b->dense_plans.empty() || b->n_tile_items || b->n_gram_tiles)) {
    CU(ctx, create(b->side_stream));
    for (Event& e : b->side_ev) CU(ctx, create(e, cudaEventDisableTiming));
  }
  CU(ctx, upload(b->d_units, plan.units, 1));
  CU(ctx, upload(b->d_items, plan.items, 1));
  CU(ctx, upload(b->d_fast_items, plan.fast_items, 1));
  CU(ctx, b->d_fast_empty.alloc(ctx->dev_pool, std::max<size_t>(1, b->n_fast)));
  CU(ctx, b->d_item_dense.alloc(ctx->dev_pool, std::max<size_t>(1, b->n_items)));
  CU(ctx, b->d_n_generic.alloc(ctx->dev_pool, 1));
  CU(ctx, upload(b->d_mean_items, plan.mean_items, 1));
  CU(ctx, b->d_planes.alloc(ctx->dev_pool, std::max<uint64_t>(4, plane_words)));
  CU(ctx, b->d_flags.alloc(ctx->dev_pool, std::max<uint64_t>(1, n_sites)));
  CU(ctx, b->d_item_cnt.alloc(ctx->dev_pool, (size_t)b->n_items + 1));
  CU(ctx, b->d_item_off.alloc(ctx->dev_pool, (size_t)b->n_items + 1));
  CU(ctx, cub::DeviceScan::ExclusiveSum(nullptr, b->scan_tmp_bytes, b->d_item_cnt.get(), b->d_item_off.get(),
                                        (int)b->n_items + 1, st));
  CU(ctx, b->d_scan_tmp.alloc(ctx->dev_pool, std::max<size_t>(b->scan_tmp_bytes, 16)));
  CU(ctx, cudaMemsetAsync(b->d_item_cnt, 0, ((size_t)b->n_items + 1) * sizeof(unsigned long long), st));
  CU(ctx, b->d_header.alloc(ctx->dev_pool, 1));
  CU(ctx, b->d_site_mean.alloc(ctx->dev_pool, std::max<uint64_t>(1, n_sites)));
  CU(ctx, b->d_site_cnt.alloc(ctx->dev_pool, std::max<uint64_t>(1, n_sites)));
  CU(ctx, b->d_dense.alloc(ctx->dev_pool, std::max<uint64_t>(1, plan.n_dense)));
  CU(ctx, b->d_unit_rec_off.alloc(ctx->dev_pool, (size_t)n_units + 1));
  if (b->n_tile_items) CU(ctx, upload(b->d_tile_items, plan.tile_items, 0));
  if (b->n_gram_tiles) {
    CU(ctx, upload(b->d_gram_tiles, plan.gram_tiles, 0));
    CU(ctx, b->d_tile_cnt.alloc(ctx->dev_pool, std::max<uint64_t>(1, plan.n_dense) * 3ull));
  }
  if (b->n_tiled_desc) CU(ctx, upload(b->d_tiled_desc, plan.tiled_desc, 0));
  if (!b->dense_plans.empty()) {
    CU(ctx, b->d_x.alloc(ctx->dev_pool, plan.x_bytes));
    CU(ctx, cudaMemsetAsync(b->d_x, 0, plan.x_bytes, st));  // rows of the site padding stay zero
    CU(ctx, b->d_gram.alloc(ctx->dev_pool, plan.gram_words));
    CU(ctx, b->d_unit_mode.alloc(ctx->dev_pool, n_units));
    if (plan.xt_words) {
      CU(ctx, b->d_xt.alloc(ctx->dev_pool, plan.xt_words));
      CU(ctx, b->d_oth_list.alloc(ctx->dev_pool, plan.oth_words));
      CU(ctx, b->d_oth_cnt.alloc(ctx->dev_pool, plan.oth_sites));
      CU(ctx, create(b->fix_stream));
      CU(ctx, create(b->fix_fork, cudaEventDisableTiming));
      CU(ctx, create(b->fix_join, cudaEventDisableTiming));
    }
    CU(ctx, upload(b->d_tiles, plan.dense_tiles, 0));
    b->tmaps.resize(b->dense_plans.size());
    for (size_t d = 0; d < b->dense_plans.size(); ++d)
      if (const int rc = encode_x_map(ctx, &b->tmaps[d], b->d_x, b->dense_plans[d], b->dense_plans[d].S_pad)) return rc;
  }
  b->rec_cap = std::max<uint64_t>(1, b->n_candidates);
  CU(ctx, b->d_records.alloc(ctx->dev_pool, b->rec_cap));
  CU(ctx, b->h_header.alloc(ctx->host_pool, 1));
  CU(ctx, b->h_site_mean.alloc(ctx->host_pool, std::max<uint64_t>(1, n_sites)));
  CU(ctx, b->h_site_cnt.alloc(ctx->host_pool, std::max<uint64_t>(1, n_sites)));
  CU(ctx, b->h_unit_rec_off.alloc(ctx->host_pool, (size_t)n_units + 1));
  CU(ctx, cudaStreamSynchronize(st));  // the plan's tables go out of scope
  if (const int rc = ensure_lntab(ctx, std::max<uint32_t>(b->max_reads, 1u))) return rc;
  *out = b.release();
  return LGMI_OK;
}

extern "C" int lgmi_batch_create(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units,
                                 uint64_t plane_words, uint64_t n_sites, lgmi_batch_t** out) {
  return batch_create(ctx, units, n_units, nullptr, plane_words, n_sites, out);
}

extern "C" int lgmi_batch_create_rows(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units,
                                      const uint32_t* row_limit, uint64_t plane_words, uint64_t n_sites,
                                      lgmi_batch_t** out) {
  if (!row_limit && n_units) return fail(ctx, LGMI_ERR_ARG, "lgmi_batch_create_rows: row_limit is NULL");
  static const uint32_t none = 0u;
  return batch_create(ctx, units, n_units, n_units ? row_limit : &none, plane_words, n_sites, out);
}

extern "C" int lgmi_batch_upload(lgmi_batch_t* b, const uint32_t* planes, const uint8_t* site_flags) {
  if (!b) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = b->ctx;
  if ((!planes && b->plane_words) || (!site_flags && b->n_sites))
    return fail(ctx, LGMI_ERR_ARG, "lgmi_batch_upload: NULL input");
  CU(ctx, cudaSetDevice(ctx->device));
  if (b->plane_words)
    CU(ctx, cudaMemcpyAsync(b->d_planes, planes, b->plane_words * sizeof(uint32_t), cudaMemcpyHostToDevice, bstream(b)));
  if (b->n_sites)
    CU(ctx, cudaMemcpyAsync(b->d_flags, site_flags, b->n_sites, cudaMemcpyHostToDevice, bstream(b)));
  b->n_het_candidates = b->n_sites ? het_candidates(b->h_units, b->h_row_limit, site_flags) : 0;
  b->het_known = true;
  b->uploaded = true;
  return plan_het(b, site_flags, bstream(b));
}

extern "C" int lgmi_batch_upload_rows(lgmi_batch_t* b, const uint32_t* planes, uint64_t word_begin, uint64_t word_end,
                                      const uint8_t* site_flags) {
  if (!b) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = b->ctx;
  if (word_begin > word_end || word_end > b->plane_words)
    return fail(ctx, LGMI_ERR_ARG, "lgmi_batch_upload_rows: words [%llu, %llu) outside the %llu plane words",
                (unsigned long long)word_begin, (unsigned long long)word_end, (unsigned long long)b->plane_words);
  if ((!planes && word_end > word_begin) || (!site_flags && b->n_sites))
    return fail(ctx, LGMI_ERR_ARG, "lgmi_batch_upload_rows: NULL input");
  CU(ctx, cudaSetDevice(ctx->device));
  if (word_end > word_begin)
    CU(ctx, cudaMemcpyAsync(b->d_planes + word_begin, planes, (word_end - word_begin) * sizeof(uint32_t),
                            cudaMemcpyHostToDevice, bstream(b)));
  if (b->n_sites)
    CU(ctx, cudaMemcpyAsync(b->d_flags, site_flags, b->n_sites, cudaMemcpyHostToDevice, bstream(b)));
  b->n_het_candidates = b->n_sites ? het_candidates(b->h_units, b->h_row_limit, site_flags) : 0;
  b->het_known = true;
  b->uploaded = true;
  return plan_het(b, site_flags, bstream(b));
}

// Direct peer copies from sdev to the current device ddev where the devices allow them; without peer access the
// runtime stages them through the host.
static void enable_peer(int ddev, int sdev) {
  if (sdev == ddev) return;
  int can = 0;
  if (cudaDeviceCanAccessPeer(&can, ddev, sdev) == cudaSuccess && can && cudaDeviceEnablePeerAccess(sdev, 0) != cudaSuccess)
    cudaGetLastError();  // (cudaErrorPeerAccessAlreadyEnabled, or no peer access: the copy works either way)
}

extern "C" int lgmi_batch_copy_planes(lgmi_batch_t* dst, uint64_t dst_word, const lgmi_batch_t* src, uint64_t src_word,
                                      uint64_t n_words) {
  if (!dst || !src) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = dst->ctx;
  if (dst_word > dst->plane_words || n_words > dst->plane_words - dst_word || src_word > src->plane_words ||
      n_words > src->plane_words - src_word)
    return fail(ctx, LGMI_ERR_ARG, "lgmi_batch_copy_planes: %llu words from %llu to %llu out of range",
                (unsigned long long)n_words, (unsigned long long)src_word, (unsigned long long)dst_word);
  if (!n_words) return LGMI_OK;
  lgmi_batch* s = const_cast<lgmi_batch*>(src);
  const int sdev = s->ctx->device, ddev = ctx->device;
  // the copy follows everything src's stream has queued so far (its upload)
  CU(ctx, cudaSetDevice(sdev));
  if (!s->copy_ev) CU(ctx, create(s->copy_ev, cudaEventDisableTiming));
  CU(ctx, cudaEventRecord(s->copy_ev.get(), bstream(s)));
  CU(ctx, cudaSetDevice(ddev));
  enable_peer(ddev, sdev);
  CU(ctx, cudaStreamWaitEvent(bstream(dst), s->copy_ev.get(), 0));
  CU(ctx, cudaMemcpyPeerAsync(dst->d_planes + dst_word, ddev, s->d_planes + src_word, sdev, n_words * sizeof(uint32_t),
                              bstream(dst)));
  dst->uploaded = true;
  return LGMI_OK;
}

// The device of this process that an exported piece lives on.
static int piece_device(lgmi_ctx* ctx, const char* fn, const lgmi_piece_ipc* p, int* dev) {
  if (!memchr(p->pci_bus_id, 0, sizeof p->pci_bus_id))
    return fail(ctx, LGMI_ERR_ARG, "%s: the piece's PCI bus id is not a string", fn);
  if (cudaDeviceGetByPCIBusId(dev, p->pci_bus_id) != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, LGMI_ERR_ARG, "%s: the piece's device (PCI bus id %s) is not visible to this process", fn,
                p->pci_bus_id);
  }
  return LGMI_OK;
}

extern "C" int lgmi_piece_export(lgmi_batch_t* b, uint32_t unit, lgmi_piece_ipc* out) {
  if (!b || !out) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = b->ctx;
  if (unit >= b->n_units || b->h_row_limit.empty() || !b->h_row_limit[unit])
    return fail(ctx, LGMI_ERR_ARG, "lgmi_piece_export: unit %u is not a unit with a row limit", unit);
  CU(ctx, cudaSetDevice(ctx->device));
  if (!b->ipc_ev) CU(ctx, create(b->ipc_ev, cudaEventInterprocess | cudaEventDisableTiming));
  if (!b->export_id) {
    std::lock_guard<std::mutex> lock(g_export_mu);
    b->export_id = ++g_export_ids;
    g_exported[b->export_id] = b;
  }
  // behind everything the batch's stream has queued: its upload, or its run
  CU(ctx, cudaEventRecord(b->ipc_ev.get(), bstream(b)));
  lgmi_piece_ipc p;
  memset(&p, 0, sizeof p);
  // A handle covers one whole allocation and the importer maps it at its base.  The pool hands out whole cudaMalloc
  // blocks (MemPool::alloc returns the raw allocation), so a PoolBuf's pointer is that base and offsets count from it.
  cudaIpcMemHandle_t mh;
  CU(ctx, cudaIpcGetMemHandle(&mh, b->d_planes.get()));
  memcpy(p.plane_mem, &mh, sizeof mh);
  CU(ctx, cudaIpcGetMemHandle(&mh, b->d_dense.get()));
  memcpy(p.dense_mem, &mh, sizeof mh);
  cudaIpcEventHandle_t eh;
  CU(ctx, cudaIpcGetEventHandle(&eh, b->ipc_ev.get()));
  memcpy(p.event, &eh, sizeof eh);
  const lgmi_unit_desc& u = b->h_units[unit];
  p.plane_word = u.plane_off;
  p.plane_words = 3ull * u.row_words * b->h_row_limit[unit];
  p.dense_off = b->h_dense_off[unit];
  p.dense_pairs = piece_pairs(b->h_row_limit[unit], u.n_sites);
  p.batch_id = b->export_id;
  p.unit = unit;
  p.n_sites = u.n_sites;
  p.row_limit = b->h_row_limit[unit];
  p.ran = b->ran ? 1u : 0u;
  p.pid = (int32_t)getpid();
  CU(ctx, cudaDeviceGetPCIBusId(p.pci_bus_id, (int)sizeof p.pci_bus_id, ctx->device));
  *out = p;
  return LGMI_OK;
}

extern "C" int lgmi_batch_copy_planes_ipc(lgmi_batch_t* dst, uint64_t dst_word, const lgmi_piece_ipc* src,
                                          uint64_t src_word, uint64_t n_words) {
  if (!dst || !src) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = dst->ctx;
  if (src->pid == (int32_t)getpid())
    return fail(ctx, LGMI_ERR_ARG,
                "lgmi_batch_copy_planes_ipc: the piece was exported by this process; copy from its batch with "
                "lgmi_batch_copy_planes");
  if (dst_word > dst->plane_words || n_words > dst->plane_words - dst_word || src_word < src->plane_word ||
      src_word - src->plane_word > src->plane_words || n_words > src->plane_words - (src_word - src->plane_word))
    return fail(ctx, LGMI_ERR_ARG, "lgmi_batch_copy_planes_ipc: %llu words from %llu to %llu out of range",
                (unsigned long long)n_words, (unsigned long long)src_word, (unsigned long long)dst_word);
  if (!n_words) return LGMI_OK;
  int sdev = 0;
  if (const int rc = piece_device(ctx, "lgmi_batch_copy_planes_ipc", src, &sdev)) return rc;
  const int ddev = ctx->device;
  void* base = nullptr;
  cudaEvent_t ev = nullptr;
  CU(ctx, dst->imports.open_mem(src->plane_mem, sdev, &base));  // (leaves sdev current: the event is opened there)
  CU(ctx, dst->imports.open_event(src->event, &ev));
  CU(ctx, cudaSetDevice(ddev));
  enable_peer(ddev, sdev);
  CU(ctx, cudaStreamWaitEvent(bstream(dst), ev, 0));
  CU(ctx, cudaMemcpyPeerAsync(dst->d_planes + dst_word, ddev, static_cast<const uint32_t*>(base) + src_word, sdev,
                              n_words * sizeof(uint32_t), bstream(dst)));
  dst->uploaded = true;
  return LGMI_OK;
}

static int run_chain(lgmi_batch* b, int min_common, uint32_t mode, bool timing);

// whether deep unit d of the batch takes the het-anchored form in a run of this mode
static bool het_form(const lgmi_batch* b, size_t d, uint32_t mode) {
  return d < b->het_plans.size() && take_het_form(b->het_plans[d], mode, b->het_known);
}

extern "C" int lgmi_batch_run(lgmi_batch_t* b, int min_common, uint32_t mode) {
  if (!b) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = b->ctx;
  if (!b->uploaded) return fail(ctx, LGMI_ERR_STATE, "lgmi_batch_run: no input uploaded");
  if ((mode & LGMI_MODE_SKIP_NONHET) && !(mode & LGMI_MODE_HET_ONLY))
    return fail(ctx, LGMI_ERR_ARG, "LGMI_MODE_SKIP_NONHET requires LGMI_MODE_HET_ONLY");
  CU(ctx, cudaSetDevice(ctx->device));
  // LGMI_MODE_GRAPH (and every group of a pipelined step): the whole launch chain as ONE cudaGraphLaunch
  const bool as_graph = (mode & LGMI_MODE_GRAPH) != 0u || (b->own_stream != nullptr && ctx->pipeline_graphs);
  mode &= ~LGMI_MODE_GRAPH;
  // the tile lists this run takes per deep unit (which of the two label forms is known after the run): what
  // dense_macs / gram_macs report, whatever is uploaded before the results are read
  b->run_macs.resize(b->dense_plans.size());
  for (size_t d = 0; d < b->dense_plans.size(); ++d) {
    const bool het = het_form(b, d, mode);
    const DensePlan& pl = b->dense_plans[d];
    b->run_macs[d] = {het ? b->het_plans[d].list4.macs : pl.list4.macs, het ? b->het_plans[d].list9.macs : pl.list9.macs};
  }
  // buffers the chain needs exist before anything is launched or captured
  if ((mode & LGMI_MODE_EMIT_COUNTS) && b->d_counts.size() < b->rec_cap * 9ull) {
    CU(ctx, cudaStreamSynchronize(bstream(b)));
    b->graphs.clear();  // they hold the addresses they were captured with
    CU(ctx, b->d_counts.alloc(ctx->dev_pool, b->rec_cap * 9ull));
  }
  if ((mode & LGMI_MODE_EMIT_COUNTS) && (b->n_tile_items || b->n_gram_tiles) && !b->d_tile_counts) {
    CU(ctx, cudaStreamSynchronize(bstream(b)));
    b->graphs.clear();
    CU(ctx, b->d_tile_counts.alloc(ctx->dev_pool, std::max<uint64_t>(1, b->n_dense) * 9ull));
  }
  if (!as_graph) return run_chain(b, min_common, mode, b->own_stream == nullptr);
  lgmi_batch::Graph* hit = nullptr;
  for (lgmi_batch::Graph& g : b->graphs)
    if (g.min_common == min_common && g.mode == mode) hit = &g;
  if (hit && hit->lntab_gen != ctx->lntab_gen) {  // the ln table has moved since the capture
    b->graphs.clear();
    hit = nullptr;
  }
  if (!hit) {
    cudaStream_t st = bstream(b);
    cudaGraph_t graph = nullptr;
    const uint64_t launches0 = ctx->launches;
    CU(ctx, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    const int rc = run_chain(b, min_common, mode, false);
    const cudaError_t e = cudaStreamEndCapture(st, &graph);
    const uint64_t n_launch = ctx->launches - launches0;
    ctx->launches = launches0;
    if (rc != LGMI_OK || e != cudaSuccess || !graph) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      return rc != LGMI_OK ? rc : fail(ctx, LGMI_ERR_CUDA, "graph capture of the launch chain failed: %s", cudaGetErrorString(e));
    }
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ei = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) return fail(ctx, LGMI_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ei));
    b->graphs.push_back(lgmi_batch::Graph{min_common, mode, ctx->lntab_gen, n_launch, GraphExec(exec)});
    hit = &b->graphs.back();
  }
  CU(ctx, cudaGraphLaunch(hit->exec.get(), bstream(b)));
  ctx->launches += hit->launches;
  b->ran = true;
  b->last_mode = mode;
  b->last_timed = false;
  return LGMI_OK;
}

// the launch chain of one run on the batch's stream (also what a graph capture records)
static int run_chain(lgmi_batch* b, int min_common, uint32_t mode, bool timing) {
  lgmi_ctx* ctx = b->ctx;
  RunParams P;
  P.units = b->d_units;
  P.items = b->d_items;
  P.n_items = b->n_items;
  P.tiled_desc = b->d_tiled_desc;
  P.n_tiled_desc = b->n_tiled_desc;
  P.n_units = b->n_units;
  P.planes = b->d_planes;
  P.site_flags = b->d_flags;
  P.lntab = ctx->d_lntab.get();
  P.ln_cap = (uint32_t)std::min<uint64_t>(ctx->ln_cap, 0xffffffffull);
  P.min_common = min_common;
  P.mode = mode;
  P.item_cnt = b->d_item_cnt;
  P.item_off = b->d_item_off;
  P.item_dense = b->d_item_dense;
  P.n_generic = b->d_n_generic;
  P.header = b->d_header;
  P.records = b->d_records;
  P.counts = b->d_counts;
  P.site_mean = b->d_site_mean;
  P.site_cnt = b->d_site_cnt;
  P.dense = b->d_dense;
  P.unit_rec_off = b->d_unit_rec_off;
  P.gram = b->d_gram;
  P.unit_mode = b->d_unit_mode;
  P.unit_het = nullptr;
  for (size_t d = 0; d < b->dense_plans.size(); ++d)
    if (het_form(b, d, mode)) P.unit_het = b->d_unit_het;
  P.unit_base = b->unit_base;
  P.tile_counts = b->d_tile_counts;

  // (pipeline groups and graph replays skip the per-kernel events)
  if (timing) CU(ctx, cudaEventRecord(b->ev[0].get(), bstream(b)));
  {
    // one launch resets the run state: header, offsets, flags, NaN means (sites of pair-less units keep them)
    const uint64_t n = std::max<uint64_t>(std::max<uint64_t>(b->n_sites, b->n_items), (uint64_t)b->n_units + 1);
    k_run_init<<<(unsigned)((n + 255) / 256), 256, 0, bstream(b)>>>(b->d_header, b->own_stream ? b->h_header.get() : nullptr,
                                                                  b->d_unit_rec_off, b->n_units + 1,
                                                                  b->d_item_dense, b->n_items, b->d_n_generic,
                                                                  b->n_items - b->n_fast - b->n_tiled_work_items, b->d_site_mean,
                                                                  b->d_site_cnt, b->n_sites);
    ++ctx->launches;
  }
  if (timing) CU(ctx, cudaEventRecord(b->ev[4].get(), bstream(b)));
  // untimed runs (graph captures, pipeline groups) of mixed batches: the small units' kernels on the side stream
  static const bool fork_ok = !(getenv("LGMI_FORK") && atoi(getenv("LGMI_FORK")) == 0);  // LGMI_FORK=0: one stream
  const bool forked = !timing && b->side_stream != nullptr && fork_ok;
  cudaStream_t small = forked ? b->side_stream.get() : bstream(b);
  if (forked) {
    CU(ctx, cudaEventRecord(b->side_ev[0].get(), bstream(b)));
    CU(ctx, cudaStreamWaitEvent(small, b->side_ev[0].get(), 0));
  }
  if (!b->dense_plans.empty())  // every dense unit starts a run in the four-block form
    CU(ctx, cudaMemsetAsync(b->d_unit_mode, 0, (size_t)b->n_units * sizeof(uint32_t), bstream(b)));
  for (const DensePlan& pl : b->dense_plans) {
    // K3: bit-planes -> 0/1 bytes -> count matrices on the tensor cores (lgmi_dense.cuh)
    const size_t d = &pl - b->dense_plans.data();
    const HetDensePlan* het = het_form(b, d, mode) ? &b->het_plans[d] : nullptr;
    const uint32_t* het_rows = het ? b->d_het_rows + b->het_rows_off[d] : nullptr;
    uint32_t* unit_mode = b->d_unit_mode + pl.unit;
    const uint32_t* planes = b->d_planes + pl.plane_off;
    const uint64_t K_pad = (uint64_t)pl.k_blocks * kDenseBK;
    if (pl.four) {
      CU(ctx, cudaMemsetAsync(b->d_oth_cnt, 0, (size_t)pl.S * sizeof(uint32_t), bstream(b)));
      k_dense_prep<<<dim3((pl.W + 7u) / 8u, pl.S_pad / 256u), 256, 0, bstream(b)>>>(planes, pl.S, pl.W, pl.S_pad, b->d_xt,
                                                                                   b->d_oth_cnt, b->d_oth_list, pl.oth_cap, unit_mode);
      ++ctx->launches;
      // the "other" cells need the lists and the transposed planes only: counted on a second stream, beside the
      // X rows and the first tiles of the GEMM; joined below, before the next unit's k_dense_prep reuses the lists and
      // before anything reads the tables.  (Measured: its three CTAs per SM hold the whole register file, so
      // k_dense_x mostly runs after it and the step costs what one fused pass cost; capping it at two CTAs per SM,
      // or k_dense_x first on a smaller grid, was slower -- tools/experiments/README.md.  The nine-block form no
      // longer pays for lists and transposes it does not use: 2.01 -> 1.65 ms.)
      CU(ctx, cudaEventRecord(b->fix_fork.get(), bstream(b)));
      CU(ctx, cudaStreamWaitEvent(b->fix_stream.get(), b->fix_fork.get(), 0));
      k_other_fix<<<pl.S, kFixThreads, 0, b->fix_stream.get()>>>(b->d_xt, K_pad, pl.S, pl.S_pad, pl.rows, b->d_oth_cnt,
                                                              b->d_oth_list, pl.oth_cap, b->d_gram + pl.gram_off, unit_mode,
                                                              het ? b->d_flags + b->h_units[pl.unit].site_off : nullptr);
      ++ctx->launches;
      CU(ctx, cudaEventRecord(b->fix_join.get(), b->fix_stream.get()));
    } else {
      CU(ctx, cudaMemsetAsync(unit_mode, 1, sizeof(uint32_t), bstream(b)));  // (any non-zero value: nine blocks)
    }
    if (!het || het->H) {  // (X is the B operand; the het form of a unit without het sites has no tiles)
      const uint64_t warps = (uint64_t)pl.S * ((pl.W + 7u) / 8u);
      const unsigned xgrid = (unsigned)std::min<uint64_t>((warps + 7) / 8, (uint64_t)ctx->num_sms * 16u);
      k_dense_x<<<xgrid, 256, 0, bstream(b)>>>(planes, pl.S, pl.W, pl.S_pad, b->d_x, unit_mode, nullptr);
      ++ctx->launches;
    }
    if (het && het->H) {  // ... and the het sites' rows, packed, the A operand
      const uint64_t warps = (uint64_t)het->H_pad * ((pl.W + 7u) / 8u);
      const unsigned xgrid = (unsigned)std::min<uint64_t>((warps + 7) / 8, (uint64_t)ctx->num_sms * 16u);
      k_dense_x<<<xgrid, 256, 0, bstream(b)>>>(planes, het->H_pad, pl.W, het->H_pad, b->d_x_het, unit_mode, het_rows);
      ++ctx->launches;
    }
    const bool last = &pl == &b->dense_plans.back();
    if (last && timing) CU(ctx, cudaEventRecord(b->ev[6].get(), bstream(b)));
    for (int form = pl.four ? 0 : 1; form < 2; ++form) {  // the launch of the form the unit is not in returns at once
      const DenseTileList& L = het ? (form ? het->list9 : het->list4) : (form ? pl.list9 : pl.list4);
      if (!L.n) continue;
      DenseParams D;
      D.tiles = (het ? b->d_het_tiles : b->d_tiles) + L.off;
      D.n_tiles = L.n;
      D.k_blocks = pl.k_blocks;
      D.S_pad = pl.S_pad;
      D.gram = b->d_gram + pl.gram_off;
      D.error = reinterpret_cast<uint32_t*>(&b->d_header->pad);
      D.mode = unit_mode;
      D.nine = (uint32_t)form;
      D.a_rows = het ? het->H_pad : pl.S_pad;
      D.rows = het_rows;
      const unsigned ggrid = (unsigned)std::min<uint32_t>(L.n, (uint32_t)ctx->num_sms);
      if (L.n > L.n_whole) {
        k_zero_partial_tiles<<<L.n - L.n_whole, 256, 0, bstream(b)>>>(D.tiles + L.n_whole, L.n - L.n_whole, pl.S_pad, D.gram,
                                                                     unit_mode, (uint32_t)form, het_rows);
        ++ctx->launches;
      }
      k_gram_i8<<<ggrid, kDenseThreads, kDenseSmemBytes, bstream(b)>>>(het ? b->het_tmaps[d] : b->tmaps[d], b->tmaps[d], D);
      ++ctx->launches;
    }
    if (last && timing) CU(ctx, cudaEventRecord(b->ev[7].get(), bstream(b)));
    if (pl.four) CU(ctx, cudaStreamWaitEvent(bstream(b), b->fix_join.get(), 0));
  }
  if (timing) CU(ctx, cudaEventRecord(b->ev[5].get(), bstream(b)));
  if (b->n_tile_items) {
    // K1 + K2 of the medium units: counts + MI per 16 x 16 block of site pairs
    const unsigned tgrid = (unsigned)std::min<uint64_t>(b->n_tile_items, (uint64_t)ctx->num_sms * 3u);
    k_tile_mi<<<tgrid, kThreads, 0, bstream(b)>>>(P, b->d_tile_items, b->n_tile_items);
    ++ctx->launches;
  }
  if (b->n_gram_tiles) {
    // K1 of the medium units on the tensor cores (batched, bits expanded in the kernel), then K2 per pair
    TileGramParams T;
    T.planes = b->d_planes;
    T.site_flags = b->d_flags;
    T.mode = mode;
    T.tiles = b->d_gram_tiles;
    T.n_tiles = b->n_gram_tiles;
    T.cnt = b->d_tile_cnt;
    T.error = reinterpret_cast<uint32_t*>(&b->d_header->pad);
    const unsigned ggrid = (unsigned)std::min<uint32_t>(b->n_gram_tiles, (uint32_t)ctx->num_sms);
    k_tile_gram_ws<<<ggrid, kTwThreads, kTwSmemBytes, bstream(b)>>>(T);
    ++ctx->launches;
    const unsigned fgrid = (unsigned)std::min<uint64_t>(b->n_items, (uint64_t)ctx->num_sms * 8u);
    k_tile_finish<<<fgrid, kThreads, 0, bstream(b)>>>(P, b->d_tile_cnt);
    ++ctx->launches;
  }
  if (b->n_fast) {
    // K0 of the small units: emitted pairs per unit from the C planes alone
    CountFastParams C;
    C.items = b->d_fast_items;
    C.n_items = b->n_fast;
    C.planes = b->d_planes;
    C.site_flags = b->d_flags;
    C.ij_tab = ctx->d_ij_tab.get();
    C.min_common = min_common;
    C.mode = mode;
    C.item_cnt = b->d_item_cnt;
    C.fast_empty = b->d_fast_empty;
    const unsigned grid = (unsigned)std::min<uint64_t>(b->n_fast, (uint64_t)ctx->num_sms * 8u);
    k_count_fast<<<grid, kThreads, 0, small>>>(C);
    ++ctx->launches;
  }
  if (forked) {  // the scan needs every item's count
    CU(ctx, cudaEventRecord(b->side_ev[1].get(), small));
    CU(ctx, cudaStreamWaitEvent(bstream(b), b->side_ev[1].get(), 0));
  }
  if (b->n_items) {
    // K0 of everything else + scan: every item's place in the ordered output
    if (b->n_items > b->n_fast) {
      const unsigned cgrid = (unsigned)std::min<uint64_t>(b->n_items, (uint64_t)ctx->num_sms * 8u);
      k_count<<<cgrid, kThreads, 0, bstream(b)>>>(P);
      ++ctx->launches;
    }
    CU(ctx, cub::DeviceScan::ExclusiveSum(b->d_scan_tmp.get(), b->scan_tmp_bytes, b->d_item_cnt.get(), b->d_item_off.get(),
                                          (int)b->n_items + 1, bstream(b)));
    ++ctx->launches;
    k_scan_finish<<<1, 32, 0, bstream(b)>>>(b->d_item_off + b->n_items, b->d_header,
                                            b->own_stream ? b->h_header.get() : nullptr, b->d_unit_rec_off + b->n_units);
    ++ctx->launches;
  }
  if (timing) CU(ctx, cudaEventRecord(b->ev[2].get(), bstream(b)));
  if (forked) {
    CU(ctx, cudaEventRecord(b->side_ev[2].get(), bstream(b)));
    CU(ctx, cudaStreamWaitEvent(small, b->side_ev[2].get(), 0));
  }
  if (b->n_fast) {
    FastParams F;
    F.items = b->d_fast_items;
    F.n_items = b->n_fast;
    F.planes = b->d_planes;
    F.site_flags = b->d_flags;
    F.lntab = ctx->d_lntab.get();
    F.ln_cap = P.ln_cap;
    F.ij_tab = ctx->d_ij_tab.get();
    F.min_common = min_common;
    F.mode = mode;
    F.item_off = b->d_item_off;
    F.fast_empty = b->d_fast_empty;
    F.item_dense = b->d_item_dense;
    F.n_generic = b->d_n_generic;
    F.records = b->d_records;
    F.counts = b->d_counts;
    F.site_mean = b->d_site_mean;
    F.site_cnt = b->d_site_cnt;
    F.unit_rec_off = b->d_unit_rec_off;
    F.unit_base = b->unit_base;
    // persistent CTAs: a whole number of CTAs per SM, never more than there are items
    const unsigned grid = (unsigned)std::min<uint64_t>(b->n_fast, (uint64_t)ctx->num_sms * ctx->pairs_ctas_per_sm);
    if ((mode & (LGMI_MODE_HET_ONLY | LGMI_MODE_SKIP_NONHET)) == (LGMI_MODE_HET_ONLY | LGMI_MODE_SKIP_NONHET))
      k_pairs_fast_het<<<grid, kFastThreads, sizeof(FastSmem), small>>>(F);
    else
      k_pairs_fast<<<grid, kFastThreads, sizeof(FastSmem), small>>>(F);
    ++ctx->launches;
  }
  if (timing) CU(ctx, cudaEventRecord(b->ev[3].get(), bstream(b)));
  if (forked) CU(ctx, cudaEventRecord(b->side_ev[3].get(), small));
  if (b->n_items) {
    // everything the small-unit kernel does not take
    if (b->n_tiled_desc) {  // ordering + emission of what k_tile_mi / k_tile_finish computed
      const unsigned grid = (unsigned)std::min<uint64_t>(b->n_tiled_desc, (uint64_t)ctx->num_sms * 4u);
      k_pairs_generic<1><<<grid, kThreads, 0, bstream(b)>>>(P);
      ++ctx->launches;
    }
    if (!b->dense_plans.empty()) {  // the deep units: tables from the count matrices
      k_pairs_generic<2><<<(unsigned)std::min<uint64_t>(b->n_items, (uint64_t)ctx->num_sms * 3u), kThreads, 0, bstream(b)>>>(P);
      ++ctx->launches;
    }
  }
  if (b->n_mean_items) {  // (units of several items: none of them is k_pairs_fast's or k_pairs_generic<0>'s)
    k_site_mean_dense<<<b->n_mean_items, kMeanThreads, 0, bstream(b)>>>(b->d_units, b->d_mean_items, b->d_flags, b->d_dense,
                                                                       b->d_site_mean, b->d_site_cnt);
    ++ctx->launches;
  }
  if (forked) CU(ctx, cudaStreamWaitEvent(bstream(b), b->side_ev[3].get(), 0));
  if (b->n_items) {
    // small units k_pairs_fast handed on (a site with too many "other" reads) and pair-less units; exits at once
    // when there is nothing
    const unsigned grid = (unsigned)std::min<uint64_t>(b->n_items, (uint64_t)ctx->num_sms * 4u);
    k_pairs_generic<0><<<grid, kThreads, 0, bstream(b)>>>(P);
    ++ctx->launches;
  }
  if (timing) CU(ctx, cudaEventRecord(b->ev[1].get(), bstream(b)));
  CU(ctx, cudaGetLastError());
  b->ran = true;
  b->last_mode = mode;
  b->last_timed = timing;
  return LGMI_OK;
}

static int fill_scalars(lgmi_batch* b, lgmi_result* out) {
  lgmi_ctx* ctx = b->ctx;
  memset(out, 0, sizeof *out);
  out->n_candidates = b->n_candidates;
  // SKIP_NONHET evaluates only the candidates next to a het_snp (counted from the host flags; a caller that
  // filled the device buffers itself gets n_candidates)
  out->n_evaluated = ((b->last_mode & LGMI_MODE_SKIP_NONHET) && b->het_known) ? b->n_het_candidates : b->n_candidates;
  out->n_records = b->h_header->n_records;
  out->n_sites = b->n_sites;
  float ms = 0.f;
  const bool timing = b->last_timed;
  if (timing) {
    CU(ctx, cudaEventElapsedTime(&ms, b->ev[0].get(), b->ev[1].get()));
    out->kernel_ms = ms;
    CU(ctx, cudaEventElapsedTime(&ms, b->ev[2].get(), b->ev[3].get()));
    out->pairs_kernel_ms = ms;
    CU(ctx, cudaEventElapsedTime(&ms, b->ev[4].get(), b->ev[5].get()));
    out->dense_kernel_ms = ms;
  }
  if (!b->dense_plans.empty()) {
    // which form each deep unit took is decided on the device: read back (the stream has been synchronised)
    std::vector<uint32_t> modes(b->n_units);
    CU(ctx, cudaMemcpy(modes.data(), b->d_unit_mode, (size_t)b->n_units * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    b->dense_macs = 0;
    out->n_dense_four = 0;
    for (size_t d = 0; d < b->dense_plans.size(); ++d) {
      const DensePlan& pl = b->dense_plans[d];
      const bool nine = modes[pl.unit] != 0u;
      const uint64_t macs = nine ? b->run_macs[d].second : b->run_macs[d].first;
      b->dense_macs += macs;
      out->n_dense_four += nine ? 0u : 1u;
      if (timing && d + 1 == b->dense_plans.size()) out->gram_macs = macs;
    }
    if (timing) {
      CU(ctx, cudaEventElapsedTime(&ms, b->ev[6].get(), b->ev[7].get()));
      out->gram_kernel_ms = ms;
    }
  }
  out->n_dense_units = (uint32_t)b->dense_plans.size();
  out->dense_macs = b->dense_macs;
  if (b->h_header->pad)
    return fail(ctx, LGMI_ERR_CUDA, "k_gram_i8 / k_tile_gram_ws: a pipeline barrier timed out (tensor-core path)");
  return LGMI_OK;
}

extern "C" int lgmi_batch_sync(lgmi_batch_t* b, lgmi_result* out) {
  if (!b || !out) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = b->ctx;
  if (!b->ran) return fail(ctx, LGMI_ERR_STATE, "lgmi_batch_sync: batch has not been run");
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaMemcpyAsync(b->h_header, b->d_header, sizeof(Header), cudaMemcpyDeviceToHost, bstream(b)));
  CU(ctx, cudaStreamSynchronize(bstream(b)));
  return fill_scalars(b, out);
}

extern "C" int lgmi_batch_download(lgmi_batch_t* b, lgmi_result* out) {
  if (!b || !out) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = b->ctx;
  if (!b->ran) return fail(ctx, LGMI_ERR_STATE, "lgmi_batch_download: batch has not been run");
  CU(ctx, cudaSetDevice(ctx->device));
  // the small per-site / per-unit outputs can go while we learn the record count
  CU(ctx, cudaMemcpyAsync(b->h_header, b->d_header, sizeof(Header), cudaMemcpyDeviceToHost, bstream(b)));
  if (b->n_sites) {
    CU(ctx, cudaMemcpyAsync(b->h_site_mean, b->d_site_mean, b->n_sites * sizeof(double), cudaMemcpyDeviceToHost, bstream(b)));
    CU(ctx, cudaMemcpyAsync(b->h_site_cnt, b->d_site_cnt, b->n_sites * sizeof(uint32_t), cudaMemcpyDeviceToHost, bstream(b)));
  }
  CU(ctx, cudaMemcpyAsync(b->h_unit_rec_off, b->d_unit_rec_off, ((size_t)b->n_units + 1) * sizeof(unsigned long long),
                          cudaMemcpyDeviceToHost, bstream(b)));
  CU(ctx, cudaStreamSynchronize(bstream(b)));
  const uint64_t nrec = b->h_header->n_records;
  if (nrec > b->rec_cap) return fail(ctx, LGMI_ERR_STATE, "record count %llu exceeds capacity", (unsigned long long)nrec);
  const uint64_t cap = std::max<uint64_t>(nrec + nrec / 8, 1024);  // (the stream is idle: synchronised above)
  if (nrec > b->h_records.size()) CU(ctx, b->h_records.alloc(ctx->host_pool, cap));
  const bool want_counts = (b->last_mode & LGMI_MODE_EMIT_COUNTS) != 0u;
  if (want_counts && nrec * 9ull > b->h_counts.size()) CU(ctx, b->h_counts.alloc(ctx->host_pool, cap * 9ull));
  if (nrec) {
    CU(ctx, cudaMemcpyAsync(b->h_records, b->d_records, nrec * sizeof(lgmi_pair_rec), cudaMemcpyDeviceToHost, bstream(b)));
    if (want_counts)
      CU(ctx, cudaMemcpyAsync(b->h_counts, b->d_counts, nrec * 9ull * sizeof(uint32_t), cudaMemcpyDeviceToHost, bstream(b)));
    CU(ctx, cudaStreamSynchronize(bstream(b)));
  }
  int rc = fill_scalars(b, out);
  if (rc) return rc;
  out->records = b->h_records;
  out->counts = want_counts ? b->h_counts.get() : nullptr;
  out->site_mean = b->h_site_mean;
  out->site_cnt = b->h_site_cnt;
  out->unit_rec_off = reinterpret_cast<const uint64_t*>(b->h_unit_rec_off.get());
  return LGMI_OK;
}

extern "C" int lgmi_batch_device_ptrs(lgmi_batch_t* b, void** d_planes, void** d_site_flags, void** d_records,
                                      void** d_site_mean) {
  if (!b) return LGMI_ERR_ARG;
  if (d_planes) *d_planes = b->d_planes;
  if (d_site_flags) *d_site_flags = b->d_flags;
  if (d_records) *d_records = b->d_records;
  if (d_site_mean) *d_site_mean = b->d_site_mean;
  b->uploaded = true;  // a device-resident caller fills the buffers itself
  b->het_known = false;
  // ... so the flags may change behind the host's back: the het plans and the graphs captured with them go, and runs
  // keep the all-pairs form
  if (!b->het_plans.empty()) {
    CU(b->ctx, cudaSetDevice(b->ctx->device));
    CU(b->ctx, cudaStreamSynchronize(bstream(b)));
    b->graphs.clear();
    b->het_plans.clear();
  }
  return LGMI_OK;
}

extern "C" int lgmi_batch_algorithmic_bytes(lgmi_batch_t* b, uint64_t* bytes) {
  if (!b || !bytes) return LGMI_ERR_ARG;
  if (!b->ran) return fail(b->ctx, LGMI_ERR_STATE, "lgmi_batch_algorithmic_bytes: batch has not been run");
  uint64_t in = 0;
  for (const lgmi_unit_desc& u : b->h_units) in += 3ull * u.n_sites * ((u.n_reads + 7ull) / 8ull) + u.n_sites;
  *bytes = in + 16ull * b->h_header->n_records + 12ull * b->n_sites;
  return LGMI_OK;
}

// --------------------------------------------------------------------------- split units
// The dense MI slices of a unit's pieces, back to back, are the whole unit's dense MI array (the pieces' pairs are
// consecutive ranges of its pair order); k_site_mean_dense over that array is the unsplit run's per-site pass.
// One piece as the checks of lgmi_split_means / lgmi_split_means_ipc see it.
struct SplitPiece {
  bool present;   // (lgmi_split_means: the batch pointer is not NULL)
  bool is_piece;  // a unit with a row limit
  bool ran;
  uint32_t sites, rows;
};

// The pieces, in row order, must be the suffixes [row, S) of the unit with row limits that cover its rows; slice[p] is
// the length of piece p's MI slice.
static int split_check(lgmi_ctx* ctx, const char* fn, uint32_t S, const std::vector<SplitPiece>& pieces,
                       std::vector<uint64_t>* slice) {
  slice->assign(pieces.size(), 0);
  uint64_t row = 0, total = 0;  // piece p: the suffix [row, S) with its row limit
  for (uint32_t p = 0; p < (uint32_t)pieces.size(); ++p) {
    const SplitPiece& v = pieces[p];
    if (!v.present) return fail(ctx, LGMI_ERR_ARG, "%s: piece %u is NULL", fn, p);
    if (!v.is_piece) return fail(ctx, LGMI_ERR_ARG, "%s: piece %u is not a unit with a row limit", fn, p);
    if (!v.ran) return fail(ctx, LGMI_ERR_STATE, "%s: piece %u has not been run", fn, p);
    if (row >= S || (uint64_t)v.sites != S - row)
      return fail(ctx, LGMI_ERR_ARG, "%s: piece %u (%u sites) is not the suffix of sites [%llu, %u)", fn, p, v.sites,
                  (unsigned long long)row, S);
    (*slice)[p] = piece_pairs(v.rows, v.sites);
    total += (*slice)[p];
    row += v.rows;
  }
  const uint64_t np = (uint64_t)S * (S - (S ? 1u : 0u)) / 2;
  if (row != S || total != np)
    return fail(ctx, LGMI_ERR_ARG, "%s: the pieces cover %llu of %llu rows (%llu of %llu pairs)", fn,
                (unsigned long long)row, (unsigned long long)S, (unsigned long long)total, (unsigned long long)np);
  return LGMI_OK;
}

// Where a piece's MI slice is read from: `src` on `device`, once `after` (if any) has completed.
struct SliceSource {
  int device;
  const double* src;
  cudaEvent_t after;
};

// The slices back to back in the context's scratch, then the unsplit run's per-site pass over them (S > 0).
static int split_gather_means(lgmi_ctx* ctx, uint32_t S, const uint8_t* site_flags, const std::vector<uint64_t>& slice,
                              const std::vector<SliceSource>& from, double* mean_out, uint32_t* cnt_out) {
  const uint64_t np = (uint64_t)S * (S - 1u) / 2;
  // scratch: dense [np] | mean [S] | cnt [S] | flags [S] | unit | mean items
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const uint32_t n_items = (S + (uint32_t)kMeanSites - 1u) / (uint32_t)kMeanSites;
  const size_t o_mean = up16(np * sizeof(double)), o_cnt = o_mean + up16((size_t)S * sizeof(double));
  const size_t o_flags = o_cnt + up16((size_t)S * sizeof(uint32_t)), o_unit = o_flags + up16(S);
  const size_t o_items = o_unit + up16(sizeof(DevUnit)), bytes = o_items + n_items * sizeof(MeanItem);
  CU(ctx, cudaSetDevice(ctx->device));
  int rc = ensure_scratch(ctx, bytes);
  if (rc) return rc;
  char* scratch = ctx->d_scratch.get();
  uint64_t at = 0;
  for (size_t p = 0; p < slice.size(); ++p) {
    if (slice[p]) {
      if (from[p].after) CU(ctx, cudaStreamWaitEvent(ctx->stream, from[p].after, 0));
      CU(ctx, cudaMemcpyPeerAsync(scratch + at * sizeof(double), ctx->device, from[p].src, from[p].device,
                                  slice[p] * sizeof(double), ctx->stream));
    }
    at += slice[p];
  }
  DevUnit u{};
  u.S = S;
  u.dense_off = 0;
  u.gram_off = kNoGram;
  std::vector<MeanItem> items(n_items);
  for (uint32_t t = 0; t < n_items; ++t) items[t] = MeanItem{0u, t * (uint32_t)kMeanSites};
  CU(ctx, cudaMemcpyAsync(scratch + o_flags, site_flags, S, cudaMemcpyHostToDevice, ctx->stream));
  CU(ctx, cudaMemcpyAsync(scratch + o_unit, &u, sizeof u, cudaMemcpyHostToDevice, ctx->stream));
  CU(ctx, cudaMemcpyAsync(scratch + o_items, items.data(), n_items * sizeof(MeanItem), cudaMemcpyHostToDevice, ctx->stream));
  k_site_mean_dense<<<n_items, kMeanThreads, 0, ctx->stream>>>(
      reinterpret_cast<const DevUnit*>(scratch + o_unit), reinterpret_cast<const MeanItem*>(scratch + o_items),
      reinterpret_cast<const uint8_t*>(scratch + o_flags), reinterpret_cast<const double*>(scratch),
      reinterpret_cast<double*>(scratch + o_mean), reinterpret_cast<uint32_t*>(scratch + o_cnt));
  ++ctx->launches;
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(mean_out, scratch + o_mean, (size_t)S * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaMemcpyAsync(cnt_out, scratch + o_cnt, (size_t)S * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return LGMI_OK;
}

extern "C" int lgmi_split_means(lgmi_t* ctx, uint32_t n_sites, const uint8_t* site_flags, uint32_t n_pieces,
                                lgmi_batch_t* const* batches, const uint32_t* unit_in_batch, double* mean_out,
                                uint32_t* cnt_out) {
  if (!ctx || !batches || !unit_in_batch || !n_pieces || (n_sites && (!site_flags || !mean_out || !cnt_out)))
    return fail(ctx, LGMI_ERR_ARG, "lgmi_split_means: NULL argument");
  std::vector<SplitPiece> pieces(n_pieces);
  for (uint32_t p = 0; p < n_pieces; ++p) {
    const lgmi_batch* b = batches[p];
    const uint32_t k = unit_in_batch[p];
    const bool is_piece = b && k < b->n_units && !b->h_row_limit.empty() && b->h_row_limit[k];
    pieces[p] = SplitPiece{b != nullptr, is_piece, b && b->ran, is_piece ? b->h_units[k].n_sites : 0u,
                           is_piece ? b->h_row_limit[k] : 0u};
  }
  std::vector<uint64_t> slice;
  if (const int rc = split_check(ctx, "lgmi_split_means", n_sites, pieces, &slice)) return rc;
  if (!n_sites) return LGMI_OK;
  std::vector<SliceSource> from(n_pieces);
  for (uint32_t p = 0; p < n_pieces; ++p) {  // the pieces' kernels have finished (they may run on other devices)
    const lgmi_batch* b = batches[p];
    CU(ctx, cudaSetDevice(b->ctx->device));
    CU(ctx, cudaStreamSynchronize(bstream(b)));
    from[p] = SliceSource{b->ctx->device, b->d_dense + b->h_dense_off[unit_in_batch[p]], nullptr};
  }
  return split_gather_means(ctx, n_sites, site_flags, slice, from, mean_out, cnt_out);
}

extern "C" int lgmi_split_means_ipc(lgmi_t* ctx, uint32_t n_sites, const uint8_t* site_flags, uint32_t n_pieces,
                                    const lgmi_piece_ipc* pieces, double* mean_out, uint32_t* cnt_out) {
  static const char fn[] = "lgmi_split_means_ipc";
  if (!ctx || !pieces || !n_pieces || (n_sites && (!site_flags || !mean_out || !cnt_out)))
    return fail(ctx, LGMI_ERR_ARG, "%s: NULL argument", fn);
  std::vector<SplitPiece> view(n_pieces);
  for (uint32_t p = 0; p < n_pieces; ++p) {
    const lgmi_piece_ipc& x = pieces[p];
    view[p] = SplitPiece{true, x.row_limit != 0u, x.ran != 0u, x.n_sites, x.row_limit};
  }
  std::vector<uint64_t> slice;
  if (const int rc = split_check(ctx, fn, n_sites, view, &slice)) return rc;
  for (uint32_t p = 0; p < n_pieces; ++p)
    if (pieces[p].dense_pairs != slice[p])
      return fail(ctx, LGMI_ERR_ARG, "%s: piece %u carries %llu MI values for %llu pairs", fn, p,
                  (unsigned long long)pieces[p].dense_pairs, (unsigned long long)slice[p]);
  if (!n_sites) return LGMI_OK;
  IpcImports imports;  // closed when this returns, after the guard below has waited for the copies that read them
  struct Drain {
    lgmi_ctx* ctx;
    ~Drain() {
      cudaSetDevice(ctx->device);
      cudaStreamSynchronize(ctx->stream);
    }
  } drain{ctx};
  const int32_t self = (int32_t)getpid();
  std::vector<SliceSource> from(n_pieces);
  for (uint32_t p = 0; p < n_pieces; ++p) {
    const lgmi_piece_ipc& x = pieces[p];
    if (x.pid == self) {  // a batch of this process: read from it, as lgmi_split_means does
      lgmi_batch* b = nullptr;
      {
        std::lock_guard<std::mutex> lock(g_export_mu);
        const auto it = g_exported.find(x.batch_id);
        if (it != g_exported.end()) b = it->second;
      }
      if (!b || x.unit >= b->n_units || b->h_row_limit.empty() || b->h_row_limit[x.unit] != x.row_limit)
        return fail(ctx, LGMI_ERR_ARG, "%s: piece %u was exported by this process from a batch that no longer exists", fn, p);
      CU(ctx, cudaSetDevice(b->ctx->device));
      CU(ctx, cudaStreamSynchronize(bstream(b)));
      from[p] = SliceSource{b->ctx->device, b->d_dense + x.dense_off, nullptr};
    } else {  // another process's batch: through its handles, behind its event
      int dev = 0;
      if (const int rc = piece_device(ctx, fn, &x, &dev)) return rc;
      void* base = nullptr;
      cudaEvent_t ev = nullptr;
      CU(ctx, imports.open_mem(x.dense_mem, dev, &base));
      CU(ctx, imports.open_event(x.event, &ev));
      from[p] = SliceSource{dev, static_cast<const double*>(base) + x.dense_off, ev};
    }
  }
  return split_gather_means(ctx, n_sites, site_flags, slice, from, mean_out, cnt_out);
}

// --------------------------------------------------------------------------- pipelined step
// The batch cut into consecutive groups of units, each a batch of its own on its own
// stream: H2D of group k+1, kernels of group k and D2H of group k-1 overlap (two copy
// engines + the SMs).  Outputs are merged into one set of pinned host arrays in the
// reference's row order, identical to upload + run + download of the whole batch.

// the input and output form of a step, decoded from its mode once (pipeline_begin)
struct StepForm {
  bool split = false;        // MI and (i, j) in arrays of their own (LGMI_MODE_SPLIT_RECORDS or COMPACT_OUTPUT)
  bool compact = false;      // LGMI_MODE_COMPACT_OUTPUT: split rows with 2-byte (i, j) where possible, no site_cnt
  bool ij16 = false;         // ... and possible: no unit has more than 256 sites
  bool tight = false;        // LGMI_MODE_TIGHT_INPUT
  bool want_counts = false;  // LGMI_MODE_EMIT_COUNTS
  uint32_t run_mode = 0;     // the mode without the bits that are a matter of the copies, not of the kernels
  size_t ij_bytes() const { return ij16 ? sizeof(uint16_t) : sizeof(uint32_t); }
};

static StepForm step_form(uint32_t mode, uint32_t max_sites) {
  StepForm f;
  f.compact = (mode & LGMI_MODE_COMPACT_OUTPUT) != 0u;
  f.split = (mode & LGMI_MODE_SPLIT_RECORDS) != 0u || f.compact;
  f.ij16 = f.compact && max_sites <= 256u;
  f.tight = (mode & LGMI_MODE_TIGHT_INPUT) != 0u;
  f.want_counts = (mode & LGMI_MODE_EMIT_COUNTS) != 0u;
  f.run_mode = mode & ~(LGMI_MODE_SPLIT_RECORDS | LGMI_MODE_COMPACT_OUTPUT | LGMI_MODE_TIGHT_INPUT);
  return f;
}

struct lgmi_pipeline {
  explicit lgmi_pipeline(lgmi_ctx* c) : ctx(c) {}
  ~lgmi_pipeline();
  lgmi_ctx* const ctx;
  uint32_t n_units = 0;
  uint64_t plane_words = 0, n_sites = 0, n_candidates = 0;
  struct Chunk {
    uint32_t unit0 = 0, n_units = 0;
    uint64_t plane0 = 0, site0 = 0;
    Event done;     // the group's kernels have finished
    Event landed;   // the group's input is in device memory
    PoolBuf<uint32_t> d_packed;   // two-plane input staging (lgmi_pipeline_step_packed)
    PoolBuf<unsigned long long> d_tight_off;  // LGMI_MODE_TIGHT_INPUT: first word of each unit, relative to the group
    uint64_t tight0 = 0, tight_words = 0;       // the group's slice of the tight two-plane input
    PoolBuf<double> d_rec_mi;     // split output (LGMI_MODE_SPLIT_RECORDS)
    PoolBuf<uint32_t> d_rec_ij;
    uint64_t base = 0;              // first row of the group in the merged output of the current step
    // declared last, so destroyed first: ~lgmi_batch synchronises the group's stream, whose kernels read and write
    // the buffers above
    std::unique_ptr<lgmi_batch> b;
  };
  std::vector<Chunk> chunks;
  // one stream per copy direction: copies of a direction run one after the other anyway, and a stream that
  // copies both ways can land on one engine with another stream's uploads in front of its downloads
  Stream h2d, d2h;
  PoolBuf<lgmi_pair_rec> h_records;
  PoolBuf<uint32_t> h_counts;     // 9 per row
  PoolBuf<double> h_rec_mi;
  PoolBuf<uint32_t> h_rec_ij;   // (2-byte entries under LGMI_MODE_COMPACT_OUTPUT when every unit has <= 256 sites)
  uint32_t max_sites = 0;
  PoolBuf<double> h_site_mean;
  PoolBuf<uint32_t> h_site_cnt;
  PoolBuf<unsigned long long> h_unit_rec_off;
  // a step between lgmi_pipeline_begin* and lgmi_pipeline_finish
  bool in_flight = false;   // begun, not finished
  bool collected = false;   // ... and its downloads queued (lgmi_pipeline_collect)
  StepForm form;
  uint64_t pend_rows = 0;
};

lgmi_pipeline::~lgmi_pipeline() {
  cudaSetDevice(ctx->device);
  // copies into the pinned output arrays and out of the groups' buffers must have landed before they go back to the
  // cache
  if (d2h) cudaStreamSynchronize(d2h.get());
  if (h2d) cudaStreamSynchronize(h2d.get());
}

extern "C" void lgmi_pipeline_destroy(lgmi_pipeline_t* p) { delete p; }

extern "C" int lgmi_pipeline_create(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units, uint64_t plane_words,
                                    uint64_t n_sites, uint32_t n_chunks, lgmi_pipeline_t** out) {
  if (!ctx || !out || (!units && n_units)) return fail(ctx, LGMI_ERR_ARG, "lgmi_pipeline_create: NULL argument");
  *out = nullptr;
  PipelinePlan plan;
  std::string err;
  if (const int rc = plan_pipeline(units, n_units, n_chunks, &plan, &err)) return fail(ctx, rc, "%s", err.c_str());
  CU(ctx, cudaSetDevice(ctx->device));

  // every failure from here on releases what the pipeline holds so far
  std::unique_ptr<lgmi_pipeline> p(new (std::nothrow) lgmi_pipeline(ctx));
  if (!p) return fail(ctx, LGMI_ERR_NOMEM, "lgmi_pipeline_create: out of host memory");
  p->n_units = n_units;
  p->plane_words = plane_words;
  p->n_sites = n_sites;
  p->n_candidates = plan.n_candidates;
  p->max_sites = plan.max_sites;
  for (const GroupPlan& g : plan.groups) {
    p->chunks.emplace_back();
    lgmi_pipeline::Chunk& c = p->chunks.back();
    lgmi_batch* b = nullptr;
    if (const int rc = lgmi_batch_create(ctx, g.units.data(), g.n_units, g.plane_words, g.n_sites, &b)) return rc;
    c.b.reset(b);
    c.b->unit_base = g.unit0;  // records carry the unit's index in the whole batch
    c.unit0 = g.unit0;
    c.n_units = g.n_units;
    c.plane0 = g.plane0;
    c.site0 = g.site0;
    c.tight0 = g.tight0;
    c.tight_words = g.tight_words;
    if (g.n_units) {
      const size_t bytes = g.tight_off.size() * sizeof(unsigned long long);
      CU(ctx, c.d_tight_off.alloc(ctx->dev_pool, g.tight_off.size()));
      CU(ctx, cudaMemcpy(c.d_tight_off, g.tight_off.data(), bytes, cudaMemcpyHostToDevice));
    }
    CU(ctx, create(c.b->own_stream));
    CU(ctx, create(c.done, cudaEventDisableTiming));
    CU(ctx, create(c.landed, cudaEventDisableTiming));
  }
  CU(ctx, create(p->h2d));
  CU(ctx, create(p->d2h));
  CU(ctx, p->h_site_mean.alloc(ctx->host_pool, std::max<uint64_t>(1, n_sites)));
  CU(ctx, p->h_site_cnt.alloc(ctx->host_pool, std::max<uint64_t>(1, n_sites)));
  CU(ctx, p->h_unit_rec_off.alloc(ctx->host_pool, (size_t)n_units + 1));
  *out = p.release();
  return LGMI_OK;
}

// grows a pinned output array of rows of `width` elements to `need` rows, keeping the `keep` rows that have already
// landed in it
template <class T>
static int grow_pinned(lgmi_pipeline* p, PoolBuf<T>& buf, uint64_t need, uint64_t keep, size_t width = 1) {
  if (need * width <= buf.size()) return LGMI_OK;
  lgmi_ctx* ctx = p->ctx;
  CU(ctx, cudaStreamSynchronize(p->d2h.get()));  // copies into the old array
  const uint64_t rows = std::max<uint64_t>(need + need / 4, 1024);
  CU(ctx, buf.alloc(ctx->host_pool, rows * width, keep * width));
  return LGMI_OK;
}

// First half of a step: everything that does not depend on a count -- the uploads, the kernels and the row split of
// every group -- is queued, group after group, and the call returns.
static int pipeline_begin(lgmi_pipeline* p, const uint32_t* planes, bool packed, const uint8_t* site_flags, int min_common,
                          uint32_t mode) {
  if (!p) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = p->ctx;
  if (p->in_flight) return fail(ctx, LGMI_ERR_STATE, "lgmi_pipeline_begin: the previous step has not been finished");
  if ((!planes && p->plane_words) || (!site_flags && p->n_sites))
    return fail(ctx, LGMI_ERR_ARG, "lgmi_pipeline_step: NULL input");
  CU(ctx, cudaSetDevice(ctx->device));
  const StepForm f = step_form(mode, p->max_sites);
  if (f.tight && !packed) return fail(ctx, LGMI_ERR_ARG, "LGMI_MODE_TIGHT_INPUT is a form of the two-plane input (lgmi_pipeline_step_packed)");
  p->form = f;
  for (lgmi_pipeline::Chunk& c : p->chunks) {
    lgmi_batch* b = c.b.get();
    cudaStream_t st = b->own_stream.get();
    // input on the upload stream, in group order; the group's own stream picks up when it has landed
    if (b->n_sites)
      CU(ctx, cudaMemcpyAsync(b->d_flags, site_flags + c.site0, b->n_sites, cudaMemcpyHostToDevice, p->h2d.get()));
    const uint64_t words2 = b->plane_words / 3u * 2u;           // staging sized for the padded form: either fits
    const uint64_t words_in = f.tight ? c.tight_words : words2;
    if (packed) {  // two planes per site over PCIe, expanded on the device
      if (!c.d_packed && words2) CU(ctx, c.d_packed.alloc(ctx->dev_pool, words2));
      if (words_in)
        CU(ctx, cudaMemcpyAsync(c.d_packed, planes + (f.tight ? c.tight0 : c.plane0 / 3u * 2u), words_in * sizeof(uint32_t),
                                cudaMemcpyHostToDevice, p->h2d.get()));
    } else if (b->plane_words) {
      CU(ctx, cudaMemcpyAsync(b->d_planes, planes + c.plane0, b->plane_words * sizeof(uint32_t), cudaMemcpyHostToDevice,
                              p->h2d.get()));
    }
    CU(ctx, cudaEventRecord(c.landed.get(), p->h2d.get()));
    CU(ctx, cudaStreamWaitEvent(st, c.landed.get(), 0));
    if (packed && words2) {
      k_unpack2<<<std::min<uint32_t>(b->n_units, (uint32_t)ctx->num_sms * 16u), 256, 0, st>>>(
          b->d_units, b->n_units, c.d_packed, b->d_planes, f.tight ? c.d_tight_off.get() : nullptr);
      ++ctx->launches;
    }
    b->uploaded = true;
    if (f.run_mode & LGMI_MODE_SKIP_NONHET) {
      b->n_het_candidates = b->n_sites ? het_candidates(b->h_units, b->h_row_limit, site_flags + c.site0) : 0;
      b->het_known = true;
      if (const int rc = plan_het(b, site_flags + c.site0, st)) return rc;
    }
    if (const int rc = lgmi_batch_run(b, min_common, f.run_mode)) return rc;
    if (f.split) {
      if (!c.d_rec_mi) {
        CU(ctx, c.d_rec_mi.alloc(ctx->dev_pool, b->rec_cap));
        CU(ctx, c.d_rec_ij.alloc(ctx->dev_pool, b->rec_cap));
      }
      k_split_records<<<(unsigned)ctx->num_sms * 8u, 256, 0, st>>>(
          b->d_header, b->d_records, c.d_rec_mi, c.d_rec_ij, f.ij16 ? reinterpret_cast<uint16_t*>(c.d_rec_ij.get()) : nullptr);
      ++ctx->launches;
    }
    CU(ctx, cudaEventRecord(c.done.get(), st));  // the group's record count is in its (host-resident) header by then
  }
  p->in_flight = true;
  return LGMI_OK;
}

// Second half: waits for the groups in order and copies their rows to the host; a group's place in the merged
// arrays is known once the groups before it have been counted.
static int pipeline_collect(lgmi_pipeline* p) {
  if (!p) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = p->ctx;
  if (!p->in_flight) return fail(ctx, LGMI_ERR_STATE, "lgmi_pipeline_collect / finish: no step has been begun");
  if (p->collected) return LGMI_OK;
  CU(ctx, cudaSetDevice(ctx->device));
  const StepForm& f = p->form;
  const size_t ij_bytes = f.ij_bytes();
  static const bool debug = getenv("LGMI_PIPE_DEBUG") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
  std::vector<double> t_done, t_issue;
  uint64_t base = 0;
  for (lgmi_pipeline::Chunk& c : p->chunks) {
    lgmi_batch* b = c.b.get();
    CU(ctx, cudaEventSynchronize(c.done.get()));
    if (debug) t_done.push_back(since());
    const uint64_t nrec = b->h_header->n_records;
    if (nrec > b->rec_cap) return fail(ctx, LGMI_ERR_STATE, "record count %llu exceeds capacity", (unsigned long long)nrec);
    int rc = LGMI_OK;
    if (f.split) {
      rc = grow_pinned(p, p->h_rec_mi, base + nrec, base);
      if (!rc) rc = grow_pinned(p, p->h_rec_ij, base + nrec, base);
    } else {
      rc = grow_pinned(p, p->h_records, base + nrec, base);
    }
    if (!rc && f.want_counts) rc = grow_pinned(p, p->h_counts, base + nrec, base, 9);
    if (rc) return rc;
    cudaStream_t st = p->d2h.get();  // the group is complete (event above): nothing here waits on a kernel
    if (nrec) {
      if (f.split) {
        CU(ctx, cudaMemcpyAsync(p->h_rec_mi + base, c.d_rec_mi, nrec * sizeof(double), cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaMemcpyAsync(reinterpret_cast<char*>(p->h_rec_ij.get()) + base * ij_bytes, c.d_rec_ij,
                                nrec * ij_bytes, cudaMemcpyDeviceToHost, st));
      } else {
        CU(ctx, cudaMemcpyAsync(p->h_records + base, b->d_records, nrec * sizeof(lgmi_pair_rec), cudaMemcpyDeviceToHost, st));
      }
      if (f.want_counts)
        CU(ctx, cudaMemcpyAsync(p->h_counts + base * 9ull, b->d_counts, nrec * 9ull * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
    CU(ctx, cudaMemcpyAsync(b->h_unit_rec_off, b->d_unit_rec_off, ((size_t)b->n_units + 1) * sizeof(unsigned long long),
                            cudaMemcpyDeviceToHost, st));
    if (b->n_sites) {
      CU(ctx, cudaMemcpyAsync(p->h_site_mean + c.site0, b->d_site_mean, b->n_sites * sizeof(double), cudaMemcpyDeviceToHost, st));
      if (!f.compact)
        CU(ctx, cudaMemcpyAsync(p->h_site_cnt + c.site0, b->d_site_cnt, b->n_sites * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
    c.base = base;
    base += nrec;
    if (debug) t_issue.push_back(since());
  }
  p->pend_rows = base;
  p->collected = true;
  if (debug) {
    fprintf(stderr, "[lgmi pipeline] (ms since lgmi_pipeline_collect) groups counted at");
    for (double t : t_done) fprintf(stderr, " %.3f", t);
    fprintf(stderr, "; D2H issued by");
    for (double t : t_issue) fprintf(stderr, " %.3f", t);
    fprintf(stderr, " ms\n");
  }
  return LGMI_OK;
}

// Third part: the copies have landed; per-unit row offsets of the merged arrays, scalars.
static int pipeline_finish(lgmi_pipeline* p, lgmi_result* out) {
  if (!p || !out) return LGMI_ERR_ARG;
  lgmi_ctx* ctx = p->ctx;
  int rc_collect = pipeline_collect(p);
  if (rc_collect) {
    p->in_flight = p->collected = false;
    return rc_collect;
  }
  p->in_flight = p->collected = false;
  const StepForm& f = p->form;
  const uint64_t base = p->pend_rows;
  CU(ctx, cudaStreamSynchronize(p->d2h.get()));
  for (lgmi_pipeline::Chunk& c : p->chunks) {
    for (uint32_t u = 0; u < c.n_units; ++u) p->h_unit_rec_off[c.unit0 + u] = c.base + c.b->h_unit_rec_off[u];
  }
  p->h_unit_rec_off[p->n_units] = base;
  memset(out, 0, sizeof *out);
  out->n_candidates = p->n_candidates;
  out->n_evaluated = 0;
  out->n_records = base;
  out->records = f.split ? nullptr : p->h_records.get();
  out->rec_mi = f.split ? p->h_rec_mi.get() : nullptr;
  out->rec_ij = f.split ? p->h_rec_ij.get() : nullptr;
  out->rec_ij_bytes = f.split ? (uint32_t)f.ij_bytes() : 0u;
  out->counts = f.want_counts ? p->h_counts.get() : nullptr;
  out->n_sites = p->n_sites;
  out->site_mean = p->h_site_mean;
  out->site_cnt = f.compact ? nullptr : p->h_site_cnt.get();
  out->unit_rec_off = reinterpret_cast<const uint64_t*>(p->h_unit_rec_off.get());
  for (lgmi_pipeline::Chunk& c : p->chunks) {
    lgmi_result r;
    int rc = fill_scalars(c.b.get(), &r);
    if (rc) return rc;
    out->n_evaluated += r.n_evaluated;
    out->kernel_ms += r.kernel_ms;
    out->pairs_kernel_ms += r.pairs_kernel_ms;
    out->dense_kernel_ms += r.dense_kernel_ms;
    out->n_dense_units += r.n_dense_units;
    out->dense_macs += r.dense_macs;
  }
  return LGMI_OK;
}

extern "C" int lgmi_pipeline_step(lgmi_pipeline_t* p, const uint32_t* planes, const uint8_t* site_flags, int min_common,
                                  uint32_t mode, lgmi_result* out) {
  if (!p || !out) return LGMI_ERR_ARG;
  int rc = pipeline_begin(p, planes, false, site_flags, min_common, mode);
  return rc ? rc : pipeline_finish(p, out);
}

extern "C" int lgmi_pipeline_step_packed(lgmi_pipeline_t* p, const uint32_t* planes2, const uint8_t* site_flags,
                                         int min_common, uint32_t mode, lgmi_result* out) {
  if (!p || !out) return LGMI_ERR_ARG;
  int rc = pipeline_begin(p, planes2, true, site_flags, min_common, mode);
  return rc ? rc : pipeline_finish(p, out);
}

extern "C" int lgmi_pipeline_begin(lgmi_pipeline_t* p, const uint32_t* planes, const uint8_t* site_flags, int min_common,
                                   uint32_t mode) {
  return pipeline_begin(p, planes, false, site_flags, min_common, mode);
}

extern "C" int lgmi_pipeline_begin_packed(lgmi_pipeline_t* p, const uint32_t* planes2, const uint8_t* site_flags,
                                          int min_common, uint32_t mode) {
  return pipeline_begin(p, planes2, true, site_flags, min_common, mode);
}

extern "C" int lgmi_pipeline_collect(lgmi_pipeline_t* p) { return pipeline_collect(p); }

extern "C" int lgmi_pipeline_finish(lgmi_pipeline_t* p, lgmi_result* out) { return pipeline_finish(p, out); }

// --------------------------------------------------------------------------- one-shot
extern "C" int lgmi_submit(lgmi_t* ctx, const lgmi_unit_desc* units, uint32_t n_units, const uint32_t* planes,
                           uint64_t plane_words, const uint8_t* site_flags, uint64_t n_sites, int min_common,
                           uint32_t mode) {
  if (!ctx) return LGMI_ERR_ARG;
  lgmi_batch_destroy(ctx->oneshot);
  lgmi_batch* b = nullptr;
  int rc = lgmi_batch_create(ctx, units, n_units, plane_words, n_sites, &b);
  if (rc) return rc;
  ctx->oneshot = b;
  rc = lgmi_batch_upload(b, planes, site_flags);
  if (rc) return rc;
  return lgmi_batch_run(b, min_common, mode);
}

extern "C" int lgmi_wait(lgmi_t* ctx, lgmi_result* out) {
  if (!ctx || !out) return LGMI_ERR_ARG;
  if (!ctx->oneshot) return fail(ctx, LGMI_ERR_STATE, "lgmi_wait: nothing submitted");
  return lgmi_batch_download(ctx->oneshot, out);
}

// --------------------------------------------------------------------------- mean of rows
extern "C" int lgmi_site_mean_csr(lgmi_t* ctx, const uint64_t* offsets, const double* values, uint64_t n_sites,
                                  double* mean_out) {
  if (!ctx || !offsets || !mean_out) return fail(ctx, LGMI_ERR_ARG, "lgmi_site_mean_csr: NULL argument");
  if (n_sites == 0) return LGMI_OK;
  CU(ctx, cudaSetDevice(ctx->device));
  const uint64_t nval = offsets[n_sites];
  if (nval && !values) return fail(ctx, LGMI_ERR_ARG, "lgmi_site_mean_csr: NULL values");
  const size_t off_bytes = (n_sites + 1) * sizeof(uint64_t);
  const size_t val_bytes = std::max<uint64_t>(1, nval) * sizeof(double);
  const size_t out_bytes = n_sites * sizeof(double);
  int rc = ensure_scratch(ctx, off_bytes + val_bytes + out_bytes + 64);
  if (rc) return rc;
  char* p = ctx->d_scratch.get();
  unsigned long long* d_off = reinterpret_cast<unsigned long long*>(p);
  double* d_val = reinterpret_cast<double*>(p + off_bytes);
  double* d_out = reinterpret_cast<double*>(p + off_bytes + val_bytes);
  CU(ctx, cudaMemcpyAsync(d_off, offsets, off_bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (nval) CU(ctx, cudaMemcpyAsync(d_val, values, nval * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  k_site_mean_csr<<<(unsigned)((n_sites + 127) / 128), 128, 0, ctx->stream>>>(d_off, d_val, n_sites, d_out);
  ++ctx->launches;
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(mean_out, d_out, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return LGMI_OK;
}

// --------------------------------------------------------------------------- ecdf
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

extern "C" int lgmi_ecdf(lgmi_t* ctx, const double* mean, const uint8_t* site_flags, uint64_t n, double threshold,
                         double* mip, uint8_t* call) {
  if (!ctx || (n && (!mean || !site_flags || !mip))) return fail(ctx, LGMI_ERR_ARG, "lgmi_ecdf: NULL argument");
  if (n == 0) return LGMI_OK;
  if (n > 0x7fffffffull) return fail(ctx, LGMI_ERR_UNSUPPORTED, "lgmi_ecdf: more than 2^31-1 sites");
  CU(ctx, cudaSetDevice(ctx->device));
  size_t sort_bytes = 0;
  CU(ctx, cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, (const double*)nullptr, (double*)nullptr, (int)n, 0, 64,
                                        ctx->stream));
  const size_t a_mean = 0;
  const size_t a_keys = align_up(a_mean + n * 8, 256);
  const size_t a_sorted = align_up(a_keys + n * 8, 256);
  const size_t a_mip = align_up(a_sorted + n * 8, 256);
  const size_t a_flags = align_up(a_mip + n * 8, 256);
  const size_t a_call = align_up(a_flags + n, 256);
  const size_t a_cnt = align_up(a_call + n, 256);
  const size_t a_tmp = align_up(a_cnt + 8, 256);
  int rc = ensure_scratch(ctx, a_tmp + sort_bytes);
  if (rc) return rc;
  char* p = ctx->d_scratch.get();
  double* d_mean = reinterpret_cast<double*>(p + a_mean);
  double* d_keys = reinterpret_cast<double*>(p + a_keys);
  double* d_sorted = reinterpret_cast<double*>(p + a_sorted);
  double* d_mip = reinterpret_cast<double*>(p + a_mip);
  uint8_t* d_flags = reinterpret_cast<uint8_t*>(p + a_flags);
  uint8_t* d_call = reinterpret_cast<uint8_t*>(p + a_call);
  unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(p + a_cnt);
  CU(ctx, cudaMemcpyAsync(d_mean, mean, n * 8, cudaMemcpyHostToDevice, ctx->stream));
  CU(ctx, cudaMemcpyAsync(d_flags, site_flags, n, cudaMemcpyHostToDevice, ctx->stream));
  CU(ctx, cudaMemsetAsync(d_cnt, 0, 8, ctx->stream));
  const unsigned grid = (unsigned)((n + 255) / 256);
  k_ecdf_keys<<<grid, 256, 0, ctx->stream>>>(d_mean, d_flags, n, d_keys, d_cnt);
  ++ctx->launches;
  CU(ctx, cub::DeviceRadixSort::SortKeys(p + a_tmp, sort_bytes, d_keys, d_sorted, (int)n, 0, 64, ctx->stream));
  ++ctx->launches;
  k_ecdf_mip<<<grid, 256, 0, ctx->stream>>>(d_mean, d_flags, n, d_sorted, d_cnt, threshold, d_mip, d_call);
  ++ctx->launches;
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(mip, d_mip, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (call) CU(ctx, cudaMemcpyAsync(call, d_call, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return LGMI_OK;
}

// sorts x on the device (NaNs canonicalised: last, as numpy.sort leaves them); d_sorted / d_nan are in the scratch
static int ecdf_sort(lgmi_ctx* ctx, const double* x, uint64_t n, size_t extra_bytes, char** scratch, double** d_sorted,
                     unsigned long long** d_nan) {
  size_t sort_bytes = 0;
  CU(ctx, cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, (const double*)nullptr, (double*)nullptr, (int)n, 0, 64,
                                        ctx->stream));
  const size_t a_x = 0;
  const size_t a_sorted = align_up(a_x + n * 8, 256);
  const size_t a_nan = align_up(a_sorted + n * 8, 256);
  const size_t a_tmp = align_up(a_nan + 8, 256);
  const size_t a_extra = align_up(a_tmp + sort_bytes, 256);
  int rc = ensure_scratch(ctx, a_extra + extra_bytes);
  if (rc) return rc;
  char* p = ctx->d_scratch.get();
  double* d_x = reinterpret_cast<double*>(p + a_x);
  *d_sorted = reinterpret_cast<double*>(p + a_sorted);
  *d_nan = reinterpret_cast<unsigned long long*>(p + a_nan);
  *scratch = p + a_extra;
  CU(ctx, cudaMemcpyAsync(d_x, x, n * 8, cudaMemcpyHostToDevice, ctx->stream));
  CU(ctx, cudaMemsetAsync(*d_nan, 0, 8, ctx->stream));
  k_canon_nan<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_x, n, *d_nan);
  ++ctx->launches;
  CU(ctx, cub::DeviceRadixSort::SortKeys(p + a_tmp, sort_bytes, d_x, *d_sorted, (int)n, 0, 64, ctx->stream));
  ++ctx->launches;
  return LGMI_OK;
}

extern "C" int lgmi_ecdf_eval(lgmi_t* ctx, const double* x, uint64_t n, const double* samples, uint64_t m,
                              double* out) {
  if (!ctx || (n && !x) || (m && (!samples || !out))) return fail(ctx, LGMI_ERR_ARG, "lgmi_ecdf_eval: NULL argument");
  if (n == 0) return fail(ctx, LGMI_ERR_ARG, "lgmi_ecdf_eval: empty x (the reference divides by len(x))");
  if (m == 0) return LGMI_OK;
  if (n > 0x7fffffffull) return fail(ctx, LGMI_ERR_UNSUPPORTED, "lgmi_ecdf_eval: more than 2^31-1 values");
  CU(ctx, cudaSetDevice(ctx->device));
  char* extra = nullptr;
  double* d_sorted = nullptr;
  unsigned long long* d_nan = nullptr;
  const size_t a_o = align_up(m * 8, 256);
  int rc = ecdf_sort(ctx, x, n, a_o + m * 8, &extra, &d_sorted, &d_nan);
  if (rc) return rc;
  double* d_s = reinterpret_cast<double*>(extra);
  double* d_o = reinterpret_cast<double*>(extra + a_o);
  CU(ctx, cudaMemcpyAsync(d_s, samples, m * 8, cudaMemcpyHostToDevice, ctx->stream));
  k_ecdf_eval<<<(unsigned)((m + 255) / 256), 256, 0, ctx->stream>>>(d_sorted, n, d_nan, d_s, m, d_o);
  ++ctx->launches;
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(out, d_o, m * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return LGMI_OK;
}

extern "C" int lgmi_ecdf_table(lgmi_t* ctx, const double* x, uint64_t n, double* sorted_out, double* y_out) {
  if (!ctx || (n && (!x || !sorted_out)) || !y_out) return fail(ctx, LGMI_ERR_ARG, "lgmi_ecdf_table: NULL argument");
  if (n == 0) return fail(ctx, LGMI_ERR_ARG, "lgmi_ecdf_table: empty x (the reference divides by len(x))");
  if (n > 0x7fffffffull) return fail(ctx, LGMI_ERR_UNSUPPORTED, "lgmi_ecdf_table: more than 2^31-1 values");
  CU(ctx, cudaSetDevice(ctx->device));
  char* extra = nullptr;
  double* d_sorted = nullptr;
  unsigned long long* d_nan = nullptr;
  int rc = ecdf_sort(ctx, x, n, (n + 1) * 8, &extra, &d_sorted, &d_nan);
  if (rc) return rc;
  double* d_y = reinterpret_cast<double*>(extra);
  k_ecdf_ordinates<<<(unsigned)((n + 256) / 256), 256, 0, ctx->stream>>>(n, d_y);
  ++ctx->launches;
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(sorted_out, d_sorted, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaMemcpyAsync(y_out, d_y, (n + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return LGMI_OK;
}

// --------------------------------------------------------------------------- site x splice-site MI
// Host side of lgmi_site_splice_mi: the triples grouped into columns (one per distinct (site, splice) of the
// triples, ascending splice id within a site), each column's triples, and the work items of k_ss_count.
namespace {
struct SsPlan {
  std::vector<uint32_t> slot_splice, slot_tri_off, tri_order;
  std::vector<uint8_t> tri_allele;
  std::vector<SsItem> items;
  uint64_t max_n = 1;  // entries of the deepest requested site
};
}  // namespace

static void ss_plan(uint32_t n_sites, const uint64_t* entry_off, uint64_t n_tri, const uint32_t* tri_site,
                    const uint32_t* tri_allele, const uint32_t* tri_splice, SsPlan& P) {
  P.tri_order.resize(n_tri);
  for (uint64_t t = 0; t < n_tri; ++t) P.tri_order[t] = (uint32_t)t;
  std::sort(P.tri_order.begin(), P.tri_order.end(), [&](uint32_t a, uint32_t b) {
    if (tri_site[a] != tri_site[b]) return tri_site[a] < tri_site[b];
    if (tri_splice[a] != tri_splice[b]) return tri_splice[a] < tri_splice[b];
    return a < b;
  });
  P.tri_allele.resize(n_tri);
  for (uint64_t t = 0; t < n_tri; ++t) P.tri_allele[t] = (uint8_t)tri_allele[t];
  for (uint64_t k = 0; k < n_tri;) {  // one site's triples: [k, end)
    const uint32_t s = tri_site[P.tri_order[k]];
    const uint32_t slot0 = (uint32_t)P.slot_splice.size();
    uint32_t rows = 0;
    uint64_t end = k;
    for (; end < n_tri && tri_site[P.tri_order[end]] == s; ++end) {
      const uint32_t t = P.tri_order[end];
      rows = std::max(rows, tri_allele[t] + 1u);
      if (end == k || tri_splice[t] != P.slot_splice.back()) {
        P.slot_splice.push_back(tri_splice[t]);
        P.slot_tri_off.push_back((uint32_t)end);
      }
    }
    const uint32_t n_slots = (uint32_t)P.slot_splice.size() - slot0;
    const uint64_t lo = entry_off[s], n = entry_off[s + 1] - lo;
    P.max_n = std::max(P.max_n, n);
    for (uint32_t c = 0; c < n_slots; c += kSsTileCols)
      for (uint64_t e = 0; e < n; e += kSsChunk)
        P.items.push_back(SsItem{lo + e, (uint32_t)std::min<uint64_t>(kSsChunk, n - e), s, slot0 + c,
                                 std::min(kSsTileCols, n_slots - c), rows, 0u});
    k = end;
  }
  P.slot_tri_off.push_back((uint32_t)n_tri);
}

static uint32_t bits_for(uint64_t n) {  // bits of the largest value below n (at least 1)
  uint32_t b = 1;
  while (b < 64 && (n - 1) >> b) ++b;
  return b;
}

extern "C" int lgmi_site_splice_mi(lgmi_t* ctx, uint32_t n_sites, const uint64_t* entry_off,
                                   const uint32_t* entry_read, const uint32_t* entry_allele, uint32_t n_reads,
                                   const uint64_t* splice_off, const uint32_t* splice_id, uint64_t n_triples,
                                   const uint32_t* tri_site, const uint32_t* tri_allele, const uint32_t* tri_splice,
                                   double* mi_out, uint32_t* table_out) {
  static const char* me = "lgmi_site_splice_mi";
  if (!ctx) return LGMI_ERR_ARG;
  if (n_triples && (!tri_site || !tri_allele || !tri_splice || !mi_out))
    return fail(ctx, LGMI_ERR_ARG, "%s: NULL triple or output array", me);
  if (!entry_off || (n_reads && !splice_off)) return fail(ctx, LGMI_ERR_ARG, "%s: NULL offsets", me);
  if (n_triples > 0xffffffffull) return fail(ctx, LGMI_ERR_UNSUPPORTED, "%s: more than 2^32-1 triples", me);
  // the site entry CSR
  if (entry_off[0] != 0) return fail(ctx, LGMI_ERR_ARG, "%s: entry_off[0] = %llu, not 0", me,
                                     (unsigned long long)entry_off[0]);
  for (uint32_t s = 0; s < n_sites; ++s)
    if (entry_off[s + 1] < entry_off[s]) return fail(ctx, LGMI_ERR_ARG, "%s: entry_off decreases at site %u", me, s);
  const uint64_t n_entries = entry_off[n_sites];
  if (n_entries && (!entry_read || !entry_allele)) return fail(ctx, LGMI_ERR_ARG, "%s: NULL entry arrays", me);
  if (n_entries > 0x7fffffffull)
    return fail(ctx, LGMI_ERR_UNSUPPORTED, "%s: %llu entries, more than the radix sort takes (2^31-1)", me,
                (unsigned long long)n_entries);
  for (uint32_t s = 0; s < n_sites; ++s)
    for (uint64_t p = entry_off[s]; p < entry_off[s + 1]; ++p) {
      if (entry_read[p] >= n_reads)
        return fail(ctx, LGMI_ERR_ARG, "%s: entry %llu names read %u of %u", me, (unsigned long long)p, entry_read[p],
                    n_reads);
      if (entry_allele[p] >= kSsMaxAlleles)
        return fail(ctx, LGMI_ERR_UNSUPPORTED,
                    "%s: site %u has allele index %u; at most 64 distinct alleles per site (the count pass keeps "
                    "one bit per allele)", me, s, entry_allele[p]);
    }
  // the read splice CSR: ids ascending, each once
  const uint64_t n_splice = n_reads ? splice_off[n_reads] : 0;
  if (n_reads && splice_off[0] != 0) return fail(ctx, LGMI_ERR_ARG, "%s: splice_off[0] is not 0", me);
  if (n_splice && !splice_id) return fail(ctx, LGMI_ERR_ARG, "%s: NULL splice_id", me);
  for (uint32_t r = 0; r < n_reads; ++r) {
    if (splice_off[r + 1] < splice_off[r]) return fail(ctx, LGMI_ERR_ARG, "%s: splice_off decreases at read %u", me, r);
    for (uint64_t k = splice_off[r] + 1; k < splice_off[r + 1]; ++k)
      if (splice_id[k] <= splice_id[k - 1])
        return fail(ctx, LGMI_ERR_ARG, "%s: splice ids of read %u are not ascending and unique", me, r);
  }
  for (uint64_t t = 0; t < n_triples; ++t) {
    if (tri_site[t] >= n_sites)
      return fail(ctx, LGMI_ERR_ARG, "%s: triple %llu names site %u of %u", me, (unsigned long long)t, tri_site[t],
                  n_sites);
    if (tri_allele[t] >= kSsMaxAlleles)
      return fail(ctx, LGMI_ERR_UNSUPPORTED, "%s: triple %llu asks for allele index %u; at most 64 per site", me,
                  (unsigned long long)t, tri_allele[t]);
  }
  if (n_triples == 0) return LGMI_OK;
  CU(ctx, cudaSetDevice(ctx->device));
  SsPlan P;
  ss_plan(n_sites, entry_off, n_triples, tri_site, tri_allele, tri_splice, P);
  if (const int rc = ensure_lntab(ctx, P.max_n)) return rc;

  const uint32_t read_bits = bits_for(std::max<uint32_t>(n_reads, 1u));
  const uint32_t key_bits = read_bits + bits_for(std::max<uint32_t>(n_sites, 1u));
  size_t sort_bytes = 0;
  CU(ctx, cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned long long*)nullptr,
                                          (unsigned long long*)nullptr, (const uint8_t*)nullptr, (uint8_t*)nullptr,
                                          (int)n_entries, 0, (int)key_bits, ctx->stream));
  MemPool& pool = ctx->dev_pool;
  const size_t ne = std::max<uint64_t>(1, n_entries), ns = std::max<uint64_t>(1, n_splice);
  PoolBuf<unsigned long long> d_entry_off, d_keys, d_keys_sorted, d_splice_off;
  PoolBuf<uint32_t> d_read, d_allele, d_splice_id, d_slot_splice, d_slot_tri_off, d_tri_order, d_tri_site, d_counts,
      d_table;
  PoolBuf<uint8_t> d_vals, d_vals_sorted, d_tri_allele;
  PoolBuf<char> d_sort_tmp;
  PoolBuf<SsItem> d_items;
  PoolBuf<double> d_mi;
  CU(ctx, d_entry_off.alloc(pool, (size_t)n_sites + 1));
  CU(ctx, d_keys.alloc(pool, ne));
  CU(ctx, d_keys_sorted.alloc(pool, ne));
  CU(ctx, d_splice_off.alloc(pool, (size_t)n_reads + 1));
  CU(ctx, d_read.alloc(pool, ne));
  CU(ctx, d_allele.alloc(pool, ne));
  CU(ctx, d_splice_id.alloc(pool, ns));
  CU(ctx, d_slot_splice.alloc(pool, P.slot_splice.size()));
  CU(ctx, d_slot_tri_off.alloc(pool, P.slot_tri_off.size()));
  CU(ctx, d_tri_order.alloc(pool, n_triples));
  CU(ctx, d_tri_site.alloc(pool, n_triples));
  CU(ctx, d_tri_allele.alloc(pool, n_triples));
  CU(ctx, d_counts.alloc(pool, 3 * n_triples));
  CU(ctx, d_vals.alloc(pool, ne));
  CU(ctx, d_vals_sorted.alloc(pool, ne));
  CU(ctx, d_sort_tmp.alloc(pool, std::max<size_t>(sort_bytes, 16)));
  CU(ctx, d_items.alloc(pool, std::max<size_t>(1, P.items.size())));
  CU(ctx, d_mi.alloc(pool, n_triples));
  if (table_out) CU(ctx, d_table.alloc(pool, 4 * n_triples));

  cudaStream_t st = ctx->stream;
  auto up = [&](void* dst, const void* src, size_t bytes) {
    return bytes ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
  };
  CU(ctx, up(d_entry_off, entry_off, ((size_t)n_sites + 1) * 8));
  CU(ctx, up(d_read, entry_read, n_entries * 4));
  CU(ctx, up(d_allele, entry_allele, n_entries * 4));
  if (n_reads) CU(ctx, up(d_splice_off, splice_off, ((size_t)n_reads + 1) * 8));
  CU(ctx, up(d_splice_id, splice_id, n_splice * 4));
  CU(ctx, up(d_slot_splice, P.slot_splice.data(), P.slot_splice.size() * 4));
  CU(ctx, up(d_slot_tri_off, P.slot_tri_off.data(), P.slot_tri_off.size() * 4));
  CU(ctx, up(d_tri_order, P.tri_order.data(), n_triples * 4));
  CU(ctx, up(d_tri_site, tri_site, n_triples * 4));
  CU(ctx, up(d_tri_allele, P.tri_allele.data(), n_triples));
  CU(ctx, up(d_items, P.items.data(), P.items.size() * sizeof(SsItem)));
  CU(ctx, cudaMemsetAsync(d_counts, 0, 3 * n_triples * 4, st));
  if (n_entries) {
    const unsigned grid = (unsigned)std::min<uint64_t>((n_entries + 255) / 256, 65536);
    k_ss_keys<<<grid, 256, 0, st>>>(d_entry_off, n_sites, d_read, d_allele, n_entries, read_bits, d_keys, d_vals);
    ++ctx->launches;
    CU(ctx, cub::DeviceRadixSort::SortPairs(d_sort_tmp.get(), sort_bytes, d_keys.get(), d_keys_sorted.get(),
                                            d_vals.get(), d_vals_sorted.get(), (int)n_entries, 0, (int)key_bits, st));
    ++ctx->launches;
  }
  if (!P.items.empty()) {
    k_ss_count<<<(unsigned)P.items.size(), kSsThreads, 0, st>>>(
        d_items, d_keys_sorted, d_vals_sorted, d_entry_off, (1ull << read_bits) - 1ull, d_splice_off, d_splice_id,
        d_slot_splice, d_slot_tri_off, d_tri_order, d_tri_allele, d_counts);
    ++ctx->launches;
  }
  k_ss_mi<<<(unsigned)((n_triples + 255) / 256), 256, 0, st>>>(d_counts, d_tri_site, d_entry_off, n_triples,
                                                                ctx->d_lntab.get(), d_mi, table_out ? d_table.get()
                                                                                                    : nullptr);
  ++ctx->launches;
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaMemcpyAsync(mi_out, d_mi, n_triples * 8, cudaMemcpyDeviceToHost, st));
  if (table_out) CU(ctx, cudaMemcpyAsync(table_out, d_table, n_triples * 16, cudaMemcpyDeviceToHost, st));
  CU(ctx, cudaStreamSynchronize(st));
  return LGMI_OK;
}

extern "C" int lgmi_device_count(void) {
  int n = 0;
  return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

// --------------------------------------------------------------------------- partitioning
extern "C" uint64_t lgmi_unit_cost(uint32_t n_sites, uint32_t n_reads) {
  if (n_sites < 2) return 0;
  return (uint64_t)n_sites * (n_sites - 1) / 2 * ((n_reads + 63ull) / 64ull);
}

extern "C" int lgmi_partition_lpt(const uint64_t* cost, uint32_t n_units, uint32_t n_bins, uint32_t* bin_of,
                                  uint64_t* bin_load) {
  if ((!cost && n_units) || !bin_of || n_bins == 0) return LGMI_ERR_ARG;
  std::vector<uint32_t> order(n_units);
  for (uint32_t k = 0; k < n_units; ++k) order[k] = k;
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return cost[a] > cost[b]; });
  typedef std::pair<uint64_t, uint32_t> Bin;  // (load, bin); min-heap, ties -> lower bin index
  std::priority_queue<Bin, std::vector<Bin>, std::greater<Bin>> heap;
  for (uint32_t k = 0; k < n_bins; ++k) heap.push(Bin(0, k));
  std::vector<uint64_t> load(n_bins, 0);
  for (uint32_t k : order) {
    Bin top = heap.top();
    heap.pop();
    bin_of[k] = top.second;
    top.first += cost[k];
    load[top.second] = top.first;
    heap.push(top);
  }
  if (bin_load) memcpy(bin_load, load.data(), n_bins * sizeof(uint64_t));
  return LGMI_OK;
}

#include "lgmi_host.inl"
