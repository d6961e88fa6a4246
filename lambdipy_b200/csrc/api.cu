// api.cu -- C ABI (include/lambdipy_b200.h) over the plan / scan / compaction kernels, the
// chunked host pipeline (pinned H2D -> kernels -> D2H on rotating streams) and the in-place tree
// walker that stands where the reference runs `find ... -name "*.so" | xargs strip`
// (/root/reference/lambdipy/project_build.py:260).
#include "lb2_common.cuh"
#include "../../include/lambdipy_b200.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cctype>
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <climits>
#include <dirent.h>
#include <regex.h>
#include <fcntl.h>
#include <spawn.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <sys/wait.h>
#include <unistd.h>

extern char **environ;

using namespace lb2;

static thread_local std::string g_create_error;

// Device workspace of one batch in flight.
struct Workspace {
  uint64_t *d_in_off = nullptr, *d_in_size = nullptr, *d_out_size = nullptr, *d_out_off = nullptr;
  int32_t *d_status = nullptr;
  uint8_t *d_scratch = nullptr;
  Tile *d_tiles = nullptr;
  BatchCounters *d_ctr = nullptr;
  UpRange *d_ranges = nullptr, *h_ranges = nullptr;  // host-buffer pipeline: input ranges to upload (pinned copy)
  BigExt *d_big = nullptr;      // extents whose tiles the scan launch's extra CTAs write
  uint32_t cap_big = 0;
  uint32_t cap_ranges = 0;
  uint64_t *h_stage = nullptr;  // pinned: 2*(n+1) offsets/sizes up
  uint8_t *h_res = nullptr;     // pinned: out_off[n+1] | out_size[n] | status[n] down (queued behind the kernels)
  BatchCounters *h_ctr = nullptr;
  cudaEvent_t done = nullptr;   // recorded behind the last result copy: collect waits on this, not on the stream
  uint32_t cap_files = 0;
  uint64_t cap_tiles = 0;
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  // last batch
  uint32_t n_files = 0;
  cudaStream_t stream = nullptr;
  bool in_flight = false;
};

struct TreeEngine;
struct lb2_ctx {
  int device = 0;
  int numa_node = -1;          // NUMA node of the GPU's PCIe root (-1: unknown / single node)
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  Workspace ws;               // lb2_strip_device_async / lb2_plan_device / even chunks of lb2_strip_device_chunked
  Workspace ws2;              // odd chunks (chunk k+1 is queued before chunk k is collected)
  int async_head = 0, async_count = 0;  // lb2_strip_device_async: up to two batches in flight (ws, ws2), collected in order
  std::string err;
  int compact_ctas_per_sm = 4;
  int use_tma = 1;             // bulk-copy engine kernel (0.97 of copy peak) ; LB2_COMPACT_TMA=0 selects the LSU kernel (0.90)
  // host pipeline slots
  struct Slot {
    Workspace ws;
    cudaStream_t stream = nullptr;
    uint8_t *d_in = nullptr, *d_out = nullptr;
    uint64_t cap_in = 0, cap_out = 0;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr}, ev_planned = nullptr;
  } slot[3];
  TreeEngine *tree = nullptr;  // lb2_strip_tree: pinned slot ring, I/O worker streams, HBM batch buffers
  // lb2_deflate_device / lb2_gzip_segments: per-chunk output slots, per-CTA match scratch, concatenation tile list,
  // and the window buffers of lb2_gzip_segments -- grown on demand and kept for the context's life, like the tree
  // engine (whose pinned slot ring and worker streams upload the windows)
  struct DeflateWs {
    uint8_t *slots = nullptr;
    uint32_t *size_crc = nullptr, *h_size_crc = nullptr;  // out_size[cap] | chunk_crc[cap], device and pinned
    uint32_t *scratch = nullptr;
    uint16_t *dists = nullptr;
    Tile *tiles = nullptr;
    BatchCounters *ctr = nullptr;
    uint64_t *out_off = nullptr;
    unsigned long long *phase = nullptr;  // DEFLATE_PHASES cycle counters
    uint64_t cap_chunks = 0, cap_tiles = 0;
    int grid = 0;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    uint8_t *d_win[2] = {nullptr, nullptr}, *d_out = nullptr, *h_out = nullptr;  // window (+ 32 KiB history) x2, output
    uint64_t cap_win[2] = {0, 0}, cap_out = 0, cap_h_out = 0;
  } gz;
};
struct TreeEngine;
static void tree_engine_free(TreeEngine *e);

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                               \
      return LB2_E_CUDA;                                                                           \
    }                                                                                              \
  } while (0)

// Pinned host arenas are placed on the NUMA node the GPU hangs off: the compaction kernel of the zero-copy
// host path reads and writes them over PCIe at ~50 GB/s per direction, and a remote-socket arena puts that
// traffic on the inter-socket link (round 1: 40 GB/s per direction at 1 GPU, half of that per GPU at 8).
// The policy is set only around the allocation (MPOL_PREFERRED: falls back to other nodes when full).
static int gpu_numa_node(int device) {
  char bus[64] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return -1; }
  for (char *c = bus; *c; c++) *c = (char)tolower(*c);
  std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
  FILE *f = fopen(path.c_str(), "r");
  if (!f) return -1;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
}
struct NumaPreferred {
  bool active = false;
  explicit NumaPreferred(int node) {
    const char *v = getenv("LB2_NUMA");
    if (node < 0 || node >= 1024 || (v && atoi(v) == 0)) return;
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    active = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, sizeof(mask) * 8 + 1) == 0;
  }
  ~NumaPreferred() { if (active) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0); }
};

// Control data of a batch (offsets up; counters, sizes, status, upload ranges down) normally rides on small
// cudaMemcpyAsync calls.  In the host-buffer DMA pipeline those would queue on the copy engines behind 100 MB
// transfers of the neighbouring chunks and stall the host for milliseconds, so there the kernels read the
// offsets through the mapping of the pinned staging buffer and this kernel stores the results into mapped
// pinned memory with ordinary SM stores: no copy engine involved.
__global__ void lb2_zero_ctr_kernel(BatchCounters *ctr) {
  if (threadIdx.x < sizeof(BatchCounters) / 4) reinterpret_cast<uint32_t *>(ctr)[threadIdx.x] = 0;
}
__global__ void __launch_bounds__(256) lb2_publish_kernel(const BatchCounters *ctr, const uint64_t *out_off, const uint64_t *out_size,
                                                          const int32_t *status, const UpRange *ranges, uint32_t n, uint32_t range_cap,
                                                          BatchCounters *h_ctr, uint64_t *h_off, uint64_t *h_size, int32_t *h_status, UpRange *h_ranges) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  if (t < sizeof(BatchCounters) / 4) reinterpret_cast<uint32_t *>(h_ctr)[t] = reinterpret_cast<const uint32_t *>(ctr)[t];
  for (uint32_t i = t; i <= n; i += stride) h_off[i] = out_off[i];
  for (uint32_t i = t; i < n; i += stride) { h_size[i] = out_size[i]; h_status[i] = status[i]; }
  if (ranges) {
    const uint32_t nr = ctr->n_ranges < range_cap ? ctr->n_ranges : range_cap;
    for (uint32_t i = t; i < nr; i += stride) h_ranges[i] = ranges[i];
  }
}

static double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static void ws_free(Workspace &w) {
  cudaFree(w.d_in_off); cudaFree(w.d_in_size); cudaFree(w.d_out_size); cudaFree(w.d_out_off); cudaFree(w.d_status);
  cudaFree(w.d_scratch); cudaFree(w.d_tiles); cudaFree(w.d_ctr);
  if (w.h_stage) cudaFreeHost(w.h_stage);
  if (w.h_res) cudaFreeHost(w.h_res);
  if (w.h_ctr) cudaFreeHost(w.h_ctr);
  cudaFree(w.d_ranges);
  cudaFree(w.d_big);
  if (w.h_ranges) cudaFreeHost(w.h_ranges);
  for (auto &e : w.ev) if (e) cudaEventDestroy(e);
  if (w.done) cudaEventDestroy(w.done);
  w = Workspace();
}

static int ws_reserve(lb2_ctx *ctx, Workspace &w, uint32_t n_files, uint64_t n_tiles) {
  if (!w.d_ctr) {
    CK(cudaMalloc(&w.d_ctr, sizeof(BatchCounters)));
    CK(cudaHostAlloc(&w.h_ctr, sizeof(BatchCounters) + 64, cudaHostAllocMapped));
    for (auto &e : w.ev) CK(cudaEventCreate(&e));
    CK(cudaEventCreateWithFlags(&w.done, cudaEventDisableTiming));
  }
  if (n_files > w.cap_files) {
    uint32_t cap = std::max<uint32_t>(n_files, 256u);
    cap = std::max<uint32_t>(cap, w.cap_files + w.cap_files / 2);
    cudaFree(w.d_in_off); cudaFree(w.d_in_size); cudaFree(w.d_out_size); cudaFree(w.d_out_off); cudaFree(w.d_status); cudaFree(w.d_scratch);
    if (w.h_stage) cudaFreeHost(w.h_stage);
    if (w.h_res) cudaFreeHost(w.h_res);
    w.h_stage = nullptr; w.h_res = nullptr;
    w.d_in_off = w.d_in_size = w.d_out_size = w.d_out_off = nullptr; w.d_status = nullptr; w.d_scratch = nullptr;
    w.cap_files = 0;
    CK(cudaMalloc(&w.d_in_off, (cap + 1) * sizeof(uint64_t)));
    CK(cudaMalloc(&w.d_in_size, (cap + 1) * sizeof(uint64_t)));
    CK(cudaMalloc(&w.d_out_size, (cap + 1) * sizeof(uint64_t)));
    CK(cudaMalloc(&w.d_out_off, (cap + 1) * sizeof(uint64_t)));
    CK(cudaMalloc(&w.d_status, (cap + 1) * sizeof(int32_t)));
    CK(cudaMalloc(&w.d_scratch, (uint64_t)cap * SCR_STRIDE));
    CK(cudaHostAlloc(&w.h_stage, (2ull * cap + 2) * sizeof(uint64_t), cudaHostAllocMapped));
    CK(cudaHostAlloc(&w.h_res, (2ull * cap + 2) * sizeof(uint64_t) + (cap + 1ull) * sizeof(int32_t), cudaHostAllocMapped));
    w.cap_files = cap;
  }
  if (n_tiles > w.cap_tiles) {
    uint64_t cap = std::max<uint64_t>(n_tiles, w.cap_tiles + w.cap_tiles / 2);
    cudaFree(w.d_tiles);
    w.d_tiles = nullptr;
    w.cap_tiles = 0;
    CK(cudaMalloc(&w.d_tiles, cap * sizeof(Tile)));
    w.cap_tiles = cap;
  }
  return LB2_OK;
}

// Upper bound on the tiles a batch can emit: an extent of l bytes yields at most l / TILE + 2 tiles, a
// file has at most MAX_EXT extents, and re-laid-out files may grow (LOAD alignment padding) -- 1 GB of
// growth per batch is allowed for before the plan kernel reports overflow.
static uint64_t tile_bound(const uint64_t *sizes, uint32_t n) {
  uint64_t t = 65536;
  for (uint32_t i = 0; i < n; i++) t += sizes[i] / TILE_BYTES + 2 * MAX_EXT + 16;
  return t;
}

// Enqueue plan -> scan -> (compact) for one batch on `s`.  h_off/h_sizes are host arrays.
static int enqueue_batch(lb2_ctx *ctx, Workspace &w, const uint8_t *d_in, const uint64_t *h_off, const uint64_t *h_sizes,
                         uint32_t n, uint8_t *d_out, uint64_t out_cap, uint32_t flags, cudaStream_t s, bool compact,
                         bool export_ranges = false, bool via_mapping = false) {
  for (uint32_t i = 0; i < n; i++)
    if (h_off[i] & 15) { ctx->err = "input offsets must be multiples of 16"; return LB2_E_ARG; }
  // sizes -> staging (pinned), upload
  std::vector<uint64_t> tmp;
  if (w.in_flight) { ctx->err = "previous batch on this workspace not collected"; return LB2_E_STATE; }
  uint64_t *st_off = nullptr, *st_size = nullptr;
  {
    // need sizes before reserve to bound tiles
    tmp.resize(n);
    for (uint32_t i = 0; i < n; i++) tmp[i] = h_sizes ? h_sizes[i] : (h_off[i + 1] - h_off[i]);
  }
  int rc = ws_reserve(ctx, w, n, tile_bound(tmp.data(), n));
  if (rc) return rc;
  st_off = w.h_stage;
  st_size = w.h_stage + (w.cap_files + 1);
  memcpy(st_off, h_off, (size_t)n * sizeof(uint64_t));
  memcpy(st_size, tmp.data(), (size_t)n * sizeof(uint64_t));
  const uint64_t *k_in_off = w.d_in_off, *k_in_size = w.d_in_size;
  if (via_mapping) {  // no copy-engine traffic for control data (see lb2_publish_kernel)
    void *alias = nullptr;
    CK(cudaHostGetDevicePointer(&alias, w.h_stage, 0));
    k_in_off = static_cast<const uint64_t *>(alias);
    k_in_size = k_in_off + (w.cap_files + 1);
    lb2_zero_ctr_kernel<<<1, 64, 0, s>>>(w.d_ctr);
  } else {
    CK(cudaMemcpyAsync(w.d_in_off, st_off, (size_t)n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(w.d_in_size, st_size, (size_t)n * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(w.d_ctr, 0, sizeof(BatchCounters), s));
  }
  CK(cudaEventRecord(w.ev[0], s));
  if (export_ranges && w.cap_ranges < 8u * n + 4096u) {
    cudaFree(w.d_ranges);
    if (w.h_ranges) cudaFreeHost(w.h_ranges);
    w.d_ranges = nullptr; w.h_ranges = nullptr; w.cap_ranges = 0;
    const uint32_t cap = 8u * std::max<uint32_t>(n, w.cap_files) + 4096u;
    CK(cudaMalloc(&w.d_ranges, (size_t)cap * sizeof(UpRange)));
    CK(cudaHostAlloc(&w.h_ranges, (size_t)cap * sizeof(UpRange), cudaHostAllocMapped));
    w.cap_ranges = cap;
  }
  PlanArgs pa;
  pa.in = d_in; pa.in_off = k_in_off; pa.in_size = k_in_size; pa.n_files = n; pa.flags = flags;
  pa.scratch = w.d_scratch; pa.out_size = w.d_out_size; pa.status = w.d_status;
  pa.tiles = w.d_tiles; pa.tile_cap = w.cap_tiles; pa.ctr = w.d_ctr;
  pa.up_ranges = export_ranges ? w.d_ranges : nullptr; pa.up_cap = export_ranges ? w.cap_ranges : 0;
  if (w.cap_big < 8u * n + 4096u) {
    cudaFree(w.d_big);
    w.d_big = nullptr; w.cap_big = 0;
    const uint32_t cap = 8u * std::max<uint32_t>(n, w.cap_files) + 4096u;
    CK(cudaMalloc(&w.d_big, (size_t)cap * sizeof(BigExt)));
    w.cap_big = cap;
  }
  pa.big = w.d_big; pa.big_cap = w.cap_big;
  launch_plan(pa, s);
  launch_scan(w.d_out_size, w.d_out_off, n, compact ? out_cap : ~0ull, w.d_ctr, w.d_big, w.cap_big, w.d_tiles, ctx->sm_count * 2, s);
  CK(cudaEventRecord(w.ev[1], s));
  if (compact) {
    CompactArgs ca;
    ca.tiles = w.d_tiles; ca.ctr = w.d_ctr; ca.out_off = w.d_out_off; ca.out = d_out;
    ca.rebase_lo = ca.rebase_len = ca.rebase_delta = 0;
    if (ctx->use_tma) launch_compact_tma(ca, ctx->sm_count, s);
    else launch_compact(ca, ctx->sm_count * ctx->compact_ctas_per_sm, s);
  }
  CK(cudaEventRecord(w.ev[2], s));
  // results ride behind the kernels into pinned staging; collect_batch only waits for `done`, so a
  // caller may queue the next batch (other workspace, same stream) before collecting this one
  {
    uint64_t *r_off = reinterpret_cast<uint64_t *>(w.h_res), *r_size = r_off + (w.cap_files + 1);
    int32_t *r_status = reinterpret_cast<int32_t *>(r_size + (w.cap_files + 1));
    if (via_mapping) {
      void *a_ctr = nullptr, *a_res = nullptr, *a_rng = nullptr;
      CK(cudaHostGetDevicePointer(&a_ctr, w.h_ctr, 0));
      CK(cudaHostGetDevicePointer(&a_res, w.h_res, 0));
      if (export_ranges) CK(cudaHostGetDevicePointer(&a_rng, w.h_ranges, 0));
      uint64_t *m_off = static_cast<uint64_t *>(a_res), *m_size = m_off + (w.cap_files + 1);
      int32_t *m_status = reinterpret_cast<int32_t *>(m_size + (w.cap_files + 1));
      lb2_publish_kernel<<<std::max(1u, std::min(32u, (n + 255u) / 256u)), 256, 0, s>>>(
          w.d_ctr, w.d_out_off, w.d_out_size, w.d_status, export_ranges ? w.d_ranges : nullptr, n, w.cap_ranges,
          static_cast<BatchCounters *>(a_ctr), m_off, m_size, m_status, static_cast<UpRange *>(a_rng));
    } else {
      CK(cudaMemcpyAsync(w.h_ctr, w.d_ctr, sizeof(BatchCounters), cudaMemcpyDeviceToHost, s));
      if (export_ranges) CK(cudaMemcpyAsync(w.h_ranges, w.d_ranges, (size_t)std::min<uint32_t>(w.cap_ranges, 8u * n + 4096u) * sizeof(UpRange), cudaMemcpyDeviceToHost, s));
      CK(cudaMemcpyAsync(r_off, w.d_out_off, (size_t)(n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
      if (n) {
        CK(cudaMemcpyAsync(r_size, w.d_out_size, (size_t)n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(r_status, w.d_status, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
      }
    }
    CK(cudaEventRecord(w.done, s));
  }
  CK(cudaGetLastError());
  w.n_files = n;
  w.stream = s;
  w.in_flight = true;
  return LB2_OK;
}

static int collect_batch(lb2_ctx *ctx, Workspace &w, uint64_t *h_out_off, uint64_t *h_out_sizes, int32_t *h_status,
                         lb2_stats *stats) {
  if (!w.in_flight) { ctx->err = "no batch in flight"; return LB2_E_STATE; }
  const uint32_t n = w.n_files;
  CK(cudaEventSynchronize(w.done));
  w.in_flight = false;
  const uint64_t *r_off = reinterpret_cast<const uint64_t *>(w.h_res), *r_size = r_off + (w.cap_files + 1);
  const int32_t *r_status = reinterpret_cast<const int32_t *>(r_size + (w.cap_files + 1));
  if (h_out_off) memcpy(h_out_off, r_off, (size_t)(n + 1) * sizeof(uint64_t));
  if (h_out_sizes && n) memcpy(h_out_sizes, r_size, (size_t)n * sizeof(uint64_t));
  if (h_status && n) memcpy(h_status, r_status, (size_t)n * sizeof(int32_t));
  if (stats) {
    const BatchCounters &c = *w.h_ctr;
    memset(stats, 0, sizeof(*stats));
    stats->n_files = n; stats->n_ok = c.n_ok; stats->n_unsupported = c.n_unsupported; stats->overflow = c.overflow;
    stats->in_bytes = c.in_bytes; stats->out_bytes = c.out_bytes; stats->copy_bytes = c.copy_bytes;
    stats->header_bytes = c.header_bytes; stats->n_tiles = c.n_tiles; stats->out_bytes_needed = r_off[n];
    cudaEventElapsedTime(&stats->plan_ms, w.ev[0], w.ev[1]);
    cudaEventElapsedTime(&stats->compact_ms, w.ev[1], w.ev[2]);
  }
  if (w.h_ctr->overflow) { ctx->err = "output arena (or tile buffer) too small for this batch"; return LB2_E_CAPACITY; }
  return LB2_OK;
}

// ============================================================================ C ABI
extern "C" {

const char *lb2_version(void) { return "lambdipy_b200 0.1 (sm_100a; GNU strip 2.42 semantics)"; }

int lb2_ctx_create(int device, lb2_ctx **out) {
  if (!out) return LB2_E_ARG;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return LB2_E_NODEVICE;
  }
  if (device < 0 || device >= count) { g_create_error = "device index out of range"; return LB2_E_ARG; }
  lb2_ctx *ctx = new lb2_ctx();
  ctx->device = device;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_create_error = std::string("cuda init: ") + cudaGetErrorString(e);
    delete ctx;
    return LB2_E_CUDA;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  ctx->sm_count = prop.multiProcessorCount;
  ctx->numa_node = gpu_numa_node(device);
  if (prop.major < 10) {
    g_create_error = "this library is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return LB2_E_NODEVICE;
  }
  if (const char *v = getenv("LB2_COMPACT_CTAS_PER_SM")) ctx->compact_ctas_per_sm = std::max(1, atoi(v));
  if (const char *v = getenv("LB2_COMPACT_TMA")) ctx->use_tma = atoi(v);
  *out = ctx;
  return LB2_OK;
}

void lb2_ctx_destroy(lb2_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  ws_free(ctx->ws);
  ws_free(ctx->ws2);
  for (auto &sl : ctx->slot) {
    ws_free(sl.ws);
    cudaFree(sl.d_in); cudaFree(sl.d_out);
    if (sl.stream) cudaStreamDestroy(sl.stream);
    for (auto &e : sl.ev_h2d) if (e) cudaEventDestroy(e);
    for (auto &e : sl.ev_d2h) if (e) cudaEventDestroy(e);
    if (sl.ev_planned) cudaEventDestroy(sl.ev_planned);
  }
  tree_engine_free(ctx->tree);
  cudaFree(ctx->gz.slots); cudaFree(ctx->gz.size_crc); cudaFreeHost(ctx->gz.h_size_crc); cudaFree(ctx->gz.scratch);
  cudaFree(ctx->gz.dists); cudaFree(ctx->gz.tiles); cudaFree(ctx->gz.ctr); cudaFree(ctx->gz.out_off);
  cudaFree(ctx->gz.phase); cudaFree(ctx->gz.d_win[0]); cudaFree(ctx->gz.d_win[1]); cudaFree(ctx->gz.d_out);
  cudaFreeHost(ctx->gz.h_out);
  for (auto &e : ctx->gz.ev) if (e) cudaEventDestroy(e);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *lb2_last_error(const lb2_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }
int lb2_sm_count(const lb2_ctx *ctx) { return ctx ? ctx->sm_count : 0; }

void *lb2_dev_alloc(lb2_ctx *ctx, uint64_t bytes) {
  void *p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes ? bytes : 256);
  if (e != cudaSuccess) { if (ctx) ctx->err = std::string("cudaMalloc: ") + cudaGetErrorString(e); return nullptr; }
  return p;
}
void lb2_dev_free(lb2_ctx *, void *p) { if (p) cudaFree(p); }
void *lb2_pinned_alloc(lb2_ctx *ctx, uint64_t bytes) {
  void *p = nullptr;
  NumaPreferred near_gpu(ctx ? ctx->numa_node : -1);
  cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 256, cudaHostAllocMapped | cudaHostAllocPortable);
  if (e != cudaSuccess) { if (ctx) ctx->err = std::string("cudaHostAlloc: ") + cudaGetErrorString(e); return nullptr; }
  return p;
}
void lb2_pinned_free(lb2_ctx *, void *p) { if (p) cudaFreeHost(p); }
int lb2_memcpy_h2d(lb2_ctx *ctx, void *d, const void *h, uint64_t n) { CK(cudaMemcpy(d, h, n, cudaMemcpyHostToDevice)); return LB2_OK; }
int lb2_memcpy_d2h(lb2_ctx *ctx, void *h, const void *d, uint64_t n) { CK(cudaMemcpy(h, d, n, cudaMemcpyDeviceToHost)); return LB2_OK; }
int lb2_memset_d(lb2_ctx *ctx, void *d, int v, uint64_t n) { CK(cudaMemset(d, v, n)); return LB2_OK; }

int lb2_strip_device_async(lb2_ctx *ctx, const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_sizes,
                           uint32_t n_files, void *d_out, uint64_t out_capacity, uint32_t flags, void *stream) {
  if (!ctx || !d_in || !h_in_off || !d_out) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  if (ctx->async_count >= 2) { ctx->err = "two batches already in flight: collect one with lb2_batch_results first"; return LB2_E_STATE; }
  cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
  Workspace &w = ((ctx->async_head + ctx->async_count) & 1) ? ctx->ws2 : ctx->ws;
  int rc = enqueue_batch(ctx, w, static_cast<const uint8_t *>(d_in), h_in_off, h_in_sizes, n_files,
                         static_cast<uint8_t *>(d_out), out_capacity, flags, s, true);
  if (rc == LB2_OK) ctx->async_count++;
  return rc;
}

int lb2_batch_results(lb2_ctx *ctx, uint64_t *h_out_off, uint64_t *h_out_sizes, int32_t *h_status, lb2_stats *stats) {
  if (!ctx) return LB2_E_ARG;
  if (ctx->async_count == 0) { ctx->err = "no batch in flight"; return LB2_E_STATE; }
  Workspace &w = (ctx->async_head & 1) ? ctx->ws2 : ctx->ws;
  ctx->async_head ^= 1;
  ctx->async_count--;
  return collect_batch(ctx, w, h_out_off, h_out_sizes, h_status, stats);
}

int lb2_plan_device(lb2_ctx *ctx, const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_sizes, uint32_t n_files,
                    uint32_t flags, uint64_t *h_out_sizes, int32_t *h_status, lb2_stats *stats) {
  if (!ctx || !d_in || !h_in_off) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  if (ctx->async_count) { ctx->err = "batches of lb2_strip_device_async still in flight"; return LB2_E_STATE; }
  int rc = enqueue_batch(ctx, ctx->ws, static_cast<const uint8_t *>(d_in), h_in_off, h_in_sizes, n_files, nullptr, 0, flags,
                         ctx->stream, false);
  if (rc) return rc;
  return collect_batch(ctx, ctx->ws, nullptr, h_out_sizes, h_status, stats);
}

// ---------------------------------------------------------------------------- shards larger than HBM
// A shard whose input plus output does not fit next to each other in HBM (BASELINE config 4 on one GPU:
// 115 GB in + 67 GB out; SURVEY D7) keeps its INPUT resident and streams the OUTPUT through a ring of two
// slots: chunk k (consecutive files, <= max_chunk_bytes of arena span) is stripped into slot k % 2 while
// the consumer still holds chunk k-1.  Chunk k+1 is queued on the stream before chunk k is collected, so
// the GPU never waits for the host between chunks.
int lb2_strip_device_chunked(lb2_ctx *ctx, const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_sizes, uint32_t n_files,
                             void *d_out_ring, uint64_t slot_capacity, uint64_t max_chunk_bytes, uint32_t flags, void *stream,
                             lb2_chunk_fn on_chunk, void *user, uint64_t *h_out_sizes, int32_t *h_status, lb2_stats *total_out) {
  if (!ctx || !d_in || !h_in_off || !d_out_ring || !slot_capacity) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  if (ctx->async_count) { ctx->err = "batches of lb2_strip_device_async still in flight"; return LB2_E_STATE; }
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
  if (!max_chunk_bytes || max_chunk_bytes > slot_capacity) max_chunk_bytes = slot_capacity;
  struct Chunk { uint32_t f0, f1; };
  std::vector<Chunk> chunks;
  for (uint32_t f = 0; f < n_files;) {
    uint32_t g = f + 1;
    while (g < n_files && h_in_off[g + 1] - h_in_off[f] <= max_chunk_bytes) g++;
    chunks.push_back({f, g});
    f = g;
  }
  lb2_stats total;
  memset(&total, 0, sizeof total);
  total.n_files = n_files;
  std::vector<uint64_t> coff, csz;
  std::vector<int32_t> cst;
  int rc = LB2_OK;
  auto enqueue = [&](size_t k) -> int {
    const Chunk &c = chunks[k];
    Workspace &w = (k & 1) ? ctx->ws2 : ctx->ws;
    uint8_t *slot = static_cast<uint8_t *>(d_out_ring) + (k & 1) * slot_capacity;
    // offsets stay absolute inside d_in: a chunk is a window of the file list, not a copy
    return enqueue_batch(ctx, w, static_cast<const uint8_t *>(d_in), h_in_off + c.f0, h_in_sizes ? h_in_sizes + c.f0 : nullptr,
                         c.f1 - c.f0, slot, slot_capacity, flags, s, true);
  };
  auto collect = [&](size_t k) -> int {
    const Chunk &c = chunks[k];
    const uint32_t n = c.f1 - c.f0;
    Workspace &w = (k & 1) ? ctx->ws2 : ctx->ws;
    coff.resize(n + 1); csz.resize(n); cst.resize(n);
    lb2_stats st;
    int r = collect_batch(ctx, w, coff.data(), csz.data(), cst.data(), &st);
    if (r) { total.out_bytes_needed = st.out_bytes_needed; total.overflow = 1; return r; }
    if (h_out_sizes) memcpy(h_out_sizes + c.f0, csz.data(), (size_t)n * sizeof(uint64_t));
    if (h_status) memcpy(h_status + c.f0, cst.data(), (size_t)n * sizeof(int32_t));
    total.n_ok += st.n_ok; total.n_unsupported += st.n_unsupported; total.in_bytes += st.in_bytes; total.out_bytes += st.out_bytes;
    total.copy_bytes += st.copy_bytes; total.header_bytes += st.header_bytes; total.n_tiles += st.n_tiles;
    total.plan_ms += st.plan_ms; total.compact_ms += st.compact_ms;
    if (st.out_bytes_needed > total.out_bytes_needed) total.out_bytes_needed = st.out_bytes_needed;
    if (on_chunk) {
      const uint8_t *slot = static_cast<const uint8_t *>(d_out_ring) + (k & 1) * slot_capacity;
      int u = on_chunk(user, (uint32_t)k, c.f0, n, slot, coff.data(), csz.data(), cst.data(), &st);
      if (u) { ctx->err = "chunk consumer returned " + std::to_string(u); return LB2_E_STATE; }
    }
    return LB2_OK;
  };
  for (size_t k = 0; k < chunks.size() && rc == LB2_OK; k++) {
    if (k >= 2) rc = collect(k - 2);           // frees workspace and output slot k % 2
    if (rc == LB2_OK) rc = enqueue(k);
  }
  for (size_t k = chunks.size() >= 2 ? chunks.size() - 2 : 0; k < chunks.size(); k++) {
    Workspace &w = (k & 1) ? ctx->ws2 : ctx->ws;
    if (!w.in_flight) continue;
    int r = collect(k);                         // always drain what was queued
    if (rc == LB2_OK) rc = r;
  }
  if (total_out) *total_out = total;
  return rc;
}

// ---------------------------------------------------------------------------- host pipeline
static uint64_t env_u64(const char *name, uint64_t dflt) {
  const char *v = getenv(name);
  return v ? strtoull(v, nullptr, 10) : dflt;
}

static int strip_host_dma(lb2_ctx *ctx, const uint8_t *h_in, const uint8_t *d_in_alias, const uint64_t *h_in_off, const uint64_t *h_in_sizes,
                          uint32_t n_files, uint8_t *h_out, uint64_t out_capacity, uint64_t *h_out_off, uint64_t *h_out_sizes,
                          int32_t *h_status, uint32_t flags, lb2_stats *stats);

int lb2_strip_host(lb2_ctx *ctx, const void *h_in_v, const uint64_t *h_in_off, const uint64_t *h_in_sizes, uint32_t n_files,
                   void *h_out_v, uint64_t out_capacity, uint64_t *h_out_off, uint64_t *h_out_sizes, int32_t *h_status,
                   uint32_t flags, lb2_stats *stats) {
  if (!ctx || !h_in_v || !h_in_off || !h_out_v || !h_out_off || !h_out_sizes || !h_status) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  const uint8_t *h_in = static_cast<const uint8_t *>(h_in_v);
  uint8_t *h_out = static_cast<uint8_t *>(h_out_v);
  // Zero-copy path: when both arenas are pinned and mapped into the device address space the
  // kernels work on them directly over PCIe -- the plan kernel pulls only headers, the compaction
  // kernel pulls only the KEPT extents and pushes the stripped files straight into host memory.
  // Dropped sections (.symtab/.strtab/.debug_*) never cross the bus, uploads and downloads run
  // concurrently in both directions, and nothing has to fit in HBM.
  if (env_u64("LB2_HOST_ZEROCOPY", 1) && n_files) {
    void *d_in_alias = nullptr, *d_out_alias = nullptr;
    cudaPointerAttributes ai, ao;
    const bool ok = cudaPointerGetAttributes(&ai, h_in) == cudaSuccess && ai.type == cudaMemoryTypeHost &&
                    cudaPointerGetAttributes(&ao, h_out) == cudaSuccess && ao.type == cudaMemoryTypeHost &&
                    cudaHostGetDevicePointer(&d_in_alias, const_cast<uint8_t *>(h_in), 0) == cudaSuccess &&
                    cudaHostGetDevicePointer(&d_out_alias, h_out, 0) == cudaSuccess;
    cudaGetLastError();  // clear "invalid value" from probing pageable memory
    if (ok && env_u64("LB2_HOST_DMA", 0)) {
      // opt-in (LB2_HOST_DMA=1): plan over the mapping, copy-engine transfers of the kept ranges, compaction in HBM.
      // Measured equal to the zero-copy path below within 3 % (67.9 vs 69.5 GB/s at 1 GPU, 312.6 vs 303.9 at 8):
      // the copy engines' edge over SM loads/stores is eaten by the per-chunk plan -> host -> DMA hand-over.
      return strip_host_dma(ctx, h_in, static_cast<const uint8_t *>(d_in_alias), h_in_off, h_in_sizes, n_files, h_out, out_capacity,
                            h_out_off, h_out_sizes, h_status, flags, stats);
    }
    if (ok) {
      int rc = enqueue_batch(ctx, ctx->ws, static_cast<const uint8_t *>(d_in_alias), h_in_off, h_in_sizes, n_files,
                             static_cast<uint8_t *>(d_out_alias), out_capacity, flags, ctx->stream, true);
      if (rc) return rc;
      lb2_stats st;
      rc = collect_batch(ctx, ctx->ws, h_out_off, h_out_sizes, h_status, &st);
      st.h2d_bytes = st.copy_bytes + st.header_bytes;   // pulled by the kernels through the mapping
      st.d2h_bytes = st.out_bytes;
      if (stats) *stats = st;
      return rc;
    }
  }
  const uint64_t chunk_bytes = env_u64("LB2_CHUNK_MB", 256) << 20;
  lb2_stats total;
  memset(&total, 0, sizeof total);
  total.n_files = n_files;

  // chunk boundaries: consecutive files, <= chunk_bytes of arena span each (a bigger file stands alone)
  struct Chunk { uint32_t f0, f1; uint64_t in_base, in_span; };
  std::vector<Chunk> chunks;
  for (uint32_t f = 0; f < n_files;) {
    uint32_t g = f + 1;
    while (g < n_files && h_in_off[g + 1] - h_in_off[f] <= chunk_bytes) g++;
    chunks.push_back({f, g, h_in_off[f], ((h_in_off[g] - h_in_off[f]) + 255) & ~255ull});
    f = g;
  }
  const int NS = 3;
  for (int k = 0; k < NS; k++) {
    auto &sl = ctx->slot[k];
    if (!sl.stream) {
      CK(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
      for (auto &e : sl.ev_h2d) CK(cudaEventCreate(&e));
      for (auto &e : sl.ev_d2h) CK(cudaEventCreate(&e));
      CK(cudaEventCreateWithFlags(&sl.ev_planned, cudaEventDisableTiming));
    }
  }
  std::vector<uint64_t> rel_off;
  uint64_t out_base = 0;  // running 256-aligned position in h_out
  int rc = LB2_OK;

  auto finish = [&](size_t ci) -> int {
    auto &sl = ctx->slot[ci % NS];
    const Chunk &c = chunks[ci];
    const uint32_t n = c.f1 - c.f0;
    // wait for plan+scan (+compact, same stream) and learn the chunk's output size
    lb2_stats st;
    std::vector<uint64_t> coff(n + 1);
    int r = collect_batch(ctx, sl.ws, coff.data(), h_out_sizes + c.f0, h_status + c.f0, &st);
    if (r == LB2_E_CAPACITY) {
      // device-side output slot too small (re-laid-out files can grow): enlarge and redo this chunk
      cudaFree(sl.d_out);
      sl.cap_out = 0;
      uint64_t need = st.out_bytes_needed + (1u << 20);
      CK(cudaMalloc(&sl.d_out, need));
      sl.cap_out = need;
      std::vector<uint64_t> ro(n + 1);
      for (uint32_t i = 0; i <= n; i++) ro[i] = h_in_off[c.f0 + i] - c.in_base;
      r = enqueue_batch(ctx, sl.ws, sl.d_in, ro.data(), h_in_sizes ? h_in_sizes + c.f0 : nullptr, n, sl.d_out, sl.cap_out, flags, sl.stream, true);
      if (r) return r;
      r = collect_batch(ctx, sl.ws, coff.data(), h_out_sizes + c.f0, h_status + c.f0, &st);
    }
    if (r) return r;
    const uint64_t bytes = coff[n];
    if (out_base + bytes > out_capacity) { ctx->err = "host output arena too small"; total.out_bytes_needed = out_base + bytes; return LB2_E_CAPACITY; }
    CK(cudaEventRecord(sl.ev_d2h[0], sl.stream));
    if (bytes) CK(cudaMemcpyAsync(h_out + out_base, sl.d_out, bytes, cudaMemcpyDeviceToHost, sl.stream));
    total.d2h_bytes += bytes;
    CK(cudaEventRecord(sl.ev_d2h[1], sl.stream));
    for (uint32_t i = 0; i < n; i++) h_out_off[c.f0 + i] = out_base + coff[i];
    out_base += bytes;
    total.n_ok += st.n_ok; total.n_unsupported += st.n_unsupported; total.in_bytes += st.in_bytes; total.out_bytes += st.out_bytes;
    total.copy_bytes += st.copy_bytes; total.header_bytes += st.header_bytes; total.n_tiles += st.n_tiles;
    total.plan_ms += st.plan_ms; total.compact_ms += st.compact_ms;
    return LB2_OK;
  };
  auto reap_copy_times = [&](size_t ci) {
    auto &sl = ctx->slot[ci % NS];
    cudaEventSynchronize(sl.ev_d2h[1]);
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, sl.ev_h2d[0], sl.ev_h2d[1]);
    cudaEventElapsedTime(&b, sl.ev_d2h[0], sl.ev_d2h[1]);
    total.h2d_ms += a; total.d2h_ms += b;
  };

  for (size_t ci = 0; ci < chunks.size() && rc == LB2_OK; ci++) {
    auto &sl = ctx->slot[ci % NS];
    const Chunk &c = chunks[ci];
    const uint32_t n = c.f1 - c.f0;
    if (ci >= (size_t)NS) reap_copy_times(ci - NS);  // slot is free once its D2H finished
    if (sl.cap_in < c.in_span + 256) {
      cudaFree(sl.d_in); sl.cap_in = 0;
      uint64_t need = std::max<uint64_t>(c.in_span + 256, std::min<uint64_t>(chunk_bytes, 64ull << 20));
      CK(cudaMalloc(&sl.d_in, need));
      sl.cap_in = need;
    }
    const uint64_t want_out = c.in_span + (uint64_t)n * 4096 + (8u << 20);
    if (sl.cap_out < want_out) {
      cudaFree(sl.d_out); sl.cap_out = 0;
      CK(cudaMalloc(&sl.d_out, want_out));
      sl.cap_out = want_out;
    }
    CK(cudaEventRecord(sl.ev_h2d[0], sl.stream));
    CK(cudaMemcpyAsync(sl.d_in, h_in + c.in_base, h_in_off[c.f1] - c.in_base, cudaMemcpyHostToDevice, sl.stream));
    total.h2d_bytes += h_in_off[c.f1] - c.in_base;
    CK(cudaEventRecord(sl.ev_h2d[1], sl.stream));
    rel_off.resize(n + 1);
    for (uint32_t i = 0; i <= n; i++) rel_off[i] = h_in_off[c.f0 + i] - c.in_base;
    rc = enqueue_batch(ctx, sl.ws, sl.d_in, rel_off.data(), h_in_sizes ? h_in_sizes + c.f0 : nullptr, n, sl.d_out, sl.cap_out, flags, sl.stream, true);
    if (rc) break;
    // with the next chunk's upload and kernels queued, turn to the previous chunk's download
    if (ci >= 1) rc = finish(ci - 1);
  }
  if (rc == LB2_OK && !chunks.empty()) rc = finish(chunks.size() - 1);
  for (size_t ci = chunks.size() >= (size_t)NS ? chunks.size() - NS : 0; ci < chunks.size(); ci++) reap_copy_times(ci);
  for (int k = 0; k < NS; k++) { cudaStreamSynchronize(ctx->slot[k].stream); ctx->slot[k].ws.in_flight = false; }
  h_out_off[n_files] = out_base;
  if (total.out_bytes_needed == 0) total.out_bytes_needed = out_base;
  if (stats) *stats = total;
  return rc;
}

}  // extern "C"


// ---- host buffers, pinned and mapped: plan over the mapping, upload only what is kept, compact in HBM ----------
// Measured on this box (profiles/r02_pcie_probe.txt): the copy engines move 49.6 GB/s per direction with both
// directions busy, SM loads/stores on mapped host memory 40.6 (what the zero-copy path gets).  So, per chunk of
// whole files (<= LB2_CHUNK_MB of arena span, three slots rotating):
//   1. plan + scan run on the host-mapped input: only headers, names and notes cross the bus; the kernel also
//      lists the input ranges its copy extents read (small files whole, neighbours merged);
//   2. those ranges are uploaded by the copy engine into a device slot laid out like the host arena -- dropped
//      sections (.symtab/.strtab/.debug_*) still never cross the bus;
//   3. the compaction kernel runs HBM -> HBM (tile sources inside the host mapping are rebased onto the slot);
//   4. one DMA brings the chunk's output down.
// The plan of chunk k+1 is queued before the host waits for chunk k's plan results, so the engines stay busy.
static int strip_host_dma(lb2_ctx *ctx, const uint8_t *h_in, const uint8_t *d_in_alias, const uint64_t *h_in_off, const uint64_t *h_in_sizes,
                          uint32_t n_files, uint8_t *h_out, uint64_t out_capacity, uint64_t *h_out_off, uint64_t *h_out_sizes,
                          int32_t *h_status, uint32_t flags, lb2_stats *stats) {
  const uint64_t chunk_bytes = env_u64("LB2_CHUNK_MB", 256) << 20;
  lb2_stats total;
  memset(&total, 0, sizeof total);
  total.n_files = n_files;
  struct Chunk { uint32_t f0, f1; uint64_t in_base, in_span; };
  std::vector<Chunk> chunks;
  for (uint32_t f = 0; f < n_files;) {
    uint32_t g = f + 1;
    while (g < n_files && h_in_off[g + 1] - h_in_off[f] <= chunk_bytes) g++;
    chunks.push_back({f, g, h_in_off[f], ((h_in_off[g] - h_in_off[f]) + 255) & ~255ull});
    f = g;
  }
  const int NS = 3;
  for (int k = 0; k < NS; k++) {
    auto &sl = ctx->slot[k];
    if (!sl.stream) {
      CK(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
      for (auto &e : sl.ev_h2d) CK(cudaEventCreate(&e));
      for (auto &e : sl.ev_d2h) CK(cudaEventCreate(&e));
      CK(cudaEventCreateWithFlags(&sl.ev_planned, cudaEventDisableTiming));
    }
  }
  uint64_t out_base = 0;
  std::vector<uint64_t> rel_off, coff;
  auto plan = [&](size_t ci) -> int {
    auto &sl = ctx->slot[ci % NS];
    const Chunk &c = chunks[ci];
    const uint32_t n = c.f1 - c.f0;
    if (ci >= (size_t)NS) {  // the slot's previous occupant must be fully downloaded
      CK(cudaEventSynchronize(sl.ev_d2h[1]));
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, sl.ev_h2d[0], sl.ev_h2d[1]);
      cudaEventElapsedTime(&b, sl.ev_d2h[0], sl.ev_d2h[1]);
      total.h2d_ms += a; total.d2h_ms += b;
    }
    rel_off.resize(n + 1);
    for (uint32_t i = 0; i <= n; i++) rel_off[i] = h_in_off[c.f0 + i] - c.in_base;
    return enqueue_batch(ctx, sl.ws, d_in_alias + c.in_base, rel_off.data(), h_in_sizes ? h_in_sizes + c.f0 : nullptr, n, nullptr, 0, flags,
                         sl.stream, false, true, true);
  };
  auto move = [&](size_t ci) -> int {
    auto &sl = ctx->slot[ci % NS];
    const Chunk &c = chunks[ci];
    const uint32_t n = c.f1 - c.f0;
    lb2_stats st;
    coff.resize(n + 1);
    int r = collect_batch(ctx, sl.ws, coff.data(), h_out_sizes + c.f0, h_status + c.f0, &st);
    if (r) return r;
    const uint64_t bytes = coff[n];
    if (out_base + bytes > out_capacity) { ctx->err = "host output arena too small"; total.out_bytes_needed = out_base + bytes; return LB2_E_CAPACITY; }
    if (sl.cap_in < c.in_span + 256) {
      cudaFree(sl.d_in); sl.d_in = nullptr; sl.cap_in = 0;
      const uint64_t need = std::max<uint64_t>(c.in_span + 256, std::min<uint64_t>(chunk_bytes, 64ull << 20));
      CK(cudaMalloc(&sl.d_in, need));
      sl.cap_in = need;
    }
    if (sl.cap_out < bytes + 256) {
      cudaFree(sl.d_out); sl.d_out = nullptr; sl.cap_out = 0;
      const uint64_t need = std::max<uint64_t>(bytes + (1u << 20), c.in_span + (8u << 20));
      CK(cudaMalloc(&sl.d_out, need));
      sl.cap_out = need;
    }
    // upload what the copy extents read
    const BatchCounters &bc = *sl.ws.h_ctr;
    CK(cudaEventRecord(sl.ev_h2d[0], sl.stream));
    if (bc.ranges_overflow || bc.n_ranges > sl.ws.cap_ranges) {
      CK(cudaMemcpyAsync(sl.d_in, h_in + c.in_base, h_in_off[c.f1] - c.in_base, cudaMemcpyHostToDevice, sl.stream));
      total.h2d_bytes += h_in_off[c.f1] - c.in_base;
    } else {
      // the kernel appended the ranges in no particular order: sort, fuse neighbours (files are 256-byte
      // padded, so runs of small files become one transfer), one DMA per fused range
      UpRange *rg = sl.ws.h_ranges;
      std::sort(rg, rg + bc.n_ranges, [](const UpRange &x, const UpRange &y) { return x.off < y.off; });
      uint64_t rs = 0, re = 0;
      auto flush = [&]() -> int {
        if (re <= rs) return LB2_OK;
        if (re > c.in_span) { ctx->err = "upload range outside the chunk"; return LB2_E_STATE; }
        CK(cudaMemcpyAsync(sl.d_in + rs, h_in + c.in_base + rs, re - rs, cudaMemcpyHostToDevice, sl.stream));
        total.h2d_bytes += re - rs;
        return LB2_OK;
      };
      for (uint32_t k = 0; k < bc.n_ranges; k++) {
        const uint64_t o = rg[k].off, e = rg[k].off + rg[k].len;
        if (re > rs && o <= re + 8192) { if (e > re) re = e; }
        else { int fr = flush(); if (fr) return fr; rs = o; re = e; }
      }
      int fr = flush();
      if (fr) return fr;
    }
    CK(cudaEventRecord(sl.ev_h2d[1], sl.stream));
    // compaction on the device copy
    CompactArgs ca;
    ca.tiles = sl.ws.d_tiles; ca.ctr = sl.ws.d_ctr; ca.out_off = sl.ws.d_out_off; ca.out = sl.d_out;
    ca.rebase_lo = reinterpret_cast<uint64_t>(d_in_alias + c.in_base);
    ca.rebase_len = c.in_span;
    ca.rebase_delta = reinterpret_cast<uint64_t>(sl.d_in) - ca.rebase_lo;
    CK(cudaEventRecord(sl.ws.ev[1], sl.stream));
    if (ctx->use_tma) launch_compact_tma(ca, ctx->sm_count, sl.stream);
    else launch_compact(ca, ctx->sm_count * ctx->compact_ctas_per_sm, sl.stream);
    CK(cudaEventRecord(sl.ws.ev[2], sl.stream));
    CK(cudaEventRecord(sl.ev_d2h[0], sl.stream));
    if (bytes) CK(cudaMemcpyAsync(h_out + out_base, sl.d_out, bytes, cudaMemcpyDeviceToHost, sl.stream));
    total.d2h_bytes += bytes;
    total.h2d_bytes += st.header_bytes;   // what the plan kernel read through the mapping
    CK(cudaEventRecord(sl.ev_d2h[1], sl.stream));
    CK(cudaGetLastError());
    for (uint32_t i = 0; i < n; i++) h_out_off[c.f0 + i] = out_base + coff[i];
    out_base += bytes;
    total.n_ok += st.n_ok; total.n_unsupported += st.n_unsupported; total.in_bytes += st.in_bytes; total.out_bytes += st.out_bytes;
    total.copy_bytes += st.copy_bytes; total.header_bytes += st.header_bytes; total.n_tiles += st.n_tiles;
    total.plan_ms += st.plan_ms;
    return LB2_OK;
  };
  int rc = LB2_OK;
  for (size_t ci = 0; ci < chunks.size() && rc == LB2_OK; ci++) {
    rc = plan(ci);
    if (rc == LB2_OK && ci >= 1) rc = move(ci - 1);
  }
  if (rc == LB2_OK && !chunks.empty()) rc = move(chunks.size() - 1);
  for (int k = 0; k < NS; k++) {
    auto &sl = ctx->slot[k];
    cudaStreamSynchronize(sl.stream);
    sl.ws.in_flight = false;
    if ((size_t)k < chunks.size()) {
      float a = 0, b = 0, cms = 0;
      if (cudaEventElapsedTime(&a, sl.ev_h2d[0], sl.ev_h2d[1]) == cudaSuccess) total.h2d_ms += a;
      if (cudaEventElapsedTime(&b, sl.ev_d2h[0], sl.ev_d2h[1]) == cudaSuccess) total.d2h_ms += b;
      if (cudaEventElapsedTime(&cms, sl.ws.ev[1], sl.ws.ev[2]) == cudaSuccess) total.compact_ms += cms;  // (last chunk of each slot only)
    }
  }
  cudaGetLastError();
  h_out_off[n_files] = out_base;
  if (total.out_bytes_needed == 0) total.out_bytes_needed = out_base;
  if (stats) *stats = total;
  return rc;
}

// ---------------------------------------------------------------------------- tree walker
static bool ends_with(const char *s, const char *suf) {
  size_t a = strlen(s), b = strlen(suf);
  return a >= b && memcmp(s + a - b, suf, b) == 0;
}

struct TreeFile { std::string path; uint64_t size; dev_t dev; ino_t ino; uint32_t times; };

// The sibling lines of the reference's script (/root/reference/lambdipy/project_build.py:256-259), done on
// the same directory walk when asked for (LB2_TREE_CLEANUP):
//   rm -rf ROOT/*.egg-info ; rm -rf ROOT/*.dist-info                  top level, shell glob (no dot files)
//   find ROOT/ -name __pycache__ | xargs rm -rf                        any depth, any type
//   find ROOT/ -name tests | grep -v "PATTERN" | xargs rm -rf          PATTERN: a grep basic regex on the path
//                                                                      line find prints ("*" keeps only paths
//                                                                      containing a literal asterisk)
// They run before the strip line, so shared objects under a removed directory are never stripped.
struct Cleanup {
  bool on = false;
  regex_t keep;          // grep -v pattern for `tests`
  bool have_keep = false;
  uint32_t n_removed = 0;
};

static void rm_rf(const std::string &p) {
  struct stat sb;
  if (lstat(p.c_str(), &sb) != 0) return;
  if (S_ISDIR(sb.st_mode)) {
    if (DIR *d = opendir(p.c_str())) {
      while (dirent *e = readdir(d)) {
        if (!strcmp(e->d_name, ".") || !strcmp(e->d_name, "..")) continue;
        rm_rf(p + "/" + e->d_name);
      }
      closedir(d);
    }
    rmdir(p.c_str());
  } else {
    unlink(p.c_str());
  }
}

// `find ROOT/ -name "*SUFFIX"`: every directory entry whose basename matches, of any type; find does
// not descend into symlinked directories.  What `strip` then does with each path decides the rest:
//   regular file           -> stripped in place: GNU strip 2.42 writes the new contents back INTO THE
//                             EXISTING INODE (smart_rename copies), so mode, owner and every other hard
//                             link of the file are kept -- `libfoo.so.1` hard-linked to `libfoo.so` ends up
//                             stripped too although its name does not match
//   symlink to a file      -> the TARGET is rewritten, the link stays
//   directory / dangling   -> strip fails -> xargs exits 123 -> the reference's script aborts
// An inode reached through k matching paths (symlinks or hard links) is stripped k times by the
// reference; `times` keeps k.  Paths are kept as found: open() follows the links like strip does.
// `shown` is the path as find would print it (ROOT as given + "/" + relative part): what grep sees.
static void walk(const std::string &dir, const std::string &shown, bool top, const char *suffix, Cleanup *cl,
                 std::vector<TreeFile> &files, lb2_tree_stats *st) {
  DIR *d = opendir(dir.c_str());
  if (!d) return;
  std::vector<std::string> names;
  while (dirent *e = readdir(d))
    if (strcmp(e->d_name, ".") && strcmp(e->d_name, "..")) names.push_back(e->d_name);
  closedir(d);
  for (const std::string &name : names) {
    const std::string p = dir + "/" + name, line = shown + name;
    struct stat lsb, sb;
    if (lstat(p.c_str(), &lsb) != 0) continue;
    if (cl && cl->on) {
      bool remove = false;
      if (top && name[0] != '.' && (ends_with(name.c_str(), ".egg-info") || ends_with(name.c_str(), ".dist-info"))) remove = true;
      else if (name == "__pycache__") remove = true;
      else if (name == "tests" && line.find('\n') == std::string::npos &&
               !(cl->have_keep && regexec(&cl->keep, line.c_str(), 0, nullptr, 0) == 0)) remove = true;
      if (remove) { rm_rf(p); cl->n_removed++; continue; }
    }
    if (suffix && ends_with(name.c_str(), suffix)) {
      st->n_selected++;
      if (stat(p.c_str(), &sb) != 0 || !S_ISREG(sb.st_mode)) {
        st->n_failed++;  // directory, dangling link, device ...: strip errors out
      } else {
        if (S_ISLNK(lsb.st_mode)) st->n_skipped++;  // the link itself is left alone
        files.push_back({p, (uint64_t)sb.st_size, sb.st_dev, sb.st_ino, 1});
      }
    }
    if (S_ISDIR(lsb.st_mode)) walk(p, line + "/", false, suffix, cl, files, st);
  }
}

static bool cleanup_init(Cleanup &cl, const char *keep_regex, std::string *err) {
  cl.on = true;
  if (keep_regex && *keep_regex) {
    if (regcomp(&cl.keep, keep_regex, REG_NOSUB) != 0) { if (err) *err = std::string("bad keep-tests pattern: ") + keep_regex; return false; }
    cl.have_keep = true;
  }
  return true;
}

static void dedupe(std::vector<TreeFile> &files) {
  std::sort(files.begin(), files.end(), [](const TreeFile &a, const TreeFile &b) {
    if (a.dev != b.dev) return a.dev < b.dev;
    if (a.ino != b.ino) return a.ino < b.ino;
    return a.path < b.path;
  });
  size_t w = 0;
  for (size_t i = 0; i < files.size(); i++) {
    if (w && files[w - 1].dev == files[i].dev && files[w - 1].ino == files[i].ino) files[w - 1].times++;
    else files[w++] = files[i];
  }
  files.resize(w);
  std::sort(files.begin(), files.end(), [](const TreeFile &a, const TreeFile &b) { return a.path < b.path; });
}

static int host_strip(const std::string &p) {
  const char *argv[] = {"strip", p.c_str(), nullptr};
  pid_t pid;
  if (posix_spawnp(&pid, "strip", nullptr, nullptr, const_cast<char *const *>(argv), environ) != 0) return 127;
  int status = 0;
  while (waitpid(pid, &status, 0) < 0 && errno == EINTR) {}
  return WIFEXITED(status) ? WEXITSTATUS(status) : 128;
}

template <class F> static void parallel_for(size_t n, int threads, F f) {
  std::atomic<size_t> next{0};
  std::vector<std::thread> pool;
  threads = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(threads, 1), n));
  for (int t = 0; t < threads; t++)
    pool.emplace_back([&] { for (size_t i; (i = next.fetch_add(1)) < n;) f(i); });
  for (auto &th : pool) th.join();
}

// ---- the streaming engine behind lb2_strip_tree ---------------------------------------------------
// File bytes travel   page cache --pread--> pinned slot --DMA--> HBM input arena   and back
//                     HBM output arena --DMA--> pinned slot --pwrite--> the file's existing inode.
// Pinned memory is only a ring of small slots (two per I/O worker, LB2_TREE_SLOT_MB each), so a
// one-shot `lambdipy build` does not pay for pinning the tree twice and a 100 GB tree needs no more
// host memory than a small one.  The tree is cut into batches of whole files (<= LB2_TREE_BATCH_MB of
// arena span; a larger file is a batch of its own) that alternate between two HBM buffer sets: while
// batch b is downloaded and written, batch b+1 is read and uploaded -- the same worker pool serves both.
struct Seg { uint32_t file; uint64_t file_off, len, slot_off; };
struct Slice { bool upload; uint8_t *dev; uint64_t len; uint32_t seg0, seg1; };

static void make_slices(bool upload, uint8_t *dev_base, const std::vector<uint32_t> &ids, const uint64_t *offs, const uint64_t *sizes,
                        uint64_t slot_bytes, std::vector<Seg> &segs, std::vector<Slice> &out) {
  // ids[k] occupies [offs[k], offs[k] + sizes[k]) of the device arena, ascending and disjoint.  A slice is
  // one contiguous DMA range of at most slot_bytes; padding between neighbouring files rides along, a
  // larger hole (files that took another route) starts a new slice.
  const size_t m = ids.size();
  size_t k = 0;
  uint64_t c = 0;  // bytes of file k already covered by earlier slices
  while (k < m) {
    if (sizes[k] == 0) { k++; c = 0; continue; }
    const uint64_t a = offs[k] + c, end = a + slot_bytes;
    Slice sl{upload, dev_base + a, 0, (uint32_t)segs.size(), 0};
    uint64_t last = a;
    while (k < m) {
      if (sizes[k] == 0) { k++; c = 0; continue; }
      const uint64_t fs = offs[k] + c, fe = offs[k] + sizes[k];
      if (fs >= end || fs - last > 65536) break;
      const uint64_t take = std::min(fe, end) - fs;
      segs.push_back({ids[k], c, take, fs - a});
      last = fs + take;
      if (last == fe) { k++; c = 0; } else { c += take; break; }  // slot full inside a big file
    }
    sl.seg1 = (uint32_t)segs.size();
    sl.len = last - a;
    out.push_back(sl);
  }
}

struct TreeWorker { cudaStream_t stream = nullptr; cudaEvent_t ev[2] = {nullptr, nullptr}; uint32_t k = 0; };

struct TreeEngine {
  uint8_t *h_ring = nullptr;
  uint64_t slot_bytes = 0;
  int n_workers = 0;
  std::vector<TreeWorker> workers;
  uint8_t *d_in[2] = {nullptr, nullptr}, *d_out[2] = {nullptr, nullptr};
  uint64_t cap_in[2] = {0, 0}, cap_out[2] = {0, 0};
};

static void tree_engine_free(TreeEngine *e) {
  if (!e) return;
  for (auto &w : e->workers) {
    if (w.stream) cudaStreamDestroy(w.stream);
    for (auto &ev : w.ev) if (ev) cudaEventDestroy(ev);
  }
  if (e->h_ring) cudaFreeHost(e->h_ring);
  for (int k = 0; k < 2; k++) { cudaFree(e->d_in[k]); cudaFree(e->d_out[k]); }
  delete e;
}

static int tree_engine_prepare(lb2_ctx *ctx, uint64_t expected_bytes) {
  if (ctx->tree) return LB2_OK;
  TreeEngine *e = new TreeEngine();
  e->slot_bytes = std::max<uint64_t>(1, env_u64("LB2_TREE_SLOT_MB", 4)) << 20;
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  int want = (int)env_u64("LB2_IO_THREADS", std::max(4u, std::min(32u, hw / 2)));
  want = std::max(want, 1);
  if (expected_bytes) want = (int)std::max<uint64_t>(2, std::min<uint64_t>((uint64_t)want, expected_bytes / (2 * e->slot_bytes) + 1));
  e->n_workers = want;
  NumaPreferred near_gpu(ctx->numa_node);
  cudaError_t err = cudaHostAlloc(&e->h_ring, (uint64_t)want * 2 * e->slot_bytes, cudaHostAllocDefault);
  if (err != cudaSuccess) { ctx->err = std::string("cudaHostAlloc(tree ring): ") + cudaGetErrorString(err); delete e; return LB2_E_CUDA; }
  e->workers.resize(want);
  for (auto &w : e->workers) {
    if (cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&w.ev[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&w.ev[1], cudaEventDisableTiming) != cudaSuccess) {
      ctx->err = "cuda stream/event creation failed"; tree_engine_free(e); return LB2_E_CUDA;
    }
  }
  ctx->tree = e;
  return LB2_OK;
}

static bool pread_all(int fd, uint8_t *dst, uint64_t n, uint64_t off) {
  uint64_t got = 0;
  while (got < n) {
    ssize_t r = pread(fd, dst + got, n - got, (off_t)(off + got));
    if (r <= 0) { if (r < 0 && errno == EINTR) continue; return false; }
    got += (uint64_t)r;
  }
  return true;
}
static bool pwrite_all(int fd, const uint8_t *src, uint64_t n, uint64_t off) {
  uint64_t put = 0;
  while (put < n) {
    ssize_t r = pwrite(fd, src + put, n - put, (off_t)(off + put));
    if (r <= 0) { if (r < 0 && errno == EINTR) continue; return false; }
    put += (uint64_t)r;
  }
  return true;
}

extern "C" {

int lb2_tree_prepare(lb2_ctx *ctx, uint64_t expected_tree_bytes) {
  if (!ctx) return LB2_E_ARG;
  CK(cudaSetDevice(ctx->device));
  int rc = tree_engine_prepare(ctx, expected_tree_bytes);
  if (rc) return rc;
  // workspaces and the compaction kernel's shared-memory opt-in are first-use costs too
  rc = ws_reserve(ctx, ctx->ws, 256, 1 << 16);
  if (rc) return rc;
  return ws_reserve(ctx, ctx->ws2, 256, 1 << 16);
}

int lb2_tree_cleanup(const char *root, const char *keep_tests_regex, uint32_t *n_removed) {
  if (!root) return LB2_E_ARG;
  struct stat rsb;
  if (stat(root, &rsb) != 0 || !S_ISDIR(rsb.st_mode)) return LB2_E_IO;
  Cleanup cl;
  if (!cleanup_init(cl, keep_tests_regex, nullptr)) return LB2_E_ARG;
  std::string r = root;
  while (r.size() > 1 && r.back() == '/') r.pop_back();
  std::vector<TreeFile> files;
  lb2_tree_stats st;
  memset(&st, 0, sizeof st);
  walk(r, r + "/", true, nullptr, &cl, files, &st);
  if (cl.have_keep) regfree(&cl.keep);
  if (n_removed) *n_removed = cl.n_removed;
  return LB2_OK;
}

int lb2_strip_tree(lb2_ctx *ctx, const char *root, const char *suffix, uint32_t flags, lb2_tree_stats *st_out) {
  return lb2_strip_tree_ex(ctx, root, suffix, flags, nullptr, st_out);
}

int lb2_strip_tree_ex(lb2_ctx *ctx, const char *root, const char *suffix, uint32_t flags, const char *keep_tests_regex,
                      lb2_tree_stats *st_out) {
  if (!ctx || !root || !suffix) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  lb2_tree_stats st;
  memset(&st, 0, sizeof st);
  double t0 = now_s();
  std::vector<TreeFile> files;
  struct stat rsb;
  if (stat(root, &rsb) != 0 || !S_ISDIR(rsb.st_mode)) { ctx->err = std::string("not a directory: ") + root; return LB2_E_IO; }
  std::string r = root;
  while (r.size() > 1 && r.back() == '/') r.pop_back();
  Cleanup cl;
  if ((flags & LB2_TREE_CLEANUP) && !cleanup_init(cl, keep_tests_regex, &ctx->err)) return LB2_E_ARG;
  walk(r, r + "/", true, suffix, &cl, files, &st);
  if (cl.have_keep) regfree(&cl.keep);
  st.n_removed = cl.n_removed;
  dedupe(files);
  const uint32_t n = (uint32_t)files.size();
  uint64_t tree_bytes = 0;
  for (auto &f : files) tree_bytes += f.size;
  st.walk_read_s = now_s() - t0;
  if (!n) { if (st_out) *st_out = st; return LB2_OK; }
  int rc = tree_engine_prepare(ctx, tree_bytes);
  if (rc) return rc;
  TreeEngine &E = *ctx->tree;
  const bool dry = (flags & LB2_TREE_DRY_RUN) != 0;

  // ---- batches of whole files
  const uint64_t batch_bytes = std::max<uint64_t>(1, env_u64("LB2_TREE_BATCH_MB", 1024)) << 20;
  struct Batch { uint32_t f0, f1; uint64_t span; };
  std::vector<Batch> batches;
  std::vector<uint64_t> off(n + 1), sizes(n), out_off(n + 1), out_sizes(n);  // offsets are relative to the batch's arena
  std::vector<int32_t> status(n, LB2_ST_MALFORMED);
  for (uint32_t f = 0; f < n;) {
    uint64_t pos = 0;
    uint32_t g = f;
    while (g < n && (g == f || pos + ((files[g].size + 255) & ~255ull) <= batch_bytes)) {
      off[g] = pos; sizes[g] = files[g].size; pos += (files[g].size + 255) & ~255ull; g++;
    }
    batches.push_back({f, g, pos});
    f = g;
  }

  // ---- worker pool: one task queue served by n_workers threads, each with two pinned slots + a stream
  std::vector<Seg> segs;
  std::vector<Slice> queue;
  std::atomic<size_t> q_next{0}, q_done{0};
  size_t q_end = 0;
  std::mutex mu;
  std::condition_variable cv_work, cv_done;
  bool quit = false;
  std::atomic<int> io_fail{0};
  std::atomic<uint64_t> ns_read{0}, ns_write{0}, ns_dma{0};  // summed over workers: where the I/O threads spend their time
  auto now_ns = [] { return (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  std::vector<std::atomic<int>> read_bad(n), write_bad(n);
  std::vector<std::atomic<uint32_t>> segs_left(n);
  for (uint32_t i = 0; i < n; i++) { read_bad[i] = 0; write_bad[i] = 0; segs_left[i] = 0; }
  std::atomic<uint32_t> n_gpu{0}, n_failed{0}, n_skipped{0};
  std::atomic<uint64_t> in_b{0}, out_b{0};
  std::vector<uint64_t> final_size(n, 0);

  auto finish_file = [&](uint32_t i) {
    // every piece of the new contents is in the inode: cut the old tail off
    bool ok = write_bad[i] == 0;
    if (ok && final_size[i] != files[i].size) ok = truncate(files[i].path.c_str(), (off_t)final_size[i]) == 0;
    if (ok) { n_gpu++; in_b += files[i].size; out_b += final_size[i]; }
    else n_failed++;
  };
  auto run_slice = [&](TreeWorker &w, int widx, const Slice &sl) {
    uint8_t *slot = E.h_ring + ((uint64_t)widx * 2 + (w.k & 1)) * E.slot_bytes;
    cudaEvent_t ev = w.ev[w.k & 1];
    w.k++;
    if (sl.upload) {
      uint64_t t0 = now_ns();
      cudaEventSynchronize(ev);  // the DMA that last read this slot has finished
      uint64_t t1 = now_ns();
      for (uint32_t q = sl.seg0; q < sl.seg1; q++) {
        const Seg &sg = segs[q];
        int fd = open(files[sg.file].path.c_str(), O_RDONLY | O_CLOEXEC);
        if (fd < 0 || !pread_all(fd, slot + sg.slot_off, sg.len, sg.file_off)) { read_bad[sg.file]++; io_fail++; }
        if (fd >= 0) close(fd);
      }
      uint64_t t2 = now_ns();
      cudaMemcpyAsync(sl.dev, slot, sl.len, cudaMemcpyHostToDevice, w.stream);
      cudaEventRecord(ev, w.stream);
      ns_dma += (t1 - t0) + (now_ns() - t2); ns_read += t2 - t1;
    } else {
      uint64_t t0 = now_ns();
      cudaMemcpyAsync(slot, sl.dev, sl.len, cudaMemcpyDeviceToHost, w.stream);
      cudaEventRecord(ev, w.stream);
      if (cudaEventSynchronize(ev) != cudaSuccess) io_fail++;
      uint64_t t1 = now_ns();
      ns_dma += t1 - t0;
      const uint64_t tw0 = t1;
      for (uint32_t q = sl.seg0; q < sl.seg1; q++) {
        const Seg &sg = segs[q];
        // no O_TRUNC, no temp file: the bytes go into the pages the file already has (see walk())
        int fd = open(files[sg.file].path.c_str(), O_WRONLY | O_CLOEXEC);
        if (fd < 0 || !pwrite_all(fd, slot + sg.slot_off, sg.len, sg.file_off)) write_bad[sg.file]++;
        if (fd >= 0) close(fd);
        if (--segs_left[sg.file] == 0) finish_file(sg.file);
      }
      ns_write += now_ns() - tw0;
    }
  };
  std::vector<std::thread> pool;
  for (int wi = 0; wi < E.n_workers; wi++)
    pool.emplace_back([&, wi] {
      cudaSetDevice(ctx->device);
      TreeWorker &w = E.workers[wi];
      for (;;) {
        size_t idx;
        {
          std::unique_lock<std::mutex> lk(mu);
          cv_work.wait(lk, [&] { return quit || q_next.load() < q_end; });
          if (q_next.load() >= q_end) { if (quit) return; continue; }
          idx = q_next.fetch_add(1);
        }
        run_slice(w, wi, queue[idx]);
        if (q_done.fetch_add(1) + 1 == q_end) { std::lock_guard<std::mutex> lk(mu); cv_done.notify_all(); }
      }
    });
  auto submit_and_wait = [&](std::vector<Slice> &a, std::vector<Slice> &b) {
    // interleave the two task lists so that downloads of batch b and uploads of batch b+1 overlap
    {
      std::lock_guard<std::mutex> lk(mu);
      size_t i = 0, j = 0;
      while (i < a.size() || j < b.size()) {
        if (i < a.size()) queue.push_back(a[i++]);
        if (j < b.size()) queue.push_back(b[j++]);
      }
      q_end = queue.size();
    }
    cv_work.notify_all();
    std::unique_lock<std::mutex> lk(mu);
    cv_done.wait(lk, [&] { return q_done.load() >= q_end; });
  };
  auto stop_pool = [&] {
    { std::lock_guard<std::mutex> lk(mu); quit = true; }
    cv_work.notify_all();
    for (auto &th : pool) th.join();
  };

  auto upload_slices = [&](size_t bi, std::vector<Slice> &out) -> int {
    const Batch &b = batches[bi];
    const int set = (int)(bi & 1);
    if (E.cap_in[set] < b.span + 256) {
      cudaFree(E.d_in[set]); E.d_in[set] = nullptr; E.cap_in[set] = 0;
      const uint64_t need = b.span + 256;
      CK(cudaMalloc(&E.d_in[set], need));
      E.cap_in[set] = need;
    }
    std::vector<uint32_t> ids(b.f1 - b.f0);
    for (uint32_t i = b.f0; i < b.f1; i++) ids[i - b.f0] = i;
    make_slices(true, E.d_in[set], ids, off.data() + b.f0, sizes.data() + b.f0, E.slot_bytes, segs, out);
    return LB2_OK;
  };

  std::vector<void *> tmp_dev;  // outputs of the re-strip passes, freed at the end
  std::vector<Slice> up, down, none;
  double t_gpu = 0, t_io0 = now_s();
  // (a lambda so that every CUDA error path still reaches stop_pool() below)
  auto run_batches = [&]() -> int {
  int rc = upload_slices(0, up);
  if (rc == LB2_OK) submit_and_wait(up, none);
  for (size_t bi = 0; bi < batches.size() && rc == LB2_OK; bi++) {
    const Batch &b = batches[bi];
    const int set = (int)(bi & 1);
    const uint32_t m = b.f1 - b.f0;
    bool bad_read = false;
    for (uint32_t i = b.f0; i < b.f1; i++) bad_read |= read_bad[i] != 0;
    if (bad_read) { ctx->err = "could not read some selected files"; rc = LB2_E_IO; break; }
    // ---- kernels on the batch, inputs in HBM
    const double tg = now_s();
    for (auto &w : E.workers) { CK(cudaStreamWaitEvent(ctx->stream, w.ev[0], 0)); CK(cudaStreamWaitEvent(ctx->stream, w.ev[1], 0)); }
    uint64_t want_out = b.span + (uint64_t)m * 4096 + (16u << 20);
    Workspace &ws = set ? ctx->ws2 : ctx->ws;
    lb2_stats bst;
    for (int attempt = 0; attempt < 2; attempt++) {
      if (E.cap_out[set] < want_out) {
        cudaFree(E.d_out[set]); E.d_out[set] = nullptr; E.cap_out[set] = 0;
        CK(cudaMalloc(&E.d_out[set], want_out));
        E.cap_out[set] = want_out;
      }
      rc = enqueue_batch(ctx, ws, E.d_in[set], off.data() + b.f0, sizes.data() + b.f0, m, E.d_out[set], E.cap_out[set], flags & 0xffu, ctx->stream, true);
      if (rc) break;
      rc = collect_batch(ctx, ws, out_off.data() + b.f0, out_sizes.data() + b.f0, status.data() + b.f0, &bst);
      if (rc != LB2_E_CAPACITY) break;
      want_out = bst.out_bytes_needed + (1u << 20);  // re-laid-out files can grow: enlarge and redo
    }
    if (rc) break;
    st.batch.n_files += m; st.batch.n_ok += bst.n_ok; st.batch.n_unsupported += bst.n_unsupported; st.batch.in_bytes += bst.in_bytes;
    st.batch.out_bytes += bst.out_bytes; st.batch.copy_bytes += bst.copy_bytes; st.batch.header_bytes += bst.header_bytes;
    st.batch.n_tiles += bst.n_tiles; st.batch.plan_ms += bst.plan_ms; st.batch.compact_ms += bst.compact_ms;
    // ---- inodes the reference strips more than once (several matching names): further passes run on
    //      the previous pass's output, still in HBM (strip is not idempotent on a few note layouts)
    std::vector<uint8_t *> src_base(m, E.d_out[set]);
    std::vector<uint64_t> src_off(out_off.begin() + b.f0, out_off.begin() + b.f1);
    for (uint32_t pass = 1; rc == LB2_OK; pass++) {
      std::vector<uint32_t> again;
      for (uint32_t i = b.f0; i < b.f1; i++) if (files[i].times > pass && status[i] == LB2_ST_OK) again.push_back(i);
      if (again.empty()) break;
      const uint32_t k2 = (uint32_t)again.size();
      std::vector<uint64_t> off2(k2 + 1), sz2(k2), ooff2(k2 + 1), osz2(k2);
      std::vector<int32_t> st2(k2);
      uint64_t p2 = 0;
      for (uint32_t k = 0; k < k2; k++) { off2[k] = p2; sz2[k] = out_sizes[again[k]]; p2 += (sz2[k] + 255) & ~255ull; }
      off2[k2] = p2;
      uint8_t *d_in2 = nullptr, *d_out2 = nullptr;
      const uint64_t cap2 = p2 + (uint64_t)k2 * 4096 + (64u << 20);
      CK(cudaMalloc(&d_in2, p2 + 256));
      tmp_dev.push_back(d_in2);
      CK(cudaMalloc(&d_out2, cap2));
      tmp_dev.push_back(d_out2);
      for (uint32_t k = 0; k < k2; k++) {
        const uint32_t i = again[k];
        CK(cudaMemcpyAsync(d_in2 + off2[k], src_base[i - b.f0] + src_off[i - b.f0], sz2[k], cudaMemcpyDeviceToDevice, ctx->stream));
      }
      lb2_stats b2;
      rc = enqueue_batch(ctx, ws, d_in2, off2.data(), sz2.data(), k2, d_out2, cap2, flags & 0xffu, ctx->stream, true);
      if (rc == LB2_OK) rc = collect_batch(ctx, ws, ooff2.data(), osz2.data(), st2.data(), &b2);
      if (rc == LB2_E_CAPACITY) { rc = LB2_OK; for (auto &x : st2) x = LB2_ST_UNSUPPORTED_LAYOUT; }  // hand them to the host strip
      if (rc) break;
      for (uint32_t k = 0; k < k2; k++) {
        const uint32_t i = again[k];
        status[i] = st2[k];
        if (st2[k] != LB2_ST_OK) continue;
        src_base[i - b.f0] = d_out2; src_off[i - b.f0] = ooff2[k]; out_sizes[i] = osz2[k];
      }
    }
    if (rc) break;
    t_gpu += now_s() - tg;
    // ---- download + write this batch, read + upload the next one
    down.clear(); up.clear();
    if (!dry) {
      // group by source buffer so that slices stay contiguous DMA ranges
      std::vector<uint8_t *> bases;
      for (uint32_t i = 0; i < m; i++) if (std::find(bases.begin(), bases.end(), src_base[i]) == bases.end()) bases.push_back(src_base[i]);
      for (uint8_t *base : bases) {
        std::vector<std::pair<uint64_t, uint32_t>> ord;
        for (uint32_t i = 0; i < m; i++)
          if (src_base[i] == base && status[b.f0 + i] == LB2_ST_OK) ord.push_back({src_off[i], b.f0 + i});
        std::sort(ord.begin(), ord.end());
        std::vector<uint32_t> ids;
        std::vector<uint64_t> o2, s2;
        for (auto &pr : ord) { ids.push_back(pr.second); o2.push_back(pr.first); s2.push_back(out_sizes[pr.second]); }
        const size_t seg_before = segs.size();
        make_slices(false, base, ids, o2.data(), s2.data(), E.slot_bytes, segs, down);
        for (size_t q = seg_before; q < segs.size(); q++) segs_left[segs[q].file]++;
        for (auto &pr : ord) {
          final_size[pr.second] = out_sizes[pr.second];
          if (out_sizes[pr.second] == 0) finish_file(pr.second);  // (cannot happen for a valid ELF; keeps the accounting total)
        }
      }
    } else {
      for (uint32_t i = b.f0; i < b.f1; i++) if (status[i] == LB2_ST_OK) { n_gpu++; in_b += files[i].size; out_b += out_sizes[i]; }
    }
    if (bi + 1 < batches.size()) rc = upload_slices(bi + 1, up);
    if (rc) break;
    submit_and_wait(down, up);
  }
  return rc;
  };
  rc = run_batches();
  stop_pool();
  cudaStreamSynchronize(ctx->stream);
  for (void *p : tmp_dev) cudaFree(p);
  st.gpu_s = t_gpu;
  st.read_cpu_s = ns_read.load() * 1e-9; st.write_cpu_s = ns_write.load() * 1e-9; st.dma_wait_s = ns_dma.load() * 1e-9;
  st.io_threads = (uint32_t)E.n_workers; st.n_batches = (uint32_t)batches.size();
  st.write_s = now_s() - t_io0 - t_gpu;  // read/upload and download/write overlap: I/O wall time next to the kernels
  if (rc) { if (st_out) *st_out = st; return rc; }

  t0 = now_s();
  std::vector<uint32_t> fallback;
  for (uint32_t i = 0; i < n; i++) if (status[i] != LB2_ST_OK) fallback.push_back(i);
  std::atomic<uint32_t> n_fb{0};
  parallel_for(fallback.size(), E.n_workers, [&](size_t k) {
    const uint32_t i = fallback[k];
    const bool non_elf = status[i] == LB2_ST_NOT_ELF;
    if (non_elf && (flags & LB2_TREE_TOLERATE_NON_ELF)) { n_skipped++; return; }
    if ((flags & LB2_TREE_FALLBACK_HOST_STRIP) && !dry) {
      // the reference's own tool decides (and fails the build exactly when the reference would)
      bool ok = true;
      for (uint32_t q = 0; q < files[i].times && ok; q++) ok = host_strip(files[i].path) == 0;
      if (ok) n_fb++; else n_failed++;
    } else {
      n_failed++;
    }
  });
  st.fallback_s = now_s() - t0;
  st.n_gpu = n_gpu; st.n_fallback = n_fb; st.n_failed += n_failed; st.n_skipped += n_skipped;
  st.in_bytes = in_b; st.out_bytes = out_b;
  if (st_out) *st_out = st;
  return LB2_OK;
}

// ---------------------------------------------------------------------------- corpus fill
int lb2_corpus_fill(lb2_ctx *ctx, void *d_arena, const lb2_fill_region *h_regions, uint32_t n_regions, uint64_t seed, void *stream) {
  if (!ctx || !d_arena || (!h_regions && n_regions)) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
  if (!n_regions) return LB2_OK;
  // split regions into <= 4 MB pieces so the grid balances
  std::vector<lb2_fill_region> pieces;
  const uint64_t P = 4ull << 20;
  for (uint32_t i = 0; i < n_regions; i++)
    for (uint64_t o = 0; o < h_regions[i].len; o += P) pieces.push_back({h_regions[i].offset + o, std::min(P, h_regions[i].len - o)});
  lb2_fill_region *d_regions = nullptr;
  CK(cudaMalloc(&d_regions, pieces.size() * sizeof(lb2_fill_region)));
  CK(cudaMemcpyAsync(d_regions, pieces.data(), pieces.size() * sizeof(lb2_fill_region), cudaMemcpyHostToDevice, s));
  launch_fill(static_cast<uint8_t *>(d_arena), reinterpret_cast<const FillRegion *>(d_regions), (uint32_t)pieces.size(), seed, ctx->sm_count * 8, s);
  CK(cudaStreamSynchronize(s));
  CK(cudaFree(d_regions));
  CK(cudaGetLastError());
  return LB2_OK;
}

int lb2_corpus_scatter(lb2_ctx *ctx, void *d_arena, const void *h_data, uint64_t data_bytes, const uint64_t *h_dst,
                       const uint64_t *h_src, const uint64_t *h_len, uint32_t n) {
  if (!ctx || !d_arena || (n && (!h_data || !h_dst || !h_src || !h_len))) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  if (!n) return LB2_OK;
  cudaStream_t s = ctx->stream;
  uint8_t *d_stage = nullptr;
  CK(cudaMalloc(&d_stage, data_bytes + 256));
  CK(cudaMemcpyAsync(d_stage, h_data, data_bytes, cudaMemcpyHostToDevice, s));
  std::vector<Tile> tiles;
  for (uint32_t i = 0; i < n; i++)
    for (uint64_t o = 0; o < h_len[i]; o += TILE_BYTES) {
      Tile t;
      t.src = reinterpret_cast<uint64_t>(d_stage) + h_src[i] + o;
      t.dst_rel = h_dst[i] + o;
      t.len = (uint32_t)std::min<uint64_t>(TILE_BYTES, h_len[i] - o);
      t.file = 0;
      tiles.push_back(t);
    }
  Tile *d_tiles = nullptr;
  BatchCounters *d_ctr = nullptr;
  uint64_t *d_off = nullptr;
  CK(cudaMalloc(&d_tiles, tiles.size() * sizeof(Tile)));
  CK(cudaMalloc(&d_ctr, sizeof(BatchCounters)));
  CK(cudaMalloc(&d_off, sizeof(uint64_t)));
  BatchCounters c;
  memset(&c, 0, sizeof c);
  c.n_tiles = tiles.size();
  uint64_t zero = 0;
  CK(cudaMemcpyAsync(d_tiles, tiles.data(), tiles.size() * sizeof(Tile), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_ctr, &c, sizeof c, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_off, &zero, sizeof zero, cudaMemcpyHostToDevice, s));
  CompactArgs ca;
  ca.tiles = d_tiles; ca.ctr = d_ctr; ca.out_off = d_off; ca.out = static_cast<uint8_t *>(d_arena);
  ca.rebase_lo = ca.rebase_len = ca.rebase_delta = 0;
  launch_compact(ca, ctx->sm_count * 4, s);
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  cudaFree(d_stage); cudaFree(d_tiles); cudaFree(d_ctr); cudaFree(d_off);
  return LB2_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- gzip: chunk concatenation, CRC combine, windows

// CRC-32 algebra (reflected polynomial 0xEDB88320): a * b mod P, and x^(8 n) mod P.  crc(A || B) =
// (x^(8 |B|) * crc(A)) ^ crc(B) for the standard (pre- and post-inverted) CRC.
static uint32_t crc_mulmod(uint32_t a, uint32_t b) {
  uint32_t p = 0;
  for (uint32_t m = 1u << 31; m; m >>= 1) {
    if (a & m) p ^= b;
    b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}
static uint32_t crc_shift(uint64_t nbytes) {
  uint32_t p = 1u << 31, sq = 1u << 23;
  for (; nbytes; nbytes >>= 1) {
    if (nbytes & 1) p = crc_mulmod(sq, p);
    sq = crc_mulmod(sq, sq);
  }
  return p;
}
static uint32_t crc_combine(uint32_t c1, uint32_t c2, uint64_t len2) {
  return len2 ? crc_mulmod(crc_shift(len2), c1) ^ c2 : c1;
}


static int deflate_reserve(lb2_ctx *ctx, uint64_t n_chunks) {
  auto &g = ctx->gz;
  if (!g.scratch) {
    deflate_smem_setup();
    CK(cudaGetLastError());
    g.grid = ctx->sm_count;   // ~210 KB of shared memory per CTA: one CTA per SM
    CK(cudaMalloc(&g.scratch, (size_t)g.grid * (DEFLATE_HIST + 2 * DEFLATE_CHUNK) * sizeof(uint32_t)));
    CK(cudaMalloc(&g.dists, (size_t)g.grid * DEFLATE_CHUNK * sizeof(uint16_t)));
    CK(cudaMalloc(&g.ctr, sizeof(BatchCounters)));
    CK(cudaMalloc(&g.out_off, sizeof(uint64_t)));
    CK(cudaMemset(g.out_off, 0, sizeof(uint64_t)));
    CK(cudaMalloc(&g.phase, DEFLATE_PHASES * sizeof(unsigned long long)));
    for (auto &e : g.ev) CK(cudaEventCreate(&e));
  }
  if (n_chunks > g.cap_chunks) {
    cudaFree(g.slots); cudaFree(g.size_crc); cudaFreeHost(g.h_size_crc); cudaFree(g.tiles);
    g.slots = nullptr; g.size_crc = nullptr; g.h_size_crc = nullptr; g.tiles = nullptr; g.cap_chunks = g.cap_tiles = 0;
    // a slot's bytes land at any offset of the stream, so they can touch one 16 KiB tile boundary more than
    // their length alone needs (a stored chunk, 65 551 bytes, can span 6 tiles)
    const uint64_t tiles_per_chunk = (DEFLATE_SLOT + TILE_BYTES - 1) / TILE_BYTES + 1;
    CK(cudaMalloc(&g.slots, n_chunks * DEFLATE_SLOT));
    CK(cudaMalloc(&g.size_crc, n_chunks * 2 * sizeof(uint32_t)));
    CK(cudaHostAlloc(&g.h_size_crc, n_chunks * 2 * sizeof(uint32_t), cudaHostAllocDefault));
    CK(cudaMalloc(&g.tiles, n_chunks * tiles_per_chunk * sizeof(Tile)));
    g.cap_chunks = n_chunks;
    g.cap_tiles = n_chunks * tiles_per_chunk;
  }
  return LB2_OK;
}

static int deflate_run(lb2_ctx *ctx, const uint8_t *d_in, uint64_t n, uint32_t hist, bool final_, uint8_t *d_out,
                       uint64_t cap, uint64_t *out_len, uint32_t *crc_out, lb2_gzip_stats *st, cudaStream_t s) {
  uint64_t nch = (n + DEFLATE_CHUNK - 1) / DEFLATE_CHUNK;
  if (!nch && final_) nch = 1;   // an empty final stream is one empty fixed block
  *out_len = 0;
  *crc_out = 0;
  if (!nch) return LB2_OK;
  int rc = deflate_reserve(ctx, nch);
  if (rc) return rc;
  auto &g = ctx->gz;
  DeflateArgs a;
  a.in = d_in; a.n = n; a.hist = std::min<uint32_t>(hist, DEFLATE_HIST); a.final_ = final_ ? 1 : 0;
  a.n_chunks = (uint32_t)nch;
  a.slots = g.slots; a.out_size = g.size_crc; a.chunk_crc = g.size_crc + nch;
  a.scratch = g.scratch; a.dists = g.dists; a.phase_cycles = g.phase;
  CK(cudaMemsetAsync(g.phase, 0, DEFLATE_PHASES * sizeof(unsigned long long), s));
  CK(cudaEventRecord(g.ev[0], s));
  launch_deflate(a, (int)std::min<uint64_t>(nch, (uint64_t)g.grid), s);
  CK(cudaGetLastError());
  CK(cudaEventRecord(g.ev[1], s));
  CK(cudaMemcpyAsync(g.h_size_crc, g.size_crc, nch * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  unsigned long long phase[DEFLATE_PHASES];
  CK(cudaMemcpyAsync(phase, g.phase, sizeof phase, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[1]));
  // exclusive scan of the slot sizes -> one tile list for the compaction kernel (the copy path of the strip)
  std::vector<Tile> tiles;
  tiles.reserve(nch * 5);
  uint64_t total = 0;
  for (uint64_t c = 0; c < nch; c++) {
    const uint64_t sz = g.h_size_crc[c];
    const uint64_t src = reinterpret_cast<uint64_t>(g.slots) + c * DEFLATE_SLOT;
    for (uint64_t k = 0; sz && k <= (total + sz - 1) / TILE_BYTES - total / TILE_BYTES; k++)
      tiles.push_back(extent_tile(src, total, sz, 0, (uint32_t)k));
    total += sz;
  }
  *out_len = total;
  if (total > cap) { ctx->err = "deflate: output capacity " + std::to_string(cap) + " < " + std::to_string(total); return LB2_E_CAPACITY; }
  if (!d_out && total) { ctx->err = "deflate: NULL output"; return LB2_E_ARG; }
  if (tiles.size() > g.cap_tiles) {   // cannot happen with the bound above; never write past the list
    ctx->err = "deflate: " + std::to_string(tiles.size()) + " concatenation tiles > " + std::to_string(g.cap_tiles);
    return LB2_E_STATE;
  }
  if (!tiles.empty()) {
    BatchCounters bc;
    memset(&bc, 0, sizeof bc);
    bc.n_tiles = tiles.size();
    CK(cudaMemcpyAsync(g.tiles, tiles.data(), tiles.size() * sizeof(Tile), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(g.ctr, &bc, sizeof bc, cudaMemcpyHostToDevice, s));
    CompactArgs ca;
    ca.tiles = g.tiles; ca.ctr = g.ctr; ca.out_off = g.out_off; ca.out = d_out;
    ca.rebase_lo = ca.rebase_len = ca.rebase_delta = 0;
    CK(cudaEventRecord(g.ev[0], s));
    launch_compact(ca, ctx->sm_count * 4, s);
    CK(cudaGetLastError());
    CK(cudaEventRecord(g.ev[1], s));
    CK(cudaStreamSynchronize(s));
    float ms2 = 0;
    CK(cudaEventElapsedTime(&ms2, g.ev[0], g.ev[1]));
    ms += ms2;
  }
  // chunks are DEFLATE_CHUNK bytes except the last: one fixed shift operator folds them
  const uint32_t op = crc_shift(DEFLATE_CHUNK);
  const uint32_t *cc = g.h_size_crc + nch;
  uint32_t crc = cc[0];
  for (uint64_t c = 1; c < nch; c++) {
    const uint64_t len = std::min<uint64_t>(DEFLATE_CHUNK, n - c * DEFLATE_CHUNK);
    crc = (len == DEFLATE_CHUNK ? crc_mulmod(op, crc) : crc_mulmod(crc_shift(len), crc)) ^ cc[c];
  }
  *crc_out = n ? crc : 0;
  if (st) {
    st->in_bytes += n; st->out_bytes += total; st->kernel_ms += ms; st->n_chunks += nch;
    for (int k = 0; k < DEFLATE_PHASES; k++) st->phase_cycles[k] += phase[k];
  }
  return LB2_OK;
}

// The concatenated segments of one lb2_gzip_segments call.  fill() is called from several I/O workers at once.
struct GzSource {
  const lb2_gz_segment *segs;
  uint32_t n_segs;
  std::vector<uint64_t> off;  // n_segs + 1 prefix sums
  // bytes [start, start + len) -> dst; "" or an error message
  std::string fill(uint8_t *dst, uint64_t start, uint64_t len) const {
    uint32_t i = (uint32_t)(std::upper_bound(off.begin(), off.end(), start) - off.begin()) - 1;
    uint64_t done = 0;
    for (; done < len && i < n_segs; i++) {
      const uint64_t in_seg = start + done - off[i];
      const uint64_t take = std::min(segs[i].len - in_seg, len - done);
      if (!take) continue;
      if (segs[i].data) {
        memcpy(dst + done, static_cast<const uint8_t *>(segs[i].data) + in_seg, take);
      } else {
        const int f = open(segs[i].path, O_RDONLY | O_CLOEXEC);
        if (f < 0) return std::string("open ") + segs[i].path + ": " + strerror(errno);
        const bool ok = pread_all(f, dst + done, take, in_seg);
        close(f);
        if (!ok) return std::string("short read (file changed since it was recorded?): ") + segs[i].path;
      }
      done += take;
    }
    return done == len ? "" : "segments shorter than their recorded total";
  }
};

// Bytes [start, start + len) of the source -> d_dst, through the tree engine's pinned slot ring: piece j
// (slot_bytes each) is read by I/O worker j % n_workers into one of its two slots and DMA'd on its stream.
// Returns LB2_OK, LB2_E_IO or LB2_E_CUDA (message in *err); *read_s += pread/memcpy time summed over workers.
static int gz_upload(lb2_ctx *ctx, const GzSource &src, uint64_t start, uint64_t len, uint8_t *d_dst, std::string *err,
                     double *read_s) {
  TreeEngine &E = *ctx->tree;
  const uint64_t sb = E.slot_bytes, n_pieces = (len + sb - 1) / sb;
  const int nw = (int)std::min<uint64_t>((uint64_t)E.n_workers, std::max<uint64_t>(1, n_pieces));
  std::vector<int> rc(nw, LB2_OK);
  std::vector<std::string> msg(nw);
  std::vector<double> rs(nw, 0.0);
  std::vector<std::thread> pool;
  for (int wi = 0; wi < nw; wi++)
    pool.emplace_back([&, wi] {
      cudaSetDevice(ctx->device);
      TreeWorker &w = E.workers[wi];
      for (uint64_t j = wi; j < n_pieces && rc[wi] == LB2_OK; j += nw) {
        uint8_t *slot = E.h_ring + ((uint64_t)wi * 2 + (w.k & 1)) * sb;
        cudaEvent_t ev = w.ev[w.k & 1];
        w.k++;
        if (cudaEventSynchronize(ev) != cudaSuccess) { rc[wi] = LB2_E_CUDA; msg[wi] = "gzip: slot DMA failed"; break; }
        const uint64_t o = j * sb, l = std::min(sb, len - o);
        const double t0 = now_s();
        msg[wi] = src.fill(slot, start + o, l);
        rs[wi] += now_s() - t0;
        if (!msg[wi].empty()) { rc[wi] = LB2_E_IO; break; }
        if (cudaMemcpyAsync(d_dst + o, slot, l, cudaMemcpyHostToDevice, w.stream) != cudaSuccess ||
            cudaEventRecord(ev, w.stream) != cudaSuccess) { rc[wi] = LB2_E_CUDA; msg[wi] = "gzip: slot DMA failed"; }
      }
      if (cudaStreamSynchronize(w.stream) != cudaSuccess && rc[wi] == LB2_OK) { rc[wi] = LB2_E_CUDA; msg[wi] = "gzip: slot DMA failed"; }
    });
  for (auto &t : pool) t.join();
  for (double r : rs) *read_s += r;
  for (int wi = 0; wi < nw; wi++)
    if (rc[wi] != LB2_OK) { *err = msg[wi]; return rc[wi]; }
  return LB2_OK;
}

static int grow_dev(lb2_ctx *ctx, uint8_t **p, uint64_t *cap, uint64_t need) {
  if (*cap >= need) return LB2_OK;
  cudaFree(*p); *p = nullptr; *cap = 0;
  CK(cudaMalloc(p, need));
  *cap = need;
  return LB2_OK;
}

extern "C" {

int lb2_deflate_device(lb2_ctx *ctx, const void *d_in, uint64_t n, uint32_t hist, uint32_t final_, void *d_out,
                       uint64_t cap, uint64_t *out_len, uint32_t *crc32, lb2_gzip_stats *stats, void *stream) {
  if (!ctx || (!d_in && (n || hist)) || !out_len || !crc32) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  if (stats) memset(stats, 0, sizeof *stats);
  cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
  int rc = deflate_run(ctx, static_cast<const uint8_t *>(d_in), n, hist, final_ != 0, static_cast<uint8_t *>(d_out), cap,
                       out_len, crc32, stats, s);
  if (stats) stats->n_windows = 1;
  return rc;
}

int lb2_gzip_segments(lb2_ctx *ctx, const lb2_gz_segment *segs, uint32_t n_segs, const char *out_path,
                      const void *gz_header, uint32_t gz_header_len, lb2_gzip_stats *stats) {
  if (!ctx || !out_path || (n_segs && !segs) || (gz_header_len && !gz_header)) { if (ctx) ctx->err = "NULL argument"; return LB2_E_ARG; }
  for (uint32_t i = 0; i < n_segs; i++)
    if (!segs[i].data && !segs[i].path && segs[i].len) { ctx->err = "segment without data or path"; return LB2_E_ARG; }
  CK(cudaSetDevice(ctx->device));
  lb2_gzip_stats st;
  memset(&st, 0, sizeof st);
  GzSource src{segs, n_segs, std::vector<uint64_t>(n_segs + 1, 0)};
  for (uint32_t i = 0; i < n_segs; i++) src.off[i + 1] = src.off[i] + segs[i].len;
  const uint64_t total = src.off[n_segs];
  uint64_t W = env_u64("LB2_GZ_WINDOW_MB", 1024) << 20;
  W = std::max<uint64_t>(DEFLATE_CHUNK, W / DEFLATE_CHUNK * DEFLATE_CHUNK);
  W = std::min<uint64_t>(W, std::max<uint64_t>(DEFLATE_CHUNK, (total + DEFLATE_CHUNK - 1) / DEFLATE_CHUNK * DEFLATE_CHUNK));
  const uint64_t n_win = std::max<uint64_t>(1, (total + W - 1) / W);
  const uint64_t out_cap = W / DEFLATE_CHUNK * DEFLATE_SLOT;
  constexpr uint64_t H_OUT = 64ull << 20;   // pinned bounce buffer of the compressed output
  cudaStream_t s = ctx->stream;
  auto &g = ctx->gz;

  int rc = LB2_OK;
  double t0 = now_s();
  if (!ctx->tree) rc = tree_engine_prepare(ctx, 0);
  for (int b = 0; rc == LB2_OK && b < (n_win > 1 ? 2 : 1); b++) rc = grow_dev(ctx, &g.d_win[b], &g.cap_win[b], DEFLATE_HIST + W);
  if (rc == LB2_OK) rc = grow_dev(ctx, &g.d_out, &g.cap_out, out_cap);
  if (rc == LB2_OK && !g.h_out) {
    cudaError_t e = cudaHostAlloc(&g.h_out, H_OUT, cudaHostAllocDefault);
    if (e != cudaSuccess) { ctx->err = std::string("cudaHostAlloc(gzip output): ") + cudaGetErrorString(e); rc = LB2_E_CUDA; }
    else g.cap_h_out = H_OUT;
  }
  st.setup_s = now_s() - t0;
  st.io_threads = ctx->tree ? (uint32_t)ctx->tree->n_workers : 0;
  if (rc != LB2_OK) { if (stats) *stats = st; return rc; }

  int fd = open(out_path, O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0644);
  if (fd < 0) { ctx->err = std::string("open ") + out_path + ": " + strerror(errno); if (stats) *stats = st; return LB2_E_IO; }
  auto fail = [&](int code, const std::string &m) { if (rc == LB2_OK) { if (!m.empty()) ctx->err = m; rc = code; } };
  std::thread uploader;
  int up_rc = LB2_OK;
  std::string up_err;
  double read_s = 0;
  do {
    uint64_t pos = 0;
    t0 = now_s();
    if (!pwrite_all(fd, static_cast<const uint8_t *>(gz_header), gz_header_len, 0)) { fail(LB2_E_IO, "write header"); break; }
    pos = gz_header_len;
    st.write_s += now_s() - t0;
    t0 = now_s();
    up_rc = gz_upload(ctx, src, 0, std::min(W, total), g.d_win[0] + DEFLATE_HIST, &up_err, &read_s);
    st.upload_s += now_s() - t0;
    if (up_rc != LB2_OK) { fail(up_rc, up_err); break; }
    uint32_t crc = 0;
    uint64_t prev_len = 0;
    for (uint64_t k = 0; k < n_win && rc == LB2_OK; k++) {
      const int b = (int)(k & 1);
      const uint64_t wlen = std::min(W, total - k * W);
      uint8_t *d_in = g.d_win[b] + DEFLATE_HIST;
      // the last 32 KiB of window k-1 become the history in front of window k
      const uint32_t hist = (uint32_t)std::min<uint64_t>(DEFLATE_HIST, k * W);
      cudaError_t e = cudaSuccess;
      if (hist && ((e = cudaMemcpyAsync(d_in - hist, g.d_win[1 - b] + DEFLATE_HIST + prev_len - hist, hist,
                                        cudaMemcpyDeviceToDevice, s)) != cudaSuccess ||
                   (e = cudaStreamSynchronize(s)) != cudaSuccess)) {
        fail(LB2_E_CUDA, std::string("gzip history copy: ") + cudaGetErrorString(e));
        break;
      }
      // window k+1 is read and uploaded (into the other buffer, behind the history copy above) while k is compressed
      if (k + 1 < n_win)
        uploader = std::thread([&, k, b] {
          cudaSetDevice(ctx->device);
          up_rc = gz_upload(ctx, src, (k + 1) * W, std::min(W, total - (k + 1) * W), g.d_win[1 - b] + DEFLATE_HIST, &up_err, &read_s);
        });
      uint64_t olen = 0;
      uint32_t wcrc = 0;
      int r = deflate_run(ctx, d_in, wlen, hist, k + 1 == n_win, g.d_out, out_cap, &olen, &wcrc, &st, s);
      if (r) fail(r, "");
      for (uint64_t o = 0; rc == LB2_OK && o < olen; o += g.cap_h_out) {
        const uint64_t l = std::min(g.cap_h_out, olen - o);
        t0 = now_s();
        if ((e = cudaMemcpyAsync(g.h_out, g.d_out + o, l, cudaMemcpyDeviceToHost, s)) != cudaSuccess ||
            (e = cudaStreamSynchronize(s)) != cudaSuccess) {
          fail(LB2_E_CUDA, std::string("gzip download: ") + cudaGetErrorString(e));
          break;
        }
        st.download_s += now_s() - t0;
        t0 = now_s();
        if (!pwrite_all(fd, g.h_out, l, pos + o)) fail(LB2_E_IO, std::string("write ") + out_path + ": " + strerror(errno));
        st.write_s += now_s() - t0;
      }
      pos += olen;
      crc = crc_combine(crc, wcrc, wlen);
      t0 = now_s();
      if (uploader.joinable()) uploader.join();
      st.upload_s += now_s() - t0;   // the part of the next window's upload the compression did not hide
      if (up_rc != LB2_OK) fail(up_rc, up_err);
      prev_len = wlen;
      st.n_windows++;
    }
    if (rc != LB2_OK) break;
    uint8_t trailer[8];
    const uint32_t isize = (uint32_t)total;
    for (int i = 0; i < 4; i++) { trailer[i] = (uint8_t)(crc >> (8 * i)); trailer[4 + i] = (uint8_t)(isize >> (8 * i)); }
    t0 = now_s();
    if (!pwrite_all(fd, trailer, 8, pos) || ftruncate(fd, (off_t)(pos + 8)) != 0) { fail(LB2_E_IO, "write trailer"); break; }
    st.write_s += now_s() - t0;
  } while (0);

  if (uploader.joinable()) uploader.join();
  if (close(fd) != 0) fail(LB2_E_IO, std::string("close ") + out_path + ": " + strerror(errno));
  if (rc != LB2_OK) unlink(out_path);
  st.read_s = read_s;
  if (stats) *stats = st;
  return rc;
}

}  // extern "C"
