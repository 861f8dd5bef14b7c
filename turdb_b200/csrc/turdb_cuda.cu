// turdb_cuda.cu — C ABI of libturdb_cuda.so (include/turdb_cuda.h).  sm_100a only.
#include "../../include/turdb_cuda.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "common.cuh"
#include "exact_search.cuh"
#include "gather_probe.cuh"
#include "search_kernels.h"

using namespace turdb;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int32_t fail(int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      int32_t _c = (_e == cudaErrorMemoryAllocation) ? TURDB_ERR_OUT_OF_MEMORY : TURDB_ERR_CUDA; \
      return fail(_c, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    }                                                                                        \
  } while (0)

static uint32_t ceil_log2(uint32_t v) {
  uint32_t b = 0;
  while (b < 31 && (1u << b) < v) ++b;
  return b;
}

// ------------------------------------------------------------------------------------------
// index
// ------------------------------------------------------------------------------------------
struct turdb_cuda_index {
  int device = 0;
  int num_sms = 0;
  int max_smem_optin = 0;
  DeviceIndex ix{};
  float* d_arena = nullptr;
  float* d_norm2 = nullptr;
  uint32_t* d_l0_adj = nullptr;
  uint32_t* d_up_base = nullptr;
  uint32_t* d_up_adj = nullptr;
  uint64_t* d_row_ids = nullptr;
  uint8_t* d_levels = nullptr;
  // per-list state the insert path's link kernels append to (graph_insert.inl): valid entries of each level-0 / upper
  // list and the node owning each upper slot; kept for the index's lifetime so that later inserts can back-link
  uint8_t* d_l0_cnt = nullptr;
  uint8_t* d_up_cnt = nullptr;
  uint32_t* d_up_owner = nullptr;
  uint64_t cap_n = 0, cap_slots = 0;       // allocated nodes / upper slots of every per-node / per-slot array (>= n, n_up_slots)
  uint8_t* d_arena_sq8 = nullptr;          // SQ8 rows: dim codes | pad | min | scale, sq8_row_bytes apart (enable_sq8)
  float* d_norm2_sq8 = nullptr;            // dot(decode(x), decode(x)) per row, AVX2 lane order
  uint32_t sq8_row_bytes = 0;
  uint16_t* d_arena_bf16 = nullptr;        // exact path operand (raw rows: L2, IP), 16-bit (FP16 or BF16), built lazily
  uint16_t* d_arena_bf16n = nullptr;       // exact path operand (rows scaled by 1/|x|: cosine), FP16, built lazily
  uint16_t* d_arena_bf16l2 = nullptr;      // exact path operand for L2: raw rows + three columns holding -|x|^2/2 (hi/mid/lo
                                           // 16-bit split, divided by l2_scale), so that the contraction itself yields the key
  int half_fp16[3] = {0, 1, 0};            // format of the copies (raw, cosine, L2): 1 FP16, 0 BF16
  float l2_scale = 1.f;                    // power of two the L2 copy's bias columns are divided by (the query side carries it)
  uint32_t* d_bf16_max2 = nullptr;         // [3 copies][2]: max |v - bf16(v)|_2, max |bf16(v)|_2 over rows (float bits); [6]: max
                                           // |value|; [7]: max |x|^2
  uint64_t* d_live = nullptr;              // turdb_cuda_index_delete: one bit per node, (cap_n + 63) / 64 words; null until the
                                           // first delete (ix.live points to it)
  uint64_t n_deleted = 0;                  // nodes in [0, n) whose live bit is clear
  cudaMemPool_t pool = nullptr;            // per-index stream-ordered scratch pool (never trimmed)
  uint64_t device_bytes = 0;
  uint64_t n_up_slots = 0;
  uint32_t tune_warps = 0, tune_slots = 0, tune_hash_bits = 0, tune_segs = 0;
  uint32_t tune_mode = 0;                  // 0 automatic, 1 staged (team + TMA staging), 2 direct (one warp per query)
  // visited-set sizing: running maximum of keys per query, one counter per ceil(log2(ef)) (device + pinned mirror
  // refreshed by an async copy after every launch; the next launch sizes its shared-memory table from it)
  TraversalStats* d_tstats = nullptr;
  TraversalStats* h_tstats = nullptr;
  // profiling ring: 3 events per call (before main, after main, after overflow pass)
  std::vector<cudaEvent_t> prof_events;
  uint32_t prof_capacity = 0, prof_used = 0;
  unsigned long long* d_dbg = nullptr;  // diagnostics: per-phase cycle counters of the traversal kernel
  std::mutex mu;
};

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// One warp per adjacency row: entries >= count become INVALID, ids are range-checked, and a repeated id
// keeps only its first occurrence (the reference's visited set skips the repeats, search.rs:338, so the
// traversal is unchanged; the kernel's lock-free visited table relies on rows without repeats).  The row is
// re-packed to a prefix in stored order, and cnt[r] becomes the number of ids it keeps.
__global__ void sanitize_adj_kernel(uint32_t* adj, uint8_t* cnt, uint64_t rows, uint32_t width,
                                    uint64_t n, uint32_t* bad) {
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (r >= rows) return;
  const uint32_t limit = min((uint32_t)cnt[r], width);
  uint32_t v = (lane < limit) ? adj[r * width + lane] : kInvalid;
  if (v != kInvalid && v >= n) {
    atomicAdd(bad, 1u);
    v = kInvalid;
  }
  bool keep = v != kInvalid;
  for (uint32_t j = 0; j < width; ++j) {
    const uint32_t o = __shfl_sync(kFullMask, v, j);
    if (j < lane && o == v) keep = false;
  }
  const uint32_t km = __ballot_sync(kFullMask, keep);
  if (lane < width) adj[r * width + lane] = kInvalid;
  __syncwarp();
  if (keep) adj[r * width + __popc(km & ((1u << lane) - 1))] = v;
  if (lane == 0) cnt[r] = (uint8_t)__popc(km);
}

// up_owner[up_base[i] + l] = i for l < levels[i] (slots no node claims keep what they held)
__global__ void up_owner_kernel(const uint8_t* levels, const uint32_t* up_base, uint64_t n, uint32_t first,
                                uint32_t* up_owner) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (uint32_t l = 0; l < levels[i]; ++l) up_owner[(size_t)up_base[i] + l] = first + (uint32_t)i;
}

// dot(b, b) per arena row in the reference's AVX2 lane order (cosine_avx2's norm_b chain)
__global__ void norm2_kernel(const float* arena, uint32_t dim, uint32_t ds, uint64_t n, float* out) {
  uint64_t quad = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  uint64_t row = quad < n ? quad : n - 1;  // keep the quad shuffles converged
  const float* b = arena + row * ds;
  float r = quad_dot(b, b, dim, threadIdx.x & 3);
  if (quad < n && (threadIdx.x & 3) == 0) out[quad] = r;
}

// SQ8Vector::from_f32 (src/hnsw/quantization.rs:68-95), one warp per row: min / max over the row, scale =
// range / 255 (1.0 when the row is constant), code = round((v - min) / scale) clamped to 0..255 (`round` = half
// away from zero, like f32::round).  Row layout: dim codes | pad to 4 | min f32 | scale f32, row_bytes apart.
__global__ void sq8_encode_kernel(const float* arena, uint32_t dim, uint32_t ds, uint64_t n, uint8_t* out, uint32_t row_bytes) {
  const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (r >= n) return;
  const float* v = arena + r * ds;
  float mn = INFINITY, mx = -INFINITY;
  for (uint32_t i = lane; i < dim; i += 32) {
    mn = fminf(mn, v[i]);
    mx = fmaxf(mx, v[i]);
  }
  for (uint32_t off = 16; off >= 1; off >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(kFullMask, mn, off));
    mx = fmaxf(mx, __shfl_xor_sync(kFullMask, mx, off));
  }
  const float range = __fsub_rn(mx, mn);
  const float scale = range > 0.f ? __fdiv_rn(range, 255.0f) : 1.0f;
  uint8_t* row = out + r * row_bytes;
  for (uint32_t i = lane; i < dim; i += 32) {
    float c = 0.f;
    if (range != 0.f) c = fminf(fmaxf(roundf(__fdiv_rn(__fsub_rn(v[i], mn), scale)), 0.f), 255.f);
    row[i] = (uint8_t)c;
  }
  const uint32_t tail = (dim + 3) & ~3u;
  for (uint32_t i = dim + lane; i < tail; i += 32) row[i] = 0;
  if (lane == 0) {
    float* ms = reinterpret_cast<float*>(row + tail);
    ms[0] = mn;
    ms[1] = scale;
  }
  for (uint32_t i = tail + 8 + lane; i < row_bytes; i += 32) row[i] = 0;
}

__global__ void sq8_norm2_kernel(const uint8_t* rows, uint32_t dim, uint32_t row_bytes, uint64_t n, float* out) {
  uint64_t quad = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  uint64_t row = quad < n ? quad : n - 1;  // keep the quad shuffles converged
  float r = quad_sq8<2>(nullptr, rows + row * row_bytes, dim, threadIdx.x & 3);
  if (quad < n && (threadIdx.x & 3) == 0) out[quad] = r;
}

// live bitmap (turdb_cuda_index_delete): bits [lo, hi) set, one thread per word
__global__ void live_set_kernel(uint64_t* live, uint64_t lo, uint64_t hi) {
  const uint64_t w = lo / 64 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w * 64 >= hi) return;
  const uint64_t a = max(lo, w * 64), b = min(hi, w * 64 + 64);
  const uint64_t run = b - a == 64 ? ~0ull : (1ull << (b - a)) - 1ull;
  live[w] |= run << (a - w * 64);
}

// clears the bits of ids[0, n); *cleared counts the bits that were set (a repeated id clears nothing the second time)
__global__ void live_clear_kernel(uint64_t* live, const uint32_t* __restrict__ ids, uint64_t n, unsigned long long* cleared) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t id = ids[i];
  const unsigned long long bit = 1ull << (id & 63);
  if (atomicAnd(reinterpret_cast<unsigned long long*>(live) + (id >> 6), ~bit) & bit) atomicAdd(cleared, 1ull);
}

__global__ void live_and_kernel(const uint64_t* __restrict__ a, const uint64_t* __restrict__ b, uint64_t words, uint64_t* out) {
  const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < words) out[w] = a[w] & b[w];
}

extern "C" {

uint32_t turdb_cuda_abi_version(void) { return TURDB_CUDA_ABI_VERSION; }

const char* turdb_cuda_last_error(void) { return g_last_error.c_str(); }

int32_t turdb_cuda_device_count(int32_t* out_count) {
  if (!out_count) return fail(TURDB_ERR_INVALID_ARGUMENT, "out_count is null");
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess) {
    *out_count = 0;
    return fail(TURDB_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  }
  *out_count = c;
  return TURDB_OK;
}

int32_t turdb_cuda_index_destroy(turdb_cuda_index* idx) {
  if (!idx) return TURDB_OK;
  {
    DeviceGuard g(idx->device);
    cudaFree(idx->d_arena);
    cudaFree(idx->d_norm2);
    cudaFree(idx->d_l0_adj);
    cudaFree(idx->d_up_base);
    cudaFree(idx->d_up_adj);
    cudaFree(idx->d_row_ids);
    cudaFree(idx->d_levels);
    cudaFree(idx->d_l0_cnt);
    cudaFree(idx->d_up_cnt);
    cudaFree(idx->d_up_owner);
    cudaFree(idx->d_arena_sq8);
    cudaFree(idx->d_norm2_sq8);
    cudaFree(idx->d_arena_bf16);
    cudaFree(idx->d_arena_bf16n);
    cudaFree(idx->d_arena_bf16l2);
    cudaFree(idx->d_bf16_max2);
    cudaFree(idx->d_live);
    for (cudaEvent_t ev : idx->prof_events) cudaEventDestroy(ev);
    cudaFree(idx->d_dbg);
    cudaFree(idx->d_tstats);
    if (idx->h_tstats) cudaFreeHost(idx->h_tstats);
    if (idx->pool) cudaMemPoolDestroy(idx->pool);
  }
  delete idx;
  return TURDB_OK;
}

int32_t turdb_cuda_index_create(const turdb_cuda_graph* g, int32_t device, turdb_cuda_index** out) {
  if (!g || !out) return fail(TURDB_ERR_INVALID_ARGUMENT, "graph/out is null");
  *out = nullptr;
  if (g->dim == 0 || g->dim > 65535) return fail(TURDB_ERR_INVALID_ARGUMENT, "dim %u out of range", g->dim);
  if (g->n >= 0x7FFFFFFFull) return fail(TURDB_ERR_UNSUPPORTED, "n %llu exceeds 2^31-2 nodes per index", (unsigned long long)g->n);
  if (g->n > 0) {
    if (!g->vectors || !g->row_ids || !g->levels || !g->l0_adj || !g->l0_cnt || !g->up_base)
      return fail(TURDB_ERR_INVALID_ARGUMENT, "graph array pointer is null");
    if (g->n_up_slots && (!g->up_adj || !g->up_cnt))
      return fail(TURDB_ERR_INVALID_ARGUMENT, "upper-level arrays are null");
    if (g->entry != TURDB_INVALID_NODE && g->entry >= g->n)
      return fail(TURDB_ERR_INVALID_ARGUMENT, "entry %u >= n", g->entry);
    if (g->entry != TURDB_INVALID_NODE && g->levels[g->entry] < g->max_level)
      return fail(TURDB_ERR_INVALID_ARGUMENT, "entry level %u < max_level %u", g->levels[g->entry], g->max_level);
    for (uint64_t i = 0; i < g->n; ++i) {
      if (g->levels[i] > 0) {
        if (g->up_base[i] == TURDB_INVALID_NODE || (uint64_t)g->up_base[i] + g->levels[i] > g->n_up_slots)
          return fail(TURDB_ERR_INVALID_ARGUMENT, "node %llu: upper slots out of range", (unsigned long long)i);
      }
    }
  }
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
    return fail(TURDB_ERR_NO_DEVICE, "no CUDA device available (libturdb_cuda has no CPU fallback)");
  if (device < 0 || device >= count) return fail(TURDB_ERR_INVALID_ARGUMENT, "device %d out of range", device);
  DeviceGuard guard(device);
  if (!guard.ok) return fail(TURDB_ERR_CUDA, "cudaSetDevice(%d) failed", device);

  turdb_cuda_index* idx = new (std::nothrow) turdb_cuda_index();
  if (!idx) return fail(TURDB_ERR_OUT_OF_MEMORY, "host allocation failed");
  idx->device = device;
  cudaDeviceProp prop{};
  cudaGetDeviceProperties(&prop, device);
  idx->num_sms = prop.multiProcessorCount;
  idx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  if (prop.major < 10) {
    delete idx;
    return fail(TURDB_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  }

  {
    cudaMemPoolProps pp{};
    pp.allocType = cudaMemAllocationTypePinned;
    pp.handleTypes = cudaMemHandleTypeNone;
    pp.location.type = cudaMemLocationTypeDevice;
    pp.location.id = device;
    if (cudaMemPoolCreate(&idx->pool, &pp) != cudaSuccess) {
      delete idx;
      return fail(TURDB_ERR_CUDA, "cudaMemPoolCreate failed");
    }
    uint64_t keep = ~0ull;  // keep freed scratch cached across synchronisations
    cudaMemPoolSetAttribute(idx->pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  if (cudaMalloc(&idx->d_tstats, 16 * sizeof(TraversalStats)) != cudaSuccess ||
      cudaMemset(idx->d_tstats, 0, 16 * sizeof(TraversalStats)) != cudaSuccess ||
      cudaMallocHost(&idx->h_tstats, 16 * sizeof(TraversalStats)) != cudaSuccess) {
    turdb_cuda_index_destroy(idx);
    return fail(TURDB_ERR_OUT_OF_MEMORY, "traversal statistics allocation failed");
  }
  memset(idx->h_tstats, 0, 16 * sizeof(TraversalStats));
  const uint64_t n = g->n;
  const uint32_t dim = g->dim, ds = (dim + 3) & ~3u;
  idx->ix.n = n;
  idx->ix.dim = dim;
  idx->ix.ds = ds;
  idx->ix.entry = n ? g->entry : kInvalid;
  idx->ix.max_level = g->max_level;

#define IDX_TRY(expr)                                                          \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) {                                                   \
      int32_t _c = (_e == cudaErrorMemoryAllocation) ? TURDB_ERR_OUT_OF_MEMORY : TURDB_ERR_CUDA; \
      fail(_c, "%s failed: %s", #expr, cudaGetErrorString(_e));                \
      turdb_cuda_index_destroy(idx);                                           \
      return _c;                                                               \
    }                                                                          \
  } while (0)

  if (n > 0) {
    const size_t arena_bytes = (size_t)n * ds * 4;
    IDX_TRY(cudaMalloc(&idx->d_arena, arena_bytes));
    if (ds == dim) {
      IDX_TRY(cudaMemcpy(idx->d_arena, g->vectors, arena_bytes, cudaMemcpyHostToDevice));
    } else {
      IDX_TRY(cudaMemset(idx->d_arena, 0, arena_bytes));
      IDX_TRY(cudaMemcpy2D(idx->d_arena, (size_t)ds * 4, g->vectors, (size_t)dim * 4, (size_t)dim * 4, n,
                           cudaMemcpyHostToDevice));
    }
    IDX_TRY(cudaMalloc(&idx->d_norm2, n * 4));
    IDX_TRY(cudaMalloc(&idx->d_l0_adj, n * kL0 * 4));
    IDX_TRY(cudaMemcpy(idx->d_l0_adj, g->l0_adj, n * kL0 * 4, cudaMemcpyHostToDevice));
    IDX_TRY(cudaMalloc(&idx->d_up_base, n * 4));
    IDX_TRY(cudaMemcpy(idx->d_up_base, g->up_base, n * 4, cudaMemcpyHostToDevice));
    IDX_TRY(cudaMalloc(&idx->d_row_ids, n * 8));
    IDX_TRY(cudaMemcpy(idx->d_row_ids, g->row_ids, n * 8, cudaMemcpyHostToDevice));
    IDX_TRY(cudaMalloc(&idx->d_levels, n));
    IDX_TRY(cudaMemcpy(idx->d_levels, g->levels, n, cudaMemcpyHostToDevice));
    const uint64_t slots = g->n_up_slots;
    IDX_TRY(cudaMalloc(&idx->d_up_adj, std::max<uint64_t>(slots, 1) * kUp * 4));
    if (slots) IDX_TRY(cudaMemcpy(idx->d_up_adj, g->up_adj, slots * kUp * 4, cudaMemcpyHostToDevice));
    IDX_TRY(cudaMalloc(&idx->d_l0_cnt, n));
    IDX_TRY(cudaMalloc(&idx->d_up_cnt, std::max<uint64_t>(slots, 1)));
    IDX_TRY(cudaMalloc(&idx->d_up_owner, std::max<uint64_t>(slots, 1) * 4));
    idx->device_bytes = arena_bytes + n * 4 + n * kL0 * 4 + n * 4 + n * 8 + n + slots * kUp * 4 + n + slots * 5;
    idx->n_up_slots = slots;
    idx->cap_n = n;
    idx->cap_slots = slots;

    // counts -> INVALID padding, id range check; the counts kept are those of the sanitised rows
    uint32_t* d_bad = nullptr;
    IDX_TRY(cudaMalloc(&d_bad, 4));
    IDX_TRY(cudaMemset(d_bad, 0, 4));
    IDX_TRY(cudaMemcpy(idx->d_l0_cnt, g->l0_cnt, n, cudaMemcpyHostToDevice));
    sanitize_adj_kernel<<<(unsigned)((n * 32 + 255) / 256), 256>>>(idx->d_l0_adj, idx->d_l0_cnt, n, kL0, n, d_bad);
    if (slots) {
      IDX_TRY(cudaMemcpy(idx->d_up_cnt, g->up_cnt, slots, cudaMemcpyHostToDevice));
      sanitize_adj_kernel<<<(unsigned)((slots * 32 + 255) / 256), 256>>>(idx->d_up_adj, idx->d_up_cnt, slots, kUp, n, d_bad);
      IDX_TRY(cudaMemset(idx->d_up_owner, 0xFF, slots * 4));
      up_owner_kernel<<<(unsigned)((n + 255) / 256), 256>>>(idx->d_levels, idx->d_up_base, n, 0, idx->d_up_owner);
    }
    norm2_kernel<<<(unsigned)((n * 4 + 255) / 256), 256>>>(idx->d_arena, dim, ds, n, idx->d_norm2);
    uint32_t bad = 0;
    IDX_TRY(cudaMemcpy(&bad, d_bad, 4, cudaMemcpyDeviceToHost));
    cudaFree(d_bad);
    IDX_TRY(cudaGetLastError());
    if (bad) {
      turdb_cuda_index_destroy(idx);
      return fail(TURDB_ERR_INVALID_ARGUMENT, "%u adjacency entries reference nodes >= n", bad);
    }
  }
#undef IDX_TRY
  idx->ix.arena = idx->d_arena;
  idx->ix.norm2 = idx->d_norm2;
  idx->ix.l0_adj = idx->d_l0_adj;
  idx->ix.up_base = idx->d_up_base;
  idx->ix.up_adj = idx->d_up_adj;
  idx->ix.row_ids = idx->d_row_ids;
  idx->ix.levels = idx->d_levels;
  *out = idx;
  return TURDB_OK;
}

int32_t turdb_cuda_index_enable_sq8(turdb_cuda_index* idx, uint8_t* out_rows, uint64_t out_capacity, uint32_t* out_row_bytes) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  DeviceGuard guard(idx->device);
  if (!guard.ok) return fail(TURDB_ERR_CUDA, "cudaSetDevice(%d) failed", idx->device);
  std::lock_guard<std::mutex> lk(idx->mu);
  const uint64_t n = idx->ix.n;
  const uint32_t dim = idx->ix.dim;
  const uint32_t row_bytes = (((dim + 3) & ~3u) + 8 + 15) & ~15u;
  if (!idx->d_arena_sq8 && n) {
    const uint64_t cap = idx->cap_n;  // sized like the arena: turdb_cuda_index_insert encodes appended rows in place
    CUDA_TRY(cudaMalloc(&idx->d_arena_sq8, cap * row_bytes));
    CUDA_TRY(cudaMalloc(&idx->d_norm2_sq8, cap * 4));
    sq8_encode_kernel<<<(unsigned)((n * 32 + 255) / 256), 256>>>(idx->d_arena, dim, idx->ix.ds, n, idx->d_arena_sq8, row_bytes);
    sq8_norm2_kernel<<<(unsigned)((n * 4 + 255) / 256), 256>>>(idx->d_arena_sq8, dim, row_bytes, n, idx->d_norm2_sq8);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
    idx->device_bytes += cap * row_bytes + cap * 4;
  }
  idx->sq8_row_bytes = row_bytes;
  if (out_row_bytes) *out_row_bytes = row_bytes;
  if (out_rows) {
    if (out_capacity < n * row_bytes) return fail(TURDB_ERR_INVALID_ARGUMENT, "out_rows holds %llu bytes, need %llu", (unsigned long long)out_capacity, (unsigned long long)(n * row_bytes));
    if (n) CUDA_TRY(cudaMemcpy(out_rows, idx->d_arena_sq8, n * row_bytes, cudaMemcpyDeviceToHost));
  }
  return TURDB_OK;
}

int32_t turdb_cuda_index_info(const turdb_cuda_index* idx, uint64_t* n, uint32_t* dim, uint32_t* max_level,
                              uint32_t* entry, uint64_t* device_bytes) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  if (n) *n = idx->ix.n;
  if (dim) *dim = idx->ix.dim;
  if (max_level) *max_level = idx->ix.max_level;
  if (entry) *entry = idx->ix.entry;
  if (device_bytes) *device_bytes = idx->device_bytes;
  return TURDB_OK;
}

// Deletion is state of the index: the live bitmap, allocated by the first delete at the node capacity (insert keeps it
// in step), every node of [0, n) set, then the deleted bits cleared.  Node ids, rows and graph stay as they are.
int32_t turdb_cuda_index_delete(turdb_cuda_index* idx, uint64_t n, const uint32_t* node_ids, uint64_t* out_n_deleted) {
  if (n && !node_ids) return fail(TURDB_ERR_INVALID_ARGUMENT, "node_ids is null");
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  const uint64_t n_nodes = idx->ix.n;
  for (uint64_t i = 0; i < n; ++i)
    if (node_ids[i] >= n_nodes)
      return fail(TURDB_ERR_INVALID_ARGUMENT, "node_ids[%llu] = %u >= n = %llu", (unsigned long long)i, node_ids[i],
                  (unsigned long long)n_nodes);
  if (n) {
    DeviceGuard guard(idx->device);
    if (!guard.ok) return fail(TURDB_ERR_CUDA, "cudaSetDevice(%d) failed", idx->device);
    const uint64_t words = (idx->cap_n + 63) / 64;
    uint64_t* fresh = nullptr;
    if (!idx->d_live) CUDA_TRY(cudaMalloc(&fresh, words * 8));
    else CUDA_TRY(cudaDeviceSynchronize());  // the bits change in place: work enqueued earlier, on any stream, reads them first
    uint64_t* live = fresh ? fresh : idx->d_live;
    cudaStream_t stream = nullptr;
    uint8_t* scr = nullptr;  // ids | cleared count
    const size_t off_cnt = (n * 4 + 15) & ~(size_t)15;
    unsigned long long cleared = 0;
    cudaError_t e = cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMallocFromPoolAsync(&scr, off_cnt + 8, idx->pool, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(scr, node_ids, n * 4, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(scr + off_cnt, 0, 8, stream);
    if (e == cudaSuccess && fresh) {
      e = cudaMemsetAsync(fresh, 0, words * 8, stream);
      live_set_kernel<<<(unsigned)((n_nodes + 64 * 256 - 1) / (64 * 256)), 256, 0, stream>>>(fresh, 0, n_nodes);
    }
    if (e == cudaSuccess) {
      live_clear_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(live, (const uint32_t*)scr, n,
                                                                         (unsigned long long*)(scr + off_cnt));
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&cleared, scr + off_cnt, 8, cudaMemcpyDeviceToHost, stream);
    if (scr) cudaFreeAsync(scr, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (stream) cudaStreamDestroy(stream);
    if (e != cudaSuccess) {
      cudaFree(fresh);
      return fail(e == cudaErrorMemoryAllocation ? TURDB_ERR_OUT_OF_MEMORY : TURDB_ERR_CUDA, "delete failed: %s",
                  cudaGetErrorString(e));
    }
    std::lock_guard<std::mutex> lk(idx->mu);
    if (fresh) {
      idx->d_live = fresh;
      idx->ix.live = fresh;
      idx->device_bytes += words * 8;
    }
    idx->n_deleted += cleared;
  }
  if (out_n_deleted) *out_n_deleted = idx->n_deleted;
  return TURDB_OK;
}

int32_t turdb_cuda_index_set_tuning(turdb_cuda_index* idx, uint32_t warps_per_cta, uint32_t staging_slots,
                                    uint32_t hash_bits, uint32_t segments) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  if (warps_per_cta > 4) return fail(TURDB_ERR_INVALID_ARGUMENT, "warps_per_cta must be <= 4");
  if (staging_slots > 32 || (staging_slots & 7)) return fail(TURDB_ERR_INVALID_ARGUMENT, "staging_slots must be 0, 8, 16, 24 or 32");
  if (hash_bits != 0 && (hash_bits < 8 || hash_bits > 15)) return fail(TURDB_ERR_INVALID_ARGUMENT, "hash_bits must be 0 or 8..15");
  if (segments > 16) return fail(TURDB_ERR_INVALID_ARGUMENT, "segments must be <= 16");
  std::lock_guard<std::mutex> lk(idx->mu);
  idx->tune_warps = warps_per_cta;
  idx->tune_slots = staging_slots;
  idx->tune_hash_bits = hash_bits;
  idx->tune_segs = segments;
  return TURDB_OK;
}

int32_t turdb_cuda_index_set_traversal_form(turdb_cuda_index* idx, uint32_t form) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  if (form > 2) return fail(TURDB_ERR_INVALID_ARGUMENT, "form must be 0 (automatic), 1 (staged) or 2 (direct)");
  std::lock_guard<std::mutex> lk(idx->mu);
  idx->tune_mode = form;
  return TURDB_OK;
}

int32_t turdb_cuda_index_debug_counters(turdb_cuda_index* idx, int32_t enable, uint64_t* out16) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  DeviceGuard guard(idx->device);
  std::lock_guard<std::mutex> lk(idx->mu);
  if (out16 && idx->d_dbg) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(out16, idx->d_dbg, 16 * 8, cudaMemcpyDeviceToHost));
  } else if (out16) {
    memset(out16, 0, 16 * 8);
  }
  if (enable && !idx->d_dbg) CUDA_TRY(cudaMalloc(&idx->d_dbg, 16 * 8));
  if (enable) CUDA_TRY(cudaMemset(idx->d_dbg, 0, 16 * 8));
  if (!enable && idx->d_dbg) {
    cudaFree(idx->d_dbg);
    idx->d_dbg = nullptr;
  }
  return TURDB_OK;
}

int32_t turdb_cuda_index_profile_begin(turdb_cuda_index* idx, uint32_t capacity) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  if (capacity > 4096) return fail(TURDB_ERR_INVALID_ARGUMENT, "capacity > 4096");
  DeviceGuard guard(idx->device);
  std::lock_guard<std::mutex> lk(idx->mu);
  while (idx->prof_events.size() < (size_t)capacity * 3) {
    cudaEvent_t ev;
    CUDA_TRY(cudaEventCreate(&ev));
    idx->prof_events.push_back(ev);
  }
  idx->prof_capacity = capacity;
  idx->prof_used = 0;
  return TURDB_OK;
}

int32_t turdb_cuda_index_profile_read(turdb_cuda_index* idx, float* main_ms, float* overflow_ms, uint32_t cap,
                                      uint32_t* out_n) {
  if (!idx || !out_n) return fail(TURDB_ERR_INVALID_ARGUMENT, "null argument");
  DeviceGuard guard(idx->device);
  std::lock_guard<std::mutex> lk(idx->mu);
  uint32_t n = std::min(idx->prof_used, cap);
  for (uint32_t i = 0; i < n; ++i) {
    float a = 0.f, b = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&a, idx->prof_events[3 * i], idx->prof_events[3 * i + 1]));
    CUDA_TRY(cudaEventElapsedTime(&b, idx->prof_events[3 * i + 1], idx->prof_events[3 * i + 2]));
    if (main_ms) main_ms[i] = a;
    if (overflow_ms) overflow_ms[i] = b;
  }
  *out_n = n;
  idx->prof_capacity = 0;
  idx->prof_used = 0;
  return TURDB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// traversal launch
// ------------------------------------------------------------------------------------------
// n_slots == 0: the direct form (one warp per query, no staging)
static TeamLayout make_layout(uint32_t dim, uint32_t ds, uint32_t ef, uint32_t hash_bits, uint32_t n_slots, uint32_t n_segs,
                              bool global_visited, uint64_t n_nodes, bool filtered = false, uint32_t sq8_row_bytes = 0,
                              bool entries32 = false) {
  TeamLayout L{};
  L.vec_bytes = sq8_row_bytes ? sq8_row_bytes : ds * 4;
  const uint32_t steps = dim >> 3;
  if (sq8_row_bytes || n_slots == 0) n_segs = 1;  // code rows are never split
  n_segs = std::max(1u, std::min(n_segs, std::max(1u, steps)));
  L.seg_steps = steps ? (steps + n_segs - 1) / n_segs : 0;
  L.n_segs = L.seg_steps ? (steps + L.seg_steps - 1) / L.seg_steps : 1;
  const uint32_t slot_words = sq8_row_bytes ? sq8_row_bytes / 4 : L.seg_steps * 8 + (ds - steps * 8);  // one piece + the < 8-element tail
  const uint32_t pad_words = (8 + 32 - (slot_words & 31)) & 31;
  L.stride = (slot_words + pad_words) * 4;
  L.hash_bits = hash_bits;
  L.n_groups = n_slots / 8;
  L.key_bits = std::max(hash_bits, ceil_log2((uint32_t)std::max<uint64_t>(n_nodes, 2)));
  L.rem_bits = L.key_bits - hash_bits;
  L.hash16 = (!global_visited && !entries32 && L.rem_bits <= 11) ? 1u : 0u;  // displacement field >= 5 bits
  // [0] mbarriers, [32] control words, [64] cand_ids[32] cand_d[32] tmp_ub[32] cand_next[32], [576] result list: fixed
  // offsets (kOffBar .. kOffList); then the filtered window, the query, the visited table, the staging slots
  uint32_t off = kOffList;
  off += filtered ? ef * 16 : ef * 8;  // result list (x2: the filtered search double-buffers it)
  L.off_clist = off; off += filtered ? ef * 16 : 0;       // search_filtered: candidate window (double-buffered)
  off = (off + 15) & ~15u;
  L.off_q = off;     off += (ds * 4 + 15) & ~15u;
  L.off_hash = off;  off += global_visited ? 0 : ((L.hash16 ? 2u : 4u) << hash_bits);
  off = (off + 127) & ~127u;
  L.off_stage = off;
  off += n_slots * L.stride;
  L.team_bytes = (off + 127) & ~127u;
  return L;
}

// Per-kernel state of the launch path: the dynamic shared-memory opt-in is raised once per kernel (monotonically,
// under a lock — concurrent callers with different ef no longer race on cudaFuncSetAttribute), occupancy is queried
// per launch.
static std::mutex g_kernel_mu;
static cudaError_t kernel_prepare(SearchKernelFn kern, size_t smem, uint32_t threads, int* occ) {
  static std::vector<std::pair<const void*, size_t>> raised;
  {
    std::lock_guard<std::mutex> lk(g_kernel_mu);
    size_t* cur = nullptr;
    for (auto& kv : raised)
      if (kv.first == (const void*)kern) cur = &kv.second;
    if (!cur) {
      raised.emplace_back((const void*)kern, 0);
      cur = &raised.back().second;
    }
    if (smem > *cur) {
      cudaError_t e = cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      *cur = smem;
    }
  }
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, (const void*)kern, (int)threads, smem);
}

static cudaError_t kernel_launch(SearchKernelFn kern, const SearchArgs& a, uint32_t grid, uint32_t threads, cudaStream_t stream) {
  void* params[1] = {const_cast<SearchArgs*>(&a)};
  return cudaLaunchKernel((const void*)kern, dim3(grid), dim3(threads), params, (size_t)a.lay.team_bytes, stream);
}

__global__ void fill_empty_results_kernel(uint64_t* rows, uint32_t* nodes, float* dist, uint32_t* counts,
                                          uint32_t* stats, uint32_t nq, uint32_t k) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (uint64_t)nq * k) {
    rows[i] = 0xFFFFFFFFFFFFFFFFull;
    if (nodes) nodes[i] = kInvalid;
    dist[i] = INFINITY;
  }
  if (i < nq) counts[i] = 0;
  if (stats && i < (uint64_t)nq * 4) stats[i] = 0;
}

// the insert path's searches (graph_insert.inl): nodes [first, first + nq) against the graph built so far
struct InsertSpec {
  uint32_t first, m, m0;
  uint32_t* sel;
  uint8_t* cnt;
};

static int32_t search_batch_device_impl(turdb_cuda_index* idx, const float* d_queries, uint32_t query_dim, uint32_t nq,
                                        uint32_t k, uint32_t ef, uint8_t metric, const uint64_t* d_visible,
                                        uint64_t* d_out_row_ids, uint32_t* d_out_node_ids, float* d_out_dist,
                                        uint32_t* d_out_counts, turdb_cuda_search_stats* d_out_stats, void* stream_,
                                        bool sq8, const InsertSpec* ins = nullptr) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  if (sq8 && idx->ix.n && !idx->d_arena_sq8) return fail(TURDB_ERR_INVALID_ARGUMENT, "call turdb_cuda_index_enable_sq8 first");
  if (query_dim != idx->ix.dim)
    return fail(TURDB_ERR_DIMENSION_MISMATCH, "query dimension %u does not match index dimension %u", query_dim, idx->ix.dim);
  if (metric > 2) return fail(TURDB_ERR_INVALID_ARGUMENT, "metric %u unknown", metric);
  if (ef == 0) return fail(TURDB_ERR_INVALID_ARGUMENT, "ef_search must be >= 1");
  if (ef > 2048) return fail(TURDB_ERR_UNSUPPORTED, "ef_search %u > 2048", ef);
  if (nq == 0) return TURDB_OK;
  if (!ins && (!d_queries || !d_out_counts || (k && (!d_out_row_ids || !d_out_dist))))
    return fail(TURDB_ERR_INVALID_ARGUMENT, "null query/output pointer");
  cudaStream_t stream = (cudaStream_t)stream_;
  DeviceGuard guard(idx->device);
  if (!guard.ok) return fail(TURDB_ERR_CUDA, "cudaSetDevice(%d) failed", idx->device);

  if (!ins && (idx->ix.n == 0 || idx->ix.entry == kInvalid || k == 0)) {  // Ok(vec![]), mod.rs:1106-1109
    uint64_t total = std::max<uint64_t>((uint64_t)nq * std::max(k, 1u), (uint64_t)nq * 4);
    fill_empty_results_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(
        d_out_row_ids, d_out_node_ids, d_out_dist, d_out_counts, (uint32_t*)d_out_stats, nq, k);
    CUDA_TRY(cudaGetLastError());
    return TURDB_OK;
  }

  uint32_t tw, ts, th, tg, tm, vis_seen;
  double rows_per_hop = 0.0;  // level-0 distance evaluations per expansion seen so far in this ef class (0: nothing seen)
  const uint32_t ef_bucket = std::min(15u, ceil_log2(ef));
  {
    std::lock_guard<std::mutex> lk(idx->mu);
    tw = idx->tune_warps;
    ts = idx->tune_slots;
    th = idx->tune_hash_bits;
    tg = idx->tune_segs;
    tm = idx->tune_mode;
    const TraversalStats hs = idx->h_tstats[ef_bucket];  // pinned mirror; refreshed asynchronously after every launch
    vis_seen = ins ? 0u : hs.vis_max;
    if (!ins && hs.sum_exp) rows_per_hop = (double)hs.sum_dist / (double)hs.sum_exp;
  }
  const uint32_t ds = idx->ix.ds, dim = idx->ix.dim;
  // Visited table: 2 << hash_bits bytes of shared memory per resident query — the item that decides how many
  // queries an SM holds at small dims.  Before anything is known about the corpus it is sized for the worst case
  // (ef * 64 keys); afterwards from the largest key count any query of this ef class has produced (+25 %: the
  // table is declared full at 7/8).  Results never depend on it: a query that outgrows its table is redone
  // exactly by the global-bitset pass below.
  // 16-bit entries need key_bits - hash_bits remainder bits and at least 6 displacement bits at the loads chosen
  // here (load <= 0.6 at the largest query); 32-bit entries have no displacement limit and may fill to 7/8.  Whichever
  // form takes fewer bytes wins (large corpora with short traversals: 32-bit entries in a small table).
  uint32_t hash_bits = std::min(15u, std::max(9u, ceil_log2(ef * 64)));
  bool entries32 = false;
  if (th) {
    hash_bits = th;
  } else if (vis_seen) {
    const uint32_t key_bits = ceil_log2((uint32_t)std::max<uint64_t>(idx->ix.n, 2));
    const uint32_t hb16 = std::min(15u, std::max({8u, ceil_log2((uint32_t)((uint64_t)vis_seen * 17 / 10 + 64)), key_bits > 10 ? key_bits - 10 : 0u}));
    const uint32_t hb32 = std::min(15u, std::max(8u, ceil_log2((uint32_t)(((uint64_t)vis_seen + 40) * 5 / 4))));
    const bool ok16 = key_bits <= hb16 + 10;
    if (ok16 && (2u << hb16) <= (4u << hb32)) {
      hash_bits = hb16;
    } else {
      hash_bits = hb32;
      entries32 = true;
    }
  }
  const uint32_t budget = (uint32_t)idx->max_smem_optin;
  const uint64_t nn = idx->ix.n;
  // deleted rows (turdb_cuda_index_delete) are rows the table no longer holds: search_filtered over `live`, or over
  // `visible AND live` (combined below, in pool scratch).  The insert path's searches read no visibility.
  const uint64_t* d_live = ins ? nullptr : idx->ix.live;
  const bool filt = d_visible != nullptr || d_live != nullptr;
  // form: short FP32 rows -> one warp per query, registers as the landing zone; long rows -> team + TMA staging
  // (measured, r02: 2M x 128 clustered, 4 new rows per hop: direct 2.64 ms, staged 3.00; 1M x 128 SIFT-like, 24 new rows
  // per hop: direct 7.9 ms, staged 4.9) — so the direct form needs short rows AND few of them per hop; until a launch
  // has reported what the corpus looks like the staged form runs.
  const bool direct = !sq8 && (tm == 2 || (tm == 0 && ds * 4 <= TURDB_DIRECT_MAX_ROW_BYTES && rows_per_hop > 0.0 &&
                                           rows_per_hop <= TURDB_DIRECT_MAX_ROWS_PER_HOP));
  uint32_t warps = direct ? 1u : (tw ? std::min(tw, 4u) : 0u);  // staged team size (0: chosen below)
  const uint32_t rb8 = sq8 ? idx->sq8_row_bytes : 0;
  TeamLayout lay{};
  bool auto_warps = false;
  if (direct) {
    lay = make_layout(dim, ds, ef, hash_bits, 0, 1, false, nn, filt, 0, entries32);
    while (lay.team_bytes > budget && hash_bits > 8) lay = make_layout(dim, ds, ef, --hash_bits, 0, 1, false, nn, filt, 0, entries32);
  } else {
    uint32_t slots = ts, segs = tg;
    if (sq8) {
      // code rows are short (dim + 8 B) but cost ~10 instructions per element pair to decode with the reference's
      // roundings: the reduce phase, not the gather, bounds a hop -> one gather round (32 slots) and the full team
      // (measured at 1M x 384: 4 warps x 32 slots 7.97 ms, 2 x 16 8.92 ms)
      if (!slots) slots = 32;
      segs = 1;
      if (!warps) warps = 4;
    }
    if (!slots || !segs) {
      // Measured at 1M x 384 (tools/sweep.py): whole vectors (1 piece) through 16 slots with 5 resident queries
      // per SM beat every split; pieces only pay when a whole vector leaves fewer than 4 queries resident
      // (large dim / large ef).  Within a piece count: resident queries x min(slots, 16) — beyond 16 slots the
      // lost residency costs more than the saved second gather round (measured) —, ties to the deeper staging.
      const uint32_t sm_bytes = budget + 1024;
      double best = -1.0;
      uint32_t bs = 8, bg = 1;
      for (uint32_t cg = tg ? tg : 1; cg <= (tg ? tg : 8); ++cg) {
        uint32_t best_occ = 0;
        for (uint32_t cs = ts ? ts : 8; cs <= (ts ? ts : 32); cs += 8) {
          TeamLayout L = make_layout(dim, ds, ef, hash_bits, cs, cg, false, nn, filt, rb8, entries32);
          if (L.n_segs != cg || L.team_bytes > budget) continue;
          if (cg > 1 && L.seg_steps * 32 < 512) continue;
          const uint32_t occ = std::min(8u, sm_bytes / (L.team_bytes + 1024));
          const double score = (double)occ * std::min(cs, 16u) / cg + 1e-6 * cs;
          if (score > best) {
            best = score;
            bs = cs;
            bg = cg;
          }
          best_occ = std::max(best_occ, occ);
        }
        if (best_occ >= 4) break;  // enough resident queries without (further) splitting
      }
      slots = bs;
      segs = bg;
    }
    lay = make_layout(dim, ds, ef, hash_bits, slots, segs, false, nn, filt, rb8, entries32);
    // Team size: warp 0 leads (control flow + speculative preparation of the next hop), the others gather and
    // reduce; every warp takes a share of a hop's bulk-copy issue.  Resident queries per SM come first (the
    // kernel is latency-bound); among equal residency the larger team wins (shorter issue phase).
    if (!warps) {
      auto_warps = true;
      warps = 4;
    }
    while (lay.team_bytes > budget && lay.n_segs < 16 && lay.seg_steps > 8)
      lay = make_layout(dim, ds, ef, hash_bits, lay.n_groups * 8, lay.n_segs + 1, false, nn, filt, rb8, entries32);
    while (lay.team_bytes > budget && lay.n_groups > 1)
      lay = make_layout(dim, ds, ef, hash_bits, lay.n_groups * 8 - 8, lay.n_segs, false, nn, filt, rb8, entries32);
    while (lay.team_bytes > budget && hash_bits > 8)
      lay = make_layout(dim, ds, ef, --hash_bits, lay.n_groups * 8, lay.n_segs, false, nn, filt, rb8, entries32);
  }
  if (lay.team_bytes > budget)
    return fail(TURDB_ERR_UNSUPPORTED, "dim %u / ef %u need %u B of shared memory per query (> %u)", idx->ix.dim, ef, lay.team_bytes, budget);

  SearchKernelFn kern = ins ? get_insert_kernel(false, direct) : get_search_kernel(metric, false, filt, sq8, direct);
  int occ = 0;
  cudaError_t e = cudaSuccess;
  if (auto_warps) {
    int best_occ = 0;
    for (uint32_t w = 4; w >= 2; --w) {
      int o = 0;
      if ((e = kernel_prepare(kern, lay.team_bytes, 32 * w, &o)) != cudaSuccess) break;
      if (o > best_occ) {
        best_occ = o;
        warps = w;
      }
    }
    occ = best_occ;
  } else {
    e = kernel_prepare(kern, lay.team_bytes, 32 * warps, &occ);
  }
  if (e != cudaSuccess || occ < 1)
    return fail(TURDB_ERR_CUDA, "traversal kernel does not fit an SM (%u B, %u threads): %s", lay.team_bytes, 32 * warps,
                cudaGetErrorString(e));
  const uint32_t grid = std::max(1u, std::min<uint32_t>(nq, (uint32_t)occ * (uint32_t)idx->num_sms));

  // fallback pass geometry (queries whose visited table or filtered-candidate buffer filled): same form, one bit
  // per node in global memory; its filtered-candidate buffer holds every node, so it cannot fail
  TeamLayout glay = direct ? make_layout(dim, ds, ef, 8, 0, 1, true, nn, filt, 0)
                           : make_layout(dim, ds, ef, 8, lay.n_groups * 8, lay.n_segs, true, nn, filt, rb8);
  const uint32_t vis_words = (uint32_t)(((nn + 31) / 32 + 3) & ~3ull);
  uint32_t fb_ctas = (uint32_t)std::min<uint32_t>((uint32_t)idx->num_sms, nq);
  const uint32_t f_ocap_main = filt ? (uint32_t)std::min<uint64_t>(nn, 32768) : 0u;
  const uint32_t f_ocap_fb = filt ? (uint32_t)nn : 0u;
  if (filt) {  // bound the fallback's scratch to ~1 GiB
    const uint64_t per_cta = (uint64_t)f_ocap_fb * sizeof(uint2) + (uint64_t)vis_words * 4;
    fb_ctas = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(fb_ctas, (1ull << 30) / std::max<uint64_t>(per_cta, 1)));
  }

  uint32_t* d_scratch = nullptr;  // [0] work counter, [1] overflow count, [2] fallback work counter, [4..] overflow list
  uint2* d_fovf = nullptr;
  uint32_t* d_gv = nullptr;
  uint2* d_fovf_fb = nullptr;
  uint64_t* d_vis_live = nullptr;
  auto release = [&]() {
    if (d_vis_live) cudaFreeAsync(d_vis_live, stream);
    if (d_fovf_fb) cudaFreeAsync(d_fovf_fb, stream);
    if (d_gv) cudaFreeAsync(d_gv, stream);
    if (d_fovf) cudaFreeAsync(d_fovf, stream);
    if (d_scratch) cudaFreeAsync(d_scratch, stream);
  };
  e = cudaMallocFromPoolAsync(&d_scratch, (size_t)(4 + nq) * 4, idx->pool, stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_scratch, 0, 16, stream);
  if (e == cudaSuccess && filt) e = cudaMallocFromPoolAsync(&d_fovf, (size_t)grid * f_ocap_main * sizeof(uint2), idx->pool, stream);
  if (e == cudaSuccess) e = cudaMallocFromPoolAsync(&d_gv, (size_t)fb_ctas * vis_words * 4, idx->pool, stream);
  if (e == cudaSuccess && filt) e = cudaMallocFromPoolAsync(&d_fovf_fb, (size_t)fb_ctas * f_ocap_fb * sizeof(uint2), idx->pool, stream);
  if (e == cudaSuccess && d_live && d_visible) {
    const uint64_t words = (nn + 63) / 64;
    e = cudaMallocFromPoolAsync(&d_vis_live, words * 8, idx->pool, stream);
    if (e == cudaSuccess) {
      live_and_kernel<<<(unsigned)((words + 255) / 256), 256, 0, stream>>>(d_visible, d_live, words, d_vis_live);
      e = cudaGetLastError();
    }
  }
  if (e != cudaSuccess) {
    release();
    return fail(e == cudaErrorMemoryAllocation ? TURDB_ERR_OUT_OF_MEMORY : TURDB_ERR_CUDA, "traversal scratch: %s", cudaGetErrorString(e));
  }

  SearchArgs a{};
  a.ix = idx->ix;
  a.lay = lay;
  a.queries = d_queries;
  a.nq = nq;
  a.k = k;
  a.ef = ef;
  a.out_row_ids = d_out_row_ids;
  a.out_node_ids = d_out_node_ids;
  a.out_dist = d_out_dist;
  a.out_counts = d_out_counts;
  a.out_stats = (uint32_t*)d_out_stats;
  a.work_counter = d_scratch;
  a.overflow_count = d_scratch + 1;
  a.overflow_list = d_scratch + 4;
  a.global_visited = nullptr;
  a.vis_words = 0;
  a.dbg = idx->d_dbg;
  a.visible = d_vis_live ? d_vis_live : (d_visible ? d_visible : d_live);
  a.rows = sq8 ? idx->d_arena_sq8 : reinterpret_cast<const uint8_t*>(idx->d_arena);
  a.row_bytes = lay.vec_bytes;
  if (sq8) a.ix.norm2 = idx->d_norm2_sq8;  // cosine's norm_b chain runs over the decoded row
  a.f_ovf = d_fovf;
  a.f_ocap = f_ocap_main;
  a.tstats = ins ? nullptr : idx->d_tstats + ef_bucket;
  if (ins) {
    a.ins_first = ins->first;
    a.ins_m = ins->m;
    a.ins_m0 = ins->m0;
    a.ins_levels = idx->d_levels + ins->first;
    a.ins_sel = ins->sel;
    a.ins_cnt = ins->cnt;
  }

  cudaEvent_t* pev = nullptr;
  {
    std::lock_guard<std::mutex> lk(idx->mu);
    if (idx->prof_used < idx->prof_capacity) pev = &idx->prof_events[3 * idx->prof_used++];
  }
  if (pev) cudaEventRecord(pev[0], stream);
  e = kernel_launch(kern, a, grid, 32 * warps, stream);
  if (pev) cudaEventRecord(pev[1], stream);
  if (e != cudaSuccess) {
    release();
    return fail(TURDB_ERR_CUDA, "traversal kernel launch failed: %s", cudaGetErrorString(e));
  }

  // exact fallback: always enqueued (no host sync); exits immediately when the list is empty
  {
    SearchKernelFn gkern = ins ? get_insert_kernel(true, direct) : get_search_kernel(metric, true, filt, sq8, direct);
    int gocc = 0;
    e = kernel_prepare(gkern, glay.team_bytes, 32 * warps, &gocc);
    if (e == cudaSuccess && gocc < 1) e = cudaErrorInvalidConfiguration;
    if (e == cudaSuccess) {
      SearchArgs b = a;
      b.lay = glay;
      b.work_counter = d_scratch + 2;
      b.vis_words = vis_words;
      b.global_visited = d_gv;
      b.f_ovf = d_fovf_fb;
      b.f_ocap = f_ocap_fb;
      e = kernel_launch(gkern, b, fb_ctas, 32 * warps, stream);
    }
    if (pev) cudaEventRecord(pev[2], stream);
    if (e != cudaSuccess) {
      release();
      return fail(TURDB_ERR_CUDA, "fallback traversal launch failed: %s", cudaGetErrorString(e));
    }
  }
  // refresh the host mirror of the visited-set statistics (read by the NEXT call; never waited for)
  if (!ins) cudaMemcpyAsync(idx->h_tstats, idx->d_tstats, 16 * sizeof(TraversalStats), cudaMemcpyDeviceToHost, stream);
  release();
  return TURDB_OK;
}

// one step of the insert path: searches of nodes [first, first + count) (squared L2, ef_construction)
static int32_t insert_search_step(turdb_cuda_index* idx, uint32_t first, uint32_t count, uint32_t ef, uint32_t m, uint32_t m0,
                                  uint32_t* d_sel, uint8_t* d_cnt, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(d_cnt, 0, (size_t)count * kInsLevels, stream);
  if (e != cudaSuccess) return fail(TURDB_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
  InsertSpec spec{first, m, m0, d_sel, d_cnt};
  return search_batch_device_impl(idx, nullptr, idx->ix.dim, count, 0, ef, kL2, nullptr, nullptr, nullptr, nullptr, nullptr,
                                  nullptr, stream, false, &spec);
}

extern "C" int32_t turdb_cuda_search_batch_device(turdb_cuda_index* idx, const float* d_queries, uint32_t query_dim,
                                                  uint32_t nq, uint32_t k, uint32_t ef, uint8_t metric,
                                                  const uint64_t* d_visible, uint64_t* d_out_row_ids,
                                                  uint32_t* d_out_node_ids, float* d_out_dist,
                                                  uint32_t* d_out_counts, turdb_cuda_search_stats* d_out_stats,
                                                  void* stream_) {
  return search_batch_device_impl(idx, d_queries, query_dim, nq, k, ef, metric, d_visible, d_out_row_ids, d_out_node_ids,
                                  d_out_dist, d_out_counts, d_out_stats, stream_, false);
}

extern "C" int32_t turdb_cuda_search_batch_sq8_device(turdb_cuda_index* idx, const float* d_queries, uint32_t query_dim,
                                                      uint32_t nq, uint32_t k, uint32_t ef, uint8_t metric,
                                                      const uint64_t* d_visible, uint64_t* d_out_row_ids,
                                                      uint32_t* d_out_node_ids, float* d_out_dist, uint32_t* d_out_counts,
                                                      turdb_cuda_search_stats* d_out_stats, void* stream_) {
  return search_batch_device_impl(idx, d_queries, query_dim, nq, k, ef, metric, d_visible, d_out_row_ids, d_out_node_ids,
                                  d_out_dist, d_out_counts, d_out_stats, stream_, true);
}

extern "C" int32_t turdb_cuda_search_batch(turdb_cuda_index* idx, const float* queries, uint32_t query_dim, uint32_t nq,
                                           uint32_t k, uint32_t ef, uint8_t metric, const uint64_t* visible,
                                           uint64_t* out_row_ids, uint32_t* out_node_ids, float* out_dist,
                                           uint32_t* out_counts, turdb_cuda_search_stats* out_stats) {
  if (!idx) return fail(TURDB_ERR_INVALID_ARGUMENT, "idx is null");
  if (query_dim != idx->ix.dim)
    return fail(TURDB_ERR_DIMENSION_MISMATCH, "query dimension %u does not match index dimension %u", query_dim, idx->ix.dim);
  if (nq == 0) return TURDB_OK;
  if (!queries || !out_counts || (k && (!out_row_ids || !out_dist)))
    return fail(TURDB_ERR_INVALID_ARGUMENT, "null query/output pointer");
  DeviceGuard guard(idx->device);
  if (!guard.ok) return fail(TURDB_ERR_CUDA, "cudaSetDevice(%d) failed", idx->device);
  cudaStream_t stream;
  CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  const size_t kk = std::max(k, 1u);
  const size_t qbytes = (size_t)nq * query_dim * 4;
  const size_t vis_bytes = visible ? ((idx->ix.n + 63) / 64) * 8 : 0;
  // one device slab: queries | rows | dist | nodes | counts | stats | visible
  size_t off_q = 0, off_rows = (qbytes + 255) & ~255ull, off_dist = off_rows + nq * kk * 8,
         off_nodes = off_dist + nq * kk * 4, off_counts = off_nodes + nq * kk * 4,
         off_stats = off_counts + ((nq * 4 + 15) & ~15ull), off_vis = off_stats + (size_t)nq * 16,
         total = off_vis + vis_bytes;
  uint8_t* slab = nullptr;
  int32_t rc = TURDB_OK;
  cudaError_t e = cudaMallocFromPoolAsync(&slab, total, idx->pool, stream);
  if (e != cudaSuccess) {
    cudaStreamDestroy(stream);
    return fail(TURDB_ERR_OUT_OF_MEMORY, "cudaMallocAsync(%zu) failed: %s", total, cudaGetErrorString(e));
  }
  auto cleanup = [&]() {
    cudaFreeAsync(slab, stream);
    cudaStreamSynchronize(stream);
    cudaStreamDestroy(stream);
  };
  e = cudaMemcpyAsync(slab + off_q, queries, qbytes, cudaMemcpyHostToDevice, stream);
  if (e == cudaSuccess && visible)
    e = cudaMemcpyAsync(slab + off_vis, visible, vis_bytes, cudaMemcpyHostToDevice, stream);
  if (e != cudaSuccess) {
    cleanup();
    return fail(TURDB_ERR_CUDA, "H2D copy failed: %s", cudaGetErrorString(e));
  }
  rc = turdb_cuda_search_batch_device(idx, (const float*)(slab + off_q), query_dim, nq, k, ef, metric,
                                      visible ? (const uint64_t*)(slab + off_vis) : nullptr,
                                      (uint64_t*)(slab + off_rows), (uint32_t*)(slab + off_nodes),
                                      (float*)(slab + off_dist), (uint32_t*)(slab + off_counts),
                                      out_stats ? (turdb_cuda_search_stats*)(slab + off_stats) : nullptr, stream);
  if (rc != TURDB_OK) {
    cleanup();
    return rc;
  }
  if (k) {
    e = cudaMemcpyAsync(out_row_ids, slab + off_rows, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_dist, slab + off_dist, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess && out_node_ids)
      e = cudaMemcpyAsync(out_node_ids, slab + off_nodes, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, stream);
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_counts, slab + off_counts, (size_t)nq * 4, cudaMemcpyDeviceToHost, stream);
  if (e == cudaSuccess && out_stats)
    e = cudaMemcpyAsync(out_stats, slab + off_stats, (size_t)nq * 16, cudaMemcpyDeviceToHost, stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  cudaFreeAsync(slab, stream);
  cudaStreamSynchronize(stream);
  cudaStreamDestroy(stream);
  if (e != cudaSuccess) return fail(TURDB_ERR_CUDA, "search failed: %s", cudaGetErrorString(e));
  return TURDB_OK;
}

// Diagnostics: random-row gather ceiling (gather_probe.cuh).  Same copies as the traversal, no dependencies.
extern "C" int32_t turdb_cuda_index_gather_probe(turdb_cuda_index* idx, uint32_t ctas_per_sm, uint32_t staging_slots,
                                                 uint32_t cta_smem_bytes, uint32_t rounds, float* out_ms,
                                                 uint64_t* out_bytes) {
  if (!idx || !out_ms || !out_bytes) return fail(TURDB_ERR_INVALID_ARGUMENT, "null argument");
  if (idx->ix.n == 0) return fail(TURDB_ERR_INVALID_ARGUMENT, "empty index");
  if (staging_slots == 0 || staging_slots > 64 * 8 || (staging_slots & 7)) return fail(TURDB_ERR_INVALID_ARGUMENT, "staging_slots must be a multiple of 8");
  if (ctas_per_sm == 0 || ctas_per_sm > 16 || rounds == 0) return fail(TURDB_ERR_INVALID_ARGUMENT, "ctas_per_sm 1..16, rounds >= 1");
  DeviceGuard guard(idx->device);
  if (!guard.ok) return fail(TURDB_ERR_CUDA, "cudaSetDevice(%d) failed", idx->device);
  TeamLayout lay = make_layout(idx->ix.dim, idx->ix.ds, 8, 8, staging_slots, 1, true, idx->ix.n, false);
  GatherProbeArgs a{};
  a.arena = idx->ix.arena;
  a.n = idx->ix.n;
  a.ds = idx->ix.ds;
  a.vec_bytes = lay.vec_bytes;
  a.stride = lay.stride;
  a.n_groups = staging_slots / 8;
  a.rounds = rounds;
  a.off_stage = 1024;
  const uint32_t need = a.off_stage + staging_slots * a.stride;
  const uint32_t smem = std::max(need, cta_smem_bytes);
  if (smem > (uint32_t)idx->max_smem_optin) return fail(TURDB_ERR_UNSUPPORTED, "%u B of shared memory per CTA", smem);
  CUDA_TRY(cudaFuncSetAttribute(gather_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gather_probe_kernel, 128, smem));
  if (occ < 1) return fail(TURDB_ERR_UNSUPPORTED, "probe does not fit an SM");
  const uint32_t per_sm = std::min<uint32_t>(ctas_per_sm, (uint32_t)occ);
  const uint32_t grid = per_sm * (uint32_t)idx->num_sms;
  uint32_t* d_sink = nullptr;
  CUDA_TRY(cudaMalloc(&d_sink, 4));
  a.sink = d_sink;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  gather_probe_kernel<<<grid, 128, smem>>>(a);  // warm-up
  cudaEventRecord(e0);
  gather_probe_kernel<<<grid, 128, smem>>>(a);
  cudaEventRecord(e1);
  cudaError_t e = cudaEventSynchronize(e1);
  float ms = 0.f;
  if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d_sink);
  if (e != cudaSuccess) return fail(TURDB_ERR_CUDA, "gather probe failed: %s", cudaGetErrorString(e));
  *out_ms = ms;
  *out_bytes = (uint64_t)grid * rounds * staging_slots * a.vec_bytes;
  return TURDB_OK;
}

// exact path + merge entry points live in exact_search.cuh / below
#include "exact_abi.inl"

#include "sql_topk.inl"
#include "sql_range.inl"
#include "sql_shards.inl"
#include "hnsw_file.inl"
#include "graph_insert.inl"
#include "graph_compact.inl"
