// turdb_cuda.hpp — header-only C++17 host mirror of TurDB's `src/hnsw` search interface over the C ABI
// (include/turdb_cuda.h).  The reference is compiled code (Rust) whose toolchain is absent from the build
// image, so this is the host side a native caller uses; names, argument meaning and error behaviour follow
// the reference (all citations into kahflane/TurDB):
//   DistanceFunction                src/hnsw/mod.rs:129-137
//   SearchResult                    src/hnsw/mod.rs:201-206 (node_id is the dense id; node_ids() maps it to (page, slot))
//   HnswSearchContext               src/hnsw/search.rs:193-225 (only ef_search survives: heaps and visited set live
//                                   in the kernel's shared memory)
//   CudaHnswIndex::search           PersistentHnswIndex::search, src/hnsw/mod.rs:1092-1174
//   CudaHnswIndex::search_filtered  src/hnsw/mod.rs:1176-1273
//   CudaHnswIndex::open             PersistentHnswIndex::open + the get_vector closure, mod.rs:811-834, 1097
//   VectorTopKExec                  DynamicExecutor::TopK open/next/close, src/sql/executor.rs:346-350, 2239-2392
// Errors: every failing call throws turdb_cuda::Error carrying the ABI status and the library's message — the
// dimension mismatch reads "query dimension {} does not match index dimension {}" as in mod.rs:1099-1104; an
// empty index yields an empty result (mod.rs:1106-1109).  There is no CPU fallback: without a CUDA device
// index creation throws with status TURDB_ERR_NO_DEVICE.
#pragma once

#include <algorithm>
#include <cstdint>
#include <functional>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "turdb_cuda.h"

namespace turdb_cuda {

enum class DistanceFunction : uint8_t { L2 = 0, Cosine = 1, InnerProduct = 2 };

struct NodeId {
  uint32_t page_no;
  uint16_t slot_index;
};

struct SearchResult {
  uint32_t node_id;  // dense id
  uint64_t row_id;
  float distance;
};

class Error : public std::runtime_error {
 public:
  Error(int32_t status, const std::string& msg) : std::runtime_error(msg), status_(status) {}
  int32_t status() const { return status_; }

 private:
  int32_t status_;
};

inline void check(int32_t rc) {
  if (rc != TURDB_OK) throw Error(rc, turdb_cuda_last_error());
}

class HnswSearchContext {
 public:
  explicit HnswSearchContext(size_t ef_search, size_t /*max_nodes*/ = 0) : ef_search_(ef_search) {}
  size_t ef_search() const { return ef_search_; }
  void set_ef_search(size_t ef) { ef_search_ = ef; }

 private:
  size_t ef_search_;
};

using GetVector = std::function<std::optional<std::vector<float>>(uint64_t row_id)>;

class CudaHnswIndex {
 public:
  CudaHnswIndex() = default;
  CudaHnswIndex(const CudaHnswIndex&) = delete;
  CudaHnswIndex& operator=(const CudaHnswIndex&) = delete;
  CudaHnswIndex(CudaHnswIndex&& o) noexcept { *this = std::move(o); }
  CudaHnswIndex& operator=(CudaHnswIndex&& o) noexcept {
    if (this != &o) {
      reset();
      h_ = o.h_;
      dim_ = o.dim_;
      n_ = o.n_;
      metric_ = o.metric_;
      node_ids_ = std::move(o.node_ids_);
      o.h_ = nullptr;
    }
    return *this;
  }
  ~CudaHnswIndex() { reset(); }

  // upload a flattened graph (the arrays stay owned by the caller and may be freed after this returns)
  static CudaHnswIndex from_graph(const turdb_cuda_graph& g, int device = 0, DistanceFunction metric = DistanceFunction::L2) {
    CudaHnswIndex idx;
    check(turdb_cuda_index_create(&g, device, &idx.h_));
    idx.dim_ = g.dim;
    idx.n_ = g.n;
    idx.metric_ = metric;
    return idx;
  }

  // PersistentHnswIndex::open(path) served from the GPU: the file is parsed once, vectors come from the table
  // through the reference's get_vector closure.  `flags` (optional) receives turdb_hnsw_file_flags.
  static CudaHnswIndex open(const std::string& path, const GetVector& get_vector, int device = 0, uint32_t* flags = nullptr) {
    turdb_cuda_hnsw_file* f = nullptr;
    check(turdb_cuda_hnsw_file_open(path.c_str(), &f));
    FileGuard guard{f};
    turdb_cuda_hnsw_file_info info{};
    check(turdb_cuda_hnsw_file_get_info(f, &info));
    if (flags) *flags = info.flags;
    CudaHnswIndex idx;
    const size_t total = (size_t)(info.n_nodes + info.n_tombstones);
    std::vector<uint32_t> pages(total);
    std::vector<uint16_t> slots(total);
    check(turdb_cuda_hnsw_file_nodes(f, nullptr, pages.data(), slots.data()));
    idx.node_ids_.resize(total);
    for (size_t i = 0; i < total; ++i) idx.node_ids_[i] = NodeId{pages[i], slots[i]};
    Trampoline tr{&get_vector, info.dimensions};
    check(turdb_cuda_hnsw_file_upload(f, nullptr, nullptr, &CudaHnswIndex::get_vector_thunk, &tr, device, &idx.h_));
    idx.dim_ = info.dimensions;
    idx.n_ = total;
    idx.metric_ = static_cast<DistanceFunction>(info.distance_fn);
    return idx;
  }

  uint32_t dimensions() const { return dim_; }
  DistanceFunction distance_fn() const { return metric_; }
  uint64_t node_count() const { return n_; }
  const std::vector<NodeId>& node_ids() const { return node_ids_; }  // dense id -> (page, slot); empty unless open()ed
  turdb_cuda_index* handle() const { return h_; }

  std::vector<SearchResult> search(const std::vector<float>& query, size_t k, const HnswSearchContext& ctx,
                                   std::optional<DistanceFunction> metric = std::nullopt) const {
    return search_one(query, k, ctx, metric, nullptr);
  }

  // is_visible is evaluated per row id into one bit per node (the MVCC predicate of mod.rs:1176-1186)
  std::vector<SearchResult> search_filtered(const std::vector<float>& query, size_t k, const HnswSearchContext& ctx,
                                            const std::vector<uint64_t>& row_ids,
                                            const std::function<bool(uint64_t)>& is_visible,
                                            std::optional<DistanceFunction> metric = std::nullopt) const {
    std::vector<uint64_t> bitmap((n_ + 63) / 64, 0);
    for (size_t i = 0; i < row_ids.size() && i < n_; ++i)
      if (is_visible(row_ids[i])) bitmap[i >> 6] |= 1ull << (i & 63);
    return search_one(query, k, ctx, metric, bitmap.data());
  }

  // nq queries at once (row-major [nq][dim]); results[q] ascend by distance
  std::vector<std::vector<SearchResult>> search_batch(const std::vector<float>& queries, size_t nq, size_t k, size_t ef_search,
                                                      std::optional<DistanceFunction> metric = std::nullopt) const {
    const uint32_t qd = nq ? (uint32_t)(queries.size() / nq) : dim_;
    std::vector<uint64_t> rows(nq * std::max<size_t>(k, 1));
    std::vector<uint32_t> nodes(rows.size()), counts(nq);
    std::vector<float> dist(rows.size());
    check(turdb_cuda_search_batch(h_, queries.data(), qd, (uint32_t)nq, (uint32_t)k, (uint32_t)ef_search,
                                  (uint8_t)metric.value_or(metric_), nullptr, rows.data(), nodes.data(), dist.data(),
                                  counts.data(), nullptr));
    std::vector<std::vector<SearchResult>> out(nq);
    for (size_t q = 0; q < nq; ++q)
      for (uint32_t i = 0; i < counts[q]; ++i) out[q].push_back(SearchResult{nodes[q * k + i], rows[q * k + i], dist[q * k + i]});
    return out;
  }

  // exact path (the SQL scan in the HNSW metric contract: squared L2 / 1 - cos / -dot)
  std::vector<SearchResult> bruteforce_topk(const std::vector<float>& query, size_t k,
                                            std::optional<DistanceFunction> metric = std::nullopt) const {
    std::vector<uint64_t> rows(std::max<size_t>(k, 1));
    std::vector<uint32_t> nodes(rows.size());
    std::vector<float> dist(rows.size());
    uint32_t count = 0;
    check(turdb_cuda_bruteforce_topk(h_, query.data(), (uint32_t)query.size(), 1, (uint32_t)k, (uint8_t)metric.value_or(metric_), 0,
                                     rows.data(), nodes.data(), dist.data(), &count));
    std::vector<SearchResult> out;
    for (uint32_t i = 0; i < count; ++i) out.push_back(SearchResult{nodes[i], rows[i], dist[i]});
    return out;
  }

 private:
  struct FileGuard {
    turdb_cuda_hnsw_file* f;
    ~FileGuard() { turdb_cuda_hnsw_file_close(f); }
  };
  struct Trampoline {
    const GetVector* fn;
    uint32_t dim;
  };
  static int32_t get_vector_thunk(void* user, uint64_t row_id, float* out) {
    auto* tr = static_cast<Trampoline*>(user);
    std::optional<std::vector<float>> v = (*tr->fn)(row_id);
    if (!v || v->size() != tr->dim) return 0;
    std::copy(v->begin(), v->end(), out);
    return 1;
  }
  std::vector<SearchResult> search_one(const std::vector<float>& query, size_t k, const HnswSearchContext& ctx,
                                       std::optional<DistanceFunction> metric, const uint64_t* visible) const {
    std::vector<uint64_t> rows(std::max<size_t>(k, 1));
    std::vector<uint32_t> nodes(rows.size());
    std::vector<float> dist(rows.size());
    uint32_t count = 0;
    check(turdb_cuda_search_batch(h_, query.data(), (uint32_t)query.size(), 1, (uint32_t)k, (uint32_t)ctx.ef_search(),
                                  (uint8_t)metric.value_or(metric_), visible, rows.data(), nodes.data(), dist.data(), &count,
                                  nullptr));
    std::vector<SearchResult> out;
    for (uint32_t i = 0; i < count; ++i) out.push_back(SearchResult{nodes[i], rows[i], dist[i]});
    return out;
  }
  void reset() {
    if (h_) turdb_cuda_index_destroy(h_);
    h_ = nullptr;
  }
  turdb_cuda_index* h_ = nullptr;
  uint32_t dim_ = 0;
  uint64_t n_ = 0;
  DistanceFunction metric_ = DistanceFunction::L2;
  std::vector<NodeId> node_ids_;
};

// `SELECT ... ORDER BY vec <op> '[...]' LIMIT limit OFFSET offset` with the reference's executor protocol.
enum class VectorOp : uint8_t { L2Distance = 0, CosineDistance = 1, InnerProduct = 2 };

class VectorTopKExec {
 public:
  VectorTopKExec(const CudaHnswIndex& index, VectorOp op, std::vector<float> literal, uint32_t limit, uint32_t offset = 0,
                 bool use_index = false, uint32_t ef_search = 0)
      : index_(index), op_(op), literal_(std::move(literal)), limit_(limit), offset_(offset), use_index_(use_index), ef_(ef_search) {}
  void open() {
    computed_ = false;
    iter_ = 0;
    result_.clear();
  }
  // (row_id, f64 sort key; NaN == NULL) or nullopt when exhausted
  std::optional<std::pair<uint64_t, double>> next() {
    if (!computed_) {  // TopKState::computed, executor.rs:2240
      std::vector<uint64_t> rows(std::max<uint32_t>(limit_, 1));
      std::vector<double> keys(rows.size());
      uint32_t count = 0;
      check(turdb_cuda_sql_topk_batch(index_.handle(), literal_.data(), (uint32_t)literal_.size(), 1, limit_, offset_,
                                      (uint8_t)op_, 0, use_index_ ? 1 : 0, ef_, rows.data(), keys.data(), nullptr, &count));
      for (uint32_t i = 0; i < count; ++i) result_.emplace_back(rows[i], keys[i]);
      computed_ = true;
    }
    if (iter_ < result_.size()) return result_[iter_++];
    return std::nullopt;
  }
  void close() { result_.clear(); }

 private:
  const CudaHnswIndex& index_;
  VectorOp op_;
  std::vector<float> literal_;
  uint32_t limit_, offset_;
  bool use_index_;
  uint32_t ef_;
  bool computed_ = false;
  size_t iter_ = 0;
  std::vector<std::pair<uint64_t, double>> result_;
};

// turdb_cuda_shards_sql_topk_batch: nq statements `ORDER BY vec <op> literal LIMIT limit OFFSET offset` over the table
// made of `shards`' live rows in shard order.  rows / keys are resized to [nq][limit], counts to [nq].
inline void shards_sql_topk(const std::vector<const CudaHnswIndex*>& shards, const std::vector<float>& literals, uint32_t dim,
                            VectorOp op, uint32_t limit, uint32_t offset, std::vector<uint64_t>& rows, std::vector<double>& keys,
                            std::vector<uint32_t>& counts) {
  std::vector<turdb_cuda_index*> handles;
  for (const CudaHnswIndex* s : shards) handles.push_back(s->handle());
  const uint32_t nq = dim ? (uint32_t)(literals.size() / dim) : 0;
  rows.assign((size_t)nq * std::max<uint32_t>(limit, 1), TURDB_INVALID_ROW);
  keys.assign(rows.size(), 0.0);
  counts.assign(nq, 0);
  check(turdb_cuda_shards_sql_topk_batch(handles.data(), (uint32_t)handles.size(), literals.data(), dim, nq, limit, offset,
                                         (uint8_t)op, 0, rows.data(), keys.data(), nullptr, counts.data()));
  rows.resize((size_t)nq * limit);
  keys.resize((size_t)nq * limit);
}

}  // namespace turdb_cuda
