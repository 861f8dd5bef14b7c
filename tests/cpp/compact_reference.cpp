// compact_reference.cpp — CPU restatement of the list repair of turdb_cuda_index_compact (test infrastructure; loaded by
// tests/compact_reference.py, which also does the per-row part of the rule).  Graph arrays in the turdb_cuda_graph
// layout.
//
// A list of live node p at level l without a deleted id is kept, in new ids.  One that holds a deleted id becomes
// select_neighbors_heuristic(p, C, cap) (operations.rs:181-233) over C = p's live neighbours at l in stored order, then,
// for each deleted neighbour d in p's stored order, d's live neighbours at l (nothing if d lacks level l); first
// occurrence kept, p excluded.  C is sorted stably ascending by squared L2 to p (the AVX2 lane order of
// euclidean_squared_avx2, NaN as +inf); the walk and the back-fill follow that order.  Every list is computed from the
// graph as it stood before the call.
#include <immintrin.h>

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <limits>
#include <vector>

namespace {

constexpr uint32_t kInvalid = 0xFFFFFFFFu;
constexpr uint32_t kL0 = 32, kUp = 16;

// euclidean_squared_avx2, distance.rs:105-129 (horizontal_sum_avx2 :150-161); the scalar tail is not contracted
float l2sq_avx2(const float* a, const float* b, size_t n) {
  size_t i = 0;
  __m256 sum = _mm256_setzero_ps();
  for (; i + 8 <= n; i += 8) {
    __m256 diff = _mm256_sub_ps(_mm256_loadu_ps(a + i), _mm256_loadu_ps(b + i));
    sum = _mm256_fmadd_ps(diff, diff, sum);
  }
  __m128 s = _mm_add_ps(_mm256_castps256_ps128(sum), _mm256_extractf128_ps(sum, 1));
  s = _mm_add_ps(s, _mm_movehl_ps(s, s));
  s = _mm_add_ss(s, _mm_shuffle_ps(s, s, 1));
  float result = _mm_cvtss_f32(s);
  for (; i < n; ++i) {
    float diff = a[i] - b[i];
    volatile float sq = diff * diff;
    result += sq;
  }
  return result;
}

struct Cand {
  uint32_t id;
  float d;
};

}  // namespace

extern "C" void tcr_compact_lists(uint32_t dim, uint64_t n, const float* vec, const uint8_t* levels,
                                  const uint32_t* l0_adj, const uint8_t* l0_cnt, const uint32_t* up_base,
                                  const uint32_t* up_adj, const uint8_t* up_cnt, const uint8_t* live,
                                  const uint32_t* o2n, const uint32_t* up_base_new, uint32_t* l0_adj_new,
                                  uint8_t* l0_cnt_new, uint32_t* up_adj_new, uint8_t* up_cnt_new) {
  auto v = [&](uint32_t i) { return vec + (size_t)i * dim; };
  auto list = [&](uint32_t i, uint32_t l, uint32_t* cnt) -> const uint32_t* {
    if (l == 0) {
      *cnt = l0_cnt[i];
      return l0_adj + (size_t)i * kL0;
    }
    if (l <= levels[i]) {
      const size_t s = (size_t)up_base[i] + l - 1;
      *cnt = up_cnt[s];
      return up_adj + s * kUp;
    }
    *cnt = 0;
    return nullptr;
  };
  for (uint64_t i = 0; i < n; ++i) {
    const uint32_t p = (uint32_t)i;
    if (!live[p]) continue;
    for (uint32_t l = 0; l <= levels[p]; ++l) {
      uint32_t cnt;
      const uint32_t* lst = list(p, l, &cnt);
      const uint32_t cap = l ? kUp : kL0;
      uint32_t* out = l ? up_adj_new + ((size_t)up_base_new[o2n[p]] + l - 1) * kUp : l0_adj_new + (size_t)o2n[p] * kL0;
      uint8_t* out_cnt = l ? up_cnt_new + up_base_new[o2n[p]] + l - 1 : l0_cnt_new + o2n[p];
      bool repair = false;
      for (uint32_t j = 0; j < cnt; ++j) repair |= !live[lst[j]];
      if (!repair) {
        for (uint32_t j = 0; j < cnt; ++j) out[j] = o2n[lst[j]];
        *out_cnt = (uint8_t)cnt;
        continue;
      }
      std::vector<Cand> cands;
      auto add = [&](uint32_t id) {
        if (id == p || !live[id]) return;
        for (const Cand& c : cands)
          if (c.id == id) return;
        cands.push_back(Cand{id, l2sq_avx2(v(p), v(id), dim)});
      };
      for (uint32_t j = 0; j < cnt; ++j) add(lst[j]);
      for (uint32_t j = 0; j < cnt; ++j) {
        if (live[lst[j]]) continue;
        uint32_t dc;
        const uint32_t* dl = list(lst[j], l, &dc);
        for (uint32_t t = 0; t < dc; ++t) add(dl[t]);
      }
      auto key = [](float d) { return std::isnan(d) ? std::numeric_limits<float>::infinity() : d; };
      std::stable_sort(cands.begin(), cands.end(), [&](const Cand& a, const Cand& b) { return key(a.d) < key(b.d); });
      // the walk (operations.rs:199-217), then the back-fill in the same order (:219-230)
      std::vector<uint32_t> sel;
      std::vector<bool> kept(cands.size(), false);
      for (size_t t = 0; t < cands.size() && sel.size() < cap; ++t) {
        bool closer = false;
        for (uint32_t e : sel)
          if (l2sq_avx2(v(cands[t].id), v(e), dim) < cands[t].d) {
            closer = true;
            break;
          }
        if (!closer) {
          sel.push_back(cands[t].id);
          kept[t] = true;
        }
      }
      for (size_t t = 0; t < cands.size() && sel.size() < cap; ++t)
        if (!kept[t]) sel.push_back(cands[t].id);
      for (size_t j = 0; j < sel.size(); ++j) out[j] = o2n[sel[j]];
      *out_cnt = (uint8_t)sel.size();
    }
  }
}
