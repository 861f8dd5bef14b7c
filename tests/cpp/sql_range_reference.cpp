// The reference's evaluation of `WHERE vec <op> literal <cmp> radius LIMIT limit OFFSET offset` over a full scan, for
// tests/test_gpu_sql_range.py: every row in primary-key (= dense id) order, its value from the oracle's restatement
// of the projected distance (tdo_sql_projection_distance, src/sql/predicate.rs:1634-1688), widened to f64 and compared
// with the f64 constant.  NULL (cosine on a zero norm) and an absent vector (a +inf row) never qualify.  Output: rows
// [offset, offset + limit) of the qualifying rows (dense ids) and their values; the count of all qualifying rows.
#include <cstddef>
#include <cstdint>
#include <limits>

extern "C" float tdo_sql_projection_distance(int op, const float* a, const float* b, uint32_t dim, int* is_null);

extern "C" void sql_range_reference(const float* vectors, uint64_t n, uint32_t dim, const float* queries, uint32_t nq, int op,
                                    int cmp, const double* radius, uint32_t limit, uint32_t offset, uint64_t* out_rows,
                                    double* out_vals, uint32_t* out_counts) {
  for (uint32_t q = 0; q < nq; ++q) {
    const float* qv = queries + (size_t)q * dim;
    const double r = radius[q];
    uint64_t count = 0;
    for (uint64_t i = 0; i < n; ++i) {
      const float* row = vectors + i * dim;
      if (row[0] == std::numeric_limits<float>::infinity()) continue;
      int is_null = 0;
      const double v = tdo_sql_projection_distance(op, row, qv, dim, &is_null);
      if (is_null) continue;
      const bool ok = cmp == 0 ? v < r : (cmp == 1 ? v <= r : (cmp == 2 ? v > r : v >= r));
      if (!ok) continue;
      if (count >= offset && count - offset < limit) {
        out_rows[(size_t)q * limit + (count - offset)] = i;
        out_vals[(size_t)q * limit + (count - offset)] = v;
      }
      ++count;
    }
    for (uint64_t j = count > offset ? count - offset : 0; j < limit; ++j) {
      out_rows[(size_t)q * limit + j] = ~0ull;
      out_vals[(size_t)q * limit + j] = std::numeric_limits<double>::quiet_NaN();
    }
    out_counts[q] = (uint32_t)count;
  }
}
