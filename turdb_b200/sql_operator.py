"""The SQL vector-scan operator: `SELECT ... ORDER BY vec <op> '[...]' LIMIT k OFFSET o` on the GPU.

Host-side mirror of the reference's TopK executor for that statement shape (kahflane/TurDB):
  - `PhysicalOperator::TopKExec{input, order_by, limit, offset}`  src/sql/planner/physical.rs:229
  - `DynamicExecutor::TopK`, pulled with open / next / close       src/sql/executor.rs:346-350, 2239-2392
  - sort-key arithmetic of `<->` and `<=>`                         src/sql/executor.rs:169-212
  - `<#>` is not a sort key there (every row evaluates to NULL)    src/sql/executor.rs:241
A planner replaces TopKExec(scan) by this operator when order_by[0] is `Column <op> literal`
(src/sql/ast.rs:907-909); many statements over one table go through ONE launch (`VectorScanBatch`,
BASELINE.json config 5's batch path).  All arithmetic is below the C ABI (csrc/sql_topk.inl).

The distance-range scan `SELECT ... WHERE vec <op> '[...]' <cmp> r [LIMIT k [OFFSET o]]` (a Filter over the scan) runs
through `VectorRangeScanBatch` (csrc/sql_range.inl), and both clauses together with one literal,
`... WHERE vec <op> '[...]' < r ORDER BY vec <op> '[...]' LIMIT k` (TopK over the Filter), through `VectorRangeTopKBatch`.
A table split into sub-indexes (one per GPU, or several on one) answers `ORDER BY ... LIMIT k` through
`ShardedVectorScanBatch` (csrc/sql_shards.inl).
"""
from __future__ import annotations

import ctypes as C
import enum

import numpy as np

from . import _lib
from .hnsw import INVALID_ROW, CudaHnswIndex, _check, _ptr


class VectorOp(enum.IntEnum):
    L2Distance = 0       # `<->`  BinaryOperator::VectorL2Distance
    CosineDistance = 1   # `<=>`  BinaryOperator::VectorCosineDistance
    InnerProduct = 2     # `<#>`  BinaryOperator::VectorInnerProduct (NULL as a sort key in the reference)


def parse_vector_literal(text: str) -> np.ndarray:
    """'[0.1, 0.2]' -> f32 vector; value_to_vec_standalone, src/sql/executor.rs:245-261."""
    t = text.strip()
    if not (t.startswith("[") and t.endswith("]")):
        raise ValueError("vector literal must be bracketed")
    return np.array([np.float32(x.strip()) for x in t[1:-1].split(",")], dtype=np.float32)


class VectorScanBatch:
    """nq statements `SELECT [vec <proj_op> literal_i] ... ORDER BY vec <op> literal_i LIMIT limit OFFSET offset` against
    one table.  `project` = the operator whose value the statement projects (predicate.rs:1634-1688), or None."""

    def __init__(self, index: CudaHnswIndex, op: VectorOp, limit: int, offset: int = 0, use_index: bool = False,
                 ef_search: int = 0, project: VectorOp | None = None):
        self.index, self.op, self.limit, self.offset = index, VectorOp(op), int(limit), int(offset)
        self.use_index, self.ef_search = bool(use_index), int(ef_search)
        self.project = None if project is None else VectorOp(project)
        self.projected = None

    def execute(self, literals) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """-> (row_ids u64 [nq, limit], keys f64 [nq, limit] (NaN = NULL), counts u32 [nq]); the projected values, when
        asked for, are left in `self.projected` (f64 [nq, limit], NaN = NULL)."""
        q = np.ascontiguousarray(literals, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        nq, qd = q.shape
        lim = max(self.limit, 1)
        rows = np.full((nq, lim), INVALID_ROW, np.uint64)
        keys = np.full((nq, lim), np.nan, np.float64)
        proj = np.full((nq, lim), np.nan, np.float64) if self.project is not None else None
        counts = np.zeros(nq, np.uint32)
        _check(_lib.load().turdb_cuda_sql_topk_batch(self.index._h, _ptr(q, C.c_float), qd, nq, self.limit, self.offset,
                                                     int(self.op), int(self.project or 0), 1 if self.use_index else 0,
                                                     self.ef_search, _ptr(rows, C.c_uint64), _ptr(keys, C.c_double),
                                                     _ptr(proj, C.c_double) if proj is not None else None,
                                                     _ptr(counts, C.c_uint32)))
        self.projected = None if proj is None else proj[:, :self.limit]
        return rows[:, :self.limit], keys[:, :self.limit], counts

    def execute_device(self, d_literals: int, nq: int, d_rows: int, d_keys: int, d_counts: int, stream: int = 0,
                       d_proj: int = 0):
        """Device-resident form: raw device addresses, enqueued on `stream` (no host synchronisation)."""
        _check(_lib.load().turdb_cuda_sql_topk_batch_device(self.index._h, d_literals, self.index.dim, nq, self.limit, self.offset,
                                                            int(self.op), int(self.project or 0), 1 if self.use_index else 0,
                                                            self.ef_search, d_rows, d_keys, d_proj or None, d_counts,
                                                            stream or None))


class RangeCmp(enum.IntEnum):
    Lt = 0   # `<`
    Le = 1   # `<=`
    Gt = 2   # `>`
    Ge = 3   # `>=`


def range_direction_supported(op: VectorOp, cmp: RangeCmp) -> bool:
    """The near direction only: `<->` / `<=>` below a radius, `<#>` above a threshold."""
    return (VectorOp(op) == VectorOp.InnerProduct) == (RangeCmp(cmp) in (RangeCmp.Gt, RangeCmp.Ge))


class VectorRangeScanBatch:
    """nq statements `SELECT ... FROM t WHERE vec <op> literal_i <cmp> radius_i LIMIT limit OFFSET offset` against one
    table (csrc/sql_range.inl).  A row qualifies iff its projected f32 value (predicate.rs:1634-1688), widened to f64,
    compares true against radius_i; NULL values and absent vectors never do.  Rows come back in scan (primary-key)
    order; limit = 0 is a COUNT.  Raises ValueError before the library is called on a bad op / cmp pair, shape or dtype."""

    def __init__(self, index: CudaHnswIndex, op: VectorOp, cmp: RangeCmp, limit: int, offset: int = 0):
        try:
            self.op, self.cmp = VectorOp(op), RangeCmp(cmp)
        except ValueError as e:
            raise ValueError(f"unknown operator: {e}") from None
        if not range_direction_supported(self.op, self.cmp):
            raise ValueError(f"{self.op.name} {self.cmp.name}: only the near direction is supported "
                             "(<-> and <=> with < or <=, <#> with > or >=)")
        limit, offset = int(limit), int(offset)
        if not (0 <= limit < 2**32 and 0 <= offset < 2**32):
            raise ValueError("limit and offset must be in [0, 2^32)")
        self.index, self.limit, self.offset = index, limit, offset

    def _inputs(self, literals, radius):
        q = np.asarray(literals)
        if q.ndim == 1:
            q = q[None, :]
        if q.dtype.kind != "f" or q.ndim != 2 or q.shape[1] != self.index.dim:
            raise ValueError(f"literals must be float [nq, {self.index.dim}], got {q.dtype} {q.shape}")
        r = np.asarray(radius)
        if r.ndim == 0:
            r = r[None]
        if r.dtype.kind not in "fiu" or r.shape != (q.shape[0],):
            raise ValueError(f"radius must be one number per statement [{q.shape[0]}], got {r.dtype} {r.shape}")
        return np.ascontiguousarray(q, dtype=np.float32), np.ascontiguousarray(r, dtype=np.float64)

    def execute(self, literals, radius) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """-> (row_ids u64 [nq, limit], values f64 [nq, limit], counts u32 [nq] = ALL qualifying rows); unused slots are
        INVALID_ROW / NaN."""
        q, r = self._inputs(literals, radius)
        nq = q.shape[0]
        lim = max(self.limit, 1)
        rows = np.full((nq, lim), INVALID_ROW, np.uint64)
        vals = np.full((nq, lim), np.nan, np.float64)
        counts = np.zeros(nq, np.uint32)
        _check(_lib.load().turdb_cuda_sql_range_batch(self.index._h, _ptr(q, C.c_float), q.shape[1], nq, int(self.op),
                                                      int(self.cmp), _ptr(r, C.c_double), self.limit, self.offset,
                                                      _ptr(rows, C.c_uint64), _ptr(vals, C.c_double), _ptr(counts, C.c_uint32)))
        return rows[:, :self.limit], vals[:, :self.limit], counts

    def execute_device(self, d_literals: int, nq: int, d_radius: int, d_rows: int, d_counts: int, stream: int = 0,
                       d_vals: int = 0):
        """Device-resident form: raw device addresses (literals f32 [nq][dim], radius f64 [nq], rows u64 [nq][limit],
        counts u32 [nq], values f64 [nq][limit] or 0), enqueued on `stream` (no host synchronisation)."""
        _check(_lib.load().turdb_cuda_sql_range_batch_device(self.index._h, d_literals, self.index.dim, nq, int(self.op),
                                                             int(self.cmp), d_radius, self.limit, self.offset,
                                                             d_rows or None, d_vals or None, d_counts, stream or None))


SQL_MAX_LIMIT_PLUS_OFFSET = 512  # TURDB_SQL_MAX_LIMIT_PLUS_OFFSET, include/turdb_cuda.h


class VectorRangeTopKBatch:
    """nq statements `SELECT [vec <project> literal_i] ... FROM t WHERE vec <where_op> literal_i <cmp> radius_i
    ORDER BY vec <order_op> literal_i LIMIT limit OFFSET offset` against one table (csrc/sql_range.inl): the reference's
    TopK over exactly the rows its Filter lets through, row for row — VectorRangeScanBatch's predicate, VectorScanBatch's
    keys and heap order.  Raises ValueError before the library is called on an unknown or unsupported operator (the far
    direction, `<#>` as the sort key), limit + offset > SQL_MAX_LIMIT_PLUS_OFFSET, or a bad literal / radius."""

    def __init__(self, index: CudaHnswIndex, where_op: VectorOp, cmp: RangeCmp, order_op: VectorOp, limit: int,
                 offset: int = 0, project: VectorOp | None = None):
        self._where = VectorRangeScanBatch(index, where_op, cmp, limit, offset)  # operator pair, window and input checks
        try:
            self.order_op = VectorOp(order_op)
            self.project = None if project is None else VectorOp(project)
        except ValueError as e:
            raise ValueError(f"unknown operator: {e}") from None
        if self.order_op == VectorOp.InnerProduct:
            raise ValueError("ORDER BY <#> is NULL for every row in the reference; only <-> and <=> are sort keys")
        w = self._where
        if w.limit + w.offset > SQL_MAX_LIMIT_PLUS_OFFSET:
            raise ValueError(f"limit + offset = {w.limit + w.offset} > {SQL_MAX_LIMIT_PLUS_OFFSET}")
        self.index, self.where_op, self.cmp, self.limit, self.offset = index, w.op, w.cmp, w.limit, w.offset
        self.projected = None

    def execute(self, literals, radius) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """-> (row_ids u64 [nq, limit], keys f64 [nq, limit] (NaN = NULL), counts u32 [nq] = rows returned); unused slots
        are INVALID_ROW / NaN.  The projected values, when asked for, are left in `self.projected` (f64 [nq, limit])."""
        q, r = self._where._inputs(literals, radius)
        nq = q.shape[0]
        lim = max(self.limit, 1)
        rows = np.full((nq, lim), INVALID_ROW, np.uint64)
        keys = np.full((nq, lim), np.nan, np.float64)
        proj = np.full((nq, lim), np.nan, np.float64) if self.project is not None else None
        counts = np.zeros(nq, np.uint32)
        _check(_lib.load().turdb_cuda_sql_range_topk_batch(self.index._h, _ptr(q, C.c_float), q.shape[1], nq,
                                                           int(self.where_op), int(self.cmp), _ptr(r, C.c_double),
                                                           int(self.order_op), int(self.project or 0), self.limit,
                                                           self.offset, _ptr(rows, C.c_uint64), _ptr(keys, C.c_double),
                                                           _ptr(proj, C.c_double) if proj is not None else None,
                                                           _ptr(counts, C.c_uint32)))
        self.projected = None if proj is None else proj[:, :self.limit]
        return rows[:, :self.limit], keys[:, :self.limit], counts

    def execute_device(self, d_literals: int, nq: int, d_radius: int, d_rows: int, d_keys: int, d_counts: int,
                       stream: int = 0, d_proj: int = 0):
        """Device-resident form: raw device addresses (literals f32 [nq][dim], radius f64 [nq], rows u64 [nq][limit],
        keys f64 [nq][limit], counts u32 [nq], projected values f64 [nq][limit] or 0), enqueued on `stream` (no host
        synchronisation)."""
        _check(_lib.load().turdb_cuda_sql_range_topk_batch_device(self.index._h, d_literals, self.index.dim, nq,
                                                                  int(self.where_op), int(self.cmp), d_radius,
                                                                  int(self.order_op), int(self.project or 0), self.limit,
                                                                  self.offset, d_rows or None, d_keys or None,
                                                                  d_proj or None, d_counts, stream or None))


class ShardedVectorScanBatch:
    """nq statements `SELECT [vec <project> literal_i] ... ORDER BY vec <op> literal_i LIMIT limit OFFSET offset` against
    one table split into sub-indexes (csrc/sql_shards.inl): the table is shard 0's live rows in node-id order, then
    shard 1's, and so on, and the result is row for row VectorScanBatch's (exact scan) on one index holding that
    concatenation.  Raises ValueError before the library is called on an unknown or unsupported operator (`<#>` as the
    sort key), limit + offset > SQL_MAX_LIMIT_PLUS_OFFSET, a shard list that is not 1..32 indexes of one dimension, or a
    bad literal."""

    def __init__(self, shards, op: VectorOp, limit: int, offset: int = 0, project: VectorOp | None = None):
        try:
            self.op = VectorOp(op)
            self.project = None if project is None else VectorOp(project)
        except ValueError as e:
            raise ValueError(f"unknown operator: {e}") from None
        if self.op == VectorOp.InnerProduct:
            raise ValueError("ORDER BY <#> is NULL for every row in the reference; only <-> and <=> are sort keys")
        limit, offset = int(limit), int(offset)
        if not (0 <= limit < 2**32 and 0 <= offset < 2**32):
            raise ValueError("limit and offset must be in [0, 2^32)")
        if limit + offset > SQL_MAX_LIMIT_PLUS_OFFSET:
            raise ValueError(f"limit + offset = {limit + offset} > {SQL_MAX_LIMIT_PLUS_OFFSET}")
        self.shards = list(shards)
        if not 1 <= len(self.shards) <= 32:
            raise ValueError(f"need 1..32 shards, got {len(self.shards)}")
        dims = {s.dim for s in self.shards}
        if len(dims) != 1:
            raise ValueError(f"shards of different dimensions: {sorted(dims)}")
        self.dim = dims.pop()
        self.limit, self.offset = limit, offset
        self.projected = None

    def execute(self, literals) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """-> (row_ids u64 [nq, limit], keys f64 [nq, limit] (NaN = NULL), counts u32 [nq]); unused slots are
        INVALID_ROW / NaN.  The projected values, when asked for, are left in `self.projected` (f64 [nq, limit])."""
        q = np.asarray(literals)
        if q.ndim == 1:
            q = q[None, :]
        if q.dtype.kind != "f" or q.ndim != 2 or q.shape[1] != self.dim:
            raise ValueError(f"literals must be float [nq, {self.dim}], got {q.dtype} {q.shape}")
        q = np.ascontiguousarray(q, dtype=np.float32)
        nq = q.shape[0]
        lim = max(self.limit, 1)
        rows = np.full((nq, lim), INVALID_ROW, np.uint64)
        keys = np.full((nq, lim), np.nan, np.float64)
        proj = np.full((nq, lim), np.nan, np.float64) if self.project is not None else None
        counts = np.zeros(nq, np.uint32)
        handles = (C.c_void_p * len(self.shards))(*[s._h for s in self.shards])
        _check(_lib.load().turdb_cuda_shards_sql_topk_batch(handles, len(self.shards), _ptr(q, C.c_float), self.dim, nq,
                                                            self.limit, self.offset, int(self.op), int(self.project or 0),
                                                            _ptr(rows, C.c_uint64), _ptr(keys, C.c_double),
                                                            _ptr(proj, C.c_double) if proj is not None else None,
                                                            _ptr(counts, C.c_uint32)))
        self.projected = None if proj is None else proj[:, :self.limit]
        return rows[:, :self.limit], keys[:, :self.limit], counts


class VectorTopKExec:
    """One statement with the executor protocol of the reference: open() / next() -> (row_id, key) | None / close()."""

    def __init__(self, index: CudaHnswIndex, op: VectorOp, literal, limit: int, offset: int = 0, use_index: bool = False,
                 ef_search: int = 0):
        self._batch = VectorScanBatch(index, op, limit, offset, use_index, ef_search)
        self._literal = parse_vector_literal(literal) if isinstance(literal, str) else np.asarray(literal, np.float32)
        self._result = None
        self._iter = 0

    def open(self):
        self._result, self._iter = None, 0

    def next(self):
        if self._result is None:  # `computed` flag of TopKState, executor.rs:2240
            rows, keys, counts = self._batch.execute(self._literal)
            self._result = [(int(rows[0, i]), float(keys[0, i])) for i in range(int(counts[0]))]
        if self._iter < len(self._result):
            self._iter += 1
            return self._result[self._iter - 1]
        return None

    def close(self):
        self._result = None


# ---- the planner rule (mirror of where the reference turns Limit(Sort(..)) into TopKExec, -------------------------
# src/sql/planner/convert.rs:348-397): a statement whose ORDER BY is `column <op> vector-literal` followed by LIMIT
# [OFFSET] is rewritten to the vector-scan operator; anything else keeps the stock plan (None).
import re as _re

_VECTOR_TOPK = _re.compile(
    r"""^\s*SELECT\s+(?P<proj>.+?)\s+FROM\s+(?P<table>[A-Za-z_][\w.]*)\s+
        ORDER\s+BY\s+(?P<col>[A-Za-z_][\w.]*)\s*(?P<op><->|<=>|<\#>)\s*'(?P<lit>\[[^']*\])'\s*(?P<dir>ASC|DESC)?\s+
        LIMIT\s+(?P<limit>\d+)(?:\s+OFFSET\s+(?P<offset>\d+))?\s*;?\s*$""",
    _re.IGNORECASE | _re.VERBOSE | _re.DOTALL)

_OPS = {"<->": VectorOp.L2Distance, "<=>": VectorOp.CosineDistance, "<#>": VectorOp.InnerProduct}


def plan_vector_topk(sql: str):
    """`SELECT .. FROM t ORDER BY col <op> '[..]' LIMIT k [OFFSET o]` -> dict(table, column, op, literal, limit, offset,
    projection) for VectorTopKExec, or None when the rule does not apply: a WHERE / JOIN / GROUP BY (the scan below the
    sort is not the bare table), a descending order (the k FARTHEST rows), a second sort key, or `<#>` — a NULL sort key
    in the reference (src/sql/executor.rs:241), which must keep the stock TopK to stay result-compatible."""
    m = _VECTOR_TOPK.match(sql)
    if not m:
        return None
    if (m.group("dir") or "ASC").upper() == "DESC":
        return None
    op = _OPS[m.group("op")]
    if op == VectorOp.InnerProduct:
        return None
    try:
        lit = parse_vector_literal(m.group("lit"))
    except ValueError:
        return None
    return dict(table=m.group("table"), column=m.group("col"), op=op, literal=lit, limit=int(m.group("limit")),
                offset=int(m.group("offset") or 0), projection=[c.strip() for c in m.group("proj").split(",")])
