"""Nearest rows within a radius (csrc/sql_range.inl, turdb_cuda_sql_range_topk_batch):
`WHERE vec <where_op> literal <cmp> r ORDER BY vec <order_op> literal LIMIT limit OFFSET offset` on the GPU against the
reference's TopK(Filter(Scan)): the oracle's TopK (`ob.sql_topk`) run per statement over exactly the rows the reference
Filter loop (tests/cpp/sql_range_reference.cpp) lets through, in scan order.  Row ids, f64 key bits, projected-value
bits and counts must be equal; rows with NULL keys are compared as a set."""
import re

import numpy as np
import pytest

from oracle import binding as ob
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import INVALID_ROW, CudaHnswIndex
from turdb_b200.sql_operator import (RangeCmp, VectorOp, VectorRangeScanBatch, VectorRangeTopKBatch, VectorScanBatch)
from test_gpu_sql_range import NEAR, radii_admitting, reference, table_index  # noqa: F401 (reference: a fixture)

pytestmark = pytest.mark.gpu
ORDER = [VectorOp.L2Distance, VectorOp.CosineDistance]


def expected(reference, x, q, where_op, cmp, radii, order_op, limit, offset):
    """(rows, keys, counts, projected, qualifying) of TopK over the Filter: dense row ids; projected = the WHERE value;
    qualifying[i] = the rows the Filter lets through for statement i, in scan order."""
    n, nq = x.shape[0], q.shape[0]
    sub, vals, qual = reference(x, q, where_op, cmp, radii, n)  # every qualifying row, in scan order, with its value
    lim = max(limit, 1)
    rows = np.full((nq, lim), INVALID_ROW, np.uint64)
    keys = np.full((nq, lim), np.nan)
    proj = np.full((nq, lim), np.nan)
    counts = np.zeros(nq, np.uint32)
    qualifying = [sub[i, :qual[i]].astype(np.int64) for i in range(nq)]
    for i, s in enumerate(qualifying):
        if limit == 0 or len(s) == 0:
            continue
        r, k, c = ob.sql_topk(x[s], q[i:i + 1], limit, op=int(order_op), offset=offset)
        c = int(c[0])
        pos = r[0, :c].astype(np.int64)
        rows[i, :c], keys[i, :c], proj[i, :c], counts[i] = s[pos], k[0, :c], vals[i, pos], c
    return rows[:, :limit], keys[:, :limit], counts, proj[:, :limit], qualifying


def null_keys(x, qv, order_op, s):
    """Which of rows s have a NULL ORDER BY key (cosine on a zero norm)."""
    if order_op != VectorOp.CosineDistance:
        return np.zeros(len(s), bool)
    return np.full(len(s), True) if not qv.any() else ~x[s].any(axis=1)


def assert_same(got, want, x, q, order_op, offset, row_ids=None, projected=None):
    """Bit for bit where no qualifying row has a NULL key.  Where one does, the reference's own order is unspecified
    (its sort treats NULL as equal to everything), so: the count, every row qualifies, NULL keys exactly on the rows
    that have them, ascending numbers; and when every qualifying key is NULL and offset = 0, the heap is never replaced
    into (nothing is strictly less than a NULL root), so the rows are the first `limit` qualifying ones, as a set."""
    rows, keys, counts = got
    w_rows, w_keys, w_counts, w_proj, qualifying = want
    assert np.array_equal(counts, w_counts)
    rid = np.arange(x.shape[0], dtype=np.uint64) if row_ids is None else row_ids
    dense = {int(r): i for i, r in enumerate(rid)}
    w_rows = np.where(w_rows == INVALID_ROW, INVALID_ROW, rid[np.minimum(w_rows, len(rid) - 1)])
    for i, s in enumerate(qualifying):
        c = int(counts[i])
        assert (rows[i, c:] == INVALID_ROW).all() and np.isnan(keys[i, c:]).all()
        null = null_keys(x, q[i], order_op, s)
        if not null.any():
            assert np.array_equal(rows[i], w_rows[i]), i
            assert np.array_equal(keys[i].view(np.uint64), w_keys[i].view(np.uint64)), i  # the f64 key bits
            if projected is not None:
                assert np.array_equal(projected[i].view(np.uint64), w_proj[i].view(np.uint64)), i
            continue
        got_dense = np.array([dense[int(r)] for r in rows[i, :c]], np.int64)
        assert np.isin(got_dense, s).all(), i
        assert np.array_equal(np.isnan(keys[i, :c]), null_keys(x, q[i], order_op, got_dense)), i
        num = keys[i, :c][~np.isnan(keys[i, :c])]
        assert (np.diff(num) >= 0).all(), i
        if null.all() and offset == 0:
            assert sorted(got_dense.tolist()) == sorted(s[:c].tolist()), i


def fallbacks(capfd):
    """Statements the streaming scan redid in the last call, from its TURDB_EXACT_VERBOSE line."""
    m = re.findall(r"\[turdb range\] statements=(\d+) fallback=(\d+)", capfd.readouterr().err)
    assert m, "no TURDB_EXACT_VERBOSE line"
    return int(m[-1][1])


def run(idx, x, q, where_op, cmp, radii, order_op, limit, offset, reference, rid=None):
    op = VectorRangeTopKBatch(idx, where_op, cmp, order_op, limit, offset, project=where_op)
    got = op.execute(q, radii)
    assert_same(got, expected(reference, x, q, where_op, cmp, radii, order_op, limit, offset), x, q, order_op, offset, rid,
                op.projected)
    return got


def test_known_answers(gpu_required, reference):
    x = np.array([[3, 4], [0, 5], [5, 0], [1, 1], [0, 0.5]], np.float32)
    rid = np.array([10, 11, 12, 13, 14], np.uint64)
    idx = table_index(x, rid)
    q = np.array([[0, 4.5]], np.float32)
    rows, keys, counts = VectorRangeTopKBatch(idx, VectorOp.L2Distance, RangeCmp.Lt, VectorOp.CosineDistance, 2).execute(q, [4.0])
    # `<-> < 4` lets (3,4), (0,5), (1,1) through ((0,0.5) is at exactly 4); by cosine: (0,5) 0, (3,4) 0.2, (1,1) 0.29.
    # The unfiltered top 2, (0,0.5) and (0,5), post-filtered would return one row.
    assert counts[0] == 2 and rows[0].tolist() == [11, 10] and keys[0, 0] == 0.0
    for cmp in (RangeCmp.Lt, RangeCmp.Le):
        for order_op in ORDER:
            for limit, offset in ((2, 0), (10, 0), (1, 2), (3, 5)):
                run(idx, x, q, VectorOp.L2Distance, cmp, [4.0], order_op, limit, offset, reference, rid)
    idx.close()


@pytest.mark.parametrize("order_op", ORDER)
@pytest.mark.parametrize("where_op,cmp", NEAR)
def test_gaussian_table_all_operator_pairs(gpu_required, reference, capfd, monkeypatch, where_op, cmp, order_op):
    """20k x 96; per statement a radius admitting 0, fewer than limit + offset, about limit + offset, 1000 or every row
    (more than the candidate buffer: the streaming scan)."""
    x = ds.gaussian_latent(20_000, 96, seed=41)
    q = ds.gaussian_latent(40, 96, seed=42)
    radii = radii_admitting(x, q, where_op, [0, 6, 12, 1000, -1] * 8)
    rid = np.arange(20_000, dtype=np.uint64) * 5 + 3
    idx = table_index(x, rid)
    monkeypatch.setenv("TURDB_EXACT_VERBOSE", "1")
    for limit, offset in ((10, 0), (5, 7), (0, 0), (10, 100), (500, 12)):
        rows, keys, counts = run(idx, x, q, where_op, cmp, radii, order_op, limit, offset, reference, rid)
        if limit:
            assert fallbacks(capfd) >= 8  # at least the every-row statements
            assert (counts[4::5] == limit).all() and (counts[0::5] == 0).all()
    idx.close()


def test_ties_on_the_filter_path_and_through_the_fallback(gpu_required, reference, capfd, monkeypatch):
    """Integer-valued vectors: hundreds of exactly equal keys across the LIMIT boundary, on the filter path.  Then 4000
    duplicates of one row inside the radius: more survivors than the buffer holds, so the streaming scan runs.  Which
    equal keys survive and in which order follows from the reference's heap alone."""
    monkeypatch.setenv("TURDB_EXACT_VERBOSE", "1")
    rng = np.random.default_rng(3)
    x = rng.integers(0, 4, (5000, 6)).astype(np.float32)
    x[np.all(x == 0, axis=1)] = 1.0  # no zero-norm rows: every key is a number
    q = rng.integers(0, 4, (24, 6)).astype(np.float32) + 0.5
    idx = table_index(x)
    for where_op, cmp in (NEAR[1], NEAR[3], NEAR[5]):
        radii = radii_admitting(x, q, where_op, [700] * 24)
        for order_op in ORDER:
            for limit, offset in ((10, 0), (7, 5), (100, 20), (300, 212)):
                run(idx, x, q, where_op, cmp, radii, order_op, limit, offset, reference)
                assert fallbacks(capfd) == 0
    idx.close()
    x = ds.gaussian_latent(9000, 32, seed=41)
    x[500:4500] = x[499]
    q = np.concatenate([x[499:500] + 1e-3, ds.gaussian_latent(5, 32, seed=42)])
    radii = np.concatenate([radii_admitting(x, q[:1], VectorOp.L2Distance, [4200]), radii_admitting(x, q[1:], VectorOp.L2Distance, [50] * 5)])
    idx = table_index(x)
    for order_op in ORDER:
        for limit, offset in ((10, 0), (25, 10), (500, 12)):
            run(idx, x, q, VectorOp.L2Distance, RangeCmp.Le, radii, order_op, limit, offset, reference)
            assert fallbacks(capfd) == 1
    idx.close()


@pytest.mark.parametrize("dim", [37, 130])
@pytest.mark.parametrize("where_op,cmp,order_op", [(*NEAR[1], VectorOp.CosineDistance), (*NEAR[2], VectorOp.L2Distance),
                                                   (*NEAR[4], VectorOp.CosineDistance), (*NEAR[0], VectorOp.L2Distance)])
def test_absent_rows_zero_norms_and_odd_dims(gpu_required, reference, dim, where_op, cmp, order_op):
    """Absent rows never qualify.  WHERE `<->` ORDER BY `<=>` lets zero-norm rows in with a NULL key."""
    x = ds.gaussian_latent(3000, dim, seed=dim)
    x[::7] = np.inf      # absent vectors
    x[3::11] = 0.0       # zero norm: NULL under cosine
    q = ds.gaussian_latent(12, dim, seed=dim + 1)
    q[5] = 0.0           # a zero literal: NULL for every row under cosine
    radii = radii_admitting(np.where(np.isfinite(x), x, 0), q, where_op, [0, 10, 200, -1] * 3)
    idx = table_index(x)
    for limit, offset in ((20, 0), (0, 0), (7, 5), (300, 100)):
        run(idx, x, q, where_op, cmp, radii, order_op, limit, offset, reference)
    idx.close()


def test_empty_index(gpu_required):
    idx = table_index(np.zeros((0, 8), np.float32))
    op = VectorRangeTopKBatch(idx, VectorOp.CosineDistance, RangeCmp.Lt, VectorOp.CosineDistance, 4, project=VectorOp.L2Distance)
    rows, keys, counts = op.execute(np.ones((3, 8), np.float32), [0.5, 1.0, 2.0])
    assert (counts == 0).all() and (rows == INVALID_ROW).all() and np.isnan(keys).all() and np.isnan(op.projected).all()
    idx.close()


@pytest.mark.parametrize("env", [{"TURDB_EXACT_PAIR": "0"}, {"TURDB_EXACT_PAIR": "1"}, {"TURDB_EXACT_FORCE_BF16": "1"}])
def test_filter_forms_give_identical_results(gpu_required, reference, monkeypatch, env):
    x = ds.gaussian_latent(20_000, 192, seed=51)
    q = ds.gaussian_latent(40, 192, seed=52)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    for (where_op, cmp), order_op in ((NEAR[0], VectorOp.CosineDistance), (NEAR[3], VectorOp.CosineDistance),
                                      (NEAR[5], VectorOp.L2Distance)):
        radii = radii_admitting(x, q, where_op, [0, 10, 1000, 3000, -1] * 8)
        idx = table_index(x)  # a fresh index: the 16-bit copies (FP16 or BF16) are built on its first call
        run(idx, x, q, where_op, cmp, radii, order_op, 25, 3, reference)
        idx.close()


def test_projection_of_another_operator(gpu_required, reference):
    x = ds.gaussian_latent(3000, 100, seed=51)
    x[7] = 0.0  # zero norm: cosine projects NULL
    q = np.concatenate([ds.gaussian_latent(30, 100, seed=52), x[7:8] + 1e-3])
    radii = radii_admitting(x, q, VectorOp.L2Distance, [40] * 31)
    idx = table_index(x)
    for proj in VectorOp:
        op = VectorRangeTopKBatch(idx, VectorOp.L2Distance, RangeCmp.Le, VectorOp.L2Distance, 8, 2, project=proj)
        rows, keys, counts = op.execute(q, radii)
        assert_same((rows, keys, counts), expected(reference, x, q, VectorOp.L2Distance, RangeCmp.Le, radii,
                                                   VectorOp.L2Distance, 8, 2), x, q, VectorOp.L2Distance, 2)
        for i in range(len(q)):
            for j in range(int(counts[i])):
                want = ob.sql_projection_distance(int(proj), x[int(rows[i, j])], q[i])
                got = op.projected[i, j]
                assert np.isnan(got) if want is None else np.float64(want) == got, (i, j, want, got)
    idx.close()


def test_results_follow_inserts(gpu_required, reference):
    x = ds.gaussian_latent(6000, 64, seed=61)
    q = ds.gaussian_latent(24, 64, seed=62)
    rid = np.arange(6000, dtype=np.uint64) + 100
    rnd = 1.0 - np.random.default_rng(3).random(6000)
    idx = CudaHnswIndex.build(x[:4000], rid[:4000], rnd[:4000], max_batch=256)
    for step, n in ((0, 4000), (1, 6000)):
        if step:
            idx.insert(x[4000:], rid[4000:], rnd[4000:])  # drops the 16-bit copies; the next call rebuilds them
        for (where_op, cmp), order_op in ((NEAR[1], VectorOp.L2Distance), (NEAR[2], VectorOp.CosineDistance),
                                          (NEAR[4], VectorOp.L2Distance)):
            radii = radii_admitting(x[:n], q, where_op, [0, 10, 300, -1] * 6)
            run(idx, x[:n], q, where_op, cmp, radii, order_op, 30, 0, reference, rid[:n])
    idx.close()


def test_every_row_admitted_is_the_unfiltered_topk(gpu_required):
    """No absent or zero-norm rows, a radius admitting every row and where_op == order_op: the statement is the plain
    ORDER BY ... LIMIT, and the result must be VectorScanBatch's exact one."""
    x = ds.gaussian_latent(20_000, 96, seed=71)
    q = ds.gaussian_latent(32, 96, seed=72)
    idx = table_index(x)
    for op in ORDER:
        for limit, offset in ((10, 0), (64, 3), (500, 12)):
            got = VectorRangeTopKBatch(idx, op, RangeCmp.Le, op, limit, offset).execute(q, np.full(32, 1e30))
            want = VectorScanBatch(idx, op, limit, offset).execute(q)
            for g, w in zip(got, want):
                assert np.array_equal(g.view(np.uint8), w.view(np.uint8))
    idx.close()


def test_range_scan_and_topk_are_unchanged_by_range_topk_calls(gpu_required):
    x = ds.gaussian_latent(20_000, 96, seed=71)
    q = ds.gaussian_latent(64, 96, seed=72)
    idx = table_index(x)

    def calls():
        out = [VectorScanBatch(idx, op, 10, 2).execute(q) for op in ORDER]
        for op, cmp in NEAR:
            out.append(VectorRangeScanBatch(idx, op, cmp, 10, 1).execute(q, radii_admitting(x, q, op, [10, 1000] * 32)))
        return out

    before = calls()
    for (op, cmp) in NEAR:
        for order_op in ORDER:
            VectorRangeTopKBatch(idx, op, cmp, order_op, 10, 2).execute(q, radii_admitting(x, q, op, [10, -1] * 32))
    after = calls()
    for b, a in zip(before, after):
        for bb, aa in zip(b, a):
            assert np.array_equal(bb.view(np.uint8), aa.view(np.uint8))
    idx.close()


def test_device_entry_matches_host_entry(gpu_required):
    import torch
    x = ds.gaussian_latent(5000, 64, seed=81)
    q = ds.gaussian_latent(16, 64, seed=82)
    idx = table_index(x)
    radii = radii_admitting(x, q, VectorOp.CosineDistance, [10, 100] * 8)
    op = VectorRangeTopKBatch(idx, VectorOp.CosineDistance, RangeCmp.Le, VectorOp.L2Distance, 12, 1,
                              project=VectorOp.InnerProduct)
    rows, keys, counts = op.execute(q, radii)
    dq, dr = torch.from_numpy(q).cuda(), torch.from_numpy(radii).cuda()
    d_rows = torch.empty((16, 12), dtype=torch.int64, device="cuda")
    d_keys = torch.empty((16, 12), dtype=torch.float64, device="cuda")
    d_proj = torch.empty((16, 12), dtype=torch.float64, device="cuda")
    d_cnt = torch.empty(16, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream()
    op.execute_device(dq.data_ptr(), 16, dr.data_ptr(), d_rows.data_ptr(), d_keys.data_ptr(), d_cnt.data_ptr(),
                      s.cuda_stream, d_proj.data_ptr())
    s.synchronize()
    assert np.array_equal(d_rows.cpu().numpy().view(np.uint64), rows)
    assert np.array_equal(d_keys.cpu().numpy().view(np.uint64), keys.view(np.uint64))
    assert np.array_equal(d_proj.cpu().numpy().view(np.uint64), op.projected.view(np.uint64))
    assert np.array_equal(d_cnt.cpu().numpy().view(np.uint32), counts)
    idx.close()
