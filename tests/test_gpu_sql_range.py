"""SQL distance-range scan (csrc/sql_range.inl): `WHERE vec <op> literal <cmp> radius LIMIT limit OFFSET offset` on the
GPU against the reference's row-by-row loop (tests/cpp/sql_range_reference.cpp over the oracle's projected distance):
row ids, the f64 value bits and the count of qualifying rows must all be equal."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import binding as ob
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import INVALID_ROW, CudaHnswIndex
from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeScanBatch, VectorScanBatch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEAR = [(VectorOp.L2Distance, RangeCmp.Lt), (VectorOp.L2Distance, RangeCmp.Le), (VectorOp.CosineDistance, RangeCmp.Lt),
        (VectorOp.CosineDistance, RangeCmp.Le), (VectorOp.InnerProduct, RangeCmp.Gt), (VectorOp.InnerProduct, RangeCmp.Ge)]


@pytest.fixture(scope="session")
def reference(tmp_path_factory):
    ob.lib()  # builds the oracle library the reference loop links against
    odir = os.path.dirname(ob._LIB_PATH)
    out = str(tmp_path_factory.mktemp("sql_range") / "libsql_range_reference.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared",
                           os.path.join(ROOT, "tests", "cpp", "sql_range_reference.cpp"), "-o", out,
                           "-L", odir, "-lturdb_oracle", f"-Wl,-rpath,{odir}"])
    L = C.CDLL(out)
    L.sql_range_reference.restype = None
    L.sql_range_reference.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_int, C.c_int,
                                      C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]

    def run(x, q, op, cmp, radius, limit, offset=0):
        x = np.ascontiguousarray(x, np.float32)
        q = np.ascontiguousarray(q, np.float32)
        r = np.ascontiguousarray(radius, np.float64)
        nq, lim = q.shape[0], max(limit, 1)
        rows = np.full((nq, lim), INVALID_ROW, np.uint64)
        vals = np.full((nq, lim), np.nan)
        counts = np.zeros(nq, np.uint32)
        L.sql_range_reference(x.ctypes.data, x.shape[0], x.shape[1], q.ctypes.data, nq, int(op), int(cmp), r.ctypes.data,
                              limit, offset, rows.ctypes.data, vals.ctypes.data, counts.ctypes.data)
        return rows[:, :limit], vals[:, :limit], counts
    return run


def table_index(x, row_ids=None):
    """A table without an HNSW graph: the scan only needs the arena (entry = none)."""
    n = x.shape[0]
    g = dict(vectors=x, row_ids=np.arange(n, dtype=np.uint64) if row_ids is None else row_ids,
             levels=np.zeros(n, np.uint8), l0_adj=np.full((n, 32), 0xFFFFFFFF, np.uint32), l0_cnt=np.zeros(n, np.uint8),
             up_base=np.full(n, 0xFFFFFFFF, np.uint32), up_adj=np.zeros((0, 16), np.uint32), up_cnt=np.zeros(0, np.uint8),
             entry=0 if n else 0xFFFFFFFF, max_level=0)
    return CudaHnswIndex.from_graph(g)


def assert_same(got, want, row_ids=None):
    rows, vals, counts = got
    o_rows, o_vals, o_counts = want
    assert np.array_equal(counts, o_counts)
    if row_ids is not None:
        o_rows = np.where(o_rows == INVALID_ROW, INVALID_ROW, row_ids[np.minimum(o_rows, len(row_ids) - 1)])
    assert np.array_equal(rows, o_rows)
    assert np.array_equal(vals.view(np.uint64), o_vals.view(np.uint64))  # the f64 value bit for bit (NaN in unused slots)


def approx_values(x, q, op):
    """float64 values for choosing radii (not the parity values)."""
    x64, q64 = x.astype(np.float64), q.astype(np.float64)
    if op == VectorOp.InnerProduct:
        return q64 @ x64.T
    if op == VectorOp.L2Distance:
        d2 = (q64 * q64).sum(1)[:, None] + (x64 * x64).sum(1)[None, :] - 2 * q64 @ x64.T
        return np.sqrt(np.maximum(d2, 0))
    nx, nq = np.linalg.norm(x64, axis=1), np.linalg.norm(q64, axis=1)
    return 1 - (q64 @ x64.T) / np.maximum(nq[:, None] * nx[None, :], 1e-300)


def radii_admitting(x, q, op, targets):
    """One radius per statement admitting about targets[i] rows (0 = none, -1 = every row)."""
    v = approx_values(x, q, op)
    far = op == VectorOp.InnerProduct
    out = np.empty(q.shape[0])
    for i, t in enumerate(targets):
        s = np.sort(v[i])[::-1] if far else np.sort(v[i])
        if t == 0:
            out[i] = s[0] + (1.0 if far else -1.0) * (abs(s[0]) + 1.0)
        elif t < 0:
            out[i] = -1e30 if far else 1e30
        else:
            out[i] = s[t - 1]
    return out


def test_known_answers(gpu_required, reference):
    x = np.array([[3, 4], [0, 5], [5, 0], [1, 1]], np.float32)
    idx = table_index(x, np.array([10, 11, 12, 13], np.uint64))
    q = np.zeros((1, 2), np.float32)
    rows, vals, counts = VectorRangeScanBatch(idx, VectorOp.L2Distance, RangeCmp.Lt, 10).execute(q, [5.0])
    assert counts[0] == 1 and rows[0, 0] == 13 and vals[0, 0] == np.float64(np.sqrt(np.float32(2)))
    assert np.all(rows[0, 1:] == INVALID_ROW) and np.all(np.isnan(vals[0, 1:]))
    rows, vals, counts = VectorRangeScanBatch(idx, VectorOp.L2Distance, RangeCmp.Le, 10).execute(q, [5.0])
    assert counts[0] == 4 and rows[0, :4].tolist() == [10, 11, 12, 13]
    for cmp in (RangeCmp.Lt, RangeCmp.Le):
        assert_same(VectorRangeScanBatch(idx, VectorOp.L2Distance, cmp, 10).execute(q, [5.0]),
                    reference(x, q, VectorOp.L2Distance, cmp, [5.0], 10), np.array([10, 11, 12, 13], np.uint64))
    idx.close()


@pytest.mark.parametrize("op,cmp", NEAR)
def test_radius_at_the_value_and_its_neighbours(gpu_required, reference, op, cmp):
    """Radii equal to rows' f32 values, their f32 neighbours and their f64 neighbours; near-duplicate rows 1e-4 apart
    (below 16-bit resolution) so that many values crowd around each radius."""
    rng = np.random.default_rng(5)
    base = rng.normal(0, 1, (8, 64)).astype(np.float32)
    x = (np.repeat(base, 400, axis=0) + rng.normal(0, 1e-4, (3200, 64))).astype(np.float32)
    x = np.concatenate([x, rng.normal(0, 1, (3000, 64)).astype(np.float32)])
    q = (base[:4] + rng.normal(0, 1e-3, (4, 64))).astype(np.float32)
    # exact f32 values of a few rows per query, by the reference itself (limit = n returns every value)
    _, all_vals, _ = reference(x, q, op, RangeCmp.Ge if op == VectorOp.InnerProduct else RangeCmp.Le,
                               [-np.inf if op == VectorOp.InnerProduct else np.inf] * 4, x.shape[0])
    lits, radii = [], []
    for i in range(4):
        for j in rng.choice(x.shape[0], 6, replace=False):
            v = np.float32(all_vals[i, j])
            for r in (float(v), float(np.nextafter(v, np.float32(np.inf))), float(np.nextafter(v, np.float32(-np.inf))),
                      np.nextafter(float(v), np.inf), np.nextafter(float(v), -np.inf)):
                lits.append(q[i])
                radii.append(r)
    lits = np.array(lits, np.float32)
    idx = table_index(x)
    for limit, offset in ((50, 0), (0, 0), (17, 900)):
        got = VectorRangeScanBatch(idx, op, cmp, limit, offset).execute(lits, radii)
        assert_same(got, reference(x, lits, op, cmp, radii, limit, offset))
    idx.close()


@pytest.mark.parametrize("op,cmp", NEAR)
def test_gaussian_table_radii_and_windows(gpu_required, reference, op, cmp):
    x = ds.gaussian_latent(20_000, 96, seed=41)
    q = ds.gaussian_latent(32, 96, seed=42)
    targets = [0, 10, 1000, -1] * 8
    radii = radii_admitting(x, q, op, targets)
    rid = np.arange(20_000, dtype=np.uint64) * 5 + 3
    idx = table_index(x, rid)
    for limit, offset in ((10, 0), (5, 7), (0, 0), (300, 2), (10, 100_000)):
        got = VectorRangeScanBatch(idx, op, cmp, limit, offset).execute(q, radii)
        want = reference(x, q, op, cmp, radii, limit, offset)
        assert_same(got, want, rid)
        if limit == 0:
            assert (want[2][3::4] == 20_000).all() and (want[2][0::4] == 0).all()
    idx.close()


@pytest.mark.parametrize("dim", [37, 130])
@pytest.mark.parametrize("op,cmp", [NEAR[1], NEAR[2], NEAR[4]])
def test_absent_rows_zero_norms_and_odd_dims(gpu_required, reference, dim, op, cmp):
    x = ds.gaussian_latent(3000, dim, seed=dim)
    x[::7] = np.inf      # absent vectors
    x[3::11] = 0.0       # zero norm: NULL under cosine
    q = ds.gaussian_latent(12, dim, seed=dim + 1)
    q[5] = 0.0           # a zero literal: NULL for every row under cosine
    radii = radii_admitting(np.where(np.isfinite(x), x, 0), q, op, [0, 10, 200, -1] * 3)
    idx = table_index(x)
    for limit, offset in ((20, 0), (0, 0), (7, 5)):
        assert_same(VectorRangeScanBatch(idx, op, cmp, limit, offset).execute(q, radii),
                    reference(x, q, op, cmp, radii, limit, offset))
    idx.close()


def test_finite_table_with_odd_dim_stays_on_the_filter(gpu_required, reference):
    x = ds.gaussian_latent(9000, 37, seed=3)
    x[4::13] = 0.0
    q = ds.gaussian_latent(16, 37, seed=4)
    for op, cmp in NEAR:
        radii = radii_admitting(x, q, op, [0, 5, 50, 500] * 4)
        idx = table_index(x)
        assert_same(VectorRangeScanBatch(idx, op, cmp, 40, 1).execute(q, radii), reference(x, q, op, cmp, radii, 40, 1))
        idx.close()


def test_empty_index_and_rejections(gpu_required):
    idx = table_index(np.zeros((0, 8), np.float32))
    rows, vals, counts = VectorRangeScanBatch(idx, VectorOp.CosineDistance, RangeCmp.Lt, 4).execute(np.ones((3, 8), np.float32),
                                                                                                      [0.5, 1.0, 2.0])
    assert (counts == 0).all() and (rows == INVALID_ROW).all() and np.isnan(vals).all()
    idx.close()
    from turdb_b200 import _lib
    x = ds.gaussian_latent(100, 8, seed=1)
    idx = table_index(x)
    L = _lib.load()
    q = np.ascontiguousarray(x[:1])
    r = np.ones(1)
    rows = np.zeros(4, np.uint64)
    cnt = np.zeros(1, np.uint32)
    args = lambda dim, op, cmp: (idx._h, q.ctypes.data_as(C.POINTER(C.c_float)), dim, 1, op, cmp,  # noqa: E731
                                 r.ctypes.data_as(C.POINTER(C.c_double)), 4, 0, rows.ctypes.data_as(C.POINTER(C.c_uint64)),
                                 None, cnt.ctypes.data_as(C.POINTER(C.c_uint32)))
    assert L.turdb_cuda_sql_range_batch(*args(7, 0, 0)) == _lib.ERR_DIMENSION_MISMATCH
    for op, cmp in ((0, 2), (0, 3), (1, 2), (1, 3), (2, 0), (2, 1)):
        assert L.turdb_cuda_sql_range_batch(*args(8, op, cmp)) == _lib.ERR_UNSUPPORTED
    assert L.turdb_cuda_sql_range_batch(*args(8, 3, 0)) == _lib.ERR_INVALID_ARGUMENT
    assert L.turdb_cuda_sql_range_batch(*args(8, 0, 4)) == _lib.ERR_INVALID_ARGUMENT
    assert L.turdb_cuda_sql_range_batch(*args(8, 0, 1)) == _lib.OK  # out_vals may be NULL
    idx.close()


@pytest.mark.parametrize("env", [{"TURDB_EXACT_PAIR": "0"}, {"TURDB_EXACT_PAIR": "1"}, {"TURDB_EXACT_FORCE_BF16": "1"}])
def test_filter_forms_give_identical_results(gpu_required, reference, monkeypatch, env):
    x = ds.gaussian_latent(20_000, 192, seed=51)
    q = ds.gaussian_latent(40, 192, seed=52)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    for op, cmp in (NEAR[0], NEAR[3], NEAR[5]):
        radii = radii_admitting(x, q, op, [0, 10, 1000, 3000, -1] * 8)
        idx = table_index(x)  # a fresh index: the 16-bit copies (FP16 or BF16) are built on its first call
        assert_same(VectorRangeScanBatch(idx, op, cmp, 25, 3).execute(q, radii), reference(x, q, op, cmp, radii, 25, 3))
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
        for op, cmp in (NEAR[1], NEAR[2], NEAR[4]):
            radii = radii_admitting(x[:n], q, op, [0, 10, 300, -1] * 6)
            assert_same(VectorRangeScanBatch(idx, op, cmp, 30).execute(q, radii),
                        reference(x[:n], q, op, cmp, radii, 30), rid[:n])
    idx.close()


def test_topk_is_unchanged_by_range_calls(gpu_required):
    x = ds.gaussian_latent(20_000, 96, seed=71)
    q = ds.gaussian_latent(64, 96, seed=72)
    idx = table_index(x)
    before = [VectorScanBatch(idx, op, 10, 2).execute(q) for op in (VectorOp.L2Distance, VectorOp.CosineDistance)]
    for op, cmp in NEAR:
        VectorRangeScanBatch(idx, op, cmp, 10).execute(q, radii_admitting(x, q, op, [10, -1] * 32))
    after = [VectorScanBatch(idx, op, 10, 2).execute(q) for op in (VectorOp.L2Distance, VectorOp.CosineDistance)]
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
    op = VectorRangeScanBatch(idx, VectorOp.CosineDistance, RangeCmp.Le, 12, 1)
    rows, vals, counts = op.execute(q, radii)
    dq, dr = torch.from_numpy(q).cuda(), torch.from_numpy(radii).cuda()
    d_rows = torch.empty((16, 12), dtype=torch.int64, device="cuda")
    d_vals = torch.empty((16, 12), dtype=torch.float64, device="cuda")
    d_cnt = torch.empty(16, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream()
    op.execute_device(dq.data_ptr(), 16, dr.data_ptr(), d_rows.data_ptr(), d_cnt.data_ptr(), s.cuda_stream, d_vals.data_ptr())
    s.synchronize()
    assert np.array_equal(d_rows.cpu().numpy().view(np.uint64), rows)
    assert np.array_equal(d_vals.cpu().numpy().view(np.uint64), vals.view(np.uint64))
    assert np.array_equal(d_cnt.cpu().numpy().view(np.uint32), counts)
    idx.close()
