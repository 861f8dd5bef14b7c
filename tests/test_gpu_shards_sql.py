"""turdb_cuda_shards_sql_topk_batch (csrc/sql_shards.inl): `ORDER BY vec <op> '[...]' LIMIT k OFFSET o` over a table split
into sub-indexes.  The table is shard 0's live rows, then shard 1's, ...; every output is compared, bit for bit, with
turdb_cuda_sql_topk_batch (exact scan) on ONE index that holds that concatenation, and a small case with the oracle's
TopKExec.  Exact results do not depend on the graph, so most shards are graph-less tables."""
import ctypes as C

import numpy as np
import pytest

from oracle import binding as ob
from turdb_b200 import _lib
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import CudaHnswIndex, _check
from turdb_b200.sql_operator import ShardedVectorScanBatch, VectorOp, VectorScanBatch

pytestmark = pytest.mark.gpu

L2, COS = VectorOp.L2Distance, VectorOp.CosineDistance


def table_index(x, row_ids, device=0):
    """A table without an HNSW graph: the exact scan only needs the arena (entry = none)."""
    n = x.shape[0]
    g = dict(vectors=x, row_ids=row_ids, levels=np.zeros(n, np.uint8), l0_adj=np.full((n, 32), 0xFFFFFFFF, np.uint32),
             l0_cnt=np.zeros(n, np.uint8), up_base=np.full(n, 0xFFFFFFFF, np.uint32), up_adj=np.zeros((0, 16), np.uint32),
             up_cnt=np.zeros(0, np.uint8), entry=0 if n else 0xFFFFFFFF, max_level=0)
    return CudaHnswIndex.from_graph(g, device=device)


class Split:
    """Rows x (row ids 3i + 7) cut into consecutive shards of the given sizes; `deleted[s]` = node ids deleted in shard s."""

    def __init__(self, x, sizes, deleted=None, devices=None, build=False):
        assert sum(sizes) == len(x)
        self.x, self.ids = x, np.arange(len(x), dtype=np.uint64) * 3 + 7
        cut = np.concatenate([[0], np.cumsum(sizes)]).astype(int)
        self.parts = [(self.x[a:b], self.ids[a:b]) for a, b in zip(cut[:-1], cut[1:])]
        devices = devices or [0] * len(sizes)
        if build:
            self.shards = [CudaHnswIndex.build(px, pid, m=8, ef_construction=64, device=d) for (px, pid), d in zip(self.parts, devices)]
        else:
            self.shards = [table_index(px, pid, d) for (px, pid), d in zip(self.parts, devices)]
        self.live = [np.ones(len(px), bool) for px, _ in self.parts]
        for s, nodes in (deleted or {}).items():
            self.shards[s].delete(np.asarray(nodes, np.uint32))
            self.live[s][np.asarray(nodes, int)] = False
        self.cat_x = np.concatenate([px[m] for (px, _), m in zip(self.parts, self.live)])
        self.cat_ids = np.concatenate([pid[m] for (_, pid), m in zip(self.parts, self.live)])
        self.one = table_index(self.cat_x, self.cat_ids)

    def close(self):
        for s in self.shards + [self.one]:
            s.close()


def assert_same(split, q, op, limit, offset=0, project=None):
    got_b = ShardedVectorScanBatch(split.shards, op, limit, offset, project=project)
    rows, keys, counts = got_b.execute(q)
    want_b = VectorScanBatch(split.one, op, limit, offset, project=project)
    w_rows, w_keys, w_counts = want_b.execute(q)
    assert np.array_equal(counts, w_counts)
    assert np.array_equal(keys.view(np.uint64), w_keys.view(np.uint64))  # f64 key bits; NaN slots included
    nn = np.array([not np.isnan(w_keys[i, :w_counts[i]]).any() for i in range(len(q))], bool)
    assert np.array_equal(rows[nn], w_rows[nn])  # order among NULL keys is unspecified
    for i in np.flatnonzero(~nn):
        assert sorted(rows[i].tolist()) == sorted(w_rows[i].tolist())
    if project is not None:
        assert np.array_equal(got_b.projected[nn].view(np.uint64), want_b.projected[nn].view(np.uint64))
    return rows, keys, counts


SIZES = {1: [3000], 2: [1800, 2200], 3: [1500, 7, 2500], 8: [900, 0, 5, 1200, 1, 1700, 300, 900]}


@pytest.mark.parametrize("n_shards", [1, 2, 3, 8])
@pytest.mark.parametrize("op", [L2, COS])
def test_matches_one_index_of_the_concatenation(gpu_required, n_shards, op):
    sizes = SIZES[n_shards]
    x = ds.gaussian_latent(sum(sizes), 64, seed=60 + n_shards)
    q = ds.gaussian_latent(48, 64, seed=70 + n_shards)
    sp = Split(x, sizes)
    for limit, offset in ((10, 0), (1, 0), (5, 7), (64, 3)):
        assert_same(sp, q, op, limit, offset)
    assert_same(sp, q, op, 0, 4)  # limit 0: counts 0
    sp.close()


@pytest.mark.parametrize("op,project", [(L2, L2), (L2, COS), (L2, VectorOp.InnerProduct), (COS, COS), (COS, L2),
                                        (COS, VectorOp.InnerProduct)])
def test_projected_values(gpu_required, op, project):
    x = ds.gaussian_latent(4000, 48, seed=81)
    x[1500] = 0.0  # a zero norm projects NULL under <=>
    q = np.concatenate([ds.gaussian_latent(20, 48, seed=82), x[1500:1501] + 1e-3])
    sp = Split(x, [1000, 1200, 1800])
    assert_same(sp, q, op, 12, 2, project=project)
    sp.close()


def test_largest_window(gpu_required):
    x = ds.gaussian_latent(3000, 32, seed=83)
    q = ds.gaussian_latent(16, 32, seed=84)
    sp = Split(x, [400, 1100, 1500])
    for op in (L2, COS):
        assert_same(sp, q, op, 500, 12)
        assert_same(sp, q, op, 1, 511)
        assert_same(sp, q, op, 512, 0, project=op)
    sp.close()


def test_ties_across_shard_boundaries(gpu_required):
    """Duplicate rows in several shards and integer-valued (SIFT-shaped) rows: many exactly equal keys inside and across
    the LIMIT boundary, in every shard.  Which survive and in which order follows from the heap procedure alone."""
    rng = np.random.default_rng(5)
    x = rng.integers(0, 4, (6000, 6)).astype(np.float32)
    q = rng.integers(0, 4, (40, 6)).astype(np.float32)
    x[100:140] = x[3000:3040] = x[5900:5940] = q[0]  # the same rows as the literal in three shards
    sp = Split(x, [2000, 1000, 3000])
    for op in (L2, COS):
        for limit, offset in ((10, 0), (7, 5), (100, 20), (300, 212)):
            assert_same(sp, q, op, limit, offset)
    sp.close()
    s = ds.sift_like(5000, 128, seed=6)
    sp = Split(s, [1700, 1600, 1700])
    assert_same(sp, s[::250] + 1.0, L2, 10)
    assert_same(sp, s[::250], L2, 25, 5)
    sp.close()


@pytest.mark.parametrize("where", ["one", "all"])
def test_mass_duplicates_take_the_streaming_relay(gpu_required, where, monkeypatch, capfd):
    """Thousands of duplicates of the nearest row overflow the candidate buffers: those shards run the reference's loop
    over every row from the relayed heap, the others replay their candidates; the result does not change."""
    x = ds.gaussian_latent(15000, 32, seed=41)
    x[600:4600] = x[599]
    if where == "all":
        x[5500:9500] = x[599]
        x[10500:14500] = x[599]
    q = np.concatenate([x[599:600] + 1e-3, ds.gaussian_latent(5, 32, seed=42)])
    sp = Split(x, [5000, 5000, 5000])
    monkeypatch.setenv("TURDB_EXACT_VERBOSE", "1")
    for limit, offset in ((10, 0), (25, 10)):
        assert_same(sp, q, L2, limit, offset)
    err = capfd.readouterr().err
    fb = np.array([int(l.split("fallback=")[1].split()[0]) for l in err.splitlines() if "[turdb shards_topk shard" in l])
    fb = fb.reshape(2, 3)  # [call][shard]
    if where == "all":
        assert (fb >= 1).all()
    else:
        assert (fb[:, 0] >= 1).all() and (fb[:, 1:] == 0).all()
    sp.close()


def test_null_keys(gpu_required):
    """Zero-norm rows have a NULL `<=>` key.  NULL rows enter the heap only while it fills, after which a NULL root is never
    replaced: here shard 0 holds fewer than limit rows, shard 1 starts with zero-norm rows; and zero-norm rows sit in
    shard 0 and in later shards of a table whose rows are close to the literals."""
    rng = np.random.default_rng(9)
    centre = rng.standard_normal(24).astype(np.float32)
    x = (centre + 0.2 * rng.standard_normal((3000, 24))).astype(np.float32)
    q = (centre + 0.2 * rng.standard_normal((30, 24))).astype(np.float32)
    x[4:10] = 0.0                     # shard 1's first rows (shard 0 = 4 rows)
    x[1000:1003] = 0.0                # later shards
    x[2990:2992] = 0.0
    sp = Split(x, [4, 1200, 1000, 796])
    for limit, offset in ((10, 0), (3, 4), (40, 0)):
        assert_same(sp, q, COS, limit, offset)
    sp.close()
    x3 = (centre + 0.2 * rng.standard_normal((3000, 24))).astype(np.float32)
    x3[[1000, 1001, 1002, 2990, 2991]] = 0.0  # only after the heap has filled with numbers: never enter
    sp = Split(x3, [4, 1200, 1000, 796])
    assert_same(sp, q, COS, 10)
    assert_same(sp, q, COS, 4, 2, project=COS)
    sp.close()
    x2 = x.copy()
    x2[:3] = 0.0                      # zero-norm rows in shard 0
    sp = Split(x2, [1500, 1500])
    assert_same(sp, q, COS, 10)
    assert_same(sp, q, COS, 5, 1)
    sp.close()


def test_deleted_rows(gpu_required):
    x = ds.gaussian_latent(6000, 40, seed=91)
    q = np.concatenate([ds.gaussian_latent(30, 40, seed=92), x[[10, 2100, 4500]]])
    rng = np.random.default_rng(93)
    deleted = {0: np.r_[10, rng.choice(2000, 300, replace=False)], 2: np.arange(1000),   # every row of shard 2
               3: np.r_[500, rng.choice(3000, 1500, replace=False)]}
    sp = Split(x, [2000, 0, 1000, 3000], deleted=deleted)
    for op in (L2, COS):
        for limit, offset in ((10, 0), (30, 5)):
            assert_same(sp, q, op, limit, offset, project=op)
    sp.close()


def test_oracle_topk_executor(gpu_required):
    x = ds.gaussian_latent(5000, 48, seed=31)
    q = ds.gaussian_latent(32, 48, seed=32)
    sp = Split(x, [1234, 2000, 1766])
    for op, oop in ((L2, ob.L2), (COS, ob.COSINE)):
        for limit, offset in ((10, 0), (5, 7)):
            rows, keys, counts = ShardedVectorScanBatch(sp.shards, op, limit, offset).execute(q)
            o_rows, o_keys, o_counts = ob.sql_topk(x, q, limit, op=oop, offset=offset, n_threads=8)
            assert np.array_equal(counts, o_counts)
            assert np.array_equal(rows, sp.ids[o_rows.astype(np.int64)])
            assert np.array_equal(keys.view(np.uint64), o_keys.view(np.uint64))
    sp.close()


def test_shards_built_by_the_insert_path(gpu_required):
    x = ds.gaussian_latent(3000, 32, seed=101)
    q = ds.gaussian_latent(24, 32, seed=102)
    sp = Split(x, [1000, 1200, 800], build=True)
    for op in (L2, COS):
        assert_same(sp, q, op, 10)
    sp.close()


def test_shards_on_several_devices(gpu_required):
    n_dev = C.c_int32(0)
    _check(_lib.load().turdb_cuda_device_count(C.byref(n_dev)))
    if n_dev.value < 2:
        pytest.skip("one visible device")
    x = ds.gaussian_latent(6000, 64, seed=111)
    q = ds.gaussian_latent(40, 64, seed=112)
    devices = [i % n_dev.value for i in range(4)]
    sp = Split(x, [1500, 1000, 2000, 1500], devices=devices)
    for op in (L2, COS):
        assert_same(sp, q, op, 10, 2, project=op)
    sp.close()


def test_dimension_mismatch(gpu_required):
    a = table_index(ds.gaussian_latent(100, 16, seed=1), np.arange(100, dtype=np.uint64))
    b = table_index(ds.gaussian_latent(100, 8, seed=2), np.arange(100, dtype=np.uint64))
    L = _lib.load()
    handles = (C.c_void_p * 2)(a._h, b._h)
    q = np.zeros((2, 16), np.float32)
    rows, keys, cnt = np.zeros(20, np.uint64), np.zeros(20), np.zeros(2, np.uint32)
    rc = L.turdb_cuda_shards_sql_topk_batch(handles, 2, q.ctypes.data_as(C.POINTER(C.c_float)), 16, 2, 10, 0, 0, 0,
                                            rows.ctypes.data_as(C.POINTER(C.c_uint64)),
                                            keys.ctypes.data_as(C.POINTER(C.c_double)), None,
                                            cnt.ctypes.data_as(C.POINTER(C.c_uint32)))
    assert rc == _lib.ERR_DIMENSION_MISMATCH and b"shard 1" in L.turdb_cuda_last_error()
    a.close()
    b.close()
