"""Exact path (tensor-core BF16 pass + FP32 rerank) vs the oracle's exact scan and vs the HNSW distance
contract.  Tolerance: the north_star's 1e-5 relative FP32 bound on distances; id sets must match except where
the boundary distance is tied within that tolerance."""
import numpy as np
import pytest

from oracle import binding as ob
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction

pytestmark = pytest.mark.gpu
REL_TOL = 1e-5


def exact_reference(x, q, k, metric):
    """k smallest oracle distances (AVX2 lane order), ties by node id."""
    out_ids = np.zeros((len(q), k), np.uint32)
    out_d = np.zeros((len(q), k), np.float32)
    for i, qq in enumerate(q):
        d = np.array([ob.distance(metric, qq, v) for v in x], np.float32)
        order = np.lexsort((np.arange(len(x)), d))[:k]
        out_ids[i], out_d[i] = order, d[order]
    return out_ids, out_d


def flat_graph(x):
    n = len(x)
    return dict(vectors=x, row_ids=np.arange(n, dtype=np.uint64) + 5, levels=np.zeros(n, np.uint8),
                l0_adj=np.full((n, 32), 0xFFFFFFFF, np.uint32), l0_cnt=np.zeros(n, np.uint8),
                up_base=np.full(n, 0xFFFFFFFF, np.uint32), up_adj=np.zeros((0, 16), np.uint32),
                up_cnt=np.zeros(0, np.uint8), entry=0, max_level=0)


@pytest.mark.parametrize("n,dim,nq,k", [(3000, 128, 40, 10), (5000, 384, 200, 10), (2500, 100, 17, 5), (700, 64, 130, 100),
                                        (2000, 768, 150, 10), (1500, 520, 33, 7)])  # > 512 dims: streamed query block
def test_exact_topk_matches_reference(gpu_required, n, dim, nq, k):
    x = ds.gaussian_latent(n, dim, seed=n, normalise=False)
    q = ds.gaussian_latent(nq, dim, seed=n + 1, normalise=False)
    idx = CudaHnswIndex.from_graph(flat_graph(x))
    for metric in (ob.L2, ob.COSINE, ob.IP):
        rows, nodes, dist, cnt = idx.bruteforce_topk(q, k, DistanceFunction(metric), rerank_factor=4)
        ref_ids, ref_d = exact_reference(x, q[:16], k, metric)
        assert (cnt == min(k, n)).all()
        assert np.array_equal(rows, nodes.astype(np.uint64) + 5)
        for i in range(16):
            # reranked distances are the reference's own arithmetic: equal bit for bit where ids agree
            same = nodes[i] == ref_ids[i]
            assert np.array_equal(dist[i][same].view(np.uint32), ref_d[i][same].view(np.uint32))
            if not same.all():  # any id difference must sit on a (near-)tie
                assert np.allclose(dist[i], ref_d[i], rtol=REL_TOL, atol=1e-6), (metric, i)
        assert (np.diff(dist, axis=1) >= 0).all()
    idx.close()


@pytest.mark.parametrize("env", [{"TURDB_EXACT_PAIR": "0"}, {"TURDB_EXACT_PAIR": "1"}, {"TURDB_EXACT_GROWTH": "2"},
                                 {"TURDB_EXACT_PAIR": "0", "TURDB_EXACT_GROWTH": "7"}])
def test_every_form_of_the_filter_gives_the_same_answer(gpu_required, monkeypatch, env):
    """One-CTA (cta_group::1) and two-CTA (cta_group::2) kernels, other slice growths: switches the library reads per call.
    The answer must not depend on any of them — ids and distance bits equal to the default configuration's and to the
    reference's exact top-k."""
    n, nq, k = 6000, 300, 10  # 300 queries: a second (partly empty) query block in both forms
    for dim in (96, 384):
        x = ds.gaussian_latent(n, dim, seed=dim, normalise=False)
        q = ds.gaussian_latent(nq, dim, seed=dim + 1, normalise=False)
        idx = CudaHnswIndex.from_graph(flat_graph(x))
        for metric in (ob.L2, ob.COSINE, ob.IP):
            base = idx.bruteforce_topk(q, k, DistanceFunction(metric))
            with monkeypatch.context() as m:
                for key, val in env.items():
                    m.setenv(key, val)
                got = idx.bruteforce_topk(q, k, DistanceFunction(metric))
            assert np.array_equal(got[1], base[1]) and np.array_equal(got[2].view(np.uint32), base[2].view(np.uint32)), (dim, metric, env)
            ref_ids, ref_d = exact_reference(x, q[:8], k, metric)
            for i in range(8):
                same = got[1][i] == ref_ids[i]
                assert np.array_equal(got[2][i][same].view(np.uint32), ref_d[i][same].view(np.uint32))
                if not same.all():
                    assert np.allclose(got[2][i], ref_d[i], rtol=REL_TOL, atol=1e-6), (dim, metric, i)
        idx.close()


def test_exact_sql_known_answers(gpu_required):
    """The reference's SQL k-NN answers (tests/hnsw_integration.rs:220-276) through the exact path."""
    x = np.array([[.1] * 4, [.5] * 4, [.9] * 4], np.float32)
    idx = CudaHnswIndex.from_graph(flat_graph(x))
    rows, nodes, dist, cnt = idx.bruteforce_topk(np.array([[.1] * 4], np.float32), 2, DistanceFunction.L2)
    assert nodes[0].tolist() == [0, 1] and cnt[0] == 2
    idx.close()
    x20 = np.array([[i / 20.0] * 4 for i in range(20)], np.float32)
    idx = CudaHnswIndex.from_graph(flat_graph(x20))
    rows, nodes, dist, cnt = idx.bruteforce_topk(np.array([[.5] * 4], np.float32), 3, DistanceFunction.L2)
    assert 8 <= nodes[0][0] <= 12 and cnt[0] == 3
    # agrees with the oracle's SQL TopK scan on the id set (SQL reports sqrt of the same squared distance)
    srows, sdist, _ = ob.sql_topk(x20, np.array([.5] * 4, np.float32), 3)
    assert set(srows[0].tolist()) == set(nodes[0].tolist())
    assert np.allclose(np.sqrt(dist[0].astype(np.float64)), sdist[0], rtol=1e-6)
    idx.close()


def test_exact_recall_against_sql_scan(gpu_required):
    x = ds.gaussian_latent(20000, 128, seed=3, normalise=True)
    q = ds.gaussian_latent(64, 128, seed=4, normalise=True)
    idx = CudaHnswIndex.from_graph(flat_graph(x))
    rows, nodes, dist, cnt = idx.bruteforce_topk(q, 10, DistanceFunction.Cosine)
    srows, _, _ = ob.sql_topk(x, q, 10, op=ob.COSINE, n_threads=8)
    rec = np.mean([len(set(nodes[i].tolist()) & set(srows[i].tolist())) / 10 for i in range(len(q))])
    assert rec >= 0.999
    idx.close()


def test_rows_closer_than_bf16_resolution_are_not_lost(gpu_required):
    """Adversarial for the BF16 filter: 600 rows within 1e-4 (relative) of one another around the query — far below
    BF16's 2^-8 resolution, so their filter keys collapse — among 6000 ordinary rows.  The certified filter widens its
    threshold by the score-error bound, so the FP32 rerank must still return exactly the reference's top-k."""
    rng = np.random.default_rng(0)
    dim, n = 96, 6000
    x = ds.gaussian_latent(n, dim, seed=21, normalise=False)
    centre = x[17].copy()
    near = rng.choice(np.arange(100, n), 600, replace=False)
    x[near] = centre * (1.0 + 1e-4 * rng.standard_normal((600, 1)).astype(np.float32)) \
        + 1e-4 * rng.standard_normal((600, dim)).astype(np.float32)
    q = np.stack([centre * (1.0 + 1e-4 * rng.standard_normal()) + 1e-4 * rng.standard_normal(dim).astype(np.float32)
                  for _ in range(24)]).astype(np.float32)
    idx = CudaHnswIndex.from_graph(flat_graph(x))
    for metric in (ob.L2, ob.COSINE, ob.IP):
        for k, rf in ((10, 4), (10, 1), (50, 2)):
            rows, nodes, dist, cnt = idx.bruteforce_topk(q, k, DistanceFunction(metric), rerank_factor=rf)
            ref_ids, ref_d = exact_reference(x, q, k, metric)
            assert np.array_equal(dist.view(np.uint32), ref_d.view(np.uint32)), (metric, k, rf)
            assert np.array_equal(nodes, ref_ids), (metric, k, rf)
    idx.close()


def test_mass_duplicates_fall_back_to_the_scan(gpu_required):
    """3000 identical rows tie at distance 0: more equal keys than the candidate buffer holds.  The flagged queries are
    redone by the streaming FP32 scan; ties order by node id."""
    dim, n = 64, 8000
    x = ds.gaussian_latent(n, dim, seed=5, normalise=False)
    dup = np.arange(1000, 4000)
    x[dup] = x[999]
    q = np.concatenate([x[999:1000], ds.gaussian_latent(7, dim, seed=6, normalise=False)])
    idx = CudaHnswIndex.from_graph(flat_graph(x))
    for metric in (ob.L2, ob.COSINE):
        rows, nodes, dist, cnt = idx.bruteforce_topk(q, 20, DistanceFunction(metric))
        ref_ids, ref_d = exact_reference(x, q, 20, metric)
        assert np.array_equal(nodes, ref_ids) and np.array_equal(dist.view(np.uint32), ref_d.view(np.uint32))
    idx.close()
