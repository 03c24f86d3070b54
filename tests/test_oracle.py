"""CPU tests of the oracle itself: known answers the restatement must reproduce (the reference
ships no tests or golden vectors, SURVEY.md section 4, so these KATs are authored here)."""
import os

import numpy as np
import pytest

import golden_inputs
from newsrecommend_b200.parity import compare_topk

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_mt19937_known_answer(oracle):
    # C++ standard, [rand.predef]: the 10000th invocation of a default mt19937 is 4123659995
    assert oracle.mt19937_nth(5489, 10000) == 4123659995


def test_rand_perm_is_permutation_and_seeded(oracle):
    p = oracle.rand_perm(1000, 1234)
    assert sorted(p.tolist()) == list(range(1000))
    assert (p == oracle.rand_perm(1000, 1234)).all()
    assert (p != oracle.rand_perm(1000, 1235)).any()
    g = np.load(os.path.join(GOLDEN, "rand_perm.npz"))
    assert (oracle.rand_perm(20, 1234) == g["perm20_seed1234"]).all()


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("nq", [1, 19, 20, 33])
def test_knn_matches_fp64_truth(oracle, metric, nq):
    rng = np.random.default_rng(nq * 7 + metric)
    xb = rng.standard_normal((3000, 250), dtype=np.float32)
    xq = rng.standard_normal((nq, 250), dtype=np.float32)
    D, I = oracle.knn(xq, xb, 50, metric)
    Dt, It = oracle.truth_topk(xq, xb, 50, metric)
    rep = compare_topk(D, I, Dt, It, metric)
    assert rep["ok"], rep
    # best-first ordering
    s = np.diff(D, axis=1)
    assert (s >= 0).all() if metric == 1 else (s <= 0).all()


def test_knn_query_block_boundary(oracle):
    rng = np.random.default_rng(5)
    xb = rng.standard_normal((1500, 16), dtype=np.float32)
    xq = rng.standard_normal((4097, 16), dtype=np.float32)
    D, I = oracle.knn(xq, xb, 5, 0)
    Dt, It = oracle.truth_topk(xq, xb, 5, 0)
    assert compare_topk(D, I, Dt, It, 0)["ok"]


def test_identity_catalog(oracle):
    d = 32
    xb = np.eye(d, dtype=np.float32)
    xq = (np.eye(d, dtype=np.float32) * 2.0)[:25]
    D, I = oracle.knn(xq, xb, 1, 0)
    assert (I[:, 0] == np.arange(25)).all() and np.allclose(D[:, 0], 2.0)
    D, I = oracle.knn(xq, xb, 1, 1)
    assert (I[:, 0] == np.arange(25)).all() and np.allclose(D[:, 0], 1.0)


@pytest.mark.parametrize("metric", [0, 1])
def test_k_larger_than_ntotal_padding(oracle, metric):
    rng = np.random.default_rng(1)
    xb = rng.standard_normal((7, 12), dtype=np.float32)
    for nq in (3, 40):
        xq = rng.standard_normal((nq, 12), dtype=np.float32)
        D, I = oracle.knn(xq, xb, 10, metric)
        assert (I[:, 7:] == -1).all() and (I[:, :7] >= 0).all()
        pad = np.float32(3.4028234663852886e38)
        assert (D[:, 7:] == (pad if metric == 1 else -pad)).all()
        assert all(sorted(r[:7].tolist()) == list(range(7)) for r in I)


def test_duplicate_rows_ties(oracle):
    rng = np.random.default_rng(2)
    base = rng.standard_normal((50, 20), dtype=np.float32)
    xb = np.concatenate([base, base, base])  # every row three times
    xq = rng.standard_normal((30, 20), dtype=np.float32)
    D, I = oracle.knn(xq, xb, 6, 0)
    for q in range(30):
        assert len(set(I[q].tolist())) == 6
        # top-6 = two triples of identical scores
        assert set((I[q, :3] % 50).tolist()).__len__() == 1 and set((I[q, 3:] % 50).tolist()).__len__() == 1


def test_l2_is_squared_and_clamped(oracle):
    xb = np.array([[3.0, 4.0], [0.0, 0.0]], dtype=np.float32)
    xq = np.zeros((21, 2), dtype=np.float32)
    D, I = oracle.knn(xq, xb, 2, 1)
    assert (I[:, 0] == 1).all() and np.allclose(D[:, 0], 0.0) and np.allclose(D[:, 1], 25.0)
    assert (D >= 0).all()


def test_compute_centroids_and_split(oracle):
    x = np.array([[0, 0], [2, 0], [10, 10], [12, 10], [11, 13]], dtype=np.float32)
    assign = np.array([0, 0, 1, 1, 1])
    cent, h = oracle.compute_centroids(x, assign, 3)
    assert np.allclose(cent[0], [1, 0]) and np.allclose(cent[1], [11, 11]) and (h == [2, 3, 0]).all()
    ns = oracle.split_clusters(cent, h, 5)
    assert ns == 1 and h.sum() == 5 and (h > 0).all()
    # the empty cluster became a +-1/1024 perturbed copy of a populated one
    src = 0 if np.allclose(cent[2], cent[0], rtol=3e-3, atol=1e-6) else 1
    assert np.allclose(cent[2], cent[src], rtol=3e-3, atol=1e-6) and not np.array_equal(cent[2], cent[src])


def test_kmeans_recovers_separated_blobs(oracle):
    rng = np.random.default_rng(3)
    k, d, per = 8, 16, 200
    centers = rng.standard_normal((k, d)).astype(np.float32) * 20
    x = (centers[:, None, :] + 0.1 * rng.standard_normal((k, per, d))).reshape(-1, d).astype(np.float32)
    x = x[rng.permutation(x.shape[0])]
    clus = oracle.Clustering(d, k)
    clus.niter = 20
    index = oracle.IndexFlatL2(d)
    clus.train(x, index)
    cent = clus.centroids.reshape(k, d)
    # Lloyd with random-row init can merge two blobs (a local minimum), but most true centres
    # must have a learned centroid within the noise radius, and the objective never increases
    dist = ((centers[:, None, :] - cent[None, :, :]) ** 2).sum(-1)
    assert (dist.min(axis=1) < 0.5).sum() >= k - 2
    assert index.ntotal == k
    objs = [s.obj for s in clus.iteration_stats]
    assert all(b <= a * (1 + 1e-6) for a, b in zip(objs, objs[1:]))


def test_kmeans_subsample_rule(oracle):
    rng = np.random.default_rng(4)
    x = rng.standard_normal((3000, 8), dtype=np.float32)
    clus = oracle.Clustering(8, 4)  # 3000 > 4*256 -> subsample to 1024 rows with rand_perm(1234)
    sub = clus.subsample(x)
    assert sub.shape == (1024, 8)
    assert np.array_equal(sub, x[oracle.rand_perm(3000, 1234)[:1024]])


def test_kmeans_too_few_points_raises(oracle):
    clus = oracle.Clustering(4, 10)
    with pytest.raises(RuntimeError, match="at least as large as number of clusters"):
        clus.train(np.zeros((5, 4), dtype=np.float32), oracle.IndexFlatL2(4))


@pytest.mark.parametrize("metric", [0, 1])
def test_ivf_full_probe_equals_flat(oracle, metric):
    rng = np.random.default_rng(6)
    xb = rng.standard_normal((2000, 24), dtype=np.float32)
    xq = rng.standard_normal((64, 24), dtype=np.float32)
    quant = oracle.IndexFlatIP(24) if metric == 0 else oracle.IndexFlatL2(24)
    ivf = oracle.IndexIVFFlat(quant, 24, 10, metric)
    with pytest.raises(RuntimeError):
        ivf.add(xb)
    ivf.train(xb)
    ivf.add(xb[:1200])
    ivf.add(xb[1200:])
    assert ivf.ntotal == 2000 and ivf.list_sizes().sum() == 2000
    ivf.nprobe = 10
    D, I = ivf.search(xq, 10)
    Df, If = oracle.knn(xq, xb, 10, metric)
    assert compare_topk(D, I, Df, If, metric)["ok"]
    ivf.nprobe = 1
    D1, I1 = ivf.search(xq, 10)
    # nprobe = 1 returns members of the nearest list only
    _, c = quant.search(xq, 1)
    a = quant.assign(xb)[:, 0]
    for q in range(64):
        got = I1[q][I1[q] >= 0]
        assert (a[got] == c[q, 0]).all()


def test_golden_flat(oracle):
    g = golden_inputs.load("flat_small")
    for metric in (0, 1):
        D, I = oracle.knn(g["xq"], g["xb"], 10, metric)
        assert np.array_equal(I, g[f"I{metric}"])
        assert np.allclose(D, g[f"D{metric}"], rtol=1e-6, atol=1e-6)
        # and the golden ids agree with fp64 truth
        assert np.array_equal(g[f"I{metric}"], g[f"It{metric}"])


def test_golden_ivf(oracle):
    """IVF-Flat fixture: the oracle retrains to the same centroids (deterministic k-means: mt19937
    subsample / init, sequential fp32 sums), builds the same lists and returns the same (D, I)."""
    g = golden_inputs.load("ivf_small")
    for metric, qcls in ((0, oracle.IndexFlatIP), (1, oracle.IndexFlatL2)):
        quant = qcls(64)
        ivf = oracle.IndexIVFFlat(quant, 64, 16, metric)
        ivf.train(g["xb"])
        assert np.allclose(quant.xb, g[f"cent{metric}"], rtol=1e-6, atol=1e-6)
        ivf.add(g["xb"])
        assert np.array_equal(ivf.list_sizes(), g[f"sizes{metric}"])
        ivf.nprobe = 4
        D, I = ivf.search(g["xq"], 10)
        assert np.array_equal(I, g[f"I{metric}"])
        assert np.allclose(D, g[f"D{metric}"], rtol=1e-6, atol=1e-6)


def test_comparator_rejects_wrong_ids():
    D = np.array([[5.0, 4.0, 3.0]])
    I = np.array([[1, 2, 3]])
    assert compare_topk(D, I, D, I, 0)["ok"]
    assert not compare_topk(D, np.array([[1, 3, 2]]), D, I, 0)["ok"]
    # a swap inside a sub-1e-5 gap is exempt
    Dt = np.array([[5.0, 4.0, 4.0 - 1e-6]])
    assert compare_topk(Dt, np.array([[1, 3, 2]]), Dt, I, 0)["ok"]
    # score off by more than 1e-4 relative
    assert not compare_topk(D * (1 + 3e-4), I, D, I, 0)["ok"]


# ------------------------------------------------------------------------------------------------
# Independent cross-checks of the ORACLE itself. faiss is not installable in this image (SURVEY 8c),
# so the restatement is pinned from several independent sides instead: torch CPU (MKL sgemm + topk),
# scikit-learn's brute-force neighbours and Lloyd step, numpy's own MT19937, and a vectorised fp64
# re-derivation of the IVF semantics -- all on the committed golden fixtures.
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("metric", [0, 1])
def test_golden_flat_against_torch_mkl_and_sklearn(metric):
    import torch
    from newsrecommend_b200.parity import compare_topk
    g = golden_inputs.load("flat_small")
    xb, xq = torch.from_numpy(g["xb"]), torch.from_numpy(g["xq"])
    ip = xq @ xb.T  # MKL sgemm: a different BLAS from the OpenBLAS behind the oracle's numpy blocks
    if metric == 0:
        D, I = torch.topk(ip, 10, dim=1, largest=True, sorted=True)
    else:
        d2 = (xq * xq).sum(1, keepdim=True) + (xb * xb).sum(1)[None, :] - 2 * ip
        D, I = torch.topk(d2.clamp_min(0), 10, dim=1, largest=False, sorted=True)
    rep = compare_topk(D.numpy(), I.numpy(), g[f"D{metric}"], g[f"I{metric}"], metric)
    assert rep["ok"], rep
    # fp64 brute force (ordered by (score, id)): the fixture's truth arrays
    rep = compare_topk(g[f"D{metric}"], g[f"I{metric}"], g[f"Dt{metric}"], g[f"It{metric}"], metric)
    assert rep["ok"], rep
    if metric == 1:
        from sklearn.neighbors import NearestNeighbors
        nn = NearestNeighbors(n_neighbors=10, algorithm="brute", metric="euclidean").fit(g["xb"].astype(np.float64))
        dist, idx = nn.kneighbors(g["xq"].astype(np.float64))
        rep = compare_topk(dist ** 2, idx, g["D1"], g["I1"], 1)  # faiss L2 is the SQUARED distance
        assert rep["ok"], rep


def test_rand_perm_against_numpy_mt19937(oracle):
    """std::mt19937(seed) raw outputs == numpy's MT19937 with legacy (init_genrand) seeding; the
    oracle's rand_perm (faiss utils/random.cpp) restated on top of numpy's generator."""
    for n, seed in [(20, 1234), (1000, 1235), (64000, 1234)]:
        bg = np.random.MT19937()
        bg._legacy_seeding(seed)
        raw = bg.random_raw(n)  # 32-bit outputs
        perm = np.arange(n, dtype=np.int64)
        for i in range(n - 1):
            j = i + int(raw[i]) % (n - i)
            perm[i], perm[j] = perm[j], perm[i]
        assert np.array_equal(oracle.rand_perm(n, seed), perm)
    assert np.array_equal(np.load(os.path.join(GOLD, "rand_perm.npz"))["perm20_seed1234"], oracle.rand_perm(20, 1234))


def test_golden_kmeans_iteration_against_sklearn_lloyd():
    """One teacher-forced Lloyd iteration of the golden k-means trace reproduced by scikit-learn
    (init = the recorded input centroids, max_iter = 1): same assignment, same means."""
    from sklearn.cluster import KMeans
    g = golden_inputs.load("kmeans_small")
    xs = g["xs"].astype(np.float64)
    for it in range(g["cin"].shape[0]):
        cin = g["cin"][it].astype(np.float64)
        # assignment by fp64 brute force
        d2 = (xs * xs).sum(1)[:, None] + (cin * cin).sum(1)[None, :] - 2 * xs @ cin.T
        a = d2.argmin(1)
        diff = np.nonzero(a != g["assign"][it])[0]
        for i in diff:  # any disagreement with the fp32 oracle must be a near-tie
            assert abs(d2[i, a[i]] - d2[i, g["assign"][it][i]]) <= 1e-5 * d2[i, a[i]]
        km = KMeans(n_clusters=cin.shape[0], init=cin, n_init=1, max_iter=1, algorithm="lloyd", tol=0.0).fit(xs)
        sizes = np.bincount(g["assign"][it], minlength=cin.shape[0])
        keep = sizes > 0  # (empty clusters: faiss splits, scikit-learn relocates)
        if diff.size == 0:
            assert np.allclose(km.cluster_centers_[keep], g["cout"][it][keep], rtol=2e-5, atol=2e-6)
        means = np.stack([xs[g["assign"][it] == c].mean(0) if sizes[c] else np.zeros(xs.shape[1]) for c in range(cin.shape[0])])
        assert np.allclose(means[keep], g["cout"][it][keep], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("metric", [0, 1])
def test_golden_ivf_against_fp64_rederivation(metric):
    """IndexIVFFlat semantics re-derived in vectorised fp64 numpy from the fixture's centroids:
    items go to their nearest centroid, a query scans the nprobe = 4 best lists, top-10 by score."""
    from newsrecommend_b200.parity import compare_topk
    g = golden_inputs.load("ivf_small")
    xb, xq, cent = g["xb"].astype(np.float64), g["xq"].astype(np.float64), g[f"cent{metric}"].astype(np.float64)

    def coarse(x):  # larger is better
        return x @ cent.T if metric == 0 else -((x * x).sum(1)[:, None] + (cent * cent).sum(1)[None, :] - 2 * x @ cent.T)

    item_list = coarse(xb).argmax(1)
    assert np.array_equal(np.bincount(item_list, minlength=cent.shape[0]), g[f"sizes{metric}"])
    probe = np.argsort(-coarse(xq), axis=1, kind="stable")[:, :4]
    D = np.empty((xq.shape[0], 10))
    I = np.empty((xq.shape[0], 10), dtype=np.int64)
    for q in range(xq.shape[0]):
        sel = np.nonzero(np.isin(item_list, probe[q]))[0]
        sc = xb[sel] @ xq[q] if metric == 0 else ((xb[sel] - xq[q]) ** 2).sum(1)
        o = np.argsort(-sc if metric == 0 else sc, kind="stable")[:10]
        D[q], I[q] = sc[o], sel[o]
    rep = compare_topk(g[f"D{metric}"], g[f"I{metric}"], D, I, metric)
    assert rep["ok"], rep
