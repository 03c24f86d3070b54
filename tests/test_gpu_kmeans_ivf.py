"""GPU parity tests of k-means (K1a assignment via K2, K1b update), list building and the IVF
search (K3) against the oracle. k-means is chaotic under ulp-level changes (SURVEY Appendix
B-E5), so bit-level parity is checked teacher-forced per iteration; free-running runs are
compared on their objective."""
import numpy as np
import pytest

import golden_inputs
from newsrecommend_b200.parity import compare_topk

pytestmark = pytest.mark.gpu


def test_kmeans_update_matches_sequential_fp32(nf, oracle):
    import torch
    rng = np.random.default_rng(0)
    n, d, k = 20000, 250, 37
    x = rng.standard_normal((n, d), dtype=np.float32)
    assign = rng.integers(0, k - 1, size=n)  # cluster k-1 stays empty
    p = nf.PackedMatrix.from_tensor(torch.from_numpy(x).cuda())
    cent, h = nf.kmeans_update(p, torch.from_numpy(assign).cuda(), k)
    co, ho = oracle.compute_centroids(x, assign, k)
    assert np.array_equal(h.cpu().numpy(), ho)
    c = cent.cpu().numpy()
    assert (c[k - 1] == 0).all()
    ref64 = np.stack([x[assign == j].astype(np.float64).mean(0) if (assign == j).any() else np.zeros(d) for j in range(k)])
    assert np.allclose(c, co, rtol=2e-6, atol=2e-7)
    # fp64 accumulation is at least as close to the exact mean as faiss's sequential fp32
    assert np.abs(c - ref64).max() <= np.abs(co - ref64).max() + 1e-7


@pytest.mark.parametrize("n,nlist", [(50001, 300), (1_000_003, 250)])  # one-block scan / grouped scan (> 256 chunks)
def test_build_lists_is_stable_counting_sort(nf, n, nlist):
    import torch
    from newsrecommend_b200._lib import check, lib
    rng = np.random.default_rng(1)
    a = rng.integers(0, nlist, size=n)
    at = torch.from_numpy(a).cuda()
    off = torch.empty(nlist + 1, dtype=torch.int32, device="cuda")
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    wsb = lib.nrb_ivf_build_lists_workspace(n, nlist)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    check(lib.nrb_ivf_build_lists(at.data_ptr(), n, nlist, off.data_ptr(), order.data_ptr(), ws.data_ptr(), wsb, None))
    torch.cuda.synchronize()
    assert np.array_equal(order.cpu().numpy(), np.argsort(a, kind="stable"))
    assert np.array_equal(off.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(a, minlength=nlist))]))


def test_kmeans_teacher_forced_against_golden(nf):
    """Each recorded oracle iteration: same input centroids -> same assignments (modulo the gap
    rule) and new centroids within 1e-6 relative."""
    import torch
    g = golden_inputs.load("kmeans_small")
    x = g["xs"]  # the rows the oracle iterated on (rand_perm subsample of g["x"])
    assert np.array_equal(x, g["x"][nf.rand_perm(g["x"].shape[0], 1234)[: x.shape[0]]])
    p = nf.PackedMatrix.from_tensor(torch.from_numpy(x).cuda())
    for it in range(g["cin"].shape[0]):
        index = nf.IndexFlatL2(x.shape[1])
        index.add(g["cin"][it])
        D, I = index.search_packed(p, 1)
        a = I.reshape(-1).cpu().numpy()
        ref = g["assign"][it]
        diff = np.nonzero(a != ref)[0]
        # any disagreement must be a near-tie between the two centroids
        for i in diff:
            d1 = ((x[i] - g["cin"][it][a[i]]) ** 2).sum()
            d2 = ((x[i] - g["cin"][it][ref[i]]) ** 2).sum()
            assert abs(d1 - d2) <= 1e-5 * max(d1, d2), (it, i, d1, d2)
        cent, h = nf.kmeans_update(p, torch.from_numpy(ref).cuda(), g["cin"].shape[1])
        assert np.allclose(cent.cpu().numpy(), g["cout"][it], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("metric", [0, 1])
def test_clustering_free_running_objective(nf, oracle, metric):
    from newsrecommend_b200 import synth
    x = synth.g_skew(30000, 250, 5, n_topics=100)
    k = 50  # 30000 > 50*256 -> exercises the rand_perm subsample
    outs = []
    for mod in (nf, oracle):
        clus = mod.Clustering(250, k)
        clus.niter = 10
        index = mod.IndexFlatIP(250) if metric == 0 else mod.IndexFlatL2(250)
        clus.train(x, index)
        assert index.ntotal == k
        outs.append((clus.centroids.reshape(k, 250).copy(), [s.obj for s in clus.iteration_stats],
                     [s.nsplit for s in clus.iteration_stats]))
    (c_g, o_g, s_g), (c_o, o_o, s_o) = outs
    # same subsample + init => first iteration objective agrees tightly, final within 1e-3
    assert abs(o_g[0] - o_o[0]) <= 1e-4 * abs(o_o[0])
    assert abs(o_g[-1] - o_o[-1]) <= 1e-3 * abs(o_o[-1])
    assert s_g[0] == s_o[0]


def test_clustering_split_path_and_errors(nf):
    rng = np.random.default_rng(3)
    # 40 distinct points repeated: k close to the number of distinct rows forces empty clusters
    base = rng.standard_normal((40, 16), dtype=np.float32)
    x = np.repeat(base, 30, axis=0)
    clus = nf.Clustering(16, 60)
    clus.niter = 5
    index = nf.IndexFlatL2(16)
    clus.train(x, index)
    assert index.ntotal == 60 and clus.centroids.shape == (60 * 16,)
    assert sum(s.nsplit for s in clus.iteration_stats) > 0
    with pytest.raises(RuntimeError, match="at least as large as number of clusters"):
        nf.Clustering(16, 100).train(x[:50], nf.IndexFlatL2(16))
    bad = x.copy()
    bad[3, 2] = np.nan
    with pytest.raises(RuntimeError, match="NaN"):
        nf.Clustering(16, 4).train(bad, nf.IndexFlatL2(16))


def _classify_ivf_mismatches(ivf_o, xq, nprobe, k, D, I, Do, Io, metric, gap=1e-5):
    """Fails unless every query whose row differs from the oracle's is explained by a near-tie at
    the coarse boundary: brute force (fp64) over each admissible probe set must reproduce the row."""
    import itertools
    off, ids, rows = ivf_o._build_csr()
    cent = ivf_o.quantizer.xb.astype(np.float64)
    explained = 0
    for q in range(xq.shape[0]):
        if compare_topk(D[q:q + 1], I[q:q + 1], Do[q:q + 1], Io[q:q + 1], metric)["ok"]:
            continue
        x = xq[q].astype(np.float64)
        cs = cent @ x if metric == 0 else -((cent - x) ** 2).sum(1)  # larger is better
        order = np.argsort(-cs, kind="stable")
        kth, nxt = cs[order[nprobe - 1]], cs[order[nprobe]]
        scale = max(abs(kth), (x * x).sum() if metric else 0.0, 1e-30)
        assert abs(kth - nxt) <= gap * scale, ("no coarse near-tie explains query", q, kth, nxt)
        lo = kth + gap * scale  # surely probed: better than the boundary by more than the gap
        sure = [l for l in order if cs[l] > lo]
        tie = [l for l in order if abs(cs[l] - kth) <= gap * scale]
        ok = False
        for pick in itertools.combinations(tie, nprobe - len(sure)):
            lists = sure + list(pick)
            sel = np.concatenate([np.arange(off[l], off[l + 1]) for l in lists])
            xr = rows[sel].astype(np.float64)
            sc = xr @ x if metric == 0 else ((xr - x) ** 2).sum(1)
            o = np.argsort(-sc if metric == 0 else sc, kind="stable")[:k]
            Dt = np.full((1, k), -3.4028235e38 if metric == 0 else 3.4028235e38)
            It = np.full((1, k), -1, dtype=np.int64)
            Dt[0, :len(o)], It[0, :len(o)] = sc[o], ids[sel][o]
            if compare_topk(D[q:q + 1], I[q:q + 1], Dt, It, metric)["ok"]:
                ok = True
                break
        assert ok, ("row matches no admissible probe set", q)
        explained += 1
    return explained


def _same_centroids_ivf(nf, oracle, xb, nlist, metric, path):
    quant_o = oracle.IndexFlatIP(xb.shape[1]) if metric == 0 else oracle.IndexFlatL2(xb.shape[1])
    ivf_o = oracle.IndexIVFFlat(quant_o, xb.shape[1], nlist, metric)
    ivf_o.train(xb)
    cent = quant_o.xb.copy()
    quant_g = nf.IndexFlatIP(xb.shape[1]) if metric == 0 else nf.IndexFlatL2(xb.shape[1])
    quant_g.add(cent)  # teacher-forced: identical coarse quantizer
    ivf_g = nf.IndexIVFFlat(quant_g, xb.shape[1], nlist, metric)
    ivf_g.path = path
    ivf_g.train(xb)  # quantizer already holds nlist centroids -> no retraining (faiss semantics)
    assert ivf_g.is_trained
    ivf_o.add(xb)
    ivf_g.add(xb[: len(xb) // 3])
    ivf_g.add(xb[len(xb) // 3:])
    return ivf_g, ivf_o


@pytest.mark.parametrize("path", [4, 2, 1, 0])  # fp16 filter + refine, 3xTF32, SIMT, auto
@pytest.mark.parametrize("metric", [0, 1])
def test_ivf_search_against_oracle(nf, oracle, metric, path):
    from newsrecommend_b200 import synth
    xb, topics = synth.g_skew(40000, 250, 21, n_topics=120, return_topics=True)
    xq = synth.user_profiles(xb, topics, 700, 22)
    ivf_g, ivf_o = _same_centroids_ivf(nf, oracle, xb, 64, metric, path)
    assert np.array_equal(ivf_g.list_sizes(), ivf_o.list_sizes())
    for nprobe in (1, 8):
        ivf_g.nprobe = ivf_o.nprobe = nprobe
        D, I = ivf_g.search(xq, 50)
        Do, Io = ivf_o.search(xq, 50)
        rep = compare_topk(D, I, Do, Io, metric)
        if not rep["ok"]:
            # every disagreement must be a COARSE-boundary near-tie (the nprobe-th and (nprobe+1)-th
            # centroid scores within 1e-5 relative, so a valid implementation may probe either list),
            # and the GPU row must be the exact answer for one of the admissible probe sets
            _classify_ivf_mismatches(ivf_o, xq, nprobe, 50, D, I, Do, Io, metric)
    # nprobe = nlist is an exact search (strongest IVF check)
    ivf_g.nprobe = 64
    D, I = ivf_g.search(xq, 50)
    Df, If = oracle.knn_fast(xq, xb, 50, metric)
    rep = compare_topk(D, I, Df, If, metric)
    assert rep["ok"], rep


def test_ivf_untrained_empty_and_small(nf, oracle):
    rng = np.random.default_rng(4)
    xb = rng.standard_normal((500, 20), dtype=np.float32)
    ivf = nf.IndexIVFFlat(nf.IndexFlatL2(20), 20, 8)
    with pytest.raises(RuntimeError):
        ivf.add(xb)
    with pytest.raises(RuntimeError):
        ivf.search(xb[:2], 1)
    ivf.train(xb)
    D, I = ivf.search(xb[:3], 4)
    assert (I == -1).all()
    ivf.add(xb)
    ivf.nprobe = 8
    D, I = ivf.search(xb[:100], 1)
    assert (I[:, 0] == np.arange(100)).all() and np.allclose(D[:, 0], 0, atol=1e-4)
    ivf.reset()
    assert ivf.ntotal == 0


def test_ivf_end_to_end_train_quality(nf, oracle):
    """Free-running IndexIVFFlat.train/add/search on the skewed generator: list-size skew like
    the README table (no singleton lists) and recall vs exact search comparable to the oracle's."""
    from newsrecommend_b200 import synth
    from newsrecommend_b200.parity import recall_at_k
    xb, topics = synth.g_skew(80000, 250, 31, return_topics=True)
    xq = synth.user_profiles(xb, topics, 500, 32)
    res = []
    for mod in (nf, oracle):
        ivf = mod.IndexIVFFlat(mod.IndexFlatIP(250), 250, 100, mod.METRIC_INNER_PRODUCT)
        ivf.train(xb)
        ivf.add(xb)
        ivf.nprobe = 16
        D, I = ivf.search(xq, 50)
        res.append((ivf.list_sizes(), I))
    _, If = oracle.knn_fast(xq, xb, 50, 0)
    sz_g, sz_o = res[0][0], res[1][0]
    assert sz_g.sum() == 80000 and sz_g.min() > 1
    r_g, r_o = recall_at_k(res[0][1], If), recall_at_k(res[1][1], If)
    assert abs(r_g - r_o) < 0.03 and r_g > 0.5, (r_g, r_o)


def test_ivf_filter_fallback_on_duplicates(nf, oracle):
    """The list scan's fp16 filter with hundreds of exact duplicates in one list: the margin sets
    overflow, the queries are flagged and recomputed by the 3xTF32 scan; still a valid top-k."""
    from newsrecommend_b200._lib import lib
    rng = np.random.default_rng(17)
    base = rng.standard_normal((20, 64), dtype=np.float32)
    xb = np.concatenate([np.repeat(base, 150, axis=0), rng.standard_normal((3000, 64), dtype=np.float32)])
    xq = base + 0.01 * rng.standard_normal((20, 64)).astype(np.float32)
    ivf = nf.IndexIVFFlat(nf.IndexFlatIP(64), 64, 8, nf.METRIC_INNER_PRODUCT)
    ivf.path = 4
    ivf.train(xb)
    ivf.add(xb)
    ivf.nprobe = 8  # = nlist: exact
    n0 = lib.nrb_fallback_query_count()
    D, I = ivf.search(xq, 10)
    assert lib.nrb_fallback_query_count() >= n0 + 20
    for q in range(20):
        assert len(set(I[q].tolist())) == 10 and (I[q] // 150 == q).all()
    Do, Io = oracle.knn_fast(xq, xb, 10, 0)
    assert np.allclose(D, Do, rtol=1e-4)


@pytest.mark.parametrize("path", [4, 2])
def test_ivf_lists_split_into_several_units(nf, oracle, path, monkeypatch):
    """Lists longer than the item run of a unit are scanned as several units whose partial results
    are merged per query: forced here with 512-row runs (default 32,768); nprobe = nlist = exact."""
    monkeypatch.setenv("NRB_IVF_CHUNK", "512")
    from newsrecommend_b200 import synth
    xb, topics = synth.g_skew(30000, 64, 71, n_topics=40, return_topics=True)
    xq = synth.user_profiles(xb, topics, 300, 72)
    ivf = nf.IndexIVFFlat(nf.IndexFlatIP(64), 64, 8, nf.METRIC_INNER_PRODUCT)
    ivf.path = path
    ivf.train(xb)
    ivf.add(xb)
    assert ivf.list_sizes().max() > 2048  # at least five runs in the longest list
    ivf.nprobe = 8
    D, I = ivf.search(xq, 20)
    Do, Io = oracle.knn_fast(xq, xb, 20, 0)
    rep = compare_topk(D, I, Do, Io, 0)
    assert rep["ok"], rep


@pytest.mark.parametrize("path", [0, 4, 2, 1])
@pytest.mark.parametrize("metric", [0, 1])
def test_ivf_golden_fixture(nf, metric, path):
    """tests/golden/ivf_small.npz (written by the oracle): with the fixture's centroids in the coarse
    quantizer the GPU index builds lists of the same sizes and returns the fixture's (D, I)."""
    g = golden_inputs.load("ivf_small")
    quant = nf.IndexFlatIP(64) if metric == 0 else nf.IndexFlatL2(64)
    quant.add(g[f"cent{metric}"])
    ivf = nf.IndexIVFFlat(quant, 64, 16, metric)
    ivf.path = path
    ivf.train(g["xb"])  # the quantizer already holds 16 centroids: no retraining
    ivf.add(g["xb"])
    assert np.array_equal(ivf.list_sizes(), g[f"sizes{metric}"])
    ivf.nprobe = 4
    D, I = ivf.search(g["xq"], 10)
    rep = compare_topk(D, I, g[f"D{metric}"], g[f"I{metric}"], metric)
    assert rep["id_mismatch_queries"] == 0 and rep["score_violations"] == 0, rep


def test_device_split_clusters_equals_host_routine(nf):
    """km_split_kernel (std::mt19937(1234) restated on the device) against nrb_split_clusters_host:
    same splits, same perturbed centroids, bit for bit; plus the imbalance factor."""
    import torch
    from newsrecommend_b200._lib import check, lib
    rng = np.random.default_rng(5)
    for k, d, n_empty in [(60, 16, 7), (300, 256, 1), (300, 250, 40), (1500, 32, 700), (50, 8, 0)]:
        sizes = rng.integers(2, 400, size=k).astype(np.float32)
        empty = rng.choice(k, size=n_empty, replace=False)
        sizes[empty] = 0
        n = int(sizes.sum())
        cent = rng.standard_normal((k, d), dtype=np.float32)
        cent[empty] = 0
        h_host, c_host = sizes.copy(), cent.copy()
        ns = check(lib.nrb_split_clusters_host(d, k, n, h_host.ctypes.data, c_host.ctypes.data))
        h_dev, c_dev = torch.from_numpy(sizes.copy()).cuda(), torch.from_numpy(cent.copy()).cuda()
        st = torch.zeros(4, dtype=torch.float64, device="cuda")
        check(lib.nrb_split_clusters(d, k, n, h_dev.data_ptr(), c_dev.data_ptr(), st.data_ptr(), None))
        st = st.cpu().numpy()
        assert int(st[2]) == ns == n_empty
        assert np.array_equal(h_dev.cpu().numpy(), h_host)
        assert np.array_equal(c_dev.cpu().numpy(), c_host)
        assert abs(st[1] - (sizes.astype(np.float64) ** 2).sum() * k / float(n) ** 2) <= 1e-12 * st[1]


@pytest.mark.parametrize("metric", [0, 1])
def test_fused_trainer_equals_stepwise_trainer(nf, metric):
    """nrb_kmeans_train with niter = 10 in one call == ten calls with niter = 1 (what the trace
    hook of the teacher-forced tests uses) == the same loop built from the separate entry points
    (search k = 1, nrb_kmeans_update, host split_clusters): bit-identical centroids and stats."""
    import torch
    from newsrecommend_b200 import synth
    from newsrecommend_b200._lib import check, lib
    x = synth.g_skew(16_000, 250, 9, n_topics=80)  # <= 256 * k rows: no subsample, so the loop below sees the same rows
    k, niter = 64, 10
    outs = []
    for stepwise in (False, True):
        clus = nf.Clustering(250, k)
        clus.niter = niter
        if stepwise:
            clus.trace = lambda it, cin, a, cout: None
        index = nf.IndexFlatIP(250) if metric == 0 else nf.IndexFlatL2(250)
        clus.train(x, index)
        outs.append((clus.centroids.copy(), [(s.obj, s.imbalance_factor, s.nsplit) for s in clus.iteration_stats]))
        assert index.ntotal == k and np.array_equal(index.reconstruct_n(0, k).reshape(-1), clus.centroids)
    assert np.array_equal(outs[0][0], outs[1][0]) and outs[0][1] == outs[1][1]
    # the loop from the separate entry points
    xt = torch.from_numpy(x).cuda()
    p = nf.PackedMatrix.from_tensor(xt)
    perm = nf.rand_perm(x.shape[0], 1235)[:k]
    cent = xt[torch.from_numpy(perm.astype(np.int64)).cuda()].contiguous()
    for it in range(niter):
        index = nf.IndexFlat(250, metric)
        index.path = nf.PATH_TC
        index.add(cent)
        _, a = index.search_packed(p, 1)
        cent, h = nf.kmeans_update(p, a.reshape(-1), k)
        hh, ch = h.cpu().numpy(), cent.cpu().numpy()
        if (hh == 0).any():
            check(lib.nrb_split_clusters_host(250, k, x.shape[0], hh.ctypes.data, ch.ctypes.data))
            cent = torch.from_numpy(ch).cuda()
    assert np.array_equal(cent.cpu().numpy().reshape(-1), outs[0][0])


def test_kmeans_partial_sums_and_means_equal_update(nf):
    """Data-parallel pieces (nrb_kmeans_partial_sums + nrb_kmeans_means) on one rank: bit-equal to
    nrb_kmeans_update; and the sum of two half-tables gives the same centroids to 1 ulp."""
    import torch
    from newsrecommend_b200._lib import check, lib
    rng = np.random.default_rng(11)
    n, d, k = 20_000, 250, 37
    x = torch.from_numpy(rng.standard_normal((n, d), dtype=np.float32)).cuda()
    assign = torch.from_numpy(rng.integers(0, k - 1, n)).cuda()  # cluster k-1 stays empty
    xs = nf.PackedMatrix.from_tensor(x, planes=("raw",))
    cent0, h0 = nf.kmeans_update(xs, assign, k)
    st = torch.cuda.current_stream().cuda_stream

    def table(lo, hi):
        t = torch.zeros(k * (d + 1), dtype=torch.float64, device="cuda")
        part = nf.PackedMatrix.from_tensor(x[lo:hi], planes=("raw",))
        wsb = lib.nrb_kmeans_update_workspace(hi - lo, k, part.kp)
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
        a = assign[lo:hi].contiguous()
        check(lib.nrb_kmeans_partial_sums(part.raw.data_ptr(), hi - lo, d, part.kp, a.data_ptr(), k, t.data_ptr(),
                                          ws.data_ptr(), wsb, st), "partial_sums")
        return t

    def means(t):
        cent = torch.empty((k, d), dtype=torch.float32, device="cuda")
        h = torch.empty(k, dtype=torch.float32, device="cuda")
        check(lib.nrb_kmeans_means(t.data_ptr(), k, d, cent.data_ptr(), h.data_ptr(), st), "means")
        return cent, h

    c1, h1 = means(table(0, n))
    assert torch.equal(c1, cent0) and torch.equal(h1, h0)
    assert float(h1[k - 1]) == 0.0 and float(c1[k - 1].abs().max()) == 0.0
    c2, h2 = means(table(0, 7_777) + table(7_777, n))
    assert torch.equal(h2, h0)
    assert torch.allclose(c2, cent0, rtol=3e-7, atol=1e-9)
