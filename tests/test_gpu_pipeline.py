"""GPU tests of the rows next to the hot path (SURVEY 8f): the batched Retrieval.py stage, the
finalize / hit-rate neighbours and the npy formats they exchange."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _synthetic_news(tmp_path, n=30000, nu=300, d=256):
    from newsrecommend_b200 import synth
    news = tmp_path / "news"
    news.mkdir()
    x, topics = synth.g_skew(n, d, 1, return_topics=True)
    ids = np.arange(100000, 100000 + n, dtype=np.int64)
    np.save(news / "article_table.npy", np.concatenate([x.astype(np.float64), ids[:, None].astype(np.float64)], axis=1))
    users = synth.user_profiles(x, topics, nu, 2)
    np.save(news / "test_user_profile.npy", {int(7 * u + 3): users[u] for u in range(nu)}, allow_pickle=True)
    rng = np.random.default_rng(5)
    gt = {int(7 * u + 3): int(ids[rng.integers(0, n)]) for u in range(nu)}
    np.save(news / "test_user_ground_truth.npy", gt, allow_pickle=True)
    return news, ids, x, users, gt


def test_batched_stage_equals_reference_script(tmp_path):
    """retrieve_candidates == the unmodified Retrieval.py run on the shim, user by user."""
    from newsrecommend_b200 import pipeline
    news, ids, x, users, gt = _synthetic_news(tmp_path)
    aids, emb = pipeline.load_article_table(news / "article_table.npy")
    assert np.array_equal(aids, ids) and emb.dtype == np.float32 and np.array_equal(emb, x)
    uids, prof = pipeline.load_user_profiles(news / "test_user_profile.npy")
    assert np.array_equal(prof, users)
    out = pipeline.retrieve_candidates(aids, emb, prof, num_clusters=300, niter=80)
    off, cand = out["offsets"].cpu().numpy(), out["candidates"].cpu().numpy()
    assert off[-1] == cand.shape[0] and int(out["list_sizes"].sum()) == len(ids)
    # the unmodified script (tests/fixtures/reference_scripts, sha256-pinned) with `import faiss` -> the shim
    ref = os.path.join(ROOT, "tests", "fixtures", "reference_scripts", "Retrieval.py")
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "shim") + os.pathsep + ROOT)
    subprocess.check_call([sys.executable, ref], cwd=tmp_path, env=env)
    u2, off2, cand2 = pipeline.load_recommendations(news / "test_user_recommendations.npy")
    assert np.array_equal(u2, uids) and np.array_equal(off2, off) and np.array_equal(cand2, cand)
    # The same call sequence the script makes (Retrieval.py:11-34), replayed in this process against
    # the shim, per-user loop included.
    sys.path.insert(0, os.path.join(ROOT, "shim"))
    try:
        import faiss
        clustering = faiss.Clustering(emb.shape[1], 300)                      # :12
        clustering.niter = 80                                                 # :13
        index = faiss.IndexHNSWFlat(emb.shape[1], 32)                         # :16
        clustering.train(np.ascontiguousarray(emb), index)                    # :17-18
        cents = faiss.vector_float_to_array(clustering.centroids).reshape(300, emb.shape[1])  # :19
        _, a = index.search(emb, 1)                                           # :21
        a = a.flatten()                                                       # :22
        cluster_to_articles = {i: aids[a == i] for i in range(300)}           # :23
        centroid_index = faiss.IndexFlatL2(emb.shape[1])                      # :25
        centroid_index.add(cents)                                             # :26
        for u in range(0, len(uids), 7):                                      # :30-34 (every 7th user)
            _, I1 = centroid_index.search(prof[u].reshape(1, -1).astype(np.float32), 1)
            assert np.array_equal(np.array(cluster_to_articles[int(I1[0, 0])]), cand[off[u]:off[u + 1]])
    finally:
        sys.path.pop(0)
        sys.modules.pop("faiss", None)
    # structural checks: a user's candidates are exactly the articles assigned to its nearest
    # centroid, in ascending row order
    assign = out["assignments"].cpu().numpy()
    ul = out["user_list"].cpu().numpy()
    for u in (0, 17, 299):
        assert np.array_equal(cand[off[u]:off[u + 1]], ids[assign == ul[u]])
    pipeline.save_recommendations(news / "rec2.npy", uids, off, cand)
    u3, off3, cand3 = pipeline.load_recommendations(news / "rec2.npy")
    assert np.array_equal(u3, uids) and np.array_equal(off3, off) and np.array_equal(cand3, cand)


def test_finalize_and_hit_rate_match_the_scripts(tmp_path):
    """finalize_candidates == finialize_retrieval.py:6-15 and hit_rate == utils.py:12-22, both
    restated here in numpy exactly as the scripts compute them."""
    from newsrecommend_b200 import pipeline
    rng = np.random.default_rng(0)
    nu = 500
    lens = rng.integers(0, 40, size=nu)
    off = np.zeros(nu + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    cand = rng.integers(0, 2000, size=off[-1]).astype(np.int64)
    gt = rng.integers(0, 2000, size=nu).astype(np.int64)
    for u in range(0, nu, 3):  # make a third of the users hits
        if lens[u]:
            gt[u] = cand[off[u] + rng.integers(0, lens[u])]
    hits, hist = pipeline.hit_rate(off, cand, gt)
    exp_hits = sum(int(gt[u] in cand[off[u]:off[u + 1]]) for u in range(nu))  # utils.py:14-16
    assert hits == exp_hits
    vals, counts = np.unique(lens, return_counts=True)
    assert hist == dict(zip(vals.tolist(), counts.tolist()))               # utils.py:19-22
    noff, ncand = pipeline.finalize_candidates(off, cand, gt)
    noff, ncand = noff.cpu().numpy(), ncand.cpu().numpy()
    for u in range(nu):                                                     # finialize_retrieval.py:10-13
        rec = cand[off[u]:off[u + 1]]
        exp = rec if gt[u] in rec else np.append(rec, gt[u])
        assert np.array_equal(ncand[noff[u]:noff[u + 1]], exp)
    assert pipeline.hit_rate(noff, ncand, gt)[0] == nu
    # the intended cap (off by default): every list <= cap (+1 for the appended ground truth)
    coff, ccand = pipeline.finalize_candidates(off, cand, gt, cap=10)
    coff, ccand = coff.cpu().numpy(), ccand.cpu().numpy()
    assert (np.diff(coff) <= 11).all()
    for u in range(nu):
        assert set(ccand[coff[u]:coff[u + 1]].tolist()) <= set(cand[off[u]:off[u + 1]].tolist()) | {int(gt[u])}


def test_finalize_cap_keeps_candidates_in_their_own_row_at_scale():
    """ADVICE r1: with >= 1e5 users the cap's shuffle must not move candidates across user rows
    (a float32 `rand + row` key collides between neighbouring rows beyond row ~2^16)."""
    from newsrecommend_b200 import pipeline
    rng = np.random.default_rng(1)
    nu = 120_000
    lens = rng.integers(20, 60, size=nu)
    off = np.zeros(nu + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    # candidate value encodes its row: every kept candidate must decode to its own row
    row = np.repeat(np.arange(nu, dtype=np.int64), lens)
    cand = row * 100 + (np.arange(off[-1]) - off[row])
    gt = np.arange(nu, dtype=np.int64) * 100 + 99  # never present: appended to every row
    coff, ccand = pipeline.finalize_candidates(off, cand, gt, cap=30, seed=3)
    coff, ccand = coff.cpu().numpy(), ccand.cpu().numpy()
    assert np.array_equal(np.diff(coff), np.minimum(lens, 30) + 1)
    crow = np.repeat(np.arange(nu, dtype=np.int64), np.diff(coff))
    assert np.array_equal(ccand // 100, crow), "a candidate moved to another user's list"
    assert np.array_equal(ccand[coff[1:] - 1], gt)
    # sampled without replacement, and not just a prefix (the sample is random)
    assert np.unique(ccand).size == ccand.size
    tail = ccand[coff[nu - 1000]:] % 100
    assert np.unique(tail[tail != 99]).size > 40  # the last rows still draw from their whole lists


def test_batched_stage_equals_the_oracle_teacher_forced(tmp_path, oracle):
    """SURVEY 8f row 2 against the ORACLE (not against the shim): the oracle runs Retrieval.py:11-34
    -- k-means (300 x 20 iterations), assign every article, lists, nearest centroid per user -- and
    retrieve_candidates gets the oracle's centroids (teacher-forced): same assignments -> same CSR."""
    from newsrecommend_b200 import pipeline
    news, ids, x, users, gt = _synthetic_news(tmp_path, n=40000, nu=2000)
    k, d = 300, x.shape[1]
    clus = oracle.Clustering(d, k)
    clus.niter = 20
    index = oracle.IndexHNSWFlat(d, 32)
    clus.train(x, index)                                              # :12-18
    cent = oracle.vector_float_to_array(clus.centroids).reshape(k, d)  # :19
    _, a = index.search(x, 1)                                         # :21
    a = a.flatten()
    cluster_to_articles = {i: ids[a == i] for i in range(k)}          # :23
    ci = oracle.IndexFlatL2(d)
    ci.add(cent)                                                      # :25-26
    _, I = ci.search(users, 1)                                        # :30-32 (batched; nq >= 20 -> BLAS path)
    out = pipeline.retrieve_candidates(ids, x, users, num_clusters=k, centroids=cent)
    off, cand = out["offsets"].cpu().numpy(), out["candidates"].cpu().numpy()
    ga, gl = out["assignments"].cpu().numpy(), out["user_list"].cpu().numpy()
    # assignments / user lists may differ only where two centroids are at (near-)equal distance
    for got, want, pts in ((ga, a, x), (gl, I[:, 0], users)):
        for i in np.nonzero(got != want)[0]:
            d1 = ((pts[i].astype(np.float64) - cent[got[i]]) ** 2).sum()
            d2 = ((pts[i].astype(np.float64) - cent[want[i]]) ** 2).sum()
            assert abs(d1 - d2) <= 1e-5 * max(d1, d2), (i, d1, d2)
    same_assign = np.array_equal(ga, a)
    n_same = 0
    for u in range(len(users)):
        ref = cluster_to_articles[int(I[u, 0])]                       # :33
        if same_assign and gl[u] == I[u, 0]:
            assert np.array_equal(cand[off[u]:off[u + 1]], ref)
            n_same += 1
    assert n_same >= 0.99 * len(users)


def test_article_table_device_loader_both_formats(tmp_path):
    """SURVEY 8f row 1: file -> page-locked staging -> HBM (no numpy array in between) for the float
    table Retrieval.py:6 can read, and the object-dtype table embedding_generate.py:124-131 writes
    (pickled Python floats: one pass through the unpickler, then the same device path). Both equal
    the host loader bit for bit."""
    from newsrecommend_b200 import pipeline
    rng = np.random.default_rng(0)
    n, d = 70_001, 250  # more than two staging chunks, ragged tail
    x = rng.standard_normal((n, d))
    ids = rng.permutation(10_000_000)[:n].astype(np.float64)
    table = np.concatenate([x, ids[:, None]], axis=1)
    np.save(tmp_path / "article_table.npy", table)
    ids_h, emb_h = pipeline.load_article_table(tmp_path / "article_table.npy")
    ids_d, emb_d = pipeline.load_article_table_device(tmp_path / "article_table.npy")
    assert ids_d.is_cuda and emb_d.is_cuda and emb_d.dtype.is_floating_point and emb_d.is_contiguous()
    assert np.array_equal(ids_d.cpu().numpy(), ids_h) and np.array_equal(emb_d.cpu().numpy(), emb_h)
    assert np.array_equal(ids_h, ids.astype(np.int64)) and np.array_equal(emb_h, x.astype(np.float32))
    # the producer's format: dtype=object rows of Python floats (needs allow_pickle)
    small = table[:3_000]
    obj = np.empty(small.shape, dtype=object)
    obj[...] = small
    np.save(tmp_path / "article_table_obj.npy", obj, allow_pickle=True)
    with pytest.raises(ValueError):
        np.load(tmp_path / "article_table_obj.npy")  # what Retrieval.py:6 would hit on the producer's file
    ids_o, emb_o = pipeline.load_article_table(tmp_path / "article_table_obj.npy")
    ids_od, emb_od = pipeline.load_article_table_device(tmp_path / "article_table_obj.npy")
    assert np.array_equal(ids_o, ids_h[:3_000]) and np.array_equal(emb_o, emb_h[:3_000])
    assert np.array_equal(ids_od.cpu().numpy(), ids_o) and np.array_equal(emb_od.cpu().numpy(), emb_o)
    # float32 tables and Fortran order fall back to the generic route and still agree
    np.save(tmp_path / "t32.npy", table[:500].astype(np.float32))
    i32, e32 = pipeline.load_article_table_device(tmp_path / "t32.npy")
    ih, eh = pipeline.load_article_table(tmp_path / "t32.npy")
    assert np.array_equal(i32.cpu().numpy(), ih) and np.array_equal(e32.cpu().numpy(), eh)
