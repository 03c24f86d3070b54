"""External ids and removal on the B200: nrb_id_select against numpy, IndexIDMap over the flat
index on every search route, remove_ids on IndexFlat / IndexIDMap / IndexIVFFlat against an index
freshly built from the survivors (bit for bit) and against the oracle, IVF add_with_ids, and one
full-size catalog case."""
import numpy as np
import pytest

from newsrecommend_b200.parity import compare_topk
from test_gpu_kmeans_ivf import _classify_ivf_mismatches

pytestmark = pytest.mark.gpu

I64_MIN, I64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max
FLT_MAX = np.float32(3.4028234663852886e38)


@pytest.fixture(scope="module")
def oracle(oracle):
    """The CPU oracle with faiss's external-id semantics added (tests/ids_oracle.py)."""
    import ids_oracle
    return ids_oracle


def _np(a):
    import torch
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else a


def _same(a, b):
    D1, I1 = map(_np, a)
    D2, I2 = map(_np, b)
    assert np.array_equal(D1.view(np.int32), D2.view(np.int32)) and np.array_equal(I1, I2)


def _rows(I, ids):
    """Labels -> positions in ids (-1 padding stays -1). The parity rule reads every negative label
    as padding, and the ids here include negative values, so oracle comparisons run on positions."""
    I = np.asarray(I)
    order = np.argsort(ids, kind="stable")
    pos = order[np.minimum(np.searchsorted(ids, I, sorter=order), len(ids) - 1)]
    assert np.array_equal(ids[pos][I != -1], I[I != -1])
    return np.where(I == -1, -1, pos)


def _translated(D, I, Dp, Ip, ids, metric):
    """An IndexIDMap result against a separate search of a plain index over the same rows. A row whose
    D is bit-identical must carry ids[plain labels] exactly. The fp16 filter recomputes the queries it
    flags with the 3xTF32 kernel, and which queries get flagged depends on the order in which
    candidates arrive, so a few rows of two searches may differ in the last bits: those must agree by
    the parity rule, and they must stay rare."""
    D, I, Dp, Ip = map(_np, (D, I, Dp, Ip))
    same = (D.view(np.int32) == Dp.view(np.int32)).all(axis=1)
    assert same.mean() >= 0.99, same.mean()
    assert np.array_equal(I[same], np.where(Ip[same] < 0, Ip[same], ids[np.maximum(Ip[same], 0)]))
    rep = compare_topk(D, _rows(I, ids), Dp, Ip, metric)
    assert rep["ok"], rep


def _id_select(ids, n, batch=None, imin=0, imax=0):
    import torch
    from newsrecommend_b200._lib import check, lib
    dev = torch.device("cuda")
    ids_t = None if ids is None else torch.from_numpy(ids).to(dev)
    b_t = None if batch is None else torch.from_numpy(batch).to(dev) if batch.size else torch.empty(1, dtype=torch.int64,
                                                                                                     device=dev)
    nb = 0 if batch is None else batch.size
    member = torch.full((max(n, 1),), 7, dtype=torch.int64, device=dev)
    wsb = lib.nrb_id_select_workspace(nb)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=dev)
    check(lib.nrb_id_select(0 if ids_t is None else ids_t.data_ptr(), n, 0 if b_t is None else b_t.data_ptr(), nb, imin,
                            imax, member.data_ptr(), ws.data_ptr(), wsb, None), "id_select")
    return member[:n].cpu().numpy()


def test_id_select_matches_numpy(nf):
    rng = np.random.default_rng(0)
    n = 200_003
    ids = rng.integers(-10 ** 6, 10 ** 6, n).astype(np.int64)
    ids[:6] = [I64_MIN, I64_MAX, -1, 0, -1, I64_MIN + 1]  # -1 is the table's empty-slot sentinel
    for batch in (ids[rng.integers(0, n, 5000)],                   # duplicates
                  np.concatenate([ids[:50], ids[:50], [-1]]),       # the sentinel itself
                  np.array([I64_MIN, I64_MAX], np.int64),
                  rng.integers(-10 ** 6, 10 ** 6, 300_000).astype(np.int64),
                  np.array([5], np.int64)):
        m = _id_select(ids, n, batch)
        assert m.dtype == np.int64 and np.array_equal(m, np.isin(ids, batch).astype(np.int64))
    assert not _id_select(ids, n, np.empty(0, np.int64)).any()  # empty batch
    for imin, imax in ((-1000, 1000), (0, 0), (5, -5), (I64_MIN, I64_MAX), (-1, 0)):
        m = _id_select(ids, n, None, imin, imax)
        assert np.array_equal(m, ((ids >= imin) & (ids < imax)).astype(np.int64)), (imin, imax)
    # ids == NULL: the id of row i is i
    m = _id_select(None, 1000, None, 100, 250)
    assert np.array_equal(np.nonzero(m)[0], np.arange(100, 250))
    m = _id_select(None, 1000, np.array([3, 3, 999, 1000, -1], np.int64))
    assert np.nonzero(m)[0].tolist() == [3, 999]


def _flat_data(n=20_000, d=64, seed=1):
    rng = np.random.default_rng(seed)
    xb = rng.standard_normal((n, d), dtype=np.float32)
    ids = (rng.permutation(n).astype(np.int64) * 1_000_003) - 7 * 10 ** 9  # shuffled, unique, some negative
    return xb, ids


@pytest.mark.parametrize("metric", [0, 1])
def test_idmap_search_every_route(nf, oracle, metric):
    import torch
    xb, ids = _flat_data()
    rng = np.random.default_rng(2)
    plain = nf.IndexFlat(64, metric)
    plain.add(xb)
    m = nf.IndexIDMap(nf.IndexFlat(64, metric))
    for lo, hi in ((0, 5000), (5000, 5001), (5001, 20_000)):
        m.add_with_ids(xb[lo:hi] if lo else torch.from_numpy(xb[lo:hi]).cuda(),
                       ids[lo:hi] if lo != 5000 else torch.from_numpy(ids[lo:hi]))
    assert (m.ntotal, m.d, m.metric_type, m.is_trained) == (20_000, 64, metric, True)
    om = oracle.IndexIDMap(oracle.IndexFlat(64, metric))
    om.add_with_ids(xb, ids)
    wave2 = 2 * nf._wave_rows()
    for nq in (1, 19, 20, 129, 5000, wave2):
        xq = rng.standard_normal((nq, 64), dtype=np.float32)
        for k in (1, 50, 112, 128):
            Dp, Ip = plain.search(xq, k)
            D, I = m.search(xq, k)
            assert isinstance(D, np.ndarray) and isinstance(I, np.ndarray)
            _translated(D, I, Dp, Ip, ids, metric)
            xt = torch.from_numpy(xq).cuda()
            Dt, It = m.search(xt, k)
            assert Dt.is_cuda and It.is_cuda
            _translated(Dt, It, *plain.search(xt, k), ids, metric)
            if nq <= 5000 and k in (1, 128) or (nq == wave2 and k == 50):
                Do, Io = om.search(xq, k)
                rep = compare_topk(D, _rows(I, ids), Do, _rows(Io, ids), metric)
                assert rep["ok"], (nq, k, rep)
    # preallocated outputs and k > ntotal
    xq = rng.standard_normal((7, 64), dtype=np.float32)
    Do, Io = np.empty((7, 50), np.float32), np.empty((7, 50), np.int64)
    D, I = m.search(xq, 50, D=Do, I=Io)
    assert D is Do and I is Io
    _translated(D, I, *plain.search(xq, 50), ids, metric)
    small = nf.IndexIDMap(nf.IndexFlat(64, metric))
    small.add_with_ids(xb[:30], ids[:30])
    for nq in (3, 40):
        D, I = small.search(xq[:1].repeat(nq, 0), 50)
        assert (I[:, 30:] == -1).all() and (D[:, 30:] == (-FLT_MAX if metric == 0 else FLT_MAX)).all()
        assert np.array_equal(np.sort(I[0, :30]), np.sort(ids[:30]))
    with pytest.raises(RuntimeError, match="add_with_ids"):
        m.add(xb[:2])
    with pytest.raises(TypeError):
        m.add_with_ids(xb[:2], ids[:3])
    with pytest.raises(RuntimeError, match="must be empty"):
        nf.IndexIDMap(plain)
    with pytest.raises(RuntimeError, match="add_with_ids not implemented"):
        plain.add_with_ids(xb[:2], ids[:2])
    m.reset()
    assert m.ntotal == 0 and (m.search(xq, 5)[1] == -1).all()


def _fresh_flat(nf, metric, xb):
    f = nf.IndexFlat(xb.shape[1], metric)
    f.add(xb)
    return f


@pytest.mark.parametrize("metric", [0, 1])
def test_flat_remove_ids(nf, oracle, metric):
    xb, _ = _flat_data(8000, 96, 3)
    big = 4321
    xb[big] *= 1000.0  # by far the largest norm: removing it must shrink max_norm and the fp16 scale
    xq = np.random.default_rng(4).standard_normal((3000, 96), dtype=np.float32)
    idx = _fresh_flat(nf, metric, xb)
    assert idx.remove_ids(nf.IDSelectorRange(9000, 20_000)) == 0
    assert idx.remove_ids(nf.IDSelectorBatch(np.empty(0, np.int64))) == 0
    assert idx.remove_ids(nf.IDSelectorBatch(np.array([big, big, -5, 10 ** 12]))) == 1
    keep = np.ones(8000, bool)
    keep[big] = False
    fresh = _fresh_flat(nf, metric, xb[keep])
    assert idx._xb.max_norm == fresh._xb.max_norm and idx._xb.h16_scale == fresh._xb.h16_scale
    assert idx._xb.max_norm < 1000.0
    for nq, k in ((5, 10), (3000, 50), (3000, 128)):
        _same(idx.search(xq[:nq], k), fresh.search(xq[:nq], k))
    # positions: a range, then a plain array (positions in the compacted index)
    assert idx.remove_ids(nf.IDSelectorRange(100, 1100)) == 1000
    pos = np.nonzero(keep)[0]
    keep[pos[100:1100]] = False
    assert idx.remove_ids(np.array([0, 17, 17, 6000], np.int64)) == 3
    pos = np.nonzero(keep)[0]
    keep[pos[[0, 17, 6000]]] = False
    assert idx.ntotal == keep.sum()
    _same(idx.search(xq, 50), _fresh_flat(nf, metric, xb[keep]).search(xq, 50))
    o = oracle.IndexFlat(96, metric)
    o.add(xb)
    assert o.remove_ids(oracle.IDSelectorBatch(np.array([big]))) == 1
    assert o.remove_ids(oracle.IDSelectorRange(100, 1100)) == 1000
    assert o.remove_ids(np.array([0, 17, 17, 6000], np.int64)) == 3
    assert compare_topk(*idx.search(xq, 50), *o.search(xq, 50), metric)["ok"]
    # add -> remove -> add
    idx.add(xb[:500])
    ref = nf.IndexFlat(96, metric)
    ref.add(xb[keep])
    ref.add(xb[:500])
    _same(idx.search(xq, 50), ref.search(xq, 50))
    # remove everything: empty results, then the index fills again
    assert idx.remove_ids(nf.IDSelectorRange(0, 10 ** 9)) == keep.sum() + 500 and idx.ntotal == 0
    D, I = idx.search(xq[:40], 5)
    assert (I == -1).all() and (D == (-FLT_MAX if metric == 0 else FLT_MAX)).all()
    idx.add(xb[:1000])
    _same(idx.search(xq, 20), _fresh_flat(nf, metric, xb[:1000]).search(xq, 20))


@pytest.mark.parametrize("metric", [0, 1])
def test_idmap_remove_ids(nf, oracle, metric):
    xb, ids = _flat_data(10_000, 64, 5)
    big = int(np.argmax(ids))
    xb[big] *= 500.0
    xq = np.random.default_rng(6).standard_normal((2000, 64), dtype=np.float32)
    m = nf.IndexIDMap(nf.IndexFlat(64, metric))
    m.add_with_ids(xb[:4000], ids[:4000])
    m.add_with_ids(xb[4000:], ids[4000:])
    om = oracle.IndexIDMap(oracle.IndexFlat(64, metric))
    om.add_with_ids(xb, ids)

    def fresh(keep):
        f = nf.IndexIDMap(nf.IndexFlat(64, metric))
        f.add_with_ids(xb[keep], ids[keep])
        return f

    keep = np.ones(10_000, bool)
    assert m.remove_ids(nf.IDSelectorBatch(np.array([12345], np.int64))) == 0  # no such id
    assert m.remove_ids(nf.IDSelectorBatch(np.array([ids[big]]))) == 1
    assert om.remove_ids(oracle.IDSelectorBatch(np.array([ids[big]]))) == 1
    keep[big] = False
    f = fresh(keep)
    assert m.index._xb.max_norm == f.index._xb.max_norm and m.index._xb.h16_scale == f.index._xb.h16_scale
    _same(m.search(xq, 50), f.search(xq, 50))
    lo, hi = -5 * 10 ** 9, 2 * 10 ** 9
    sel = (ids >= lo) & (ids < hi) & keep
    assert m.remove_ids(nf.IDSelectorRange(lo, hi)) == sel.sum() == om.remove_ids(oracle.IDSelectorRange(lo, hi))
    keep &= ~sel
    batch = ids[keep][::7]
    assert m.remove_ids(batch) == batch.size == om.remove_ids(batch)
    keep &= ~np.isin(ids, batch)
    assert np.array_equal(m.id_map.cpu().numpy(), ids[keep])
    for nq, k in ((3, 50), (2000, 50), (2000, 128)):
        D, I = m.search(xq[:nq], k)
        _same((D, I), fresh(keep).search(xq[:nq], k))
        Do, Io = om.search(xq[:nq], k)
        rep = compare_topk(D, _rows(I, ids), Do, _rows(Io, ids), metric)
        assert rep["ok"], rep
    m.add_with_ids(xb[:10], ids[:10] + 1)  # add -> remove -> add
    f = nf.IndexIDMap(nf.IndexFlat(64, metric))
    f.add_with_ids(xb[keep], ids[keep])
    f.add_with_ids(xb[:10], ids[:10] + 1)
    _same(m.search(xq, 50), f.search(xq, 50))
    assert m.remove_ids(nf.IDSelectorRange(I64_MIN, I64_MAX)) == keep.sum() + 10 and m.ntotal == 0
    D, I = m.search(xq[:5], 4)
    assert (I == -1).all() and (D == (-FLT_MAX if metric == 0 else FLT_MAX)).all()


def _ivf_pair(nf, oracle, xb, nlist, metric, seed=0):
    """GPU and oracle IVF over identical centroids (teacher-forced quantizer)."""
    d = xb.shape[1]
    qo = oracle.IndexFlatIP(d) if metric == 0 else oracle.IndexFlatL2(d)
    ivf_o = oracle.IndexIVFFlat(qo, d, nlist, metric)
    ivf_o.train(xb)
    cent = qo.xb.copy()

    def make():
        q = nf.IndexFlatIP(d) if metric == 0 else nf.IndexFlatL2(d)
        q.add(cent)
        ivf = nf.IndexIVFFlat(q, d, nlist, metric)
        ivf.train(xb)
        return ivf
    return make, ivf_o


def _ivf_data(n=30_000, nq=700, seed=21):
    from newsrecommend_b200 import synth
    xb, topics = synth.g_skew(n, 250, seed, n_topics=120, return_topics=True)
    xq = synth.user_profiles(xb, topics, nq, seed + 1)
    ids = np.random.default_rng(seed).permutation(10 * n)[:n].astype(np.int64) * 3 + 10 ** 10
    return xb, xq, ids


def _ivf_check(ivf, ivf_o, xq, k, metric, nprobes, xb_exact, ids_exact, oracle):
    for nprobe in nprobes:
        ivf.nprobe = ivf_o.nprobe = nprobe
        for nq in (64, xq.shape[0]):  # the small-batch list scan and the tcgen05 scan
            D, I = ivf.search(xq[:nq], k)
            Do, Io = ivf_o.search(xq[:nq], k)
            if not compare_topk(D, I, Do, Io, metric)["ok"]:
                _classify_ivf_mismatches(ivf_o, xq[:nq], nprobe, k, D, I, Do, Io, metric)
    ivf.nprobe = ivf.nlist
    D, I = ivf.search(xq, k)
    Df, If = oracle.knn_fast(xq, xb_exact, k, metric)
    rep = compare_topk(D, I, Df, np.where(If < 0, -1, ids_exact[np.maximum(If, 0)]), metric)
    assert rep["ok"], rep


@pytest.mark.parametrize("metric", [0, 1])
def test_ivf_add_with_ids(nf, oracle, metric):
    xb, xq, ids = _ivf_data()
    nlist = 64
    make, ivf_o = _ivf_pair(nf, oracle, xb, nlist, metric)
    ivf = make()
    ivf.add_with_ids(xb[:10_000], ids[:10_000])
    ivf.add_with_ids(xb[10_000:], ids[10_000:])
    ivf_o.add_with_ids(xb, ids)
    assert np.array_equal(ivf.list_sizes(), ivf_o.list_sizes())
    _ivf_check(ivf, ivf_o, xq, 50, metric, (1, 16, nlist), xb, ids, oracle)
    # add() numbers rows from ntotal, whatever ids came before
    plain = make()
    plain.add(xb[:5000])
    mixed = make()
    mixed.add_with_ids(xb[:2000], np.arange(2000, dtype=np.int64))
    mixed.add(xb[2000:5000])
    plain.nprobe = mixed.nprobe = 8
    _same(plain.search(xq, 20), mixed.search(xq, 20))
    with pytest.raises(TypeError):
        ivf.add_with_ids(xb[:5], ids[:5].astype(np.int32))


@pytest.mark.parametrize("metric", [0, 1])
def test_ivf_remove_ids(nf, oracle, metric):
    xb, xq, ids = _ivf_data(seed=31)
    nlist = 64
    make, ivf_o = _ivf_pair(nf, oracle, xb, nlist, metric)
    ivf = make()
    ivf.add_with_ids(xb, ids)
    ivf_o.add_with_ids(xb, ids)
    assert ivf.remove_ids(nf.IDSelectorRange(0, 10)) == 0 == ivf_o.remove_ids(oracle.IDSelectorRange(0, 10))
    keep = np.ones(len(ids), bool)
    lo, hi = int(np.quantile(ids, 0.2)), int(np.quantile(ids, 0.35))
    sel = (ids >= lo) & (ids < hi)
    assert ivf.remove_ids(nf.IDSelectorRange(lo, hi)) == sel.sum() == ivf_o.remove_ids(oracle.IDSelectorRange(lo, hi))
    keep &= ~sel
    batch = np.concatenate([ids[keep][::5], ids[keep][::5], [-1, 7]])
    sel = np.isin(ids, batch) & keep
    assert ivf.remove_ids(nf.IDSelectorBatch(batch.size, batch)) == sel.sum() == ivf_o.remove_ids(batch)
    keep &= ~sel
    assert ivf.ntotal == keep.sum() == ivf_o.ntotal
    fresh = make()
    fresh.add_with_ids(xb[keep], ids[keep])
    for nprobe in (1, 16, nlist):
        ivf.nprobe = fresh.nprobe = nprobe
        for nq in (30, 700):
            _same(ivf.search(xq[:nq], 50), fresh.search(xq[:nq], 50))
    _ivf_check(ivf, ivf_o, xq, 50, metric, (1, 16), xb[keep], ids[keep], oracle)
    # add -> remove -> add: new rows get ids from ntotal, like faiss
    n0 = ivf.ntotal
    ivf.add(xb[:100])
    ivf_o.add(xb[:100])
    fresh.add(xb[:100])
    ivf.nprobe = fresh.nprobe = 16
    _same(ivf.search(xq, 50), fresh.search(xq, 50))
    assert np.array_equal(ivf._ids[-100:].cpu().numpy(), np.arange(n0, n0 + 100))
    assert ivf.remove_ids(nf.IDSelectorRange(I64_MIN, I64_MAX)) == n0 + 100 and ivf.ntotal == 0
    D, I = ivf.search(xq[:10], 5)
    assert (I == -1).all() and (D == (-FLT_MAX if metric == 0 else FLT_MAX)).all()
    ivf.add_with_ids(xb[:50], ids[:50])
    f50 = make()
    f50.add_with_ids(xb[:50], ids[:50])
    f50.nprobe = ivf.nprobe
    _same(ivf.search(xq, 5), f50.search(xq, 5))


def test_fullsize_idmap_remove_by_range(nf, oracle):
    """The 364,047 x 250 catalog keyed by synthetic article ids in publication order; the oldest
    10 % leave by IDSelectorRange, then 2,048 queries are checked against the oracle."""
    from newsrecommend_b200 import synth
    xb, topics = synth.g_skew(synth.N_ARTICLES, 250, 42, return_topics=True)
    xq = synth.user_profiles(xb, topics, 2048, 43)
    n = xb.shape[0]
    ids = 100_000 + np.arange(n, dtype=np.int64) * 3
    cut = int(ids[n // 10])
    m = nf.IndexIDMap(nf.IndexFlatIP(250))
    m.add_with_ids(xb, ids)
    assert m.remove_ids(nf.IDSelectorRange(0, cut)) == n // 10
    om = oracle.IndexIDMap(oracle.IndexFlatIP(250))
    om.add_with_ids(xb[n // 10:], ids[n // 10:])
    D, I = m.search(xq, 50)
    assert I.min() >= cut
    rep = compare_topk(D, I, *om.search(xq, 50), 0)
    assert rep["ok"] and rep["recall"] >= 0.9999, rep
