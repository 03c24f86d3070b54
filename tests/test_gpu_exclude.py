"""Per-query exclusion lists on the B200: nrb_exclude_topk against its numpy restatement bit for bit,
every route of search(exclude=...) against the same route at its group's k' followed by the numpy
exclusion (and the long group against one masked call per query), parity with the oracle restatement
(tests/exclude_oracle.py), IndexIDMap, IndexIVFFlat, exclusion combined with a freshness window,
empty lists, and the config-1 catalog with the synthetic click histories."""
import numpy as np
import pytest

from newsrecommend_b200.parity import compare_topk

pytestmark = pytest.mark.gpu

FLT_MAX = np.float32(3.4028234663852886e38)


@pytest.fixture(scope="module")
def eo(oracle):
    import exclude_oracle
    return exclude_oracle


@pytest.fixture(scope="module")
def io(oracle):
    import ids_oracle
    return ids_oracle


def _np(a):
    import torch
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else a


def _same(a, b, what=""):
    D1, I1 = map(_np, a)
    D2, I2 = map(_np, b)
    assert D1.shape == D2.shape, what
    assert np.array_equal(D1.view(np.int32), D2.view(np.int32)) and np.array_equal(I1, I2), what


def _rows(x, rows):
    import torch
    if isinstance(x, torch.Tensor):
        return x.index_select(0, torch.from_numpy(rows).to(x.device))
    return np.ascontiguousarray(x[rows])


def _route_reference(eo, search, x, k, off, ids, metric, long_search):
    """What search(x, k, exclude=(off, ids)) must return: each group searched at its own k' by
    search(x_group, k') and excluded in numpy; each long query answered by long_search(q)."""
    nq = off.size - 1
    need = k + np.diff(off)
    D = np.full((nq, k), np.nan, np.float32)
    I = np.full((nq, k), -2, np.int64)
    for group in (need <= 112, (need > 112) & (need <= 128)):
        rows = np.nonzero(group)[0]
        if rows.size:
            Dg, Ig = search(_rows(x, rows), int(need[rows].max()))
            eo.exclude_topk(_np(Dg), _np(Ig), rows, off, ids, metric, k, D, I)
    for q in np.nonzero(need > 128)[0]:
        Dq, Iq = long_search(q)
        D[q], I[q] = _np(Dq)[0], _np(Iq)[0]
    return D, I


def _not_listed(I, off, ids):
    I = _np(I)
    for q in range(I.shape[0]):
        assert not np.isin(I[q][I[q] >= 0], ids[off[q]:off[q + 1]]).any(), q


def _parity(D, I, Do, Io, metric, what):
    rep = compare_topk(_np(D), _np(I), Do, Io, metric)
    assert rep["ok"], (what, rep)


def _make_lists(rng, top, lens, n_labels, absent):
    """Query q's list: lens[q] labels, most from its own plain top results (so the exclusion bites),
    the rest random labels, duplicates, -1 and an absent label."""
    lists = []
    for q, L in enumerate(lens):
        own = top[q][top[q] >= 0]
        l = np.concatenate([rng.choice(own, min(L, own.size) * 2 // 3, replace=False) if L else own[:0],
                            rng.choice(n_labels, L, replace=True)])[:max(L - 2, 0)]
        extra = [-1, absent] if L >= 2 else ([-1] if L == 1 else [])
        lists.append(np.concatenate([l, np.asarray(extra, np.int64)]).astype(np.int64))
    return lists


def _lens(rng, nq, lo, hi):
    return rng.integers(lo, hi + 1, nq)


# ------------------------------------------------------------------ the kernel against numpy
@pytest.mark.parametrize("metric", [0, 1])
def test_exclude_topk_kernel(eo, metric):
    import torch
    from newsrecommend_b200 import _lib
    rng = np.random.default_rng(11 + metric)
    L = _lib.lib
    stream = torch.cuda.current_stream().cuda_stream
    pad = FLT_MAX if metric == 1 else -FLT_MAX
    for nq, nrows, kin, k, maxlen in ((40, 40, 128, 50, 300), (500, 173, 77, 60, 17), (33, 33, 5, 5, 1),
                                      (1000, 1000, 128, 128, 0), (64, 20, 100, 1, 2000)):
        Din = np.sort(rng.standard_normal((nrows, kin)).astype(np.float32), axis=1)
        Din = Din[:, ::-1] if metric == 0 else Din
        Iin = rng.integers(0, 500, (nrows, kin)).astype(np.int64)
        npad = rng.integers(0, kin + 1, nrows)  # padding in the input's tail
        for r in range(nrows):
            if npad[r]:
                Din[r, kin - npad[r]:], Iin[r, kin - npad[r]:] = pad, -1
        Din = np.ascontiguousarray(Din)
        qidx = np.sort(rng.choice(nq, nrows, replace=False)).astype(np.int64) if nrows < nq else None
        lists = []
        for q in range(nq):
            Lq = int(rng.integers(0, maxlen + 1))
            l = rng.integers(-2, 520, Lq)
            if Lq:
                l[: Lq // 2] = rng.choice(Iin[0], Lq // 2)  # hits
            lists.append(l)
        off, ids = eo.csr(lists)
        D = np.full((nq, k), 7.0, np.float32)
        I = np.full((nq, k), -9, np.int64)
        Dref, Iref = eo.exclude_topk(Din, Iin, qidx, off, ids, metric, k, D.copy(), I.copy())
        dev = torch.device("cuda")
        t = [torch.from_numpy(a).to(dev) for a in (Din, Iin, off, ids if ids.size else np.zeros(1, np.int64), D, I)]
        qd = torch.from_numpy(qidx).to(dev) if qidx is not None else None
        rc = L.nrb_exclude_topk(t[0].data_ptr(), t[1].data_ptr(), nrows, kin, 0 if qd is None else qd.data_ptr(),
                                t[2].data_ptr(), t[3].data_ptr(), metric, k, t[4].data_ptr(), t[5].data_ptr(), stream)
        assert rc == 0, _lib.last_error()
        _same((t[4], t[5]), (Dref, Iref), (nq, nrows, kin, k))


# ------------------------------------------------------------------ flat routes
@pytest.fixture(scope="module")
def flat_data():
    rng = np.random.default_rng(21)
    n, d = 20_000, 96
    xb = rng.standard_normal((n, d), dtype=np.float32)
    xq = rng.standard_normal((600, d), dtype=np.float32)
    return xb, xq


def _flat_cases(rng, top, n, k):
    """(name, query rows, list lengths): the routes and the three groups. The fp16-filter batch stays at
    k' <= 96: near k' = 112 the filter has few margin slots left, and whether a query overflows them and
    is recomputed by the 3xTF32 kernel (same ids, other last bits) can differ between two searches, so
    two calls are not bit-comparable there (config 1 below checks k' = 112 by parity)."""
    return [
        ("numpy_small", np.arange(7), _lens(rng, 7, 0, 40), "numpy"),
        ("device_small", np.arange(7, 19), _lens(rng, 12, 0, 40), "cuda"),
        ("filter_batch", np.arange(300), _lens(rng, 300, 0, 96 - k), "numpy"),
        ("wide", np.arange(100, 400), _lens(rng, 300, 113 - k, 128 - k), "cuda"),
        ("long", np.arange(3), _lens(rng, 3, 129 - k, 400), "numpy"),
        ("mixed", np.arange(600), np.concatenate([_lens(rng, 400, 0, 30), _lens(rng, 150, 113 - k, 128 - k),
                                                  _lens(rng, 50, 129 - k, 300)])[rng.permutation(600)], "numpy"),
    ]


@pytest.mark.parametrize("metric", [0, 1])
def test_exclude_flat_routes(nf, io, eo, flat_data, metric):
    import torch
    xb, xq = flat_data
    n, k = xb.shape[0], 50
    index = nf.IndexFlat(xb.shape[1], metric)
    index.add(xb)
    o = io.IndexFlat(xb.shape[1], metric)
    o.add(xb)
    top = index.search(xq, 128)[1]
    rng = np.random.default_rng(31 + metric)
    for name, rows, lens, kind in _flat_cases(rng, top, n, k):
        lists = _make_lists(rng, top[rows], lens, n, n + 5)
        off, ids = eo.csr(lists)
        x = xq[rows] if kind == "numpy" else torch.from_numpy(xq[rows]).cuda()
        D, I = index.search(x, k, exclude=(off, ids))
        assert isinstance(D, np.ndarray) == (kind == "numpy")

        def long_search(q, x=x, off=off, ids=ids):
            sel = nf.IDSelectorNot(nf.IDSelectorBatch(ids[off[q]:off[q + 1]]))
            return index.search(_rows(x, np.array([q])), k, params=nf.SearchParameters(sel=sel))

        _same((D, I), _route_reference(eo, index.search, x, k, off, ids, metric, long_search), name)
        _not_listed(I, off, ids)
        _parity(D, I, *eo.search_excluded(o.search, xq[rows], k, off, ids, metric), metric, name)
        if name == "mixed":  # CUDA tensors in and out, lists on the device: the same bits
            Dt, It = index.search(torch.from_numpy(xq[rows]).cuda(), k,
                                  exclude=(torch.from_numpy(off).cuda(), torch.from_numpy(ids).cuda()))
            assert Dt.is_cuda
            _same((Dt, It), (D, I), name)


def test_exclude_idmap_large_ids(nf, eo, flat_data):
    """IndexIDMap with ids >= 2^32: the same bits as the plain index with the lists and labels mapped."""
    xb, xq = flat_data
    n, k = xb.shape[0], 50
    ext = np.random.default_rng(3).permutation(10 * n)[:n].astype(np.int64) * 7 + 2 ** 33
    plain = nf.IndexFlatIP(xb.shape[1])
    plain.add(xb)
    m = nf.IndexIDMap(nf.IndexFlatIP(xb.shape[1]))
    m.add_with_ids(xb, ext)
    top = plain.search(xq, 128)[1]
    rng = np.random.default_rng(4)
    for name, rows, lens, kind in _flat_cases(rng, top, n, k):
        lists = _make_lists(rng, top[rows], lens, n, n + 5)
        off, ids = eo.csr(lists)
        ids_ext = np.where((ids >= 0) & (ids < n), ext[np.clip(ids, 0, n - 1)], ids)  # absent stays absent
        D, I = plain.search(xq[rows], k, exclude=(off, ids))
        De, Ie = m.search(xq[rows], k, exclude=(off, ids_ext))
        _same((De, Ie), (D, np.where(I < 0, -1, ext[np.maximum(I, 0)])), name)


# ------------------------------------------------------------------ IVF
@pytest.mark.parametrize("metric", [0, 1])
def test_exclude_ivf_routes(nf, io, eo, metric):
    import torch
    from test_gpu_ids import _ivf_data, _ivf_pair
    xb, xq, ids_b = _ivf_data(20_000, 400, seed=51)
    nlist, k = 32, 50
    make, ivf_o = _ivf_pair(nf, io, xb, nlist, metric)
    ivf = make()
    ivf.add_with_ids(xb, ids_b)
    ivf_o.add_with_ids(xb, ids_b)
    top = ivf.search(xq, 128, params=nf.SearchParametersIVF(nprobe=8))[1]
    rng = np.random.default_rng(61 + metric)
    cases = [("small", np.arange(40), _lens(rng, 40, 0, 40)),
             ("small_mixed", np.arange(40, 64), np.concatenate([_lens(rng, 12, 0, 50), _lens(rng, 6, 70, 78),
                                                               _lens(rng, 6, 79, 200)])),
             ("batch_mixed", np.arange(400), np.concatenate([_lens(rng, 250, 0, 40), _lens(rng, 100, 63, 78),
                                                            _lens(rng, 50, 79, 300)])[rng.permutation(400)])]
    for nprobe in (4, nlist):
        p = nf.SearchParametersIVF(nprobe=nprobe)
        for name, rows, lens in cases:
            off, ids = eo.csr(_make_lists(rng, _np(top)[rows], lens, 10 ** 9, 5))
            x = torch.from_numpy(xq[rows]).cuda()
            D, I = ivf.search(x, k, params=p, exclude=(off, ids))

            def long_search(q, x=x, off=off, ids=ids):
                sel = nf.IDSelectorNot(nf.IDSelectorBatch(ids[off[q]:off[q + 1]]))
                return ivf.search(x[q:q + 1], k, params=nf.SearchParametersIVF(sel=sel, nprobe=nprobe))

            ref = _route_reference(eo, lambda xs, kk: ivf.search(xs, kk, params=p), x, k, off, ids, metric,
                                   long_search)
            _same((D, I), ref, (name, nprobe))
            _not_listed(I, off, ids)
            Dn, In = ivf.search(xq[rows], k, params=p, exclude=(off, ids))  # numpy in, numpy out
            _same((Dn, In), (D, I), (name, nprobe))
            if nprobe == nlist:  # every list probed: the oracle restatement has no coarse near-ties to explain
                ivf_o.nprobe = nlist
                _parity(D, I, *eo.search_excluded(ivf_o.search, xq[rows], k, off, ids, metric), metric, name)


# ------------------------------------------------------------------ exclusion with a freshness window
def test_exclude_with_freshness_window(nf, io, eo, flat_data):
    """A row is returned only if the window keeps it and the list misses it. Groups: the filtered route
    at k'; the long group: an index built from the rows that pass both filters."""
    import torch
    from test_gpu_ids import _ivf_data, _ivf_pair
    xb, xq = flat_data
    n, d, k = xb.shape[0], xb.shape[1], 50
    lo, hi = n // 3, n  # the newest two thirds (ids in publication order)
    ext = np.arange(n, dtype=np.int64) * 3 + 2 ** 34
    flat = nf.IndexFlatIP(d)
    flat.add(xb)
    m = nf.IndexIDMap(nf.IndexFlatIP(d))
    m.add_with_ids(xb, ext)
    rng = np.random.default_rng(71)
    top = flat.search(xq, 128, params=nf.SearchParameters(sel=nf.IDSelectorRange(lo, hi)))[1]
    rows = np.arange(300)
    lens = np.concatenate([_lens(rng, 200, 0, 40), _lens(rng, 90, 63, 78), _lens(rng, 10, 79, 250)])
    off, ids = eo.csr(_make_lists(rng, top[rows], lens, n, n + 1))
    ids_ext = np.where((ids >= 0) & (ids < n), ext[np.clip(ids, 0, n - 1)], ids)

    def subset_search(q, keep_rows, labels):
        sub = nf.IndexFlatIP(d)
        sub.add(xb[keep_rows])
        Dq, Iq = sub.search(xq[q:q + 1], k)
        return Dq, np.where(Iq < 0, -1, labels[np.maximum(Iq, 0)])

    for index, sel, lids, labels in ((flat, nf.IDSelectorRange(lo, hi), ids, np.arange(n)),
                                     (m, nf.IDSelectorRange(ext[lo], ext[-1] + 1), ids_ext, ext)):
        p = nf.SearchParameters(sel=sel)
        D, I = index.search(xq[rows], k, params=p, exclude=(off, lids))

        def long_search(q, lids=lids, labels=labels):
            keep = np.nonzero((np.arange(n) >= lo) & ~np.isin(labels, lids[off[q]:off[q + 1]]))[0]
            return subset_search(q, keep, labels[keep])

        ref = _route_reference(eo, lambda xs, kk: index.search(xs, kk, params=p), xq[rows], k, off, lids, 0,
                               long_search)
        _same((D, I), ref, type(index).__name__)
        _not_listed(I, off, lids)
        assert (_np(I)[_np(I) >= 0] >= labels[lo]).all()
    # IVF: stored ids in publication order, a window over them
    xb2, xq2, _ = _ivf_data(20_000, 200, seed=81)
    ids2 = np.arange(xb2.shape[0], dtype=np.int64) + 2 ** 35
    make, _ = _ivf_pair(nf, io, xb2, 32, 0)
    ivf = make()
    ivf.add_with_ids(xb2, ids2)
    w0 = ids2[xb2.shape[0] // 2]
    p = nf.SearchParametersIVF(sel=nf.IDSelectorRange(w0, 2 ** 40), nprobe=6)
    top = _np(ivf.search(xq2, 128, params=p)[1])
    lens = np.concatenate([_lens(rng, 150, 0, 40), _lens(rng, 40, 63, 78), _lens(rng, 10, 79, 250)])
    off, lids = eo.csr(_make_lists(rng, top, lens, 2 ** 36, 3))
    D, I = ivf.search(xq2, k, params=p, exclude=(off, lids))

    def long_ivf(q):
        keep = np.nonzero((ids2 >= w0) & ~np.isin(ids2, lids[off[q]:off[q + 1]]))[0]
        sub = make()
        sub.add_with_ids(xb2[keep], ids2[keep])
        return sub.search(xq2[q:q + 1], k, params=nf.SearchParametersIVF(nprobe=6))

    ref = _route_reference(eo, lambda xs, kk: ivf.search(xs, kk, params=p), xq2, k, off, lids, 0, long_ivf)
    _same((D, I), ref, "ivf")
    _not_listed(I, off, lids)
    assert (I[I >= 0] >= w0).all()


# ------------------------------------------------------------------ empty lists
def test_exclude_empty_lists_change_nothing(nf, io, flat_data):
    import torch
    from test_gpu_ids import _ivf_data, _ivf_pair
    xb, xq = flat_data
    for metric in (0, 1):
        index = nf.IndexFlat(xb.shape[1], metric)
        index.add(xb)
        for nq, k in ((1, 50), (19, 10), (500, 50), (500, 120)):
            ex = (np.zeros(nq + 1, np.int64), np.empty(0, np.int64))
            _same(index.search(xq[:nq], k, exclude=ex), index.search(xq[:nq], k), (metric, nq, k))
            xt = torch.from_numpy(xq[:nq]).cuda()
            _same(index.search(xt, k, exclude=ex), index.search(xt, k), (metric, nq, k, "cuda"))
    xb2, xq2, ids2 = _ivf_data(20_000, 300, seed=91)
    make, _ = _ivf_pair(nf, io, xb2, 32, 1)
    ivf = make()
    ivf.add_with_ids(xb2, ids2)
    for nq, k in ((5, 50), (64, 20), (300, 50)):
        ex = (np.zeros(nq + 1, np.int64), np.empty(0, np.int64))
        p = nf.SearchParametersIVF(nprobe=8)
        _same(ivf.search(xq2[:nq], k, params=p, exclude=ex), ivf.search(xq2[:nq], k, params=p), ("ivf", nq, k))


# ------------------------------------------------------------------ config 1 at full size
def test_config1_click_history_excluded(nf, oracle, eo):
    from newsrecommend_b200 import synth
    from test_gpu_fullsize import _all_threads
    _all_threads()
    xb, topics = synth.g_skew(synth.N_ARTICLES, 250, 42, return_topics=True)
    xq, (off, clicks) = synth.user_profiles(xb, topics, synth.N_TEST_USERS, 43, return_clicks=True)
    index = nf.IndexFlatIP(250)
    index.add(xb)
    k = 50
    D, I = index.search(xq, k, exclude=(off, clicks))
    assert (I >= 0).all()
    owner = np.repeat(np.arange(xq.shape[0]), np.diff(off))
    # (user, row) pairs: a returned row the user clicked would appear in both sets
    ret = I.astype(np.int64) + np.arange(xq.shape[0])[:, None] * np.int64(synth.N_ARTICLES)
    assert not np.isin(ret, clicks + owner * np.int64(synth.N_ARTICLES)).any()
    sample = np.random.default_rng(5).choice(xq.shape[0], 4096, replace=False)
    so = np.zeros(sample.size + 1, np.int64)
    np.cumsum(np.diff(off)[sample], out=so[1:])
    sids = np.concatenate([clicks[off[u]:off[u + 1]] for u in sample])
    Do, Io = oracle.knn_fast(xq[sample], xb, k + 64, 0)  # k + the longest list: the first k survivors are exact
    Dx, Ix = eo.exclude_topk(Do, Io, None, so, sids, 0, k, np.empty((sample.size, k), np.float32),
                             np.empty((sample.size, k), np.int64))
    _parity(D[sample], I[sample], Dx, Ix, 0, "config1")
