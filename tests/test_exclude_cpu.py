"""CPU checks of per-query exclusion lists: the numpy restatement of nrb_exclude_topk and of the whole
feature (tests/exclude_oracle.py) against fp64 brute force, the argument errors of search(exclude=...),
the C-ABI argument checks of nrb_exclude_topk, and synth.user_profiles(return_clicks=True)."""
import numpy as np
import pytest
import torch

from newsrecommend_b200 import _lib, synth

FLT_MAX = np.float32(3.4028234663852886e38)


@pytest.fixture(scope="module")
def eo(oracle):
    import exclude_oracle
    return exclude_oracle


@pytest.fixture(scope="module")
def io(oracle):
    import ids_oracle
    return ids_oracle


def _brute_excluded(xq, xb, labels, k, metric, off, ids, cand=None):
    """fp64 top k of the rows query q may see: not listed (and in cand[q] when given), ties by row."""
    nq = xq.shape[0]
    D = np.full((nq, k), -FLT_MAX if metric == 0 else FLT_MAX, dtype=np.float64)
    I = np.full((nq, k), -1, dtype=np.int64)
    x64, b64 = xq.astype(np.float64), xb.astype(np.float64)
    for q in range(nq):
        ok = ~np.isin(labels, ids[off[q]:off[q + 1]])
        if cand is not None:
            ok &= cand[q]
        rows = np.nonzero(ok)[0]
        sc = b64[rows] @ x64[q] if metric == 0 else ((b64[rows] - x64[q]) ** 2).sum(1)
        o = np.argsort(-sc if metric == 0 else sc, kind="stable")[:k]
        D[q, :o.size], I[q, :o.size] = sc[o], labels[rows[o]]
    return D, I


def _check(D, I, Dt, It, metric):
    from newsrecommend_b200.parity import compare_topk
    rep = compare_topk(D, I, Dt, It, metric)
    assert rep["ok"], rep


def _lists(rng, labels, nq, n_absent):
    """Lists with duplicates, -1, ids absent from the index, empty lists, one list of every label and
    one longer than the index."""
    lists = []
    for q in range(nq):
        kind = q % 6
        if kind == 0:
            lists.append([])
        elif kind == 1:
            l = rng.choice(labels, 5)
            lists.append(np.concatenate([l, l[:3], [-1, -1]]))  # duplicates and -1
        elif kind == 2:
            lists.append(np.concatenate([rng.choice(labels, 12), n_absent + rng.integers(0, 50, 4), [-7]]))
        elif kind == 3:
            lists.append(rng.permutation(labels))  # every row: only padding is left
        elif kind == 4:
            lists.append(rng.choice(labels, labels.size - 10, replace=False))  # k + E_q > ntotal
        else:
            lists.append(rng.choice(labels, 40))
    return lists


def test_exclude_topk_restatement(eo):
    Din = np.array([[9, 8, 7, 6, 5, 4], [3, 2, 1, -FLT_MAX, -FLT_MAX, -FLT_MAX]], np.float32)
    Iin = np.array([[10, 11, 12, 13, 14, 15], [20, 21, 22, -1, -1, -1]], np.int64)
    off, ids = eo.csr([[11, 11, -1, 99], [], [21, 22, -1, 20, 13]])
    D = np.zeros((3, 3), np.float32)
    I = np.zeros((3, 3), np.int64)
    eo.exclude_topk(Din, Iin, np.array([0, 2]), off, ids, 0, 3, D, I)
    assert I[0].tolist() == [10, 12, 13] and D[0].tolist() == [9, 7, 6]
    assert I[2].tolist() == [-1, -1, -1] and (D[2] == -FLT_MAX).all()  # -1 in the list keeps the padding
    assert (I[1] == 0).all()  # no row of the input is query 1's
    D2, I2 = np.zeros((2, 2), np.float32), np.zeros((2, 2), np.int64)
    eo.exclude_topk(Din, Iin, None, off, ids, 1, 2, D2, I2)
    assert I2.tolist() == [[10, 12], [20, 21]]


@pytest.mark.parametrize("metric", [0, 1])
def test_oracle_excluded_flat_and_idmap(eo, io, metric):
    rng = np.random.default_rng(7)
    n, d, k, nq = 300, 16, 20, 36
    xb = rng.standard_normal((n, d), dtype=np.float32)
    xq = rng.standard_normal((nq, d), dtype=np.float32)
    flat = io.IndexFlat(d, metric)
    flat.add(xb)
    pos = np.arange(n, dtype=np.int64)
    off, ids = eo.csr(_lists(rng, pos, nq, n))
    D, I = eo.search_excluded(flat.search, xq, k, off, ids, metric)
    _check(D, I, *_brute_excluded(xq, xb, pos, k, metric, off, ids), metric)
    for q in range(nq):
        assert not np.isin(I[q][I[q] >= 0], ids[off[q]:off[q + 1]]).any()
    assert (I[3::6] == -1).all()  # every row listed
    ext = rng.permutation(10 * n)[:n].astype(np.int64) * 3 + 2 ** 33
    m = io.IndexIDMap(io.IndexFlat(d, metric))
    m.add_with_ids(xb, ext)
    off, ids = eo.csr(_lists(rng, ext, nq, 2 ** 40))
    D, I = eo.search_excluded(m.search, xq, k, off, ids, metric)
    _check(D, I, *_brute_excluded(xq, xb, ext, k, metric, off, ids), metric)


@pytest.mark.parametrize("metric", [0, 1])
def test_oracle_excluded_ivf(eo, io, metric):
    """The coarse search is the unexcluded one; the scan of the probed lists skips the listed ids."""
    rng = np.random.default_rng(8)
    n, d, nlist, k, nq = 2000, 16, 10, 15, 24
    xb = rng.standard_normal((n, d), dtype=np.float32)
    xq = rng.standard_normal((nq, d), dtype=np.float32)
    ids_b = rng.permutation(4 * n)[:n].astype(np.int64) + 10 ** 6
    qz = io.IndexFlatIP(d) if metric == 0 else io.IndexFlatL2(d)
    ivf = io.IndexIVFFlat(qz, d, nlist, metric)
    ivf.train(xb)
    ivf.add_with_ids(xb, ids_b)
    lists = _lists(rng, ids_b, nq, 0)
    lists = [l if q % 6 != 4 else rng.choice(ids_b, 60) for q, l in enumerate(lists)]
    off, ids = eo.csr(lists)
    cent = qz.xb.astype(np.float64)
    assign = qz.assign(xb, 1).reshape(-1)
    for nprobe in (1, 3, nlist):
        ivf.nprobe = nprobe
        D, I = eo.search_excluded(ivf.search, xq, k, off, ids, metric)
        cs = xq.astype(np.float64) @ cent.T if metric == 0 else -((xq[:, None].astype(np.float64) - cent) ** 2).sum(-1)
        probed = np.argsort(-cs, axis=1, kind="stable")[:, :nprobe]
        cand = np.stack([np.isin(assign, probed[q]) for q in range(nq)])
        _check(D, I, *_brute_excluded(xq, xb, ids_b, k, metric, off, ids, cand), metric)


def test_exclude_argument_errors():
    import newsrecommend_b200.faiss as nf
    x = np.zeros((3, 8), np.float32)
    ok_off, ok_ids = np.array([0, 1, 1, 3], np.int64), np.array([4, 5, 6], np.int64)
    ivf = nf.IndexIVFFlat(nf.IndexFlatL2(8), 8, 4)
    for index in (nf.IndexFlatIP(8), nf.IndexIDMap(nf.IndexFlatL2(8)), ivf):
        bad = [
            (TypeError, [ok_off, ok_ids][:1]),
            (TypeError, ok_off),
            (TypeError, (ok_off.astype(np.int32), ok_ids)),
            (TypeError, (ok_off, ok_ids.astype(np.float64))),
            (TypeError, (ok_off.tolist(), ok_ids)),
            (TypeError, (torch.from_numpy(ok_off).int(), ok_ids)),
            (ValueError, (ok_off[:-1], ok_ids)),
            (ValueError, (np.array([0, 1, 1, 2, 3], np.int64), ok_ids)),
            (ValueError, (np.array([1, 1, 1, 3], np.int64), ok_ids)),
            (ValueError, (np.array([0, 1, 1, 2], np.int64), ok_ids)),
            (ValueError, (np.array([0, 2, 1, 3], np.int64), ok_ids)),
            (ValueError, (ok_off.reshape(1, 4), ok_ids)),
            (ValueError, (ok_off, ok_ids.reshape(3, 1))),
        ]
        for err, ex in bad:
            with pytest.raises(err):
                index.search(x, 2, exclude=ex)
    with pytest.raises(TypeError):  # exclude is keyword-only
        nf.IndexFlatL2(8).search(x, 2, None, None, None, (ok_off, ok_ids))
    assert nf._exclude_arg((torch.from_numpy(ok_off), torch.from_numpy(ok_ids)), 3)[0].tolist() == ok_off.tolist()


def test_exclude_topk_rejects_bad_arguments():
    L = _lib.lib
    D = np.empty(8, np.float32)
    I = np.empty(8, np.int64)
    p = (D.ctypes.data, I.ctypes.data)
    off = np.array([0, 0], np.int64)
    assert L.nrb_exclude_topk(None, None, 0, 4, None, None, None, 0, 2, None, None, None) == 0  # nothing to do
    for nrows, kin, metric, k in ((-1, 4, 0, 2), (1, 0, 0, 1), (1, 129, 0, 2), (1, 4, 0, 5), (1, 4, 0, 0),
                                  (1, 4, 2, 2), (1, 4, -1, 2)):
        assert L.nrb_exclude_topk(*p, nrows, kin, None, off.ctypes.data, I.ctypes.data, metric, k, *p, None) == -1
        assert "exclude_topk" in _lib.last_error()
    for miss in range(5):
        args = [D.ctypes.data, I.ctypes.data, off.ctypes.data, I.ctypes.data, D.ctypes.data, I.ctypes.data]
        args[[0, 1, 2, 3, 5][miss]] = None
        rc = L.nrb_exclude_topk(args[0], args[1], 1, 4, None, args[2], args[3], 0, 2, args[4], args[5], None)
        assert rc == -1 and "null" in _lib.last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_exclude_topk_without_device():
    D = np.empty(8, np.float32)
    I = np.empty(8, np.int64)
    off = np.array([0, 0], np.int64)
    assert _lib.lib.nrb_exclude_topk(D.ctypes.data, I.ctypes.data, 1, 4, None, off.ctypes.data, I.ctypes.data, 1, 4,
                                     D.ctypes.data, I.ctypes.data, None) == -3


@pytest.mark.parametrize("topics", [True, False])
def test_user_profiles_return_clicks(topics):
    xb, tp = synth.g_skew(3000, 24, 42, return_topics=True)
    tp = tp if topics else None
    plain = synth.user_profiles(xb, tp, 500, 43)
    prof, (off, rows) = synth.user_profiles(xb, tp, 500, 43, return_clicks=True)
    assert np.array_equal(prof.view(np.int32), plain.view(np.int32))
    assert off.dtype == np.int64 and rows.dtype == np.int64 and off.shape == (501,)
    assert off[0] == 0 and off[-1] == rows.size and (np.diff(off) >= 1).all() and (np.diff(off) <= 64).all()
    assert rows.min() >= 0 and rows.max() < xb.shape[0]
    for u in range(500):
        mean = xb[rows[off[u]:off[u + 1]]].astype(np.float64).mean(0)
        assert np.allclose(prof[u], mean, rtol=1e-5, atol=1e-5)
