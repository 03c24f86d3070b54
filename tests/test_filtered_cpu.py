"""CPU checks of search-time ID selectors: SearchParameters / SearchParametersIVF and their argument
errors, IDSelectorNot, the shim's new names, the argument checks of the new C-ABI entry points, and
the numpy restatement of filtered flat / IndexIDMap / IVF search (tests/filtered_oracle.py) against
brute force."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from newsrecommend_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLT_MAX = 3.4028235e38


@pytest.fixture(scope="module")
def fo(oracle):
    import filtered_oracle
    return filtered_oracle


@pytest.fixture(scope="module")
def io(oracle):
    import ids_oracle
    return ids_oracle


def _nf():
    import newsrecommend_b200.faiss as nf
    return nf


def _brute(xq, xb, ids, k, metric):
    """fp64 top-k over the rows xb labelled ids, ties by position; -1 / -+FLT_MAX padding."""
    nq = xq.shape[0]
    D = np.full((nq, k), -FLT_MAX if metric == 0 else FLT_MAX)
    I = np.full((nq, k), -1, dtype=np.int64)
    if xb.shape[0] == 0:
        return D, I
    sc = xq.astype(np.float64) @ xb.astype(np.float64).T if metric == 0 else \
        ((xq[:, None, :].astype(np.float64) - xb[None].astype(np.float64)) ** 2).sum(-1)
    for q in range(nq):
        o = np.argsort(-sc[q] if metric == 0 else sc[q], kind="stable")[:k]
        D[q, :len(o)], I[q, :len(o)] = sc[q, o], ids[o]
    return D, I


def _check(D, I, Dt, It, metric):
    from newsrecommend_b200.parity import compare_topk
    rep = compare_topk(D, I, Dt, It, metric)
    assert rep["ok"], rep


def test_search_parameters():
    nf = _nf()
    p = nf.SearchParameters()
    assert p.sel is None
    r = nf.IDSelectorRange(0, 10)
    assert nf.SearchParameters(sel=r).sel is r
    q = nf.SearchParametersIVF(sel=r, nprobe=7)
    assert isinstance(q, nf.SearchParameters) and q.sel is r and q.nprobe == 7 and q.max_codes == 0
    assert nf.SearchParametersIVF().nprobe is None
    assert nf.SearchParametersIVF(max_codes=0).max_codes == 0
    with pytest.raises(NotImplementedError):
        nf.SearchParametersIVF(max_codes=1000)
    for cls, kw in ((nf.SearchParameters, {"nprobe": 4}), (nf.SearchParameters, {"quantizer_params": None}),
                    (nf.SearchParametersIVF, {"quantizer_params": None}),
                    (nf.SearchParametersIVF, {"inverted_list_context": None}), (nf.SearchParametersIVF, {"bogus": 1})):
        with pytest.raises(TypeError):
            cls(**kw)
    with pytest.raises(TypeError):
        nf.SearchParameters(sel=np.arange(3))
    # IndexIVFFlat wants SearchParametersIVF (checked before any device work); flat indexes take either
    ivf = nf.IndexIVFFlat(nf.IndexFlatL2(8), 8, 4)
    with pytest.raises(RuntimeError, match="IndexIVF params have incorrect type"):
        ivf.search(np.zeros((1, 8), np.float32), 1, params=nf.SearchParameters(sel=r))
    with pytest.raises(TypeError):
        nf.IndexFlatL2(8).search(np.zeros((1, 8), np.float32), 1, params=object())
    with pytest.raises(TypeError):  # params is keyword-only
        nf.IndexFlatL2(8).search(np.zeros((1, 8), np.float32), 1, None, None, nf.SearchParameters())


def test_idselector_not():
    nf = _nf()
    r = nf.IDSelectorRange(10, 20)
    b = nf.IDSelectorBatch(np.array([3, 15, -7], np.int64))
    n1, n2, n3 = nf.IDSelectorNot(r), nf.IDSelectorNot(nf.IDSelectorNot(b)), nf.IDSelectorNot(nf.IDSelectorNot(
        nf.IDSelectorNot(b)))
    for i in (-7, 0, 3, 9, 10, 15, 19, 20):
        assert n1.is_member(i) == (not r.is_member(i))
        assert n2.is_member(i) == b.is_member(i)
        assert n3.is_member(i) == (not b.is_member(i))
    assert nf._unwrap_not(n1) == (r, 0) and nf._unwrap_not(n2) == (b, 1) and nf._unwrap_not(n3) == (b, 0)
    with pytest.raises(TypeError):
        nf.IDSelectorNot(np.arange(3))
    assert nf._selector(n1) is n1  # remove_ids accepts it
    # host-side count of kept positions (the small route skips the search when it is 0)
    assert nf._positions_kept(r, 15) == 5 and nf._positions_kept(n1, 15) == 10
    assert nf._positions_kept(b, 100) == 2 and nf._positions_kept(n3, 100) == 98
    assert nf._positions_kept(nf.IDSelectorRange(5, 5), 10) == 0
    assert nf._positions_kept(nf.IDSelectorNot(nf.IDSelectorRange(-5, 50)), 10) == 0


def test_shim_exports_selectors():
    sys.path.insert(0, os.path.join(ROOT, "shim"))
    try:
        import faiss
        import newsrecommend_b200.faiss as nf
        for name in ("IDSelectorNot", "SearchParameters", "SearchParametersIVF"):
            assert getattr(faiss, name) is getattr(nf, name) and name in nf.__all__
    finally:
        sys.path.pop(0)


def test_sel_entry_points_reject_bad_arguments():
    L = _lib.lib
    m = _lib.Matrix()
    D = np.empty(1, np.float32)
    I = np.empty(1, np.int64)
    # member == NULL is refused before any device work
    rc = L.nrb_search_small_sel(None, 8, 1, 8, C.byref(m), 0, 1, 0, D.ctypes.data, I.ctypes.data, None, 0, None, None, 1)
    assert rc == -1 and "member" in _lib.last_error()
    rc = L.nrb_search_small_host_sel(C.byref(m), D.ctypes.data, 1, 8, 0, 1, 0, D.ctypes.data, I.ctypes.data, None, None, 1)
    assert rc == -1 and "member" in _lib.last_error()
    rc = L.nrb_ivf_scan_small_sel(None, 8, 1, 8, C.byref(m), None, 4, 1, None, None, 1, 0, 1, None, None, None, 0, None,
                                  None, 1)
    assert rc == -1 and "member" in _lib.last_error()
    assert L.nrb_sel_keys(None, 1, None, 0, 4, None, None) == 0  # nothing to do
    assert L.nrb_sel_keys(None, 1, None, 10, 4, None, None) == -1
    assert L.nrb_sel_keys(None, 1, None, -1, 4, None, None) == -1


@pytest.mark.parametrize("metric", [0, 1])
def test_oracle_filtered_flat_and_idmap(fo, io, metric):
    rng = np.random.default_rng(3)
    n, d, k = 400, 16, 30
    xb = rng.standard_normal((n, d), dtype=np.float32)
    xq = rng.standard_normal((23, d), dtype=np.float32)
    ids = rng.permutation(10 * n)[:n].astype(np.int64) * 7 - 900
    flat = io.IndexFlat(d, metric)
    flat.add(xb)
    m = io.IndexIDMap(io.IndexFlat(d, metric))
    m.add_with_ids(xb, ids)
    pos = np.arange(n, dtype=np.int64)
    for sel in (io.IDSelectorRange(100, 300), io.IDSelectorBatch(pos[::9]), fo.IDSelectorNot(io.IDSelectorRange(20, 390)),
                fo.IDSelectorNot(fo.IDSelectorNot(io.IDSelectorBatch(pos[5:12]))), io.IDSelectorRange(5, 5),
                io.IDSelectorRange(-10, 10 ** 6)):
        keep = sel.members(pos)
        D, I = fo.search_flat(flat, xq, k, sel)
        _check(D, I, *_brute(xq, xb[keep], pos[keep], k, metric), metric)
        assert np.isin(I[I >= 0], pos[keep]).all()
        if keep.sum() < k:
            assert (I[:, keep.sum():] == -1).all()
    for sel in (io.IDSelectorRange(int(np.median(ids)), 10 ** 9), io.IDSelectorBatch(ids[::4]),
                fo.IDSelectorNot(io.IDSelectorBatch(ids[::3])), fo.IDSelectorNot(io.IDSelectorRange(-10 ** 9, 10 ** 9))):
        keep = sel.members(ids)
        D, I = fo.search_idmap(m, xq, k, sel)
        _check(D, I, *_brute(xq, xb[keep], ids[keep], k, metric), metric)
        assert np.isin(I[I >= 0], ids[keep]).all()


@pytest.mark.parametrize("metric", [0, 1])
def test_oracle_filtered_ivf(fo, io, metric):
    """The coarse search ranks every centroid; the scan is restricted to the selected ids."""
    rng = np.random.default_rng(4)
    n, d, nlist, k = 3000, 16, 12, 20
    xb = rng.standard_normal((n, d), dtype=np.float32)
    xq = rng.standard_normal((40, d), dtype=np.float32)
    ids = rng.permutation(5 * n)[:n].astype(np.int64) + 10 ** 6
    q = io.IndexFlatIP(d) if metric == 0 else io.IndexFlatL2(d)
    ivf = io.IndexIVFFlat(q, d, nlist, metric)
    ivf.train(xb)
    ivf.add_with_ids(xb, ids)
    cent = q.xb.astype(np.float64)
    assign = q.assign(xb, 1).reshape(-1)
    for sel in (io.IDSelectorRange(int(np.quantile(ids, 0.4)), 10 ** 9), io.IDSelectorBatch(ids[::10]),
                fo.IDSelectorNot(io.IDSelectorBatch(ids[::2])), io.IDSelectorBatch(ids[:5])):
        keep = sel.members(ids)
        for nprobe in (1, 4, nlist):
            D, I = fo.search_ivf(ivf, xq, k, sel, nprobe)
            assert np.isin(I[I >= 0], ids[keep]).all()
            for qi in range(xq.shape[0]):
                x = xq[qi].astype(np.float64)
                cs = cent @ x if metric == 0 else -((cent - x) ** 2).sum(1)
                probed = np.argsort(-cs, kind="stable")[:nprobe]  # over ALL centroids
                cand = keep & np.isin(assign, probed)
                _check(D[qi:qi + 1], I[qi:qi + 1], *_brute(xq[qi:qi + 1], xb[cand], ids[cand], k, metric), metric)
        if nprobe == nlist:
            _check(D, I, *_brute(xq, xb[keep], ids[keep], k, metric), metric)
    assert fo.filtered_ivf(ivf, io.IDSelectorRange(0, 0)).ntotal == 0
    D, I = fo.search_ivf(ivf, xq, k, io.IDSelectorRange(0, 0), nlist)
    assert (I == -1).all()
