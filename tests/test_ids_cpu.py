"""CPU checks of external ids and removal: the oracle's faiss semantics (IndexFlat.remove_ids,
IndexIVFFlat.add_with_ids / remove_ids, IndexIDMap, IDSelectorBatch / IDSelectorRange) against numpy
brute force, the argument checks of nrb_id_select / nrb_map_ids, and the shim's new names."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from newsrecommend_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def oracle(oracle):
    """The CPU oracle with faiss's external-id semantics added (tests/ids_oracle.py)."""
    import ids_oracle
    return ids_oracle


def _brute(xq, xb, ids, k, metric):
    """fp64 top-k over the rows xb labelled ids, ties by position; -1 / -+FLT_MAX padding."""
    sc = xq.astype(np.float64) @ xb.astype(np.float64).T if metric == 0 else \
        ((xq[:, None, :].astype(np.float64) - xb[None].astype(np.float64)) ** 2).sum(-1)
    nq = xq.shape[0]
    D = np.full((nq, k), -3.4028235e38 if metric == 0 else 3.4028235e38)
    I = np.full((nq, k), -1, dtype=np.int64)
    for q in range(nq):
        o = np.argsort(-sc[q] if metric == 0 else sc[q], kind="stable")[:k]
        D[q, :len(o)], I[q, :len(o)] = sc[q, o], ids[o]
    return D, I


def _check(D, I, Dt, It, metric):
    from newsrecommend_b200.parity import compare_topk
    rep = compare_topk(D, I, Dt, It, metric)
    assert rep["ok"], rep


@pytest.mark.parametrize("metric", [0, 1])
def test_oracle_flat_remove_renumbers(oracle, metric):
    rng = np.random.default_rng(1)
    xb = rng.standard_normal((300, 12), dtype=np.float32)
    xq = rng.standard_normal((25, 12), dtype=np.float32)
    idx = oracle.IndexFlat(12, metric)
    idx.add(xb)
    with pytest.raises(RuntimeError, match="add_with_ids not implemented"):
        idx.add_with_ids(xb, np.arange(300))
    assert idx.remove_ids(oracle.IDSelectorRange(50, 100)) == 50
    assert idx.remove_ids(np.array([0, 0, 7, 10_000], dtype=np.int64)) == 2  # positions after the first removal
    keep = np.ones(300, bool)
    keep[50:100] = False
    pos = np.nonzero(keep)[0]
    keep[pos[[0, 7]]] = False
    assert idx.ntotal == keep.sum() and np.array_equal(idx.xb, xb[keep])
    D, I = idx.search(xq, 10)
    _check(D, I, *_brute(xq, xb[keep], np.arange(keep.sum()), 10, metric), metric)  # renumbered 0..n-1
    assert idx.remove_ids(oracle.IDSelectorBatch(np.empty(0, np.int64))) == 0
    assert idx.remove_ids(oracle.IDSelectorRange(0, 10 ** 9)) == keep.sum() and idx.ntotal == 0


@pytest.mark.parametrize("metric", [0, 1])
def test_oracle_idmap_translates_and_removes(oracle, metric):
    rng = np.random.default_rng(2)
    xb = rng.standard_normal((400, 10), dtype=np.float32)
    xq = rng.standard_normal((30, 10), dtype=np.float32)
    ids = rng.permutation(10 ** 6)[:400].astype(np.int64) - 500_000
    with pytest.raises(RuntimeError, match="must be empty"):
        flat = oracle.IndexFlat(10, metric)
        flat.add(xb[:1])
        oracle.IndexIDMap(flat)
    m = oracle.IndexIDMap(oracle.IndexFlat(10, metric))
    with pytest.raises(RuntimeError, match="add_with_ids"):
        m.add(xb)
    m.add_with_ids(xb[:150], ids[:150])
    m.add_with_ids(xb[150:], ids[150:])
    D, I = m.search(xq, 20)
    _check(D, I, *_brute(xq, xb, ids, 20, metric), metric)
    # remove by external id: a range, a batch (SWIG form, n < len) and a plain array
    r = m.remove_ids(oracle.IDSelectorRange(-100_000, 100_000))
    gone = (ids >= -100_000) & (ids < 100_000)
    assert r == gone.sum()
    batch = ids[~gone][:40]
    assert m.remove_ids(oracle.IDSelectorBatch(20, batch)) == 20
    assert m.remove_ids(batch[20:]) == 20
    gone |= np.isin(ids, batch)
    assert m.ntotal == (~gone).sum() and np.array_equal(m.id_map, ids[~gone])
    D, I = m.search(xq, 20)
    _check(D, I, *_brute(xq, xb[~gone], ids[~gone], 20, metric), metric)
    m.reset()
    assert m.ntotal == 0 and m.id_map.size == 0
    D, I = m.search(xq[:3], 5)
    assert (I == -1).all()


@pytest.mark.parametrize("metric", [0, 1])
def test_oracle_ivf_keeps_ids_through_removal(oracle, metric):
    rng = np.random.default_rng(3)
    d, nlist = 8, 6
    cent = rng.standard_normal((nlist, d), dtype=np.float32)
    xb = rng.standard_normal((500, d), dtype=np.float32)
    xq = rng.standard_normal((20, d), dtype=np.float32)
    q = oracle.IndexFlatIP(d) if metric == 0 else oracle.IndexFlatL2(d)
    q.add(cent)
    ivf = oracle.IndexIVFFlat(q, d, nlist, metric)
    ivf.train(xb)
    ids = rng.permutation(5000)[:500].astype(np.int64) * 7
    ivf.add_with_ids(xb[:200], ids[:200])
    ivf.add_with_ids(xb[200:], ids[200:])
    ivf.nprobe = nlist  # exact
    D, I = ivf.search(xq, 15)
    _check(D, I, *_brute(xq, xb, ids, 15, metric), metric)
    gone = np.isin(ids, ids[::3])
    assert ivf.remove_ids(ids[::3]) == gone.sum() == 500 - ivf.ntotal
    assert ivf.remove_ids(oracle.IDSelectorRange(0, 7000)) == ((ids < 7000) & ~gone).sum()
    gone |= ids < 7000
    assert ivf.list_sizes().sum() == ivf.ntotal == (~gone).sum()
    off, cids, rows = ivf._build_csr()
    assert sorted(cids.tolist()) == sorted(ids[~gone].tolist())
    for i, c in zip(cids[:50], rows[:50]):
        assert np.array_equal(c, xb[ids == i][0])  # every id still names its own row
    D, I = ivf.search(xq, 15)
    _check(D, I, *_brute(xq, xb[~gone], ids[~gone], 15, metric), metric)
    # add() after removals numbers from ntotal, as faiss does
    n0 = ivf.ntotal
    ivf.add(xb[:3])
    assert set(np.concatenate([c[0] for l in ivf._lists for c in l]).tolist()) >= {n0, n0 + 1, n0 + 2}


def test_oracle_ivf_remove_fills_holes_with_the_last_entry(oracle):
    d = 4
    q = oracle.IndexFlatL2(d)
    q.add(np.zeros((1, d), np.float32))
    ivf = oracle.IndexIVFFlat(q, d, 1)
    ivf.train(np.zeros((1, d), np.float32))
    x = np.arange(6 * d, dtype=np.float32).reshape(6, d)
    ivf.add_with_ids(x, np.array([10, 11, 12, 13, 14, 15]))
    assert ivf.remove_ids(np.array([11])) == 1
    off, ids, rows = ivf._build_csr()
    assert ids.tolist() == [10, 15, 12, 13, 14] and np.array_equal(rows[1], x[5])


def _ws(nbytes):
    return np.zeros(max(nbytes, 1), dtype=np.uint8)


def test_id_select_argument_checks():
    L = _lib.lib
    ids = np.arange(10, dtype=np.int64)
    batch = np.array([1, 2, 3], dtype=np.int64)
    member = np.zeros(10, dtype=np.int64)
    assert L.nrb_id_select_workspace(0) == 0
    wsb = L.nrb_id_select_workspace(3)
    assert wsb >= 3 * 8 * 2 and L.nrb_id_select_workspace(1000) >= 2000 * 8
    ws = _ws(wsb)
    a = (ids.ctypes.data, 10, batch.ctypes.data, 3, 0, 0, member.ctypes.data, ws.ctypes.data, wsb, None)
    bad = [(1, -1), (3, -1)]  # n < 0, nbatch < 0
    for pos, val in bad:
        args = list(a)
        args[pos] = val
        assert L.nrb_id_select(*args) == -1, pos
    args = list(a)
    args[2] = None  # nbatch > 0 with no batch
    assert L.nrb_id_select(*args) == -1
    args = list(a)
    args[8] = wsb - 1  # workspace too small
    assert L.nrb_id_select(*args) == -4
    args[8], args[7] = 0, None
    assert L.nrb_id_select(*args) == -4
    # a range and an empty batch need no workspace
    assert L.nrb_id_select_workspace(0) == 0
    assert L.nrb_map_ids(None, member.ctypes.data, -1, None) == -1
    assert L.nrb_map_ids(None, member.ctypes.data, 10, None) == -1
    assert L.nrb_map_ids(ids.ctypes.data, member.ctypes.data, 0, None) == 0
    assert L.nrb_id_select(ids.ctypes.data, 0, batch.ctypes.data, 3, 0, 0, None, ws.ctypes.data, wsb, None) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_id_entry_points_need_a_device():
    L = _lib.lib
    ids = np.arange(10, dtype=np.int64)
    batch = np.array([1, 2, 3], dtype=np.int64)
    member = np.zeros(10, dtype=np.int64)
    wsb = L.nrb_id_select_workspace(3)
    ws = _ws(wsb)
    assert L.nrb_id_select(ids.ctypes.data, 10, batch.ctypes.data, 3, 0, 0, member.ctypes.data, ws.ctypes.data, wsb,
                           None) == -3
    assert L.nrb_id_select(None, 10, None, 0, 2, 5, member.ctypes.data, None, 0, None) == -3
    assert L.nrb_map_ids(ids.ctypes.data, member.ctypes.data, 10, None) == -3
    assert "no CPU fallback" in _lib.last_error()


def test_selector_arguments():
    import newsrecommend_b200.faiss as nf
    r = nf.IDSelectorRange(3, 9, True)
    assert (r.imin, r.imax, r.assume_sorted) == (3, 9, True) and r.is_member(3) and not r.is_member(9)
    b = nf.IDSelectorBatch(2, np.array([5, 6, 7]))
    assert b.ids.tolist() == [5, 6] and b.ids.dtype == np.int64 and b.is_member(6) and not b.is_member(7)
    assert nf.IDSelectorBatch(torch.tensor([1, 2])).ids.tolist() == [1, 2]
    assert nf.IDSelectorBatch([]).ids.size == 0
    with pytest.raises(TypeError):
        nf.IDSelectorBatch(np.array([1.5, 2.0]))
    with pytest.raises(ValueError):
        nf.IDSelectorBatch(5, np.array([1, 2]))
    with pytest.raises(TypeError):
        nf._selector("1, 2")
    assert isinstance(nf._selector(np.array([4], np.int64)), nf.IDSelectorBatch)
    with pytest.raises(TypeError, match="IndexIVFFlat has add_with_ids"):
        nf.IndexIDMap(nf.IndexIVFFlat(nf.IndexFlatL2(4), 4, 2))
    with pytest.raises(TypeError, match="int64"):
        nf._ids_arg(np.arange(3, dtype=np.int32), 3, "cpu")
    with pytest.raises(TypeError, match="length 3"):
        nf._ids_arg(np.arange(4, dtype=np.int64), 3, "cpu")
    with pytest.raises(TypeError):
        nf._ids_arg([0, 1, 2], 3, "cpu")


def test_shim_exports_id_names():
    sys.path.insert(0, os.path.join(ROOT, "shim"))
    try:
        import faiss  # the shim
        for name in ("IndexIDMap", "IDSelectorBatch", "IDSelectorRange"):
            assert hasattr(faiss, name), name
        assert hasattr(faiss.IndexFlatIP, "remove_ids") and hasattr(faiss.IndexIVFFlat, "add_with_ids")
        assert hasattr(faiss.IndexIVFFlat, "remove_ids") and hasattr(faiss.IndexFlatL2, "add_with_ids")
    finally:
        sys.path.pop(0)
        sys.modules.pop("faiss", None)
