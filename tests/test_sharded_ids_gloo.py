"""world_size-2 gloo tests (CPU) of external ids, removal and search-time selectors on the sharded
indexes: add_with_ids / add_with_ids_local (called repeatedly), remove_ids, search(params=...), the
16-byte wire format of id-carrying results, and the plain indexes' selectors and removals by global
position. The rank-local indexes are the oracle's (tests/ids_oracle.py, tests/filtered_oracle.py),
wrapped so that they take the library's selector and params objects; the codec is a numpy
restatement of nrb_pack_topk_ids / nrb_merge_topk_packed_ids. Every answer is compared with the
single oracle index of the same kind holding the same rows, ids and removals."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import filtered_oracle as fl
import ids_oracle as io
from oracle import faiss_oracle as fo
from test_sharded_gloo import NumpyCodec, _free_port

I64_MIN, I64_MAX = -(1 << 63), (1 << 63) - 1
FLT_MAX = np.float32(3.4028235e38)


class NumpyIdCodec(NumpyCodec):
    """numpy restatement of nrb_pack_topk_ids / nrb_merge_topk_packed_ids (include/nrb200.h)."""

    @staticmethod
    def pack_ids(D, I):
        d = np.ascontiguousarray(D.numpy(), dtype=np.float32).view(np.uint32).astype(np.uint64)
        i = np.ascontiguousarray(I.numpy(), dtype=np.int64)
        w0 = (d << np.uint64(32)) | np.where(i < 0, 0xFFFFFFFF, 0).astype(np.uint64)
        return torch.from_numpy(np.stack([w0.view(np.int64), i], axis=-1))

    @staticmethod
    def merge_ids(P, metric):
        P = np.ascontiguousarray(P.numpy())
        G, nq, k, _ = P.shape
        D = np.empty((nq, k), dtype=np.float32)
        I = np.empty((nq, k), dtype=np.int64)
        for q in range(nq):
            w0 = P[:, q, :, 0].reshape(-1).view(np.uint64)  # part-major: ties resolve by part, then position
            ids = P[:, q, :, 1].reshape(-1)
            keep = (w0 & np.uint64(0xFFFFFFFF)) != np.uint64(0xFFFFFFFF)
            d = (w0 >> np.uint64(32)).astype(np.uint32).view(np.float32)[keep]
            ids = ids[keep]
            o = np.argsort(-d if metric == 0 else d, kind="stable")[:k]
            D[q, :len(o)], I[q, :len(o)] = d[o], ids[o]
            D[q, len(o):], I[q, len(o):] = (FLT_MAX if metric else -FLT_MAX), -1
        return torch.from_numpy(D), torch.from_numpy(I)


def _osel(sel):
    """The library's selector as the oracle's (an oracle selector passes through)."""
    import newsrecommend_b200.faiss as nf
    if hasattr(sel, "members"):
        return sel
    if isinstance(sel, nf.IDSelectorNot):
        return fl.IDSelectorNot(_osel(sel.sel))
    if isinstance(sel, nf.IDSelectorRange):
        return io.IDSelectorRange(sel.imin, sel.imax)
    if isinstance(sel, nf.IDSelectorBatch):
        return io.IDSelectorBatch(sel.ids)
    return io.IDSelectorBatch(np.asarray(sel, dtype=np.int64))


class OFlat(io.IndexFlat):
    def search(self, x, k, params=None):
        if params is None or params.sel is None:
            return super().search(x, k)
        return fl.search_flat(self, x, k, _osel(params.sel))

    def remove_ids(self, sel):
        return super().remove_ids(_osel(sel))


class OIDMap(io.IndexIDMap):
    def search(self, x, k, params=None):
        if params is None or params.sel is None:
            return super().search(x, k)
        return fl.search_idmap(self, x, k, _osel(params.sel))

    def remove_ids(self, sel):
        return super().remove_ids(_osel(sel))


class OIVF(io.IndexIVFFlat):
    def search(self, x, k, params=None):
        if params is None:
            return super().search(x, k)
        sel = _osel(params.sel) if params.sel is not None else io.IDSelectorRange(I64_MIN, I64_MAX)
        return fl.search_ivf(self, x, k, sel, params.nprobe)

    def remove_ids(self, sel):
        return super().remove_ids(_osel(sel))


def _same(a, b, what):
    Da, Ia = (t.numpy() if isinstance(t, torch.Tensor) else t for t in a)
    Db, Ib = b
    assert np.array_equal(Ia, Ib), (what, "ids differ from the single index")
    assert np.allclose(Da, Db, rtol=1e-5, atol=1e-5), (what, "scores differ")


def _all_equal(v):
    """The value on every rank (an int), checked equal across ranks."""
    t = torch.tensor([v], dtype=torch.int64)
    out = [torch.zeros(1, dtype=torch.int64) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    assert all(int(o) == v for o in out), ("ranks disagree", [int(o) for o in out])
    return v


def _selectors(nf, ids, owned_by_rank1):
    """(name, selector) pairs over ids: a freshness window, a blocklist, rows of one shard, nothing."""
    s = np.sort(ids)
    return [
        ("newest10", nf.IDSelectorRange(int(s[int(0.9 * len(s))]), I64_MAX)),
        ("blocklist", nf.IDSelectorNot(nf.IDSelectorBatch(ids[::7].copy()))),
        ("one_shard", nf.IDSelectorBatch(owned_by_rank1)),
        ("nothing", nf.IDSelectorRange(0, 0) if not (ids == 0).any() else nf.IDSelectorBatch(np.array([-12345]))),
    ]


def _flat_ids_case(rank, world, metric, exchange, form, nf):
    from newsrecommend_b200.sharded import ShardedIndexFlat, shard_range
    rng = np.random.default_rng(10 + metric)
    d, k, n1, n2 = 16, 10, 301, 200
    x = rng.standard_normal((n1 + n2 + 50, d), dtype=np.float32)
    xq = rng.standard_normal((37, d), dtype=np.float32)
    ids = (np.sort(rng.choice(1 << 40, n1 + n2 + 50, replace=False)) + (1 << 33)).astype(np.int64)  # beyond 32 bits
    idx = ShardedIndexFlat(d, metric, make_index=OFlat, make_idmap=OIDMap, codec=NumpyIdCodec, exchange=exchange,
                           chunk_queries=16)
    single = OIDMap(OFlat(d, metric))
    owned1 = []
    for a, b in ((0, n1), (n1, n1 + n2)):  # two adds: each rank appends its slice of every batch
        lo, hi = shard_range(b - a, world, rank)
        if form == "global":
            idx.add_with_ids(x[a:b], ids[a:b])
        else:
            idx.add_with_ids_local(x[a + lo:a + hi], ids[a + lo:a + hi])
        single.add_with_ids(x[a:b], ids[a:b])
        owned1.append(ids[a:b][slice(*shard_range(b - a, world, 1))][:4])
    assert idx.with_ids and _all_equal(idx.ntotal) == n1 + n2
    with pytest.raises(RuntimeError, match="add_with_ids"):
        idx.add_global(x)
    with pytest.raises(RuntimeError, match="add_with_ids"):
        idx.add_local(x[:3], 0, 3)
    with pytest.raises(TypeError):
        idx.search(xq, k, params="sel")
    _same(idx.search(xq, k), single.search(xq, k), "unfiltered")
    for name, sel in _selectors(nf, ids[:n1 + n2], np.concatenate(owned1)):
        p = nf.SearchParameters(sel=sel)
        D, I = idx.search(xq, k, params=p)
        _same((D, I), single.search(xq, k, params=p), name)
        if name == "one_shard":
            assert (I.numpy()[:, 8:] == -1).all()  # 8 rows qualify: the tail is padding
        if name == "nothing":
            assert (I.numpy() == -1).all() and (D.numpy() == (FLT_MAX if metric else -FLT_MAX)).all()
        Dr, Ir, spans = idx.search(xq, k, gather=False, params=p)
        rows = np.concatenate([np.arange(a, b) for a, b in spans])
        assert np.array_equal(Ir.numpy(), I.numpy()[rows])
    # removals by external id: a range, a batch, Not and a plain array
    s = np.sort(ids[:n1 + n2])
    removals = [nf.IDSelectorRange(int(s[10]), int(s[40])), nf.IDSelectorBatch(ids[100:400:9].copy()),
                nf.IDSelectorNot(nf.IDSelectorRange(I64_MIN, int(s[-15]))), ids[200:260:2].copy(),
                nf.IDSelectorBatch(np.array([-1, 5], dtype=np.int64))]
    for sel in removals:
        r = idx.remove_ids(sel)
        assert _all_equal(r) == single.remove_ids(sel)
        assert _all_equal(idx.ntotal) == single.ntotal
    assert single.ntotal < n1 + n2 - 60
    _same(idx.search(xq, k), single.search(xq, k), "after removal")
    # a second round of adds after the removals
    a, b = n1 + n2, n1 + n2 + 50
    lo, hi = shard_range(b - a, world, rank)
    idx.add_with_ids_local(x[a + lo:a + hi], ids[a + lo:a + hi])
    single.add_with_ids(x[a:b], ids[a:b])
    assert _all_equal(idx.ntotal) == single.ntotal
    _same(idx.search(xq, k), single.search(xq, k), "re-added")
    p = nf.SearchParameters(sel=nf.IDSelectorRange(int(ids[n1 + n2 - 30]), I64_MAX))
    _same(idx.search(xq, k, params=p), single.search(xq, k, params=p), "re-added newest")


def _flat_plain_case(rank, world, metric, exchange, nf):
    from newsrecommend_b200.sharded import ShardedIndexFlat, shard_range
    rng = np.random.default_rng(20 + metric)
    d, k, nb = 16, 10, 401
    x = rng.standard_normal((nb, d), dtype=np.float32)
    xq = rng.standard_normal((37, d), dtype=np.float32)
    idx = ShardedIndexFlat(d, metric, make_index=OFlat, make_idmap=OIDMap, codec=NumpyIdCodec, exchange=exchange,
                           chunk_queries=16)
    idx.add_global(x)
    single = OFlat(d, metric)
    single.add(x)
    assert not idx.with_ids
    with pytest.raises(RuntimeError, match="carries no ids"):
        idx.add_with_ids(x, np.arange(nb))
    with pytest.raises(RuntimeError, match="carries no ids"):
        idx.add_with_ids_local(x[:2], np.arange(2))
    pos = np.arange(nb, dtype=np.int64)
    for name, sel in _selectors(nf, pos, pos[slice(*shard_range(nb, world, 1))][3:9]):
        p = nf.SearchParameters(sel=sel)
        _same(idx.search(xq, k, params=p), single.search(xq, k, params=p), "plain " + name)
    for sel in (nf.IDSelectorRange(150, 260), nf.IDSelectorNot(nf.IDSelectorRange(-5, 330)),
                np.array([0, 3, 3, 199, 200, 10_000], dtype=np.int64)):
        r = idx.remove_ids(sel)
        assert _all_equal(r) == single.remove_ids(sel)
        assert _all_equal(idx.ntotal) == single.ntotal
        # positions renumbered: every shard's first global position is the rows before it
        counts = torch.tensor([idx.local.ntotal], dtype=torch.int64)
        allc = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(allc, counts)
        assert idx.id_base == sum(int(c) for c in allc[:rank]) and idx._bases_host[rank] == idx.id_base
        _same(idx.search(xq, k), single.search(xq, k), "plain after removal")
        p = nf.SearchParameters(sel=nf.IDSelectorRange(100, 180))
        _same(idx.search(xq, k, params=p), single.search(xq, k, params=p), "plain window after removal")


def _ivf_case(rank, world, metric, exchange, nf):
    from newsrecommend_b200.sharded import ShardedIndexIVFFlat, shard_range
    rng = np.random.default_rng(30 + metric)
    d, nlist, k, n1, n2 = 16, 4, 10, 400, 201
    topics = rng.standard_normal((6, d)).astype(np.float32) * 3
    x = (topics[rng.integers(0, 6, n1 + n2)] + rng.standard_normal((n1 + n2, d))).astype(np.float32)
    xq = (topics[rng.integers(0, 6, 37)] + rng.standard_normal((37, d))).astype(np.float32)
    ids = rng.permutation(1 << 20)[: n1 + n2].astype(np.int64) * 4099 + (1 << 32)
    idx = ShardedIndexIVFFlat(d, nlist, metric, make_index=fo.IndexFlat, make_ivf=OIVF, codec=NumpyIdCodec,
                              exchange=exchange, chunk_queries=16)
    idx.train_global(x)
    q2 = fo.IndexFlat(d, metric)
    q2.add(np.array(idx.quantizer.xb, copy=True))
    single = OIVF(q2, d, nlist, metric)
    single.train(x)
    plain = ShardedIndexIVFFlat(d, nlist, metric, make_index=fo.IndexFlat, make_ivf=OIVF, codec=NumpyIdCodec,
                                exchange=exchange, chunk_queries=16)
    plain.train_global(x)
    q3 = fo.IndexFlat(d, metric)
    q3.add(np.array(idx.quantizer.xb, copy=True))
    single_plain = OIVF(q3, d, nlist, metric)
    single_plain.train(x)
    plain.add_global(x)
    single_plain.add(x)
    owned1 = []
    for a, b in ((0, n1), (n1, n1 + n2)):
        lo, hi = shard_range(b - a, world, rank)
        idx.add_with_ids_local(x[a + lo:a + hi], ids[a + lo:a + hi])
        single.add_with_ids(x[a:b], ids[a:b])
        owned1.append(ids[a:b][slice(*shard_range(b - a, world, 1))][:4])
    assert _all_equal(idx.ntotal) == n1 + n2
    with pytest.raises(RuntimeError, match="incorrect type"):
        idx.search(xq, k, params=nf.SearchParameters(sel=nf.IDSelectorRange(0, 10)))
    with pytest.raises(RuntimeError, match="add_with_ids"):
        idx.add_global(x)
    with pytest.raises(RuntimeError, match="carries no ids"):
        plain.add_with_ids_local(x[:2], ids[:2])
    for nprobe in (1, 3):
        idx.nprobe = single.nprobe = plain.nprobe = single_plain.nprobe = nprobe
        _same(idx.search(xq, k), single.search(xq, k), ("ivf", nprobe))
        for name, sel in _selectors(nf, ids, np.concatenate(owned1)):
            p = nf.SearchParametersIVF(sel=sel)
            _same(idx.search(xq, k, params=p), single.search(xq, k, params=p), ("ivf", nprobe, name))
        pos = np.arange(n1 + n2, dtype=np.int64)
        for name, sel in _selectors(nf, pos, pos[slice(*shard_range(n1 + n2, world, 1))][2:9]):
            p = nf.SearchParametersIVF(sel=sel)
            _same(plain.search(xq, k, params=p), single_plain.search(xq, k, params=p), ("plain ivf", nprobe, name))
    # SearchParametersIVF.nprobe overrides index.nprobe for the call
    idx.nprobe = single.nprobe = 1
    p = nf.SearchParametersIVF(nprobe=nlist)
    xr = rng.standard_normal((23, d)).astype(np.float32) * 3  # between the topics: one list is not enough
    ex = single.search(xr, k, params=p)
    _same(idx.search(xr, k, params=p), ex, "nprobe override")
    assert not np.array_equal(ex[1], single.search(xr, k)[1])
    p = nf.SearchParametersIVF(sel=nf.IDSelectorRange(int(np.sort(ids)[300]), I64_MAX), nprobe=3)
    _same(idx.search(xq, k, params=p), single.search(xq, k, params=p), "nprobe + window")
    for sel in (nf.IDSelectorRange(int(np.sort(ids)[20]), int(np.sort(ids)[90])), nf.IDSelectorBatch(ids[::11].copy()),
                nf.IDSelectorNot(nf.IDSelectorRange(I64_MIN, int(np.sort(ids)[-10]))), ids[5:60:3].copy()):
        assert _all_equal(idx.remove_ids(sel)) == single.remove_ids(sel)
        assert _all_equal(idx.ntotal) == single.ntotal
    idx.nprobe = single.nprobe = 2
    _same(idx.search(xq, k), single.search(xq, k), "ivf after removal")
    # plain IVF: stored ids are global positions, and survivors keep them
    for sel in (nf.IDSelectorRange(100, 300), nf.IDSelectorNot(nf.IDSelectorRange(0, 550)), np.arange(0, 40, 3)):
        assert _all_equal(plain.remove_ids(sel)) == single_plain.remove_ids(sel)
    plain.nprobe = single_plain.nprobe = 2
    _same(plain.search(xq, k), single_plain.search(xq, k), "plain ivf after removal")
    p = nf.SearchParametersIVF(sel=nf.IDSelectorRange(250, 500))
    _same(plain.search(xq, k, params=p), single_plain.search(xq, k, params=p), "plain ivf window after removal")


def _empty_shard_case(rank, world, metric, exchange, nf):
    """nb = 1: rank 0's shard is empty."""
    from newsrecommend_b200.sharded import ShardedIndexFlat
    rng = np.random.default_rng(40)
    x = rng.standard_normal((1, 8), dtype=np.float32)
    xq = rng.standard_normal((5, 8), dtype=np.float32)
    idx = ShardedIndexFlat(8, metric, make_index=OFlat, make_idmap=OIDMap, codec=NumpyIdCodec, exchange=exchange)
    idx.add_with_ids(x, np.array([(1 << 40) + 7], dtype=np.int64))
    single = OIDMap(OFlat(8, metric))
    single.add_with_ids(x, np.array([(1 << 40) + 7], dtype=np.int64))
    assert idx.local.ntotal == rank and _all_equal(idx.ntotal) == 1
    _same(idx.search(xq, 4), single.search(xq, 4), "empty shard")
    p = nf.SearchParameters(sel=nf.IDSelectorNot(nf.IDSelectorBatch(np.array([(1 << 40) + 7]))))
    _same(idx.search(xq, 4, params=p), single.search(xq, 4, params=p), "empty shard, nothing selected")
    assert _all_equal(idx.remove_ids(np.array([(1 << 40) + 7]))) == 1 and _all_equal(idx.ntotal) == 0


def _worker(rank, world, port, metric, exchange, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import newsrecommend_b200.faiss as nf
        fo.build()
        _flat_ids_case(rank, world, metric, exchange, "global", nf)
        _flat_ids_case(rank, world, metric, exchange, "local", nf)
        _flat_plain_case(rank, world, metric, exchange, nf)
        _ivf_case(rank, world, metric, exchange, nf)
        _empty_shard_case(rank, world, metric, exchange, nf)
        out.put((rank, True))
    except Exception as e:  # noqa: BLE001
        import traceback
        out.put((rank, repr(e) + traceback.format_exc()[-1500:]))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("metric,exchange", [(0, "alltoall"), (1, "alltoall"), (0, "allgather"), (1, "allgather")])
def test_sharded_ids_world2_gloo(metric, exchange):
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, metric, exchange, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
    res = sorted(out.get(timeout=5) for _ in range(2))
    assert res == [(0, True), (1, True)], res


def test_numpy_id_codec_roundtrip():
    """The 16-byte words keep every int64 id (also >= 2^32 and negative padding) and the fp32 bits."""
    D = torch.tensor([[3.5, -1.0, 0.0]], dtype=torch.float32)
    I = torch.tensor([[(1 << 40) + 3, -5, -1]], dtype=torch.int64)
    P = NumpyIdCodec.pack_ids(D, I)
    assert P.shape == (1, 3, 2) and P[0, 0, 1] == (1 << 40) + 3
    assert (P[0, :, 0].numpy().view(np.uint64) & np.uint64(0xFFFFFFFF)).tolist() == [0, 0xFFFFFFFF, 0xFFFFFFFF]
    Dm, Im = NumpyIdCodec.merge_ids(P.unsqueeze(0), 0)
    assert Im.tolist() == [[(1 << 40) + 3, -1, -1]] and Dm[0, 0] == 3.5


def test_shift_selector():
    import newsrecommend_b200.faiss as nf
    from newsrecommend_b200.sharded import shift_selector
    r = shift_selector(nf.IDSelectorRange(10, 20), 15)
    assert (r.imin, r.imax) == (-5, 5)
    r = shift_selector(nf.IDSelectorRange(I64_MIN, I64_MAX), 100)
    assert (r.imin, r.imax) == (I64_MIN, I64_MAX - 100)
    b = shift_selector(nf.IDSelectorBatch(np.array([3, 100, 107, I64_MIN])), 100)
    assert b.ids.tolist() == [0, 7]
    n = shift_selector(nf.IDSelectorNot(nf.IDSelectorNot(nf.IDSelectorBatch(np.array([5])))), 2)
    assert isinstance(n.sel.sel, nf.IDSelectorBatch) and n.sel.sel.ids.tolist() == [3]
    with pytest.raises(TypeError):
        shift_selector("0-5", 0)


def test_sharded_id_entry_point_argument_checks():
    from newsrecommend_b200 import _lib
    L = _lib.lib
    D = np.zeros(6, dtype=np.float32)
    I = np.zeros(6, dtype=np.int64)
    P = np.zeros(12, dtype=np.uint64)
    d, i, p = D.ctypes.data, I.ctypes.data, P.ctypes.data
    assert L.nrb_pack_topk_ids(d, i, -1, p, None) == -1
    assert L.nrb_pack_topk_ids(None, i, 6, p, None) == -1
    assert L.nrb_pack_topk_ids(d, i, 6, None, None) == -1
    assert L.nrb_pack_topk_ids(None, None, 0, None, None) == 0
    for nparts, nq, k in ((0, 2, 3), (257, 2, 3), (2, -1, 3), (2, 2, 0), (2, 2, 129)):
        assert L.nrb_merge_topk_packed_ids(p, nparts, nq, k, 0, d, i, None) == -1, (nparts, nq, k)
    assert L.nrb_merge_topk_packed_ids(p, 256, 0, 128, 1, d, i, None) == 0
    assert L.nrb_merge_topk_packed_ids(None, 2, 1, 3, 0, d, i, None) == -1
    assert L.nrb_merge_topk_packed_ids(p, 2, 1, 3, 0, None, i, None) == -1
    assert L.nrb_merge_topk_packed_ids(p, 2, 1, 3, 0, d, None, None) == -1
    assert "merge_topk_packed_ids" in _lib.last_error()
    for name in ("nrb_pack_topk_ids", "nrb_merge_topk_packed_ids"):
        assert name in _lib.SYMBOLS and hasattr(L, name)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_sharded_id_entry_points_need_a_device():
    from newsrecommend_b200 import _lib
    L = _lib.lib
    D = np.zeros(6, dtype=np.float32)
    I = np.zeros(6, dtype=np.int64)
    P = np.zeros(12, dtype=np.uint64)
    assert L.nrb_pack_topk_ids(D.ctypes.data, I.ctypes.data, 6, P.ctypes.data, None) == -3
    assert L.nrb_merge_topk_packed_ids(P.ctypes.data, 2, 1, 3, 0, D.ctypes.data, I.ctypes.data, None) == -3
    assert "no CPU fallback" in _lib.last_error()


def test_refused_arguments_without_a_group():
    """Checks that raise before any collective, on a one-rank index with no process group."""
    import newsrecommend_b200.faiss as nf
    from newsrecommend_b200.sharded import ShardedIndexFlat, ShardedIndexIVFFlat
    idx = ShardedIndexFlat(4, 1, make_index=OFlat, make_idmap=OIDMap, codec=NumpyIdCodec)
    with pytest.raises(TypeError):
        idx.remove_ids("1, 2")
    with pytest.raises(TypeError, match="ids for"):
        idx.add_with_ids(np.zeros((3, 4), np.float32), np.arange(2, dtype=np.int64))
    ivf = ShardedIndexIVFFlat(4, 2, 1, make_index=fo.IndexFlat, make_ivf=OIVF, codec=NumpyIdCodec)
    with pytest.raises(RuntimeError, match="incorrect type"):
        ivf.search(np.zeros((1, 4), np.float32), 1, params=nf.SearchParameters())
    with pytest.raises(RuntimeError, match="is_trained"):
        ivf.add_with_ids_local(np.zeros((3, 4), np.float32), np.arange(3, dtype=np.int64))
