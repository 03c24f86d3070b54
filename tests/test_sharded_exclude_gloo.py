"""world_size-2 gloo tests (CPU) of per-query exclusion lists on the sharded indexes:
search(..., exclude=(offsets, ids)) with both exchange forms and 16-query chunks (lists cross chunk
boundaries), gathered and per-rank results, on plain and id-carrying ShardedIndexFlat and
ShardedIndexIVFFlat. The rank-local indexes are the oracle's, wrapped so that they take params and
exclude (tests/exclude_oracle.py); the localization is a numpy restatement of nrb_id_select +
nrb_csr_compact. Every answer is compared with the single oracle index of the same kind holding the
same rows, ids and removals, searched with the same lists and params."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import exclude_oracle as xo
from oracle import faiss_oracle as fo
from test_sharded_gloo import _free_port
from test_sharded_ids_gloo import I64_MAX, NumpyIdCodec, OFlat, OIDMap, OIVF, _all_equal, _same

FLT_MAX = np.float32(3.4028235e38)


def csr_compact(off, ids, member, shift):
    """numpy restatement of nrb_csr_compact: entry i of every row is kept when member[i] == 1 and
    written as ids[i] - shift, in order. Returns (offsets, ids) int64."""
    off = np.asarray(off, dtype=np.int64)
    keep = np.asarray(member) == 1
    before = np.zeros(keep.size + 1, dtype=np.int64)  # kept entries before position i
    np.cumsum(keep, out=before[1:])
    return before[off], (np.asarray(ids, dtype=np.int64)[keep] - np.int64(shift)).astype(np.int64)


def localize_numpy(ex, held, shift):
    """GpuCodec.localize restated: membership (a label range, or the stored ids), then csr_compact."""
    off_h, _, ids = ex
    ids = ids.cpu().numpy() if isinstance(ids, torch.Tensor) else np.asarray(ids)
    if isinstance(held, tuple):
        member = (ids >= held[0]) & (ids < held[1])
    else:
        stored = np.empty(0, np.int64) if held is None else (
            held.cpu().numpy() if isinstance(held, torch.Tensor) else np.asarray(held))
        member = np.isin(ids, stored)
    return csr_compact(off_h, ids, member.astype(np.int64), shift)


class NumpyExcludeCodec(NumpyIdCodec):
    @staticmethod
    def localize(ex, held, shift, dev):
        return localize_numpy(ex, held, shift)


def _excluded(cls, index, x, k, params, exclude):
    """cls.search of an oracle wrapper, with per-query exclusion lists restated by exclude_oracle."""
    if exclude is None:
        return cls.search(index, x, k, params)
    off, ids = (np.asarray(a) for a in exclude)
    return xo.search_excluded(lambda xs, kq: cls.search(index, xs, kq, params), np.asarray(x), k, off, ids,
                              index.metric_type)


class XFlat(OFlat):
    def search(self, x, k, params=None, exclude=None):
        return _excluded(OFlat, self, x, k, params, exclude)


class XIDMap(OIDMap):
    @property
    def metric_type(self):
        return self.index.metric_type

    def search(self, x, k, params=None, exclude=None):
        return _excluded(OIDMap, self, x, k, params, exclude)


class XIVF(OIVF):
    @property
    def _ids(self):
        """The stored ids, as IndexIVFFlat keeps them (order does not matter to membership)."""
        chunks = [c[0] for lst in self._lists for c in lst]
        return np.concatenate(chunks) if chunks else np.empty(0, np.int64)

    def search(self, x, k, params=None, exclude=None):
        return _excluded(OIVF, self, x, k, params, exclude)


def make_lists(rng, nq, k, labels, top, shard0, shard1, absent):
    """nq exclusion lists that cover the cases, cycling by query: the query's own plain top hits with
    random labels of both shards; labels of one shard only; empty; -1, duplicates and absent ids; a
    list longer than 128 - k held by shard 1 alone (the long group there); every label of shard 0."""
    lists = []
    for q in range(nq):
        c = q % 6
        if c == 0:
            lst = np.concatenate([top[q, :4], rng.choice(labels, int(rng.integers(0, 9)))])
        elif c == 1:
            lst = np.concatenate([top[q, :2][np.isin(top[q, :2], shard1)], rng.choice(shard1, 6)])
        elif c == 2:
            lst = []
        elif c == 3:
            lst = np.concatenate([[-1], top[q, :3], top[q, :2], absent[:3], [-1]])
        elif c == 4:
            lst = np.resize(shard1, 129 - k + 3)
        else:
            lst = shard0
        lists.append(rng.permutation(np.asarray(lst, dtype=np.int64)))
    return xo.csr(lists)


def _check_excluded(idx, single, xq, k, ex, params, what):
    """The sharded search (gathered and per-rank) against the single index with the same lists."""
    D, I = idx.search(xq, k, params=params, exclude=ex)
    _same((D, I), single.search(xq, k, params, ex), what)
    off, ids = ex
    for q in range(xq.shape[0]):
        got = I.numpy()[q]
        lst = ids[off[q]:off[q + 1]]
        assert not np.isin(got[got >= 0], lst[lst >= 0]).any(), (what, q)
    Dr, Ir, spans = idx.search(xq, k, gather=False, params=params, exclude=ex)
    rows = np.concatenate([np.arange(a, b) for a, b in spans])
    assert np.array_equal(Ir.numpy(), I.numpy()[rows]) and np.array_equal(Dr.numpy(), D.numpy()[rows]), what
    return D, I


def _lists_for(rng, single, xq, k, labels, shard0, shard1):
    top = single.search(xq, 4)[1]
    absent = np.array([labels.max() + 11, labels.max() + 12, -5], dtype=np.int64)
    return make_lists(rng, xq.shape[0], k, labels, top, shard0, shard1, absent)


def _flat_case(rank, world, metric, exchange, form, nf):
    """form: "plain" (add_global, labels are global row positions), "global" / "local" (add_with_ids /
    add_with_ids_local, labels are external ids)."""
    from newsrecommend_b200.sharded import ShardedIndexFlat, shard_range
    rng = np.random.default_rng(50 + metric)
    d, k, nb = 16, 10, 401
    x = rng.standard_normal((nb, d), dtype=np.float32)
    xq = rng.standard_normal((37, d), dtype=np.float32)
    idx = ShardedIndexFlat(d, metric, make_index=XFlat, make_idmap=XIDMap, codec=NumpyExcludeCodec, exchange=exchange,
                           chunk_queries=16)
    lo, hi = shard_range(nb, world, rank)
    if form == "plain":
        labels = np.arange(nb, dtype=np.int64)
        idx.add_global(x)
        single = XFlat(d, metric)
        single.add(x)
    else:
        labels = (np.sort(rng.choice(1 << 40, nb, replace=False)) + (1 << 33)).astype(np.int64)
        if form == "global":
            idx.add_with_ids(x, labels)
        else:
            idx.add_with_ids_local(x[lo:hi], labels[lo:hi])
        single = XIDMap(XFlat(d, metric))
        single.add_with_ids(x, labels)
    shard0, shard1 = labels[slice(*shard_range(nb, world, 0))], labels[slice(*shard_range(nb, world, 1))]
    ex = _lists_for(rng, single, xq, k, labels, shard0, shard1)
    D, I = _check_excluded(idx, single, xq, k, ex, None, (form, "lists"))
    assert not np.array_equal(I.numpy(), single.search(xq, k)[1])  # the lists hit the plain top k
    # the rows of shard 0 excluded: those queries draw from shard 1 only
    assert np.isin(I.numpy()[5::6], shard1).all()
    empty = (np.zeros(xq.shape[0] + 1, dtype=np.int64), np.empty(0, np.int64))
    D0, I0 = _check_excluded(idx, single, xq, k, empty, None, (form, "all empty"))
    _same((D0, I0), single.search(xq, k), (form, "all empty = no exclude"))
    s = np.sort(labels)
    window = nf.SearchParameters(sel=nf.IDSelectorRange(int(s[int(0.6 * nb)]), I64_MAX))
    block = nf.SearchParameters(sel=nf.IDSelectorNot(nf.IDSelectorBatch(labels[::7].copy())))
    for name, p in (("window", window), ("blocklist", block)):
        _check_excluded(idx, single, xq, k, ex, p, (form, name))
    # removals: plain positions renumber, ids stay
    for sel in (nf.IDSelectorRange(int(s[150]), int(s[260])), labels[[0, 3, 199, 200, 390]].copy()):
        assert _all_equal(idx.remove_ids(sel)) == single.remove_ids(sel)
    n = single.ntotal
    if form == "plain":
        labels = np.arange(n, dtype=np.int64)
        cut = idx._bases_host[1]
        shard0, shard1 = labels[:cut], labels[cut:]
    else:
        keep = np.isin(labels, single.id_map)
        shard0, shard1 = shard0[np.isin(shard0, labels[keep])], shard1[np.isin(shard1, labels[keep])]
        labels = labels[keep]
    ex = _lists_for(rng, single, xq, k, labels, shard0, shard1)
    _check_excluded(idx, single, xq, k, ex, None, (form, "after removal"))
    _check_excluded(idx, single, xq, k, ex, window, (form, "window after removal"))


def _ivf_case(rank, world, metric, exchange, with_ids, nf):
    from newsrecommend_b200.sharded import ShardedIndexIVFFlat, shard_range
    rng = np.random.default_rng(60 + metric)
    d, nlist, k, nb = 16, 4, 10, 601
    topics = rng.standard_normal((6, d)).astype(np.float32) * 3
    x = (topics[rng.integers(0, 6, nb)] + rng.standard_normal((nb, d))).astype(np.float32)
    xq = (topics[rng.integers(0, 6, 37)] + rng.standard_normal((37, d))).astype(np.float32)
    labels = rng.permutation(1 << 20)[:nb].astype(np.int64) * 4099 + (1 << 32) if with_ids else \
        np.arange(nb, dtype=np.int64)
    idx = ShardedIndexIVFFlat(d, nlist, metric, make_index=fo.IndexFlat, make_ivf=XIVF, codec=NumpyExcludeCodec,
                              exchange=exchange, chunk_queries=16)
    idx.train_global(x)
    q = fo.IndexFlat(d, metric)
    q.add(np.array(idx.quantizer.xb, copy=True))
    single = XIVF(q, d, nlist, metric)
    single.train(x)
    if with_ids:
        lo, hi = shard_range(nb, world, rank)
        idx.add_with_ids_local(x[lo:hi], labels[lo:hi])
        single.add_with_ids(x, labels)
    else:
        idx.add_global(x)
        single.add(x)
    shard0, shard1 = labels[slice(*shard_range(nb, world, 0))], labels[slice(*shard_range(nb, world, 1))]
    idx.nprobe = single.nprobe = 2
    ex = _lists_for(rng, single, xq, k, labels, shard0, shard1)
    what = "ivf ids" if with_ids else "ivf plain"
    _check_excluded(idx, single, xq, k, ex, None, (what, "lists"))
    s = np.sort(labels)
    for name, p in (("nprobe", nf.SearchParametersIVF(nprobe=3)),
                    ("window", nf.SearchParametersIVF(sel=nf.IDSelectorRange(int(s[nb // 2]), I64_MAX), nprobe=3)),
                    ("blocklist", nf.SearchParametersIVF(sel=nf.IDSelectorNot(nf.IDSelectorBatch(labels[::5].copy()))))):
        _check_excluded(idx, single, xq, k, ex, p, (what, name))
    for sel in (nf.IDSelectorRange(int(s[100]), int(s[300])), labels[5:60:3].copy()):
        assert _all_equal(idx.remove_ids(sel)) == single.remove_ids(sel)
    _check_excluded(idx, single, xq, k, ex, None, (what, "after removal"))  # removed labels match nothing
    empty = (np.zeros(xq.shape[0] + 1, dtype=np.int64), np.empty(0, np.int64))
    _same(_check_excluded(idx, single, xq, k, empty, None, (what, "all empty")), single.search(xq, k), what)


def _empty_shard_case(rank, world, metric, exchange, nf):
    """nb = 1: rank 0's shard is empty; its lists localize to nothing."""
    from newsrecommend_b200.sharded import ShardedIndexFlat
    rng = np.random.default_rng(70)
    x = rng.standard_normal((1, 8), dtype=np.float32)
    xq = rng.standard_normal((5, 8), dtype=np.float32)
    one = np.array([(1 << 40) + 7], dtype=np.int64)
    idx = ShardedIndexFlat(8, metric, make_index=XFlat, make_idmap=XIDMap, codec=NumpyExcludeCodec, exchange=exchange)
    idx.add_with_ids(x, one)
    single = XIDMap(XFlat(8, metric))
    single.add_with_ids(x, one)
    assert idx.local.ntotal == rank
    ex = xo.csr([[], one, [-1, 3], one, [one[0], one[0]]])
    D, I = _check_excluded(idx, single, xq, 4, ex, None, "empty shard")
    assert (I.numpy()[[1, 3, 4]] == -1).all() and (I.numpy()[[0, 2], 0] == one[0]).all()
    pad = FLT_MAX if metric else -FLT_MAX
    assert (D.numpy()[1] == pad).all()


def _malformed_case(rank, world, metric, exchange, nf):
    """Bad lists raise the same error on every rank before any collective; the group stays usable."""
    from newsrecommend_b200.sharded import ShardedIndexFlat
    rng = np.random.default_rng(80)
    x = rng.standard_normal((50, 8), dtype=np.float32)
    xq = rng.standard_normal((3, 8), dtype=np.float32)
    idx = ShardedIndexFlat(8, metric, make_index=XFlat, make_idmap=XIDMap, codec=NumpyExcludeCodec, exchange=exchange)
    idx.add_global(x)
    single = XFlat(8, metric)
    single.add(x)
    off, ids = xo.csr([[1], [2, 30], []])
    bad = [(TypeError, (off, ids.astype(np.int32))), (TypeError, (off,)), (TypeError, [off, ids.tolist()]),
           (ValueError, (off[:-1], ids)), (ValueError, (np.array([0, 2, 1, 3]), ids)),
           (ValueError, (off + 1, ids)), (ValueError, (off, ids.reshape(1, -1)))]
    for err, ex in bad:
        with pytest.raises(err):
            idx.search(xq, 4, exclude=ex)
        with pytest.raises(err):
            idx.search(xq, 4, gather=False, exclude=ex)
    _check_excluded(idx, single, xq, 4, (off, ids), None, "after the refused lists")


def _worker(rank, world, port, metric, exchange, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import newsrecommend_b200.faiss as nf
        fo.build()
        for form in ("plain", "global", "local"):
            _flat_case(rank, world, metric, exchange, form, nf)
        _ivf_case(rank, world, metric, exchange, False, nf)
        _ivf_case(rank, world, metric, exchange, True, nf)
        _empty_shard_case(rank, world, metric, exchange, nf)
        _malformed_case(rank, world, metric, exchange, nf)
        out.put((rank, True))
    except Exception as e:  # noqa: BLE001
        import traceback
        out.put((rank, repr(e) + traceback.format_exc()[-1500:]))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("metric,exchange", [(0, "alltoall"), (1, "alltoall"), (0, "allgather"), (1, "allgather")])
def test_sharded_exclude_world2_gloo(metric, exchange):
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


def _compact_brute(off, ids, member, shift):
    lists = [[int(ids[i]) - shift for i in range(off[r], off[r + 1]) if member[i] == 1] for r in range(len(off) - 1)]
    return xo.csr(lists)


@pytest.mark.parametrize("case", ["random", "empty_rows", "all_kept", "none_kept", "no_rows", "big_ids"])
def test_csr_compact_restatement_matches_brute_force(case):
    rng = np.random.default_rng(hash(case) % 1000)
    lens = rng.integers(0, 70, 300)
    if case == "empty_rows":
        lens[rng.random(300) < 0.7] = 0
    if case == "no_rows":
        lens = lens[:0]
    off = np.zeros(lens.size + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    ids = rng.integers(-1, 1000, off[-1], dtype=np.int64)
    if case == "big_ids":
        ids = ids + (1 << 40)
    member = {"all_kept": np.ones(ids.size), "none_kept": np.zeros(ids.size)}.get(case, rng.integers(0, 2, ids.size))
    member = member.astype(np.int64)
    shift = (1 << 35) if case == "big_ids" else 17
    o, i = csr_compact(off, ids, member, shift)
    ob, ib = _compact_brute(off, ids, member, shift)
    assert np.array_equal(o, ob) and np.array_equal(i, ib)
    assert o.dtype == np.int64 and i.dtype == np.int64


def test_localize_restatement():
    """Range membership (plain indexes) shifts into the shard's positions; id membership keeps ids."""
    off, ids = xo.csr([[5, 12, -1, 9, 12], [], [100, 11]])
    ex = (off, off, ids)
    o, i = localize_numpy(ex, (9, 13), 9)
    assert o.tolist() == [0, 3, 3, 4] and i.tolist() == [3, 0, 3, 2]
    o, i = localize_numpy(ex, np.array([100, 12], dtype=np.int64), 0)
    assert o.tolist() == [0, 2, 2, 3] and i.tolist() == [12, 12, 100]
    o, i = localize_numpy(ex, None, 0)
    assert o.tolist() == [0, 0, 0, 0] and i.size == 0


def test_chunk_lists():
    from newsrecommend_b200.sharded import chunk_lists
    off, ids = xo.csr([[1, 2], [], [3], [4, 5, 6]])
    o, i = chunk_lists((off, ids), 1, 4)
    assert o.tolist() == [0, 0, 1, 4] and i.tolist() == [3, 4, 5, 6]
    o, i = chunk_lists((off, ids), 1, 2)
    assert o.tolist() == [0, 0] and i.size == 0


def test_csr_compact_entry_point_argument_checks():
    from newsrecommend_b200 import _lib
    L = _lib.lib
    off = np.array([0, 2, 3], dtype=np.int64)
    ids = np.array([4, 5, 6], dtype=np.int64)
    mem = np.ones(3, dtype=np.int64)
    oo = np.zeros(3, dtype=np.int64)
    oi = np.zeros(3, dtype=np.int64)
    ws = np.zeros(64, dtype=np.uint8)
    o, i, m, a, b, w = off.ctypes.data, ids.ctypes.data, mem.ctypes.data, oo.ctypes.data, oi.ctypes.data, ws.ctypes.data
    assert L.nrb_csr_compact_workspace(0) == 0
    assert L.nrb_csr_compact_workspace(1) == 8 and L.nrb_csr_compact_workspace(257) == 16
    assert L.nrb_csr_compact(o, i, -1, 3, m, 0, a, b, w, 64, None) == -1
    assert L.nrb_csr_compact(o, i, 2, -1, m, 0, a, b, w, 64, None) == -1
    assert L.nrb_csr_compact(None, i, 2, 3, m, 0, a, b, w, 64, None) == -1
    assert L.nrb_csr_compact(o, i, 2, 3, m, 0, None, b, w, 64, None) == -1
    for args in ((None, m, b), (i, None, b), (i, m, None)):
        assert L.nrb_csr_compact(o, args[0], 2, 3, args[1], 0, a, args[2], w, 64, None) == -1
    assert "csr_compact" in _lib.last_error()
    assert L.nrb_csr_compact(o, i, 2, 3, m, 0, a, b, w, 4, None) == -4  # workspace too small
    assert L.nrb_csr_compact(o, i, 2, 3, m, 0, a, b, None, 64, None) == -4
    for name in ("nrb_csr_compact_workspace", "nrb_csr_compact"):
        assert name in _lib.SYMBOLS and hasattr(L, name)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_csr_compact_needs_a_device():
    from newsrecommend_b200 import _lib
    L = _lib.lib
    off = np.array([0, 0], dtype=np.int64)
    oo = np.zeros(2, dtype=np.int64)
    ws = np.zeros(8, dtype=np.uint8)
    assert L.nrb_csr_compact(off.ctypes.data, None, 1, 0, None, 0, oo.ctypes.data, None, ws.ctypes.data, 8, None) == -3
    assert L.nrb_csr_compact(off.ctypes.data, None, 0, 0, None, 0, oo.ctypes.data, None, None, 0, None) == -3
    assert "no CPU fallback" in _lib.last_error()


def test_refused_lists_without_a_group():
    """A one-rank index with no process group checks the lists before anything else."""
    from newsrecommend_b200.sharded import ShardedIndexFlat, ShardedIndexIVFFlat
    idx = ShardedIndexFlat(4, 1, make_index=XFlat, make_idmap=XIDMap, codec=NumpyExcludeCodec)
    idx.add_global(np.zeros((3, 4), np.float32))
    with pytest.raises(ValueError, match="nq \\+ 1"):
        idx.search(np.zeros((2, 4), np.float32), 1, exclude=(np.zeros(2, np.int64), np.empty(0, np.int64)))
    ivf = ShardedIndexIVFFlat(4, 2, 1, make_index=fo.IndexFlat, make_ivf=XIVF, codec=NumpyExcludeCodec)
    with pytest.raises(TypeError, match="pair"):
        ivf.search(np.zeros((1, 4), np.float32), 1, exclude=np.zeros(2, np.int64))
