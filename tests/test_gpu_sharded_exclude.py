"""GPU tests of per-query exclusion lists on the sharded indexes: nrb_csr_compact against its numpy
restatement, the localization (nrb_id_select + nrb_csr_compact) against numpy, G = 2, 4, 8 virtual
shards in one process (localize, per-shard excluded search, pack, exchange by hand, merge) against
the single-GPU index with the same lists and the oracle, and the NCCL path under torchrun
(tests/sharded_exclude_nccl_worker.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _compact_gpu(off, ids, member, shift):
    import torch
    from newsrecommend_b200 import _lib
    nq, n = off.size - 1, ids.size
    off_d, ids_d, mem_d = (torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).cuda() for a in (off, ids, member))
    out_off = torch.full((nq + 1,), -7, dtype=torch.int64, device="cuda")
    out_ids = torch.full((max(n, 1),), -7, dtype=torch.int64, device="cuda")
    wsb = _lib.lib.nrb_csr_compact_workspace(nq)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib.nrb_csr_compact(off_d.data_ptr(), ids_d.data_ptr() if n else None, nq, n,
                                        mem_d.data_ptr() if n else None, shift, out_off.data_ptr(),
                                        out_ids.data_ptr() if n else None, ws.data_ptr(), wsb,
                                        torch.cuda.current_stream().cuda_stream), "csr_compact")
    o = out_off.cpu().numpy()
    return o, out_ids[: int(o[-1])].cpu().numpy()


@pytest.mark.parametrize("case", ["random", "empty_rows", "all_kept", "none_kept", "no_rows", "big_ids",
                                  "rows_250k", "rows_300k"])
def test_csr_compact_kernel_matches_numpy(nf, case):
    """Bit for bit against the restatement. 300k rows take two tiles of the block-sum scan."""
    from test_sharded_exclude_gloo import csr_compact
    rng = np.random.default_rng(len(case))
    nrows = {"rows_250k": 250_000, "rows_300k": 300_001, "no_rows": 0}.get(case, 3_000)
    lens = rng.integers(0, 70, nrows) if nrows < 100_000 else rng.geometric(0.15, nrows) - 1
    if case == "empty_rows":
        lens[rng.random(nrows) < 0.8] = 0
        lens[:300] = 0  # whole blocks of empty rows
    off = np.zeros(nrows + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    ids = rng.integers(-1, 1 << 20, int(off[-1]), dtype=np.int64)
    if case == "big_ids":
        ids = ids * 4099 + (1 << 40)
    member = {"all_kept": np.ones(ids.size), "none_kept": np.zeros(ids.size)}.get(case, rng.integers(0, 2, ids.size))
    member = member.astype(np.int64)
    member[np.nonzero(member == 0)[0][::5]] = 2  # only the value 1 keeps an entry
    shift = (1 << 36) if case == "big_ids" else 1_000
    o, i = _compact_gpu(off, ids, member, shift)
    on, i_n = csr_compact(off, ids, member, shift)
    assert np.array_equal(o, on) and np.array_equal(i, i_n)
    o2, i2 = _compact_gpu(off, ids, member, shift)
    assert np.array_equal(o, o2) and np.array_equal(i, i2)  # deterministic
    if case == "big_ids":
        assert (i >= (1 << 32)).any()


@pytest.mark.parametrize("form", ["range", "ids", "no_ids"])
def test_localize_matches_numpy(nf, form):
    import torch
    from newsrecommend_b200.sharded import GpuCodec
    from test_sharded_exclude_gloo import localize_numpy
    import exclude_oracle as xo
    rng = np.random.default_rng(5)
    stored = rng.choice(1 << 45, 20_000, replace=False).astype(np.int64) + (1 << 33)
    pool = np.concatenate([stored, stored[:50] + 1, [-1]])
    lists = [rng.choice(pool, int(rng.integers(0, 40))) for _ in range(2_001)]
    off, ids = xo.csr(lists)
    if form == "range":
        ids = ids % 30_000
        held, shift = (10_000, 20_000), 10_000
    else:
        held, shift = (torch.from_numpy(stored).cuda() if form == "ids" else None), 0
    for ex in ((off, off, ids), (off, torch.from_numpy(off).cuda(), torch.from_numpy(ids).cuda())):
        o, i = GpuCodec.localize(ex, held, shift, torch.device("cuda"))
        on, i_n = localize_numpy(ex, held.cpu().numpy() if isinstance(held, torch.Tensor) else held, shift)
        assert isinstance(o, np.ndarray) and i.is_cuda
        assert np.array_equal(o, on) and np.array_equal(i.cpu().numpy(), i_n)
    assert (form == "no_ids") == (o[-1] == 0)


class VirtualShards:
    """G shards of one catalog in one process, searched as ShardedIndex*.search(exchange="alltoall")
    does: localize the lists per shard, per-shard excluded search, pack, every rank's query range from
    every shard, merge. kind: flat (global row positions), idmap, ivf (stored global positions),
    ivf_ids."""

    def __init__(self, nf, kind, metric, xb, labels, G, single):
        from newsrecommend_b200.sharded import shard_range
        self.nf, self.kind, self.metric, self.G = nf, kind, metric, G
        self.with_ids = kind in ("idmap", "ivf_ids")
        d = xb.shape[1]
        self.shards, self.bases, self.pos_end = [], [], []
        for r in range(G):
            lo, hi = shard_range(xb.shape[0], G, r)
            if kind in ("flat", "idmap"):
                ix = nf.IndexFlat(d, metric)
                if kind == "idmap":
                    ix = nf.IndexIDMap(ix)
            else:
                q = nf.IndexFlat(d, metric)
                q.add(single.quantizer.reconstruct_n())
                ix = nf.IndexIVFFlat(q, d, single.nlist, metric)
                ix.train(xb[:1])
                ix.nprobe = single.nprobe
            if self.with_ids:
                ix.add_with_ids(xb[lo:hi], labels[lo:hi])
            else:
                ix.add(xb[lo:hi])
            self.shards.append(ix)
            self.bases.append(lo)
            self.pos_end.append(hi)

    def held(self, r):
        ix = self.shards[r]
        if self.kind == "idmap":
            return ix.id_map, 0
        if self.kind == "ivf_ids":
            return ix._ids, 0
        hi = self.bases[r] + ix.ntotal if self.kind == "flat" else self.pos_end[r]
        return (self.bases[r], hi), self.bases[r]

    def local_params(self, r, params):
        from newsrecommend_b200.sharded import shift_selector
        if params is None or params.sel is None or self.with_ids:
            return params
        sel = shift_selector(params.sel, self.bases[r])
        if self.kind == "flat":
            return self.nf.SearchParameters(sel=sel)
        return self.nf.SearchParametersIVF(sel=sel, nprobe=params.nprobe)

    def remove(self, labels):
        """Removes the rows with these labels from every shard (plain flat: positions renumber)."""
        from newsrecommend_b200.sharded import shift_selector
        n = 0
        for r, ix in enumerate(self.shards):
            sel = self.nf.IDSelectorBatch(labels)
            n += ix.remove_ids(sel if self.with_ids else shift_selector(sel, self.bases[r]))
        if self.kind == "flat":
            self.bases = [0] + np.cumsum([ix.ntotal for ix in self.shards])[:-1].tolist()
        return n

    def search(self, xq, k, params=None, ex=None, check_local=True):
        import torch
        from newsrecommend_b200.faiss import _exclude_arg
        from newsrecommend_b200.sharded import GpuCodec, chunk_lists, chunk_slices
        from test_sharded_exclude_gloo import localize_numpy
        nq, dev = xq.shape[0], xq.device
        lists, lists_np = [None] * self.G, [None] * self.G
        if ex is not None:
            exa = _exclude_arg(ex, nq)
            for r in range(self.G):
                held, shift = self.held(r)
                lists[r] = GpuCodec.localize(exa, held, shift, dev)
                lists_np[r] = localize_numpy(exa, held.cpu().numpy() if isinstance(held, torch.Tensor) else held,
                                             shift)
                assert np.array_equal(lists[r][0], lists_np[r][0])
                assert np.array_equal(lists[r][1].cpu().numpy(), lists_np[r][1])
        D = torch.empty((nq, k), dtype=torch.float32, device=dev)
        I = torch.empty((nq, k), dtype=torch.int64, device=dev)
        bases = torch.tensor(self.bases, dtype=torch.int64, device=dev)
        for c0, c1, per in chunk_slices(nq, self.G, 512):
            packed = []
            for r, ix in enumerate(self.shards):
                lp = self.local_params(r, params)
                if ex is None:
                    if self.kind == "flat" and lp is None:  # ShardedIndexFlat.search_local's fast path
                        q = self.nf.PackedMatrix.from_tensor(xq[c0:c1], planes=ix._query_planes(k))
                        Dl, Il = ix.search_packed(q, k, self.bases[r])
                    else:
                        Dl, Il = ix.search(xq[c0:c1], k, params=lp)
                else:
                    Dl, Il = ix.search(xq[c0:c1], k, params=lp, exclude=chunk_lists(lists[r], c0, c1))
                    if check_local:  # the same shard given the numpy-localized lists, as host arrays
                        Dn, In = ix.search(xq[c0:c1], k, params=lp, exclude=chunk_lists(lists_np[r], c0, c1))
                        assert torch.equal(Dl, Dn) and torch.equal(Il, In), ("shard", r, c0)
                if self.with_ids:
                    packed.append(GpuCodec.pack_ids(Dl, Il))
                else:
                    if not (ex is None and self.kind == "flat" and lp is None):
                        Il = torch.where(Il >= 0, Il + self.bases[r], Il)
                    packed.append(GpuCodec.pack(Dl, Il, self.bases[r]))
            for j in range(self.G):
                lo, hi = min(c1 - c0, j * per), min(c1 - c0, (j + 1) * per)
                P = torch.stack([p[lo:hi] for p in packed])
                Dm, Im = GpuCodec.merge_ids(P, self.metric) if self.with_ids else GpuCodec.merge(P, bases, self.metric)
                D[c0 + lo:c0 + hi], I[c0 + lo:c0 + hi] = Dm, Im
        return D, I


def _lists(rng, nq, labels, top):
    """Exclusion lists that do not depend on G: the query's own top hits with random labels; labels
    of the last eighth of the rows (held by the last shard for every G); empty; -1, duplicates and
    absent ids. Query 4 lists 90 labels of the last eighth (k + 90 > 128: the long group on that
    shard only), query 9 every label of the first eighth (every row of shard 0 at G = 8). Every
    other list holds at most 40 labels, so each shard's filter group stays at k' <= 90."""
    n = labels.size
    first, last = labels[: n // 8], labels[n - n // 8:]
    absent = labels.max() + np.arange(1, 4)
    lists = []
    for q in range(nq):
        c = q % 5
        if q == 4:
            lst = last[:90]
        elif q == 9:
            lst = first
        elif c == 0:
            lst = np.concatenate([top[q, :10], rng.choice(labels, 10)])
        elif c == 1:
            lst = np.concatenate([rng.choice(last, 30), [-1]])
        elif c == 2:
            lst = []
        elif c == 3:
            lst = np.concatenate([top[q, :5], top[q, :5], absent, [-1]])
        else:
            lst = rng.choice(labels, 40)
        lists.append(rng.permutation(np.asarray(lst, dtype=np.int64)))
    import exclude_oracle as xo
    return xo.csr(lists)


def _no_listed_label(I, ex):
    off, ids = ex
    I = I.cpu().numpy()
    for q in range(I.shape[0]):
        lst = ids[off[q]:off[q + 1]]
        got = I[q][I[q] >= 0]
        assert not np.isin(got, lst[lst >= 0]).any(), q


def _oracle(kind, metric, xb, labels, single, nf, oracle):
    """The single oracle index with the same rows and labels, taking params and exclude."""
    from test_sharded_exclude_gloo import XFlat, XIDMap, XIVF
    d = xb.shape[1]
    if kind == "flat":
        o = XFlat(d, metric)
        o.add(xb)
    elif kind == "idmap":
        o = XIDMap(XFlat(d, metric))
        o.add_with_ids(xb, labels)
    else:
        q = oracle.IndexFlat(d, metric)
        q.add(single.quantizer.reconstruct_n())
        o = XIVF(q, d, single.nlist, metric)
        o.train(xb[:1])
        if kind == "ivf_ids":
            o.add_with_ids(xb, labels)
        else:
            o.add(xb)
        o.nprobe = single.nprobe
    return o


@pytest.mark.parametrize("kind,metric", [("flat", 0), ("idmap", 1), ("ivf", 1), ("ivf_ids", 0)])
@pytest.mark.parametrize("nq", [1_003, 13])
def test_virtual_shards_exclude(nf, oracle, kind, metric, nq):
    """G = 2, 4, 8 virtual shards against the single-GPU index with the same lists (and selector, and
    removals) and the oracle. nq = 13 takes the small-batch routes."""
    import torch
    from newsrecommend_b200.parity import compare_topk
    rng = np.random.default_rng(11)
    nb, d, k, nlist = 50_003, 128, 50, 64
    xb = rng.standard_normal((nb, d), dtype=np.float32)
    xq = rng.standard_normal((nq, d), dtype=np.float32)
    xq_dev = torch.from_numpy(xq).cuda()
    if kind in ("flat", "ivf"):
        labels = np.arange(nb, dtype=np.int64)
    elif kind == "idmap":
        labels = (np.sort(rng.choice(1 << 45, nb, replace=False)) + (1 << 33)).astype(np.int64)
    else:
        labels = rng.permutation(1 << 30)[:nb].astype(np.int64) * 1031 + (1 << 34)
    if kind in ("flat", "idmap"):
        single = nf.IndexFlat(d, metric) if kind == "flat" else nf.IndexIDMap(nf.IndexFlat(d, metric))
        window = nf.SearchParameters(sel=nf.IDSelectorRange(int(np.sort(labels)[int(0.7 * nb)]), 1 << 62))
    else:
        single = nf.IndexIVFFlat(nf.IndexFlat(d, metric), d, nlist, metric)
        single.train(xb)
        single.nprobe = 4
        window = nf.SearchParametersIVF(sel=nf.IDSelectorNot(nf.IDSelectorBatch(labels[::5].copy())), nprobe=8)
    if kind in ("flat", "ivf"):
        single.add(xb)
    else:
        single.add_with_ids(xb, labels)
    top = single.search(xq_dev, 10)[1].cpu().numpy()
    ex = _lists(rng, nq, labels, top)
    empty = (np.zeros(nq + 1, dtype=np.int64), np.empty(0, np.int64))
    ref = {None: single.search(xq_dev, k, exclude=ex), "window": single.search(xq_dev, k, params=window, exclude=ex)}
    orc = _oracle(kind, metric, xb, labels, single, nf, oracle)
    ref_o = {None: orc.search(xq, k, None, ex), "window": orc.search(xq, k, window, ex)}
    for name, (Dr, Ir) in ref.items():
        rep = compare_topk(Dr.cpu().numpy(), Ir.cpu().numpy(), *ref_o[name], metric)
        assert rep["ok"], ("single vs oracle", name, rep)
    for G in (2, 4, 8):
        vs = VirtualShards(nf, kind, metric, xb, labels, G, single)
        for name, p in ((None, None), ("window", window)):
            D, I = vs.search(xq_dev, k, p, ex)
            Dh, Ih = D.cpu().numpy(), I.cpu().numpy()
            rep = compare_topk(Dh, Ih, ref[name][0].cpu().numpy(), ref[name][1].cpu().numpy(), metric)
            assert rep["ok"], (G, name, "vs single", rep)
            rep = compare_topk(Dh, Ih, *ref_o[name], metric)
            assert rep["ok"], (G, name, "vs oracle", rep)
            _no_listed_label(I, ex)
        if G == 8:  # query 9 excludes every row of shard 0; query 4's 90 labels sit on shard 7
            assert not np.isin(Ih[9], labels[: nb // 8]).any()
        D0, I0 = vs.search(xq_dev, k, None, empty, check_local=False)
        Dp, Ip = vs.search(xq_dev, k)
        if nq >= 20:
            assert torch.equal(D0, Dp) and torch.equal(I0, Ip), (G, "all-empty lists")
        else:
            rep = compare_topk(D0.cpu().numpy(), I0.cpu().numpy(), Dp.cpu().numpy(), Ip.cpu().numpy(), metric)
            assert rep["ok"], (G, "all-empty lists", rep)
    # removals, then the same lists (removed labels match nothing) on the last G
    gone = labels[3::7].copy()
    assert vs.remove(gone) == single.remove_ids(nf.IDSelectorBatch(gone))
    if kind == "flat":  # positions renumbered: lists over the new positions
        labels = np.arange(single.ntotal, dtype=np.int64)
        top = single.search(xq_dev, 10)[1].cpu().numpy()
        ex = _lists(rng, nq, labels, top)
    for p in (None, window):
        D, I = vs.search(xq_dev, k, p, ex)
        Ds, Is = single.search(xq_dev, k, params=p, exclude=ex)
        rep = compare_topk(D.cpu().numpy(), I.cpu().numpy(), Ds.cpu().numpy(), Is.cpu().numpy(), metric)
        assert rep["ok"], ("after removal", rep)
        _no_listed_label(I, ex)


def test_sharded_exclude_nccl_torchrun():
    """ShardedIndexFlat / ShardedIndexIVFFlat (plain and id-carrying) search and search_host with
    exclusion lists over NCCL, one rank per visible GPU (2 ranks when the box has more than one;
    world size 1 still runs the process group, the localization and the host-array entry point)."""
    import torch
    n = min(torch.cuda.device_count(), 2)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29523",
           os.path.join(ROOT, "tests", "sharded_exclude_nccl_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and f"SHARDED_EXCLUDE_NCCL_OK world={n}" in r.stdout, (r.stdout[-2000:], r.stderr[-4000:])
