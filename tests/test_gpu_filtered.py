"""Search-time ID selectors on the B200: the masked HBM-regime kernels against the numpy restatement
(tests/filtered_oracle.py), bit-for-bit equivalence of every filtered route with the same route on an
index built from only the selected rows, SearchParametersIVF.nprobe, remove_ids with IDSelectorNot,
and one full-size catalog case."""
import numpy as np
import pytest

from newsrecommend_b200.parity import compare_topk
from test_gpu_kmeans_ivf import _classify_ivf_mismatches

pytestmark = pytest.mark.gpu

FLT_MAX = np.float32(3.4028234663852886e38)


@pytest.fixture(scope="module")
def fo(oracle):
    import filtered_oracle
    return filtered_oracle


@pytest.fixture(scope="module")
def io(oracle):
    import ids_oracle
    return ids_oracle


def _np(a):
    import torch
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else a


def _same(a, b):
    D1, I1 = map(_np, a)
    D2, I2 = map(_np, b)
    assert D1.shape == D2.shape and np.array_equal(D1.view(np.int32), D2.view(np.int32)) and np.array_equal(I1, I2)


def _sel_pair(nf, io, fo, kind, arg):
    """The same selector for the GPU index and for the oracle."""
    if kind == "range":
        return nf.IDSelectorRange(*arg), io.IDSelectorRange(*arg)
    if kind == "batch":
        return nf.IDSelectorBatch(arg), io.IDSelectorBatch(arg)
    if kind == "not_batch":
        return nf.IDSelectorNot(nf.IDSelectorBatch(arg)), fo.IDSelectorNot(io.IDSelectorBatch(arg))
    return nf.IDSelectorNot(nf.IDSelectorRange(*arg)), fo.IDSelectorNot(io.IDSelectorRange(*arg))


def _parity(D, I, Do, Io, metric, xq, xb, what):
    """The parity rule; a selection smaller than k returns every selected row, also rows whose IP
    score is a near-zero cancellation, where the rule's relative score tolerance is meaningless. Such
    rows must still carry exactly the oracle's ids and padding, with scores within 1e-4 of
    |q| * max|x|."""
    rep = compare_topk(D, I, Do, Io, metric)
    if rep["ok"]:
        return
    assert metric == 0 and rep["id_mismatch_queries"] == 0 and rep["pad_ok"], (what, rep)
    bound = 1e-4 * np.linalg.norm(xq, axis=1)[:, None] * np.linalg.norm(xb, axis=1).max()
    assert (np.abs(D.astype(np.float64) - Do) <= bound)[Io >= 0].all(), (what, rep)


def _mapped(D, I, labels):
    D, I = _np(D), _np(I)
    return D, np.where(I < 0, -1, labels[np.maximum(I, 0)])


# ------------------------------------------------------------------ masked kernels against numpy
@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("n", [6000, 40_000])  # fused kernel (n <= 8,192) and two-level selection
def test_masked_small_flat(nf, io, fo, metric, n):
    import torch
    rng = np.random.default_rng(n + metric)
    d = 96
    xb = rng.standard_normal((n, d), dtype=np.float32)
    ids = np.arange(n, dtype=np.int64) * 5 + 3  # IndexIDMap: the selector reaches the kernel without a host count
    plain = nf.IndexFlat(d, metric)
    plain.add(xb)
    m = nf.IndexIDMap(nf.IndexFlat(d, metric))
    m.add_with_ids(xb, ids)
    o = io.IndexFlat(d, metric)
    o.add(xb)
    pos = np.arange(n, dtype=np.int64)
    rand = np.sort(rng.choice(n, n // 10, replace=False))
    cases = {"none": pos[:0], "fewer_than_k": rand[:30], "all": pos, "ten_percent": rand}
    for nq in (1, 5, 19):
        xq = rng.standard_normal((nq, d), dtype=np.float32)
        for name, rows in cases.items():
            for k in (1, 50, 128):
                Do, Io = fo.search_flat(o, xq, k, io.IDSelectorBatch(rows))
                # plain index, numpy: the single-call host route (positions)
                D, I = plain.search(xq, k, params=nf.SearchParameters(sel=nf.IDSelectorBatch(rows)))
                _parity(D, I, Do, Io, metric, xq, xb, (nq, name, k))
                assert np.isin(I[I >= 0], rows).all()
                nk = min(k, rows.size)
                assert (I[:, :nk] >= 0).all() and (I[:, nk:] == -1).all()
                assert (D[:, nk:] == (-FLT_MAX if metric == 0 else FLT_MAX)).all()
                # IndexIDMap, CUDA tensors: the device route, selector on the ids
                Dt, It = m.search(torch.from_numpy(xq).cuda(), k,
                                  params=nf.SearchParameters(sel=nf.IDSelectorNot(nf.IDSelectorNot(
                                      nf.IDSelectorBatch(ids[rows])))))
                assert Dt.is_cuda
                _same((Dt, It), (D, np.where(I < 0, -1, ids[np.maximum(I, 0)])))


@pytest.mark.parametrize("metric", [0, 1])
def test_masked_small_ivf(nf, io, fo, metric):
    from test_gpu_ids import _ivf_data, _ivf_pair
    xb, xq, ids = _ivf_data(20_000, 64, seed=41)
    nlist, k = 32, 50
    make, ivf_o = _ivf_pair(nf, io, xb, nlist, metric)
    ivf = make()
    ivf.add_with_ids(xb, ids)
    ivf_o.add_with_ids(xb, ids)
    rng = np.random.default_rng(5)
    cases = {"none": ids[:0], "fewer_than_k": ids[rng.choice(len(ids), 20, replace=False)],
             "all": ids, "ten_percent": ids[rng.choice(len(ids), len(ids) // 10, replace=False)]}
    for name, batch in cases.items():
        sel, sel_o = nf.IDSelectorBatch(batch), io.IDSelectorBatch(batch)
        for nq in (1, 64):
            for nprobe in (4, nlist):
                D, I = ivf.search(xq[:nq], k, params=nf.SearchParametersIVF(sel=sel, nprobe=nprobe))
                assert np.isin(I[I >= 0], batch).all()
                view = fo.filtered_ivf(ivf_o, sel_o)
                view.nprobe = nprobe
                Do, Io = view.search(xq[:nq], k)
                if not compare_topk(D, I, Do, Io, metric)["ok"]:
                    _classify_ivf_mismatches(view, xq[:nq], nprobe, k, D, I, Do, Io, metric)
                if name == "none":
                    assert (I == -1).all() and (D == (-FLT_MAX if metric == 0 else FLT_MAX)).all()


# ------------------------------------------------------------------ equivalence, bit for bit
def _flat_selectors(n, rng):
    """Range, Batch, Not(Batch), Not(Range) over positions, each keeping > 8,192 of n = 30,000 rows
    so that the filtered and the subset-built index take the same low-latency kernel family."""
    return [("range", (5000, 25_000)), ("batch", np.sort(rng.choice(n, n // 2, replace=False))),
            ("not_batch", rng.choice(n, 3000)), ("not_range", (0, 10_000))]


@pytest.mark.parametrize("metric", [0, 1])
def test_flat_equivalence_every_route(nf, io, fo, metric):
    import torch
    n, d = 30_000, 64
    rng = np.random.default_rng(10 + metric)
    xb = rng.standard_normal((n, d), dtype=np.float32)
    pos = np.arange(n, dtype=np.int64)
    ids = (rng.permutation(n).astype(np.int64) * 1_000_003) - 7 * 10 ** 9  # random, non-contiguous
    plain = nf.IndexFlat(d, metric)
    plain.add(xb)
    m = nf.IndexIDMap(nf.IndexFlat(d, metric))
    m.add_with_ids(xb, ids)
    wave2 = 2 * nf._wave_rows()
    xq_all = rng.standard_normal((wave2 + 100, d), dtype=np.float32)
    routes = [("numpy_small", xq_all[:19], False), ("cuda_small", xq_all[:19], True),
              ("cuda_batch", xq_all[:700], True), ("numpy_pipelined", xq_all, False)]
    o = io.IndexFlat(d, metric)
    o.add(xb)
    for kind, arg in _flat_selectors(n, rng):
        sel, sel_o = _sel_pair(nf, io, fo, kind, arg)
        keep = sel_o.members(pos)
        sub = nf.IndexFlat(d, metric)
        sub.add(xb[keep])
        sub_m = nf.IndexIDMap(nf.IndexFlat(d, metric))
        sub_m.add_with_ids(xb[keep], ids[keep])
        # the same rows named by their ids, for the IndexIDMap
        sel_ids = nf.IDSelectorNot(nf.IDSelectorBatch(ids[~keep])) if kind.startswith("not") else \
            nf.IDSelectorBatch(ids[keep])
        for route, xq, cuda in routes:
            x = torch.from_numpy(xq).cuda() if cuda else xq
            for k in (1, 50):
                D, I = plain.search(x, k, params=nf.SearchParameters(sel=sel))
                assert isinstance(D, torch.Tensor) == cuda
                _same((D, I), _mapped(*sub.search(x, k), pos[keep]))
                _same(m.search(x, k, params=nf.SearchParameters(sel=sel_ids)), sub_m.search(x, k))
            if route in ("numpy_small", "cuda_batch"):
                Do, Io = fo.search_flat(o, xq[:300], 50, sel_o)
                rep = compare_topk(_np(D)[:300], _np(I)[:300], Do, Io, metric)
                assert rep["ok"], (kind, route, rep)
    # a selector that keeps every row is the unfiltered search
    every = nf.IDSelectorNot(nf.IDSelectorRange(n, 2 * n))
    for route, xq, cuda in routes:
        x = torch.from_numpy(xq).cuda() if cuda else xq
        _same(plain.search(x, 50, params=nf.SearchParameters(sel=every)), plain.search(x, 50))
        _same(m.search(x, 50, params=nf.SearchParameters(sel=nf.IDSelectorRange(-10 ** 18, 10 ** 18))), m.search(x, 50))


@pytest.mark.parametrize("metric", [0, 1])
def test_flat_equivalence_every_path(nf, io, fo, metric):
    """The batch route on each index.path searches the compacted subset on that same path."""
    import torch
    from newsrecommend_b200._lib import PATH_SIMT, PATH_TC, PATH_TC1, PATH_TC16
    n, d = 12_000, 128
    rng = np.random.default_rng(20 + metric)
    xb = rng.standard_normal((n, d), dtype=np.float32)
    xq = rng.standard_normal((600, d), dtype=np.float32)
    pos = np.arange(n, dtype=np.int64)
    for kind, arg in (("range", (2000, 9000)), ("not_batch", rng.choice(n, 5000)), ("batch", pos[::3]),
                      ("not_range", (100, 11_000))):
        sel, sel_o = _sel_pair(nf, io, fo, kind, arg)
        keep = sel_o.members(pos)
        for path in (PATH_TC16, PATH_TC1, PATH_TC, PATH_SIMT):
            idx, sub = nf.IndexFlat(d, metric), nf.IndexFlat(d, metric)
            idx.path = sub.path = path
            idx.add(xb)
            sub.add(xb[keep])
            for nq in (5, 600):  # with an explicit path even nq < 20 takes the batch route
                for x in (xq[:nq], torch.from_numpy(xq[:nq]).cuda()):
                    _same(idx.search(x, 50, params=nf.SearchParameters(sel=sel)), _mapped(*sub.search(x, 50), pos[keep]))


@pytest.mark.parametrize("metric", [0, 1])
def test_ivf_filtered_equivalence_and_nprobe(nf, io, fo, metric):
    from test_gpu_ids import _ivf_data, _ivf_pair
    xb, xq, ids = _ivf_data(30_000, 700, seed=51)
    nlist = 64
    make, ivf_o = _ivf_pair(nf, io, xb, nlist, metric)
    ivf = make()
    ivf.add_with_ids(xb[:12_000], ids[:12_000])
    ivf.add_with_ids(xb[12_000:], ids[12_000:])
    ivf_o.add_with_ids(xb, ids)
    rng = np.random.default_rng(6)
    # SearchParametersIVF(nprobe=p) is index.nprobe = p for the call, and leaves index.nprobe alone
    ivf.nprobe = 3
    for p in (1, 16, nlist):
        for nq in (30, 700):
            D, I = ivf.search(xq[:nq], 50, params=nf.SearchParametersIVF(nprobe=p))
            assert ivf.nprobe == 3
            ivf.nprobe = p
            _same((D, I), ivf.search(xq[:nq], 50))
            ivf.nprobe = 3
    _same(ivf.search(xq, 50, params=nf.SearchParametersIVF()), ivf.search(xq, 50))
    lo = int(np.quantile(ids, 0.5))
    for kind, arg in (("range", (lo, 10 ** 12)), ("batch", ids[rng.choice(len(ids), 9000, replace=False)]),
                      ("not_batch", ids[::4]), ("not_range", (0, lo))):
        sel, sel_o = _sel_pair(nf, io, fo, kind, arg)
        keep = sel_o.members(ids)
        fresh = make()  # shares the trained quantizer's centroids
        fresh.add_with_ids(xb[keep], ids[keep])
        for nprobe in (1, 16):
            fresh.nprobe = nprobe
            for nq in (30, 700):  # the masked small scan and the tcgen05 scan over filtered lists
                D, I = ivf.search(xq[:nq], 50, params=nf.SearchParametersIVF(sel=sel, nprobe=nprobe))
                _same((D, I), fresh.search(xq[:nq], 50))
                view = fo.filtered_ivf(ivf_o, sel_o)
                view.nprobe = nprobe
                Do, Io = view.search(xq[:nq], 50)
                if not compare_topk(D, I, Do, Io, metric)["ok"]:
                    _classify_ivf_mismatches(view, xq[:nq], nprobe, 50, D, I, Do, Io, metric)
    every = nf.IDSelectorRange(-10 ** 18, 10 ** 18)
    for nq in (30, 700):
        _same(ivf.search(xq[:nq], 50, params=nf.SearchParametersIVF(sel=every)), ivf.search(xq[:nq], 50))
        D, I = ivf.search(xq[:nq], 50, params=nf.SearchParametersIVF(sel=nf.IDSelectorNot(every)))
        assert (I == -1).all() and (D == (-FLT_MAX if metric == 0 else FLT_MAX)).all()


# ------------------------------------------------------------------ remove_ids with IDSelectorNot
@pytest.mark.parametrize("metric", [0, 1])
def test_remove_ids_not(nf, io, fo, metric):
    from test_gpu_ids import _flat_data, _ivf_data, _ivf_pair
    xb, ids = _flat_data(9000, 64, 61)
    xq = np.random.default_rng(7).standard_normal((500, 64), dtype=np.float32)
    pos = np.arange(9000, dtype=np.int64)
    s_pos = pos[(pos % 7 == 0) | (pos > 8000)]
    # flat: Not(s) selects positions; remove_ids(Not(s)) == remove_ids(complement of s)
    a, b = nf.IndexFlat(64, metric), nf.IndexFlat(64, metric)
    a.add(xb)
    b.add(xb)
    assert a.remove_ids(nf.IDSelectorNot(nf.IDSelectorBatch(s_pos))) == b.remove_ids(np.setdiff1d(pos, s_pos)) \
        == 9000 - s_pos.size
    _same(a.search(xq, 50), b.search(xq, 50))
    # IndexIDMap: on the ids
    a, b = nf.IndexIDMap(nf.IndexFlat(64, metric)), nf.IndexIDMap(nf.IndexFlat(64, metric))
    a.add_with_ids(xb, ids)
    b.add_with_ids(xb, ids)
    lo, hi = int(np.quantile(ids, 0.3)), int(np.quantile(ids, 0.6))
    out = ids[(ids < lo) | (ids >= hi)]
    assert a.remove_ids(nf.IDSelectorNot(nf.IDSelectorRange(lo, hi))) == b.remove_ids(out) == out.size
    assert np.array_equal(a.id_map.cpu().numpy(), b.id_map.cpu().numpy())
    _same(a.search(xq, 50), b.search(xq, 50))
    # IVF
    xb2, xq2, ids2 = _ivf_data(20_000, 300, seed=62)
    make, _ = _ivf_pair(nf, io, xb2, 32, metric)
    a, b = make(), make()
    a.add_with_ids(xb2, ids2)
    b.add_with_ids(xb2, ids2)
    s = ids2[::3]
    assert a.remove_ids(nf.IDSelectorNot(nf.IDSelectorBatch(s))) == b.remove_ids(np.setdiff1d(ids2, s)) \
        == len(ids2) - s.size
    a.nprobe = b.nprobe = 8
    _same(a.search(xq2, 50), b.search(xq2, 50))


# ------------------------------------------------------------------ full size
def test_fullsize_newer_half(nf, io, fo):
    """The 364,047 x 250 catalog with article ids in publication order, all 50,000 queries, and a
    freshness window keeping the newer half, against the index built from that half."""
    from newsrecommend_b200 import synth
    xb, topics = synth.g_skew(synth.N_ARTICLES, 250, 42, return_topics=True)
    xq = synth.user_profiles(xb, topics, 50_000, 43)
    n = xb.shape[0]
    ids = 100_000 + np.arange(n, dtype=np.int64) * 3
    cut = int(ids[n // 2])
    m = nf.IndexIDMap(nf.IndexFlatIP(250))
    m.add_with_ids(xb, ids)
    sub = nf.IndexIDMap(nf.IndexFlatIP(250))
    sub.add_with_ids(xb[n // 2:], ids[n // 2:])
    D, I = m.search(xq, 50, params=nf.SearchParameters(sel=nf.IDSelectorRange(cut, 1 << 62)))
    assert I.min() >= cut
    _same((D, I), sub.search(xq, 50))
    Do, Io = fo.search_idmap(_fullsize_oracle(io, xb, ids), xq[:1000], 50, io.IDSelectorRange(cut, 1 << 62))
    rep = compare_topk(D[:1000], I[:1000], Do, Io, 0)
    assert rep["ok"] and rep["recall"] >= 0.9999, rep
    # the single-query numpy route of Retrieval.py:32, masked
    D1, I1 = m.search(xq[:1], 50, params=nf.SearchParameters(sel=nf.IDSelectorRange(cut, 1 << 62)))
    assert compare_topk(D1, I1, D[:1], I[:1], 0)["ok"]


def _fullsize_oracle(io, xb, ids):
    om = io.IndexIDMap(io.IndexFlatIP(xb.shape[1]))
    om.add_with_ids(xb, ids)
    return om
