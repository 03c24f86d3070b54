"""GPU parity tests of the exact top-k path (K0 pack, K2 distance+selection, select) against the
oracle, through the faiss-compatible surface and the C-ABI. Bit-exact ids outside sub-1e-5 gaps,
scores within 1e-4 relative (tolerances of BASELINE.json's north_star, see parity.py)."""
import numpy as np
import pytest

import golden_inputs
from newsrecommend_b200.parity import compare_topk

pytestmark = pytest.mark.gpu
PATHS = {"tc": 2, "simt": 1, "tc1": 3, "tc16": 4, "auto": 0}


def _l2_scale(xq, xb):
    """|q|^2 + max |x|^2: the size of the terms the norm trick cancels (tolerance scale for L2)."""
    if xb.shape[0] == 0:
        return None
    return (xq.astype(np.float64) ** 2).sum(1, keepdims=True) + (xb.astype(np.float64) ** 2).sum(1).max()


def _search(nf, xb, xq, k, metric, path):
    index = nf.IndexFlatIP(xb.shape[1]) if metric == 0 else nf.IndexFlatL2(xb.shape[1])
    index.path = PATHS[path]
    index.add(xb)
    assert index.ntotal == xb.shape[0]
    return index.search(xq, k)


def test_pack_rows_split_is_exact(nf):
    import torch
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1000, 250), dtype=np.float32) * np.float32(3.0)
    p = nf.PackedMatrix.from_tensor(torch.from_numpy(x).cuda())
    raw, hi, lo = p.raw[:1000].cpu().numpy(), p.hi[:1000].cpu().numpy(), p.lo[:1000].cpu().numpy()
    assert p.kp == 256 and np.array_equal(raw[:, :250], x) and (raw[:, 250:] == 0).all()
    assert (hi.view(np.uint32) & 0x1FFF == 0).all() and (lo.view(np.uint32) & 0x1FFF == 0).all()
    # hi + lo reproduces x to ~2^-22 relative (two tf32 mantissas)
    err = np.abs((hi.astype(np.float64) + lo.astype(np.float64))[:, :250] - x)
    assert (err <= np.abs(x) * 2.0 ** -21 + 1e-30).all()
    assert np.allclose(p.norms[:1000].cpu().numpy(), (x.astype(np.float64) ** 2).sum(1), rtol=1e-5)


def test_pack_rows_h16_scales(nf):
    """fp16 plane of the fp16 filter: power-of-two scales (per row for queries, one for index
    storage, re-packed when a later append outgrows it), relative rounding error <= 2^-11."""
    import torch
    rng = np.random.default_rng(1)
    x = (rng.standard_normal((777, 250)) * np.exp(rng.uniform(-20, 20, size=(777, 1)))).astype(np.float32)
    x[5] = 0
    q = nf.PackedMatrix.from_tensor(torch.from_numpy(x).cuda(), planes=("raw", "norms", "h16"))
    s = q.row_scale[:777].cpu().numpy().astype(np.float64)
    h = q.h16[:777].cpu().numpy().astype(np.float64)
    nrm = np.sqrt((x.astype(np.float64) ** 2).sum(1))
    assert (np.log2(s) == np.round(np.log2(s))).all() and s[5] == 1.0
    live = nrm > 0
    assert ((nrm * s)[live] >= 2.0 ** 14 * (1 - 1e-6)).all() and ((nrm * s)[live] < 2.0 ** 15 * (1 + 1e-6)).all()
    assert np.isfinite(h).all() and (h[:, 250:] == 0).all()
    err = np.abs(h[:, :250] / s[:, None] - x)
    assert (err <= np.abs(x) * 2.0 ** -11 + 2.0 ** -25 / s[:, None]).all()
    # index storage: one scale; a 1000x larger second batch forces a re-pack of the first
    b = nf.PackedMatrix(250, planes=("raw", "hi", "lo", "norms", "h16"), track_max_norm=True)
    x1 = rng.standard_normal((300, 250), dtype=np.float32)
    b.append(torch.from_numpy(x1).cuda())
    s1 = b.h16_scale
    x2 = x1 * np.float32(1000.0)
    b.append(torch.from_numpy(x2).cuda())
    s2 = b.h16_scale
    assert s2 < s1 and b.max_norm * s2 < 2.0 ** 15 * (1 + 1e-6)
    hb = b.h16[:600].cpu().numpy().astype(np.float64) / s2
    xa = np.concatenate([x1, x2])
    assert np.isfinite(hb).all()
    assert (np.abs(hb[:, :250] - xa) <= np.abs(xa) * 2.0 ** -11 + 2.0 ** -25 / s2).all()


@pytest.mark.parametrize("path", ["tc", "simt", "tc1", "tc16", "auto"])
@pytest.mark.parametrize("metric", [0, 1])
def test_golden_fixture(nf, path, metric):
    g = golden_inputs.load("flat_small")
    D, I = _search(nf, g["xb"], g["xq"], 10, metric, path)
    assert D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (48, 10)
    rep = compare_topk(D, I, g[f"D{metric}"], g[f"I{metric}"], metric)
    assert rep["ok"], rep


@pytest.mark.parametrize("path", ["tc", "simt", "tc1", "tc16", "auto"])
@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("nq,nb,d,k", [
    (1, 5000, 250, 50), (19, 5000, 250, 50), (20, 5000, 256, 50), (129, 3001, 250, 20),
    (300, 255, 64, 1), (300, 256, 64, 16), (257, 257, 3, 5), (64, 1000, 1, 10), (33, 2000, 257, 100),
    (130, 7, 12, 10), (5, 1, 40, 3), (1000, 20000, 250, 128),
    (70, 3000, 96, 20), (300, 5000, 160, 50),  # fp16 rows of 192 / 320 bytes: the last 128-byte K chunk is zero-filled by TMA
])
def test_shapes_against_oracle(nf, oracle, path, metric, nq, nb, d, k):
    if path in ("tc1", "tc16") and (k > 112 or d > 256):
        pytest.skip("the filter paths cover k <= 112 and d <= 256 (PATH_AUTO routes the rest to 3xTF32)")
    rng = np.random.default_rng(nq * 1000 + nb + d + k)
    xb = rng.standard_normal((nb, d), dtype=np.float32)
    xq = rng.standard_normal((nq, d), dtype=np.float32)
    D, I = _search(nf, xb, xq, k, metric, path)
    Do, Io = oracle.knn_fast(xq, xb, k, metric)
    rep = compare_topk(D, I, Do, Io, metric, scale=_l2_scale(xq, xb) if metric == 1 else None)
    assert rep["ok"], rep
    assert rep["recall"] == 1.0 or rep["tie_exempt_queries"] > 0


@pytest.mark.parametrize("path", ["tc", "simt", "tc1", "tc16"])
def test_identity_duplicates_and_padding(nf, path):
    d = 32
    eye = np.eye(d, dtype=np.float32)
    D, I = _search(nf, eye, (eye * 2)[:25], 1, 0, path)
    assert (I[:, 0] == np.arange(25)).all() and np.allclose(D[:, 0], 2.0)
    D, I = _search(nf, eye, (eye * 2)[:25], 1, 1, path)
    assert (I[:, 0] == np.arange(25)).all() and np.allclose(D[:, 0], 1.0)
    # duplicates: ids are a valid choice from the tied set, no repeats
    rng = np.random.default_rng(2)
    base = rng.standard_normal((50, 20), dtype=np.float32)
    xb = np.concatenate([base, base, base])
    xq = rng.standard_normal((30, 20), dtype=np.float32)
    D, I = _search(nf, xb, xq, 6, 0, path)
    for q in range(30):
        assert len(set(I[q].tolist())) == 6
        assert len(set((I[q, :3] % 50).tolist())) == 1 and len(set((I[q, 3:] % 50).tolist())) == 1
    # k > ntotal: -1 / -+FLT_MAX padding
    fmax = np.float32(3.4028234663852886e38)
    xb = rng.standard_normal((7, 12), dtype=np.float32)
    xq = rng.standard_normal((40, 12), dtype=np.float32)
    for metric in (0, 1):
        D, I = _search(nf, xb, xq, 10, metric, path)
        assert (I[:, 7:] == -1).all() and all(sorted(r[:7].tolist()) == list(range(7)) for r in I)
        assert (D[:, 7:] == (fmax if metric == 1 else -fmax)).all()


def test_incremental_add_reset_and_errors(nf, oracle):
    rng = np.random.default_rng(9)
    xb = rng.standard_normal((3000, 250), dtype=np.float32)
    xq = rng.standard_normal((40, 250), dtype=np.float32)
    index = nf.IndexFlatIP(250)
    index.add(xb[:1000])
    index.add(xb[1000:])
    D, I = index.search(xq, 10)
    Do, Io = oracle.knn(xq, xb, 10, 0)
    assert compare_topk(D, I, Do, Io, 0)["ok"]
    assert np.array_equal(index.reconstruct_n(0, 5), xb[:5])
    index.reset()
    assert index.ntotal == 0
    D, I = index.search(xq, 3)
    assert (I == -1).all()
    with pytest.raises(AssertionError):
        index.search(xq[:, :10], 3)
    with pytest.raises(AssertionError):
        index.search(xq, 0)
    with pytest.raises(RuntimeError):
        index.search(xq, 1000)


def test_cuda_tensor_in_cuda_tensor_out(nf, oracle):
    import torch
    rng = np.random.default_rng(10)
    xb = rng.standard_normal((2000, 250), dtype=np.float32)
    xq = rng.standard_normal((100, 250), dtype=np.float32)
    index = nf.IndexFlatL2(250)
    index.add(torch.from_numpy(xb).cuda())
    D, I = index.search(torch.from_numpy(xq).cuda(), 5)
    assert D.is_cuda and I.is_cuda and I.dtype == torch.int64
    Do, Io = oracle.knn(xq, xb, 5, 1)
    assert compare_topk(D.cpu().numpy(), I.cpu().numpy(), Do, Io, 1)["ok"]


@pytest.mark.parametrize("metric", [0, 1])
def test_midsize_skewed_catalog(nf, oracle, metric):
    from newsrecommend_b200 import synth
    xb, topics = synth.g_skew(60000, 250, 42, return_topics=True)
    xq = synth.user_profiles(xb, topics, 3000, 43)
    D, I = _search(nf, xb, xq, 50, metric, "tc")
    Do, Io = oracle.knn_fast(xq, xb, 50, metric)
    rep = compare_topk(D, I, Do, Io, metric)
    assert rep["ok"], rep


def test_full_catalog_config1_sample(nf, oracle):
    """BASELINE config 1 catalog at full size (364,047 x 250), a 1,536-query sample against the
    oracle, plus tcgen05-vs-SIMT agreement on a second sample."""
    from newsrecommend_b200 import synth
    xb, topics = synth.g_skew(synth.N_ARTICLES, 250, 42, return_topics=True)
    xq = synth.user_profiles(xb, topics, 4096, 43)
    index = nf.IndexFlatIP(250)
    index.add(xb)
    D, I = index.search(xq, 50)
    Do, Io = oracle.knn_fast(xq[:1536], xb, 50, 0)
    rep = compare_topk(D[:1536], I[:1536], Do, Io, 0)
    assert rep["ok"], rep
    assert (np.diff(D, axis=1) <= 0).all() and I.min() >= 0 and I.max() < synth.N_ARTICLES
    index.path = PATHS["simt"]
    Ds, Is = index.search(xq[1536:2048], 50)
    rep = compare_topk(D[1536:2048], I[1536:2048], Ds, Is, 0)
    assert rep["ok"], rep


def test_item_item_cosine_self_match(nf):
    """Config 4 shape (cosine neighbours of L2-normalised items): the self match is rank 0 with
    score ~1 and idempotent normalisation."""
    from newsrecommend_b200 import synth
    x = synth.g_skew(20000, 250, 11)
    nf.normalize_L2(x)
    assert np.allclose((x.astype(np.float64) ** 2).sum(1), 1.0, atol=1e-5)
    index = nf.IndexFlatIP(250)
    index.add(x)
    D, I = index.search(x[:4000], 20)
    assert (I[:, 0] == np.arange(4000)).mean() > 0.999  # exact duplicates aside
    assert np.allclose(D[:, 0], 1.0, atol=1e-5)


@pytest.mark.parametrize("metric", [0, 1])
def test_tc_kernel_variants(nf, oracle, metric):
    """The 3xTF32 tcgen05 kernel (CTA pairs, cta_group::2) against the oracle on shapes with odd
    query-tile counts, partial item tiles and several item chunks."""
    rng = np.random.default_rng(77 + metric)
    for nq, nb, d, k in ((48, 2000, 250, 10), (385, 30011, 250, 50), (1, 70000, 96, 7), (129, 513, 32, 128)):
        xb = rng.standard_normal((nb, d), dtype=np.float32)
        xq = rng.standard_normal((nq, d), dtype=np.float32)
        D, I = _search(nf, xb, xq, k, metric, "tc")
        Do, Io = oracle.knn_fast(xq, xb, k, metric)
        rep = compare_topk(D, I, Do, Io, metric, scale=_l2_scale(xq, xb) if metric == 1 else None)
        assert rep["ok"], (nq, nb, d, k, rep)


@pytest.mark.parametrize("filt", ["tc1", "tc16"])
def test_tc1_filter_margin_and_fallback(nf, oracle, filt):
    """The 1xTF32 filter: (a) on ordinary data no query needs the 3xTF32 fallback, i.e. every
    estimate stayed inside the assumed error bound and the margin set fitted its slots;
    (b) with hundreds of exact duplicates the margin set overflows, the queries are flagged,
    recomputed by the 3xTF32 kernel, and the result is still a valid top-k."""
    from newsrecommend_b200 import synth
    from newsrecommend_b200._lib import lib
    xb, topics = synth.g_skew(50000, 250, 3, return_topics=True)
    xq = synth.user_profiles(xb, topics, 2000, 4)
    for metric in (0, 1):
        n0 = lib.nrb_fallback_query_count()
        D, I = _search(nf, xb, xq, 50, metric, filt)
        assert lib.nrb_fallback_query_count() == n0, "fallback used on ordinary data"
        Do, Io = oracle.knn_fast(xq, xb, 50, metric)
        rep = compare_topk(D, I, Do, Io, metric, scale=_l2_scale(xq, xb) if metric == 1 else None)
        assert rep["ok"], rep
    rng = np.random.default_rng(8)
    base = rng.standard_normal((20, 64), dtype=np.float32)
    xb = np.concatenate([np.repeat(base, 150, axis=0), rng.standard_normal((2000, 64), dtype=np.float32)])
    xq = base + 0.01 * rng.standard_normal((20, 64), dtype=np.float32)
    n0 = lib.nrb_fallback_query_count()
    D, I = _search(nf, xb, xq, 10, 0, filt)
    assert lib.nrb_fallback_query_count() >= n0 + 20
    for q in range(20):
        assert len(set(I[q].tolist())) == 10 and (I[q] // 150 == q).all()  # ten of the 150 copies of base[q]
    Do, Io = oracle.knn_fast(xq, xb, 10, 0)
    assert np.allclose(D, Do, rtol=1e-4)


@pytest.mark.parametrize("path", ["tc16", "tc1", "tc"])
@pytest.mark.parametrize("metric", [0, 1])
def test_adversarial_item_order(nf, oracle, path, metric):
    """Worst case for a streaming top-k: the catalog is sorted so that every query's scores improve
    monotonically along the scan (every item beats the running threshold: candidate buffers fill
    up inside the tiles and the overflow guard has to prune over and over), and, separately, a
    catalog sorted the other way (the first tile already holds the answer)."""
    rng = np.random.default_rng(123)
    d, nb, nq, k = 64, 30000, 200, 50
    u = rng.standard_normal(d).astype(np.float32)
    u /= np.linalg.norm(u)
    xb = rng.standard_normal((nb, d), dtype=np.float32)
    t = np.sort(rng.standard_normal(nb).astype(np.float32) * 4)  # strength along u, ascending
    xb = xb - np.outer(xb @ u, u) + np.outer(t, u)
    if metric == 1:
        xq = 40.0 * u[None, :] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)  # far along u: nearest = last rows
    else:
        xq = 3.0 * u[None, :] + 0.05 * rng.standard_normal((nq, d)).astype(np.float32)
    for order in (slice(None), slice(None, None, -1)):
        xs = np.ascontiguousarray(xb[order])
        D, I = _search(nf, xs, xq.astype(np.float32), k, metric, path)
        Do, Io = oracle.knn_fast(xq.astype(np.float32), xs, k, metric)
        rep = compare_topk(D, I, Do, Io, metric, scale=_l2_scale(xq, xs) if metric == 1 else None)
        assert rep["ok"], rep


def test_host_pipelined_search_matches_single_shot(nf):
    """numpy in / numpy out with >= 2 waves of queries takes the chunked copy/compute pipeline:
    same (D, I) as the packed single-shot search, with and without caller-provided outputs."""
    import torch
    rng = np.random.default_rng(31)
    d, nb, k = 64, 4000, 10
    nq = 2 * nf._wave_rows() + 1234
    xb = rng.standard_normal((nb, d), dtype=np.float32)
    xq = rng.standard_normal((nq, d), dtype=np.float32)
    index = nf.IndexFlatIP(d)
    index.add(xb)
    q = nf.PackedMatrix.from_tensor(torch.from_numpy(xq).cuda(), planes=index._query_planes(k))
    Dr, Ir = index.search_packed(q, k)
    Dr, Ir = Dr.cpu().numpy(), Ir.cpu().numpy()
    D1, I1 = index.search(xq, k)
    assert np.array_equal(I1, Ir) and np.array_equal(D1, Dr)
    Dp = torch.empty((nq, k), dtype=torch.float32, pin_memory=True).numpy()
    Ip = torch.empty((nq, k), dtype=torch.int64, pin_memory=True).numpy()
    D2, I2 = index.search(xq, k, D=Dp, I=Ip)
    assert D2 is Dp and I2 is Ip and np.array_equal(I2, Ir) and np.array_equal(D2, Dr)


def test_growing_norms_repack_fp16_plane(nf, oracle):
    """add() of rows 1000x larger than the first batch outgrows the fp16 plane's scale: the plane is
    re-packed from the raw plane and the search still matches the oracle on the whole catalog."""
    rng = np.random.default_rng(55)
    x1 = rng.standard_normal((3000, 128), dtype=np.float32)
    x2 = rng.standard_normal((3000, 128), dtype=np.float32) * np.float32(1000.0)
    xq = rng.standard_normal((200, 128), dtype=np.float32)
    for metric in (0, 1):
        index = nf.IndexFlatIP(128) if metric == 0 else nf.IndexFlatL2(128)
        index.path = PATHS["tc16"]
        index.add(x1)
        s1 = index._xb.h16_scale
        D, I = index.search(xq, 20)
        Do, Io = oracle.knn_fast(xq, x1, 20, metric)
        assert compare_topk(D, I, Do, Io, metric, scale=_l2_scale(xq, x1) if metric == 1 else None)["ok"]
        index.add(x2)
        assert index._xb.h16_scale < s1
        xb = np.concatenate([x1, x2])
        D, I = index.search(xq, 20)
        Do, Io = oracle.knn_fast(xq, xb, 20, metric)
        rep = compare_topk(D, I, Do, Io, metric, scale=_l2_scale(xq, xb) if metric == 1 else None)
        assert rep["ok"], rep


@pytest.mark.parametrize("metric", [0, 1])
def test_single_cta_filter_kernel(nf, oracle, metric, monkeypatch):
    """The single-CTA (cta_group::1, M = 128) form of the fp16 filter kernel, which the planner picks
    for single partial waves where CTA pairs cannot cut the catalog finely enough: forced here on
    shapes with odd tile counts, ragged tiles and several item chunks."""
    monkeypatch.setenv("NRB_FORCE_SINGLE_CTA", "1")
    rng = np.random.default_rng(90 + metric)
    for nq, nb, d, k in ((1, 3000, 250, 50), (129, 70000, 250, 50), (385, 30011, 96, 20), (6250, 20000, 64, 10)):
        xb = rng.standard_normal((nb, d), dtype=np.float32)
        xq = rng.standard_normal((nq, d), dtype=np.float32)
        D, I = _search(nf, xb, xq, k, metric, "tc16")
        Do, Io = oracle.knn_fast(xq, xb, k, metric)
        rep = compare_topk(D, I, Do, Io, metric, scale=_l2_scale(xq, xb) if metric == 1 else None)
        assert rep["ok"], (nq, nb, d, k, rep)
