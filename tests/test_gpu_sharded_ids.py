"""GPU tests of the id-carrying sharded search: the 16-byte wire-format kernels against their numpy
restatement, G virtual shards in one process (the data flow of the all-to-all by query range,
exchanged by hand) for IndexIDMap and IndexIVFFlat shards, filtered and unfiltered, against the
single-GPU index with the same ids and the oracle, and the NCCL path under torchrun
(tests/sharded_ids_nccl_worker.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("metric", [0, 1])
def test_pack_and_merge_ids_kernels(nf, metric):
    import torch
    from newsrecommend_b200.sharded import GpuCodec
    from test_sharded_ids_gloo import NumpyIdCodec
    rng = np.random.default_rng(0)
    G, nq, k = 8, 300, 50
    Dp = np.sort(rng.standard_normal((G, nq, k)).astype(np.float32), axis=2)
    Dp = Dp[:, :, ::-1].copy() if metric == 0 else np.sort(np.abs(Dp), axis=2)
    Ip = rng.integers(0, 1 << 50, (G, nq, k), dtype=np.int64)  # ids far beyond 32 bits, in no shard order
    Ip[3, :, 40:] = -1  # a shard with fewer than k results
    Dp[3, :, 40:] = 3.4028235e38 if metric else -3.4028235e38
    Ip[5] = -1  # a shard with none
    Dp[0, :, 5] = Dp[1, :, 7]  # exact score ties between shards: the lower part wins
    Dp[0] = -np.sort(-Dp[0], axis=1) if metric == 0 else np.sort(Dp[0], axis=1)
    packs, packs_np = [], []
    for s in range(G):
        P = GpuCodec.pack_ids(torch.from_numpy(Dp[s]).cuda(), torch.from_numpy(Ip[s]).cuda())
        Pn = NumpyIdCodec.pack_ids(torch.from_numpy(Dp[s]), torch.from_numpy(Ip[s]))
        assert torch.equal(P.cpu(), Pn)  # bit-exact wire format
        packs.append(P)
        packs_np.append(Pn)
    D, I = GpuCodec.merge_ids(torch.stack(packs), metric)
    Dn, In = NumpyIdCodec.merge_ids(torch.stack(packs_np), metric)
    assert torch.equal(I.cpu(), In) and torch.equal(D.cpu(), Dn)
    assert (In.numpy() >= (1 << 32)).any()


def _shards(nf, kind, metric, xb, ids, G, single):
    from newsrecommend_b200.sharded import shard_range
    d = xb.shape[1]
    shards = []
    for r in range(G):
        lo, hi = shard_range(xb.shape[0], G, r)
        if kind == "flat":
            ix = nf.IndexIDMap(nf.IndexFlat(d, metric))
        else:
            q = nf.IndexFlat(d, metric)
            q.add(single.quantizer.reconstruct_n())  # the shared coarse quantizer
            ix = nf.IndexIVFFlat(q, d, single.nlist, metric)
            ix.train(xb[:1])
            ix.nprobe = single.nprobe
        ix.add_with_ids(xb[lo:hi], ids[lo:hi])
        shards.append(ix)
    return shards


@pytest.mark.parametrize("kind", ["flat", "ivf"])
@pytest.mark.parametrize("filtered", [False, True])
@pytest.mark.parametrize("metric,nq", [(0, 1_003), (1, 1_003), (0, 13)])
def test_virtual_id_shards_match_single_index_and_oracle(nf, oracle, kind, filtered, metric, nq):
    """ShardedIndex*.search(exchange="alltoall") with G = 4 id-carrying shards in one process:
    per-shard search (params included) -> nrb_pack_topk_ids -> every rank's query range from every
    shard -> nrb_merge_topk_packed_ids. nq = 13 takes the masked small-batch kernels."""
    import filtered_oracle as fl
    import ids_oracle as io
    import torch
    from newsrecommend_b200.parity import compare_topk
    from newsrecommend_b200.sharded import GpuCodec, chunk_slices
    rng = np.random.default_rng(3)
    nb, d, k, G, nlist = 50_003, 128, 50, 4, 64
    xb = rng.standard_normal((nb, d), dtype=np.float32)
    xq = rng.standard_normal((nq, d), dtype=np.float32)
    ids = (np.sort(rng.choice(1 << 45, nb, replace=False)) + (1 << 33)).astype(np.int64)
    xq_dev = torch.from_numpy(xq).cuda()
    if kind == "flat":
        single = nf.IndexIDMap(nf.IndexFlat(d, metric))
        sel = nf.IDSelectorRange(int(ids[int(0.7 * nb)]), 1 << 62)  # the newest 30 %
        params = nf.SearchParameters(sel=sel) if filtered else None
    else:
        single = nf.IndexIVFFlat(nf.IndexFlat(d, metric), d, nlist, metric)
        single.train(xb)
        single.nprobe = 4
        sel = nf.IDSelectorNot(nf.IDSelectorBatch(ids[::5].copy()))  # a blocklist of a fifth of the rows
        params = nf.SearchParametersIVF(sel=sel, nprobe=8) if filtered else None
    single.add_with_ids(xb, ids)
    Ds, Is = single.search(xq_dev, k, params=params)
    shards = _shards(nf, kind, metric, xb, ids, G, single)
    D = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    I = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    for c0, c1, per in chunk_slices(nq, G, 512):
        packed = []
        for r in range(G):
            Dl, Il = shards[r].search(xq_dev[c0:c1], k, params=params)
            packed.append(GpuCodec.pack_ids(Dl, Il))
        for j in range(G):
            lo, hi = min(c1 - c0, j * per), min(c1 - c0, (j + 1) * per)
            Dm, Im = GpuCodec.merge_ids(torch.stack([p[lo:hi] for p in packed]), metric)
            D[c0 + lo:c0 + hi], I[c0 + lo:c0 + hi] = Dm, Im
    Dh, Ih = D.cpu().numpy(), I.cpu().numpy()
    assert compare_topk(Dh, Ih, Ds.cpu().numpy(), Is.cpu().numpy(), metric)["ok"]
    assert torch.equal(D, Ds)  # random-normal rows: the single index's scores, position for position
    # the oracle: the same rows, ids (and selector) on the CPU
    osel = None if not filtered else (io.IDSelectorRange(sel.imin, sel.imax) if kind == "flat" else
                                      fl.IDSelectorNot(io.IDSelectorBatch(sel.sel.ids)))
    if kind == "flat":
        om = io.IndexIDMap(io.IndexFlat(d, metric))
        om.add_with_ids(xb, ids)
        Do, Io = om.search(xq, k) if osel is None else fl.search_idmap(om, xq, k, osel)
    else:
        q = oracle.IndexFlat(d, metric)
        q.add(single.quantizer.reconstruct_n())
        ov = io.IndexIVFFlat(q, d, nlist, metric)
        ov.train(xb[:1])
        ov.add_with_ids(xb, ids)
        ov.nprobe = 4
        Do, Io = ov.search(xq, k) if osel is None else fl.search_ivf(ov, xq, k, osel, 8)
    rep = compare_topk(Dh, Ih, Do, Io, metric)
    assert rep["ok"], rep


def test_sharded_ids_nccl_torchrun():
    """The id-carrying and plain sharded indexes with ids, selectors and removals over NCCL, one rank
    per visible GPU (2 ranks when the box has more than one; world size 1 still runs the process
    group, the 16-byte codec and the host-array entry point)."""
    import torch
    n = min(torch.cuda.device_count(), 2)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", "29521",
           os.path.join(ROOT, "tests", "sharded_ids_nccl_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and f"SHARDED_IDS_NCCL_OK world={n}" in r.stdout, (r.stdout[-2000:], r.stderr[-4000:])
