"""Worker of tests/test_gpu_sharded_ids.py::test_sharded_ids_nccl_torchrun (launched with torchrun,
one rank per GPU, NCCL): external ids, search-time selectors and removals on ShardedIndexFlat and
ShardedIndexIVFFlat must answer like the single-GPU index of the same kind holding the same rows,
ids and removals -- both exchange forms, gathered and per-rank results, the host-array entry point
with selectors, removals followed by more add_with_ids_local, and the plain indexes' selectors and
removals by global position. Prints SHARDED_IDS_NCCL_OK on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

I64_MAX = (1 << 63) - 1


def _check(got, ref, what, compare_topk, metric, exact_d=True):
    D, I = got
    Ds, Is = ref
    rep = compare_topk(D.cpu().numpy(), I.cpu().numpy(), Ds.cpu().numpy(), Is.cpu().numpy(), metric)
    assert rep["ok"], (what, rep)
    if exact_d:
        assert torch.equal(D, Ds), (what, "scores differ from the single index")


def _same_on_all_ranks(v):
    t = torch.tensor([v], dtype=torch.int64, device="cuda")
    out = torch.empty(dist.get_world_size(), dtype=torch.int64, device="cuda")
    dist.all_gather_into_tensor(out, t)
    assert (out == v).all(), ("ranks disagree", out.tolist())
    return v


def flat_checks(rank, world, nf, compare_topk):
    from newsrecommend_b200.sharded import ShardedIndexFlat, owned_rows, shard_range
    rng = np.random.default_rng(7)
    n1, n2, n3, d, nq, k = 30_001, 20_000, 5_001, 128, 2_001, 50
    x = rng.standard_normal((n1 + n2 + n3, d), dtype=np.float32)
    xq = rng.standard_normal((nq, d), dtype=np.float32)
    ids = (np.sort(rng.choice(1 << 45, x.shape[0], replace=False)) + (1 << 33)).astype(np.int64)
    xq_dev = torch.from_numpy(xq).cuda()
    xq_pin = torch.from_numpy(xq).pin_memory().numpy()
    window = nf.SearchParameters(sel=nf.IDSelectorRange(int(ids[int(0.9 * (n1 + n2))]), I64_MAX))
    block = nf.SearchParameters(sel=nf.IDSelectorNot(nf.IDSelectorBatch(ids[: n1 + n2][::50].copy())))
    for metric in (0, 1):
        for exchange in ("alltoall", "allgather"):
            idx = ShardedIndexFlat(d, metric, exchange=exchange, chunk_queries=1024)
            single = nf.IndexIDMap(nf.IndexFlat(d, metric))
            for a, b in ((0, n1), (n1, n1 + n2)):
                lo, hi = shard_range(b - a, world, rank)
                idx.add_with_ids_local(x[a + lo:a + hi], ids[a + lo:a + hi])
                single.add_with_ids(x[a:b], ids[a:b])
            assert _same_on_all_ranks(idx.ntotal) == n1 + n2
            for name, p in (("unfiltered", None), ("window", window), ("blocklist", block)):
                D, I = idx.search(xq_dev, k, params=p)
                _check((D, I), single.search(xq_dev, k, params=p), (metric, exchange, name), compare_topk, metric)
                Dr, Ir, spans = idx.search(xq_dev, k, gather=False, params=p)
                rows = np.concatenate([np.arange(a, b) for a, b in spans])
                assert spans == owned_rows(nq, world, rank, idx._chunk())
                assert torch.equal(Ir, I[torch.from_numpy(rows).cuda()])
                D_pin = torch.full((nq, k), float("nan"), dtype=torch.float32).pin_memory().numpy()
                I_pin = torch.full((nq, k), -7, dtype=torch.int64).pin_memory().numpy()
                assert idx.search_host(xq_pin, k, D_pin, I_pin, params=p) == spans
                assert np.array_equal(I_pin[rows], I.cpu().numpy()[rows])
                assert np.array_equal(D_pin[rows], D.cpu().numpy()[rows])
            # removals, then more rows
            for sel in (nf.IDSelectorRange(int(ids[100]), int(ids[5_000])), ids[20_000:40_000:3].copy()):
                assert _same_on_all_ranks(idx.remove_ids(sel)) == single.remove_ids(sel)
            lo, hi = shard_range(n3, world, rank)
            a = n1 + n2
            idx.add_with_ids_local(x[a + lo:a + hi], ids[a + lo:a + hi])
            single.add_with_ids(x[a:], ids[a:])
            assert _same_on_all_ranks(idx.ntotal) == single.ntotal
            for name, p in (("unfiltered", None), ("window", window)):
                _check(idx.search(xq_dev, k, params=p), single.search(xq_dev, k, params=p),
                       (metric, exchange, "after removal", name), compare_topk, metric)
        # plain index: selectors and removals by global row position
        idx = ShardedIndexFlat(d, metric, chunk_queries=1024)
        idx.add_global(x[:n1])
        single = nf.IndexFlat(d, metric)
        single.add(x[:n1])
        p = nf.SearchParameters(sel=nf.IDSelectorRange(n1 // 3, n1 - 100))
        _check(idx.search(xq_dev, k, params=p), single.search(xq_dev, k, params=p), (metric, "plain window"),
               compare_topk, metric)
        for sel in (nf.IDSelectorRange(1_000, 9_000), nf.IDSelectorNot(nf.IDSelectorRange(0, 25_000))):
            assert _same_on_all_ranks(idx.remove_ids(sel)) == single.remove_ids(sel)
        _check(idx.search(xq_dev, k), single.search(xq_dev, k), (metric, "plain after removal"), compare_topk, metric)
        _check(idx.search(xq_dev, k, params=p), single.search(xq_dev, k, params=p),
               (metric, "plain window after removal"), compare_topk, metric)


def ivf_checks(rank, world, nf, compare_topk):
    from newsrecommend_b200 import synth
    from newsrecommend_b200.sharded import ShardedIndexIVFFlat, shard_range
    nb, d, nq, k, nlist = 40_003, 128, 2_001, 50, 32
    xb, topics = synth.g_skew(nb, d, 7, return_topics=True)
    xq = synth.user_profiles(xb, topics, nq, 8)
    xq_dev = torch.from_numpy(xq).cuda()
    rng = np.random.default_rng(8)
    ids = rng.permutation(1 << 30)[:nb].astype(np.int64) * 1031 + (1 << 34)
    lo, hi = shard_range(nb, world, rank)
    for metric in (0, 1):
        single = nf.IndexIVFFlat(nf.IndexFlat(d, metric), d, nlist, metric)
        single.train(xb)
        idx = ShardedIndexIVFFlat(d, nlist, metric, chunk_queries=1024)
        idx.train_global(xb)  # gather mode: the single index's centroids, bit for bit
        assert np.array_equal(idx.quantizer.reconstruct_n(), single.quantizer.reconstruct_n())
        single.add_with_ids(xb, ids)
        idx.add_with_ids_local(xb[lo:hi], ids[lo:hi])
        sel = nf.IDSelectorNot(nf.IDSelectorBatch(ids[::13].copy()))
        for p in (None, nf.SearchParametersIVF(sel=sel), nf.SearchParametersIVF(sel=sel, nprobe=8)):
            idx.nprobe = single.nprobe = 2
            _check(idx.search(xq_dev, k, params=p), single.search(xq_dev, k, params=p), (metric, "ivf"), compare_topk,
                   metric, exact_d=False)
        assert _same_on_all_ranks(idx.remove_ids(ids[1::4].copy())) == single.remove_ids(ids[1::4].copy())
        _check(idx.search(xq_dev, k), single.search(xq_dev, k), (metric, "ivf after removal"), compare_topk, metric,
               exact_d=False)
        # plain: the stored ids are global positions and survive removal
        plain = ShardedIndexIVFFlat(d, nlist, metric, chunk_queries=1024)
        plain.train_global(xb)
        plain.add_global(xb)
        sp = nf.IndexIVFFlat(nf.IndexFlat(d, metric), d, nlist, metric)
        sp.train(xb)
        sp.add(xb)
        plain.nprobe = sp.nprobe = 4
        p = nf.SearchParametersIVF(sel=nf.IDSelectorRange(nb // 2, nb))
        _check(plain.search(xq_dev, k, params=p), sp.search(xq_dev, k, params=p), (metric, "plain ivf window"),
               compare_topk, metric, exact_d=False)
        assert _same_on_all_ranks(plain.remove_ids(nf.IDSelectorRange(0, nb // 3))) == \
            sp.remove_ids(nf.IDSelectorRange(0, nb // 3))
        _check(plain.search(xq_dev, k), sp.search(xq_dev, k), (metric, "plain ivf after removal"), compare_topk,
               metric, exact_d=False)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import newsrecommend_b200.faiss as nf
    from newsrecommend_b200.parity import compare_topk
    flat_checks(rank, world, nf, compare_topk)
    ivf_checks(rank, world, nf, compare_topk)
    dist.barrier()
    if rank == 0:
        print("SHARDED_IDS_NCCL_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
