"""Worker of tests/test_gpu_sharded_exclude.py::test_sharded_exclude_nccl_torchrun (launched with
torchrun, one rank per GPU, NCCL): per-query exclusion lists on plain and id-carrying
ShardedIndexFlat and ShardedIndexIVFFlat must answer like the single-GPU index of the same kind with
the same rows, ids, lists and params -- both exchange forms, gathered and per-rank results, and the
host-array entry point. Prints SHARDED_EXCLUDE_NCCL_OK on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

I64_MAX = (1 << 63) - 1


def _lists(rng, nq, labels, top):
    """Each query's own top hits, random labels, -1 and absent ids, some empty lists, and one list
    longer than 128 - k (the long group)."""
    import exclude_oracle as xo
    lists = []
    for q in range(nq):
        if q % 4 == 0:
            lst = []
        elif q == 5:
            lst = labels[-100:]
        else:
            lst = np.concatenate([top[q, :6], rng.choice(labels, 12), [-1, labels.max() + 3]])
        lists.append(np.asarray(lst, dtype=np.int64))
    return xo.csr(lists)


def _check(got, ref, what, compare_topk, metric, ex):
    D, I = got
    Ds, Is = ref
    rep = compare_topk(D.cpu().numpy(), I.cpu().numpy(), Ds.cpu().numpy(), Is.cpu().numpy(), metric)
    assert rep["ok"], (what, rep)
    off, ids = ex
    Ih = I.cpu().numpy()
    for q in range(Ih.shape[0]):
        lst = ids[off[q]:off[q + 1]]
        assert not np.isin(Ih[q][Ih[q] >= 0], lst[lst >= 0]).any(), (what, q)


def _all_forms(idx, single, xq, k, p, ex, what, compare_topk, metric):
    """search (gather True / False, numpy and CUDA lists) and search_host, against the single index."""
    nq = xq.shape[0]
    ref = single.search(xq, k, params=p, exclude=ex)
    D, I = idx.search(xq, k, params=p, exclude=ex)
    _check((D, I), ref, what, compare_topk, metric, ex)
    ex_d = tuple(torch.from_numpy(a).cuda() for a in ex)
    D2, I2 = idx.search(xq, k, params=p, exclude=ex_d)
    assert torch.equal(D2, D) and torch.equal(I2, I), (what, "CUDA lists")
    Dr, Ir, spans = idx.search(xq, k, gather=False, params=p, exclude=ex)
    rows = np.concatenate([np.arange(a, b) for a, b in spans])
    assert torch.equal(Ir, I[torch.from_numpy(rows).cuda()]), what
    xq_pin = torch.from_numpy(xq.cpu().numpy()).pin_memory().numpy()
    D_pin = torch.full((nq, k), float("nan"), dtype=torch.float32).pin_memory().numpy()
    I_pin = torch.full((nq, k), -7, dtype=torch.int64).pin_memory().numpy()
    assert idx.search_host(xq_pin, k, D_pin, I_pin, params=p, exclude=ex) == spans
    assert np.array_equal(I_pin[rows], I.cpu().numpy()[rows]), (what, "search_host")
    assert np.array_equal(D_pin[rows], D.cpu().numpy()[rows]), (what, "search_host")


def flat_checks(rank, world, nf, compare_topk):
    from newsrecommend_b200.sharded import ShardedIndexFlat, shard_range
    rng = np.random.default_rng(17)
    nb, d, nq, k = 40_001, 128, 2_001, 50
    x = rng.standard_normal((nb, d), dtype=np.float32)
    xq = torch.from_numpy(rng.standard_normal((nq, d), dtype=np.float32)).cuda()
    ids = (np.sort(rng.choice(1 << 45, nb, replace=False)) + (1 << 33)).astype(np.int64)
    lo, hi = shard_range(nb, world, rank)
    for metric in (0, 1):
        for exchange in ("alltoall", "allgather"):
            for with_ids in (False, True):
                idx = ShardedIndexFlat(d, metric, exchange=exchange, chunk_queries=512)
                if with_ids:
                    idx.add_with_ids_local(x[lo:hi], ids[lo:hi])
                    single = nf.IndexIDMap(nf.IndexFlat(d, metric))
                    single.add_with_ids(x, ids)
                    labels = ids
                else:
                    idx.add_global(x)
                    single = nf.IndexFlat(d, metric)
                    single.add(x)
                    labels = np.arange(nb, dtype=np.int64)
                ex = _lists(rng, nq, labels, single.search(xq, 10)[1].cpu().numpy())
                window = nf.SearchParameters(sel=nf.IDSelectorRange(int(labels[nb // 2]), I64_MAX))
                for name, p in (("lists", None), ("window", window)):
                    _all_forms(idx, single, xq, k, p, ex, (metric, exchange, with_ids, name), compare_topk, metric)
                gone = labels[7::9].copy()
                assert idx.remove_ids(gone) == single.remove_ids(gone)
                if not with_ids:
                    labels = np.arange(single.ntotal, dtype=np.int64)
                    ex = _lists(rng, nq, labels, single.search(xq, 10)[1].cpu().numpy())
                _all_forms(idx, single, xq, k, None, ex, (metric, exchange, with_ids, "after removal"), compare_topk,
                           metric)


def ivf_checks(rank, world, nf, compare_topk):
    from newsrecommend_b200 import synth
    from newsrecommend_b200.sharded import ShardedIndexIVFFlat, shard_range
    nb, d, nq, k, nlist = 40_003, 128, 2_001, 50, 32
    xb, topics = synth.g_skew(nb, d, 7, return_topics=True)
    xq = torch.from_numpy(synth.user_profiles(xb, topics, nq, 8)).cuda()
    rng = np.random.default_rng(18)
    ids = rng.permutation(1 << 30)[:nb].astype(np.int64) * 1031 + (1 << 34)
    lo, hi = shard_range(nb, world, rank)
    for metric in (0, 1):
        for with_ids in (False, True):
            single = nf.IndexIVFFlat(nf.IndexFlat(d, metric), d, nlist, metric)
            single.train(xb)
            idx = ShardedIndexIVFFlat(d, nlist, metric, exchange="alltoall" if metric else "allgather",
                                      chunk_queries=512)
            idx.train_global(xb)
            if with_ids:
                single.add_with_ids(xb, ids)
                idx.add_with_ids_local(xb[lo:hi], ids[lo:hi])
                labels = ids
            else:
                single.add(xb)
                idx.add_global(xb)
                labels = np.arange(nb, dtype=np.int64)
            idx.nprobe = single.nprobe = 4
            ex = _lists(rng, nq, labels, single.search(xq, 10)[1].cpu().numpy())
            sel = nf.IDSelectorNot(nf.IDSelectorBatch(labels[::13].copy()))
            for name, p in (("lists", None), ("blocklist", nf.SearchParametersIVF(sel=sel, nprobe=8))):
                _all_forms(idx, single, xq, k, p, ex, ("ivf", metric, with_ids, name), compare_topk, metric)
            gone = labels[1::4].copy()
            assert idx.remove_ids(gone) == single.remove_ids(gone)
            _all_forms(idx, single, xq, k, None, ex, ("ivf", metric, with_ids, "after removal"), compare_topk, metric)


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
        print("SHARDED_EXCLUDE_NCCL_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
