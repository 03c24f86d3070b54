"""world_size-2 gloo tests (CPU) of the catalog-sharding host logic: row ranges, global ids, the
8-byte wire format, all-to-all by query range (and the all-gather form), chunking with per-chunk
ownership, the final gather, and the merge contract. The per-rank index and the codec are
injected (the oracle index and numpy pack / merge stand in for the CUDA kernels, which need a
GPU); the GPU suite covers the real kernels (tests/test_gpu_sharded.py) and bench.py --gpus N
asserts parity of the NCCL path on every run."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class NumpyCodec:
    """numpy restatement of nrb_pack_topk / nrb_merge_topk_packed (include/nrb200.h)."""

    @staticmethod
    def pack(D, I, id_base):
        d = np.ascontiguousarray(D.numpy(), dtype=np.float32).view(np.uint32).astype(np.uint64)
        i = I.numpy()
        lo = np.where(i < 0, 0xFFFFFFFF, i - id_base).astype(np.uint64)
        return torch.from_numpy(((d << np.uint64(32)) | lo).view(np.int64))

    @staticmethod
    def merge(P, bases, metric):
        P = P.numpy().view(np.uint64)
        G, nq, k = P.shape
        bases = bases.numpy()
        D = np.empty((nq, k), dtype=np.float32)
        I = np.empty((nq, k), dtype=np.int64)
        for q in range(nq):
            w = P[:, q, :]
            d = (w >> np.uint64(32)).astype(np.uint32).view(np.float32).reshape(G, k)
            lo = (w & np.uint64(0xFFFFFFFF)).astype(np.int64)
            ids = np.where(lo == 0xFFFFFFFF, -1, lo + bases[:, None])
            d, ids = d.reshape(-1), ids.reshape(-1)
            keep = ids >= 0
            d, ids = d[keep], ids[keep]
            o = np.argsort(-d if metric == 0 else d, kind="stable")[:k]
            D[q, :len(o)], I[q, :len(o)] = d[o], ids[o]
            D[q, len(o):], I[q, len(o):] = (np.float32(3.4028235e38) if metric else -np.float32(3.4028235e38)), -1
        return torch.from_numpy(D), torch.from_numpy(I)


def _worker(rank, world, port, metric, exchange, nb, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from newsrecommend_b200.sharded import ShardedIndexFlat, owned_rows, shard_range
        from oracle import faiss_oracle as fo
        rng = np.random.default_rng(0)
        xb = rng.standard_normal((nb, 24), dtype=np.float32)  # odd size: uneven shards
        xq = rng.standard_normal((37, 24), dtype=np.float32)
        # chunk_queries=16: three chunks (16, 16, 5 rows), the last one smaller than the world is wide
        idx = ShardedIndexFlat(24, metric, make_index=fo.IndexFlat, codec=NumpyCodec, exchange=exchange,
                               chunk_queries=16)
        idx.add_global(xb)
        lo, hi = shard_range(nb, world, rank)
        assert idx.id_base == lo and idx.local.ntotal == hi - lo and idx.ntotal == nb
        k = 10
        Do, Io = fo.knn(xq, xb, k, metric)
        D, I = idx.search(xq, k)  # gathered: every rank holds the full answer
        assert np.array_equal(I.numpy(), Io), "merged ids differ from the single-index answer"
        assert np.allclose(D.numpy(), Do, rtol=1e-5, atol=1e-5)
        Dr, Ir, spans = idx.search(xq, k, gather=False)  # only the rows this rank owns
        assert spans == owned_rows(37, world, rank, 16)
        rows = np.concatenate([np.arange(a, b) for a, b in spans]) if spans else np.empty(0, np.int64)
        assert np.array_equal(Ir.numpy(), Io[rows]) and np.allclose(Dr.numpy(), Do[rows], rtol=1e-5, atol=1e-5)
        # every query row is owned by exactly one rank
        own = torch.zeros(37, dtype=torch.int64)
        own[torch.from_numpy(rows)] += 1
        dist.all_reduce(own)
        assert bool((own == 1).all())
        # add_local: each rank passes only its rows
        idx2 = ShardedIndexFlat(24, metric, make_index=fo.IndexFlat, codec=NumpyCodec, exchange=exchange)
        idx2.add_local(xb[lo:hi], lo, nb)
        D2, I2 = idx2.search(xq, k)
        assert np.array_equal(I2.numpy(), Io)
        out.put((rank, True))
    except Exception as e:  # noqa: BLE001
        out.put((rank, repr(e)))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("metric,exchange,nb", [
    (0, "alltoall", 1001), (1, "alltoall", 1001), (0, "allgather", 1001), (1, "allgather", 1001),
    (0, "alltoall", 1), (1, "allgather", 1),  # nb = 1 < world: one shard is empty
])
def test_sharded_search_world2_gloo(metric, exchange, nb):
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, metric, exchange, nb, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
    res = sorted(out.get(timeout=5) for _ in range(2))
    assert res == [(0, True), (1, True)], res


def test_shard_range_covers_catalog():
    from newsrecommend_b200.sharded import shard_range
    for nb in (0, 1, 7, 9, 364047):
        for world in (1, 2, 3, 8):
            spans = [shard_range(nb, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == nb
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1  # balanced: no empty trailing shard while nb >= world


def test_chunk_ownership_partitions_the_batch():
    from newsrecommend_b200.sharded import chunk_slices, owned_rows
    for nq in (0, 1, 5, 37, 50_000):
        for world in (1, 2, 8):
            for chunk in (16, 18_944, 1 << 17):
                seen = np.zeros(nq, dtype=np.int64)
                for r in range(world):
                    for lo, hi in owned_rows(nq, world, r, chunk):
                        seen[lo:hi] += 1
                assert (seen == 1).all()
                assert sum(c1 - c0 for c0, c1, _ in chunk_slices(nq, world, chunk)) == nq


def _bench():
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_default_layout():
    """bench.py's default multi-GPU layout: shards of >= 180,000 rows, at least 2 per replica group, a
    divisor of the world size (config 1 -> groups of 2; a 10M-row catalog -> one group of N)."""
    bench = _bench()
    assert [bench.default_shards(w, 364_047) for w in (1, 2, 4, 8)] == [1, 2, 2, 2]
    assert [bench.default_shards(w, 10_000_000) for w in (1, 2, 4, 8)] == [1, 2, 4, 8]
    assert bench.default_shards(3, 364_047) == 1 and bench.default_shards(6, 364_047) == 2
    assert bench.default_shards(8, 1_000) == 2


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: float32 scores stay float32, int64 ids become float64 with the same
    values, one <name>.npy per array (per rank with N > 1)."""
    bench = _bench()
    D = np.arange(6, dtype=np.float32).reshape(2, 3) / 7
    I = np.array([[364_046, 0, -1], [5, 4, 3]], dtype=np.int64)
    bench.dump_outputs(str(tmp_path / "one"), {"D": D, "I": I})
    d, i = np.load(tmp_path / "one" / "D.npy"), np.load(tmp_path / "one" / "I.npy")
    assert d.dtype == np.float32 and np.array_equal(d, D)
    assert i.dtype == np.float64 and np.array_equal(i.astype(np.int64), I)
    bench.dump_outputs(str(tmp_path / "two"), {"D": D, "I": I, "query_rows": np.arange(2)}, rank=1, world=2)
    assert sorted(os.listdir(tmp_path / "two")) == ["D.rank1.npy", "I.rank1.npy", "query_rows.rank1.npy"]
