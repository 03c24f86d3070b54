"""External ids, selectors and removal on the sharded flat index, against the plain sharded index, in
the same run. Every rank generates ITS catalog rows on its GPU (seeded per 1M-row chunk, as
scripts/bench_config5.py does, so the catalog does not depend on N) and the full query batch.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
      --master-port P scripts/bench_sharded_ids.py --config 1|5 [--steps 2] [--out path]

Per step, plain and id-carrying alternated: the unfiltered search, the newest-10 % window, a
1,000-id blocklist, remove_ids of 1 % of the catalog and add_with_ids_local of 1 % new rows (the
plain index cannot take more rows, so its add is not timed). Times are the max over ranks of a
host clock around work that ends in a device synchronise, median over steps. Parity: a query
sample of every search is checked on rank 0 against the single IndexIDMap over the whole
catalog when it fits one GPU (config 1). The record, with the card name and power limit read in
the same run, is merged into profiles/sharded_ids_bench.json under "config<c>_n<N>"."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import numpy as np
import torch
import torch.distributed as dist

CONFIGS = {1: dict(nb=364_047, d=250, nq=50_000, k=50), 5: dict(nb=10_000_000, d=256, nq=1_000_000, k=100)}
CH = 1_000_000


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, mhz = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=mhz)
    except Exception as e:  # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def rows(lo, hi, d, model, dev):
    """Catalog rows [lo, hi): chunk c of CH rows always comes from seed 1000 + c, whatever the sharding."""
    from bench_config5 import gen_rows
    out = [torch.empty((0, d), device=dev)]
    for c in range(lo // CH, -(-hi // CH)):
        full = gen_rows(CH, 1000 + c, model, dev)
        out.append(full[max(lo - c * CH, 0):min(hi - c * CH, CH), :d])
    return torch.cat(out).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS))
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--nq", type=int, default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sharded_ids_bench.json"))
    args = ap.parse_args()
    world, rank, local = (int(os.environ.get(v, dflt)) for v, dflt in (("WORLD_SIZE", 1), ("RANK", 0), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import newsrecommend_b200.faiss as nf
    from bench_config5 import topic_model
    from newsrecommend_b200.parity import compare_topk
    from newsrecommend_b200.sharded import ShardedIndexFlat, shard_range
    cfg = dict(CONFIGS[args.config])
    nb, d, k = cfg["nb"], cfg["d"], cfg["k"]
    nq = args.nq or cfg["nq"]
    model = topic_model(dev)
    lo, hi = shard_range(nb, world, rank)
    x = rows(lo, hi, d, model, dev)
    xq = torch.randn((nq, d), generator=torch.Generator(device=dev).manual_seed(7), device=dev)
    ids_all = np.arange(nb, dtype=np.int64) * 3 + (1 << 33)  # publication order, beyond 32 bits
    ids = torch.from_numpy(ids_all[lo:hi]).to(dev)
    plain = ShardedIndexFlat(d, 0)
    plain.add_local(x, lo, nb)
    withids = ShardedIndexFlat(d, 0)
    withids.add_with_ids_local(x, ids)
    rng = np.random.default_rng(11)
    window_p = nf.SearchParameters(sel=nf.IDSelectorRange(int(ids_all[int(0.9 * nb)]), 1 << 62))
    window_plain = nf.SearchParameters(sel=nf.IDSelectorRange(int(0.9 * nb), nb))
    blk = np.sort(rng.choice(nb, 1000, replace=False))
    block_p = nf.SearchParameters(sel=nf.IDSelectorNot(nf.IDSelectorBatch(ids_all[blk])))
    block_plain = nf.SearchParameters(sel=nf.IDSelectorNot(nf.IDSelectorBatch(blk)))
    single = None
    if args.config == 1 and rank == 0:
        single = nf.IndexIDMap(nf.IndexFlat(d, 0))
        single.add_with_ids(rows(0, nb, d, model, dev), torch.from_numpy(ids_all).to(dev))
    sample = torch.arange(0, nq, max(1, nq // 512), device=dev)

    def timed(fn):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ms = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), out

    times = {}
    parity = {}

    def record(name, ms):
        times.setdefault(name, []).append(ms)

    for step in range(args.steps + 1):  # step 0 warms every shape up and is not recorded
        keep = step > 0
        for name, idx, p in (("search_plain", plain, None), ("search_ids", withids, None),
                             ("window10_plain", plain, window_plain), ("window10_ids", withids, window_p),
                             ("blocklist_plain", plain, block_plain), ("blocklist_ids", withids, block_p)):
            ms, (D, I) = timed(lambda: idx.search(xq, k, params=p))
            if keep:
                record(name, ms)
            if single is not None and name.endswith("_ids") and step == 1:
                Ds, Is = single.search(xq[sample], k, params=p)
                rep = compare_topk(D[sample].cpu().numpy(), I[sample].cpu().numpy(), Ds.cpu().numpy(),
                                   Is.cpu().numpy(), 0)
                parity[name] = dict(ok=bool(rep["ok"]), queries=int(sample.numel()))
                assert rep["ok"], (name, rep)
            del D, I
        # remove 1 % of the catalog (every 100th live id, drawn from this step's id range)
        gone = ids_all[step::100].copy()
        ms, r = timed(lambda: withids.remove_ids(gone))
        if keep:
            record("remove1pct_ids", ms)
        ms, _ = timed(lambda: plain.remove_ids(nf.IDSelectorRange(0, nb // 100)))
        if keep:
            record("remove1pct_plain", ms)
        # add 1 % new rows with fresh ids on every rank
        n_new = (nb // 100) * (rank + 1) // world - (nb // 100) * rank // world
        xn = rows(lo, lo + n_new, d, model, dev) * 0.5
        new_ids = torch.arange(n_new, device=dev, dtype=torch.int64) + (1 << 50) + step * nb + lo
        ms, _ = timed(lambda: withids.add_with_ids_local(xn, new_ids))
        if keep:
            record("add1pct_ids", ms)
        if single is not None:
            single.remove_ids(gone)
            xs = torch.cat([rows(shard_range(nb, world, r)[0], shard_range(nb, world, r)[0] +
                                 (nb // 100) * (r + 1) // world - (nb // 100) * r // world, d, model, dev)
                            for r in range(world)]) * 0.5
            ids_s = torch.cat([torch.arange((nb // 100) * (r + 1) // world - (nb // 100) * r // world, device=dev,
                                            dtype=torch.int64) + (1 << 50) + step * nb + shard_range(nb, world, r)[0]
                               for r in range(world)])
            single.add_with_ids(xs, ids_s)
    med = {n: float(np.median(v)) for n, v in times.items()}
    res = dict(config=args.config, n_gpus=world, nb=nb, d=d, nq=nq, k=k, metric="IP", steps=args.steps,
               exchange=plain.exchange_mode, card=card(), ms_median=med, ms_all=times, parity=parity or "not run",
               id_overhead_ms=med["search_ids"] - med["search_plain"],
               wire_bytes_per_search=dict(plain=nq * k * 8 * world, ids=nq * k * 16 * world))
    if rank == 0:
        path = args.out
        allres = json.load(open(path)) if os.path.exists(path) else {}
        allres[f"config{args.config}_n{world}"] = res
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            json.dump(allres, f, indent=1)
        print(json.dumps(dict(config=args.config, n_gpus=world, ms=med, parity=parity)))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
