"""Per-query exclusion lists on the sharded indexes (search(..., exclude=(offsets, ids))) with the
synthetic click histories, under torchrun with the catalog sharded over the N ranks. Writes
profiles/sharded_exclude_bench.json (or the path given) from rank 0, with every rank's card name and
power limit read in the same run. Device-resident queries and lists, CUDA-event timing, plain and
excluded calls alternated (medians and every run):
  - config-1 flat IP (364,047 x 250, 50,000 users, k = 50) on ShardedIndexFlat, plain and
    id-carrying (ids >= 2^33);
  - config-2 IVF (nlist 250, nprobe 16, IP, 250,000 users) on plain ShardedIndexIVFFlat;
  - per rank: the localized lists' groups (query count and k' of the k + E <= 112 filter group, the
    112 < k + E <= 128 group, and the count of longer lists), the localization time (list check,
    membership, compaction, offsets to the host), nrb_fallback_query_count of one plain and one
    excluded call;
  - per rank, the localization A/B: the rank's local searches over the whole batch driven by the
    localized lists against the same searches driven by the whole lists shifted into the rank's
    label space (correct too, since entries of other shards match no local row; it only over-fetches
    more);
  - full size: no returned article is in the user's history, and a 4,096-query sample of the flat
    result matches the oracle.

  torchrun --nproc-per-node N scripts/bench_sharded_exclude.py [out.json]
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from bench_exclude import card, clicked_share, event_ms  # noqa: E402
from newsrecommend_b200 import _lib, synth  # noqa: E402
from newsrecommend_b200.sharded import (ShardedIndexFlat, ShardedIndexIVFFlat, chunk_lists,  # noqa: E402
                                        chunk_slices)

K, D = 50, 250


def alternate(plain, excluded, reps):
    plain()
    excluded()
    tp, te = [], []
    for _ in range(reps):
        dist.barrier()
        tp.append(event_ms(plain))
        dist.barrier()
        te.append(event_ms(excluded))
    return dict(plain_ms=float(np.median(tp)), excluded_ms=float(np.median(te)),
                plain_ms_all=[round(t, 3) for t in tp], excluded_ms_all=[round(t, 3) for t in te])


def groups(loc_off):
    need = K + np.diff(loc_off)
    out = {}
    for name, m in (("filter", need <= 112), ("wide", (need > 112) & (need <= _lib.MAX_K))):
        out[name] = dict(nq=int(m.sum()), k_prime=int(need[m].max()) if m.any() else None)
    out["long"] = dict(nq=int((need > _lib.MAX_K).sum()))
    out["list_len_max"] = int(np.diff(loc_off).max()) if loc_off.size > 1 else 0
    return out


def fallbacks(fn):
    torch.cuda.synchronize()
    f0 = _lib.lib.nrb_fallback_query_count()
    fn()
    torch.cuda.synchronize()
    return int(_lib.lib.nrb_fallback_query_count() - f0)


def per_rank(idx, xq_d, ex, whole_local, reps):
    """The rank's localization cost, groups, fallbacks and the localization A/B of its local searches."""
    nq = xq_d.shape[0]
    lists = idx._localize(ex, nq)
    loc_ms = [event_ms(lambda: idx._localize(ex, nq)) for _ in range(reps)]
    chunk = idx._chunk()
    lp = idx._local_params(None)

    def local_pass(l):
        for c0, c1, _ in chunk_slices(nq, idx.world, chunk):
            idx.search_local(xq_d[c0:c1], K, lp, chunk_lists(l, c0, c1))

    tl, tw = [], []
    local_pass(lists)
    local_pass(whole_local)
    for _ in range(reps):
        tl.append(event_ms(lambda: local_pass(lists)))
        tw.append(event_ms(lambda: local_pass(whole_local)))
    ab = dict(localized_ms=float(np.median(tl)), whole_shifted_ms=float(np.median(tw)),
              localized_ms_all=[round(t, 3) for t in tl], whole_shifted_ms_all=[round(t, 3) for t in tw],
              whole_shifted_groups=groups(whole_local[0]),
              fallback_queries_localized=fallbacks(lambda: local_pass(lists)),
              fallback_queries_whole_shifted=fallbacks(lambda: local_pass(whole_local)))
    return dict(rank=idx.rank, local_rows=int(idx.local.ntotal), groups=groups(lists[0]),
                localize_ms=float(np.median(loc_ms)), localize_ms_all=[round(t, 3) for t in loc_ms],
                fallback_queries_plain=fallbacks(lambda: idx.search(xq_d, K)),
                fallback_queries_excluded=fallbacks(lambda: idx.search(xq_d, K, exclude=ex)),
                localization_ab=ab)


def gathered(obj):
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, obj)
    return out


def no_clicked(I, off, clicks, n):
    """True when no returned row (I: catalog rows, -1 padding) is in its user's click history."""
    owner = np.repeat(np.arange(off.size - 1), np.diff(off))
    ret = np.where(I >= 0, I.astype(np.int64) + np.arange(I.shape[0])[:, None] * np.int64(n), -1)
    return bool(not np.isin(ret, clicks + owner * np.int64(n)).any())


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "sharded_exclude_bench.json")
    xb, topics = synth.g_skew(synth.N_ARTICLES, D, 42, return_topics=True)
    n = xb.shape[0]
    xq, (off, clicks) = synth.user_profiles(xb, topics, synth.N_TEST_USERS, 43, return_clicks=True)
    xq_d = torch.from_numpy(xq).to(dev)
    off_d, clicks_d = torch.from_numpy(off).to(dev), torch.from_numpy(clicks).to(dev)
    res = dict(bench="sharded_exclude", world=world, cards=gathered(card()), catalog=[n, D], k=K,
               timing="CUDA events around each call on every rank (device-resident queries and lists); median of "
                      "the listed runs, plain and excluded calls alternated; the tables report rank 0's call times",
               lists="synth.user_profiles(..., return_clicks=True): each user's clicked rows, duplicates kept",
               list_len_mean=float(np.diff(off).mean()), list_len_max=int(np.diff(off).max()))
    # config 1, flat IP, plain: labels are global row positions
    flat = ShardedIndexFlat(D, 0)
    flat.add_global(xb)
    ex = (off_d, clicks_d)
    r = alternate(lambda: flat.search(xq_d, K), lambda: flat.search(xq_d, K, exclude=ex), 7)
    r["ranks"] = gathered(per_rank(flat, xq_d, ex, (off, clicks_d - flat.id_base), 5))
    Dd, I = flat.search(xq_d, K, exclude=ex)
    Ih = I.cpu().numpy()
    r["no_clicked_article_returned"] = no_clicked(Ih, off, clicks, n)
    if rank == 0:
        from newsrecommend_b200.parity import compare_topk
        from oracle import faiss_oracle as fo
        import exclude_oracle as xo
        fo.build()
        sample = np.random.default_rng(5).choice(xq.shape[0], 4096, replace=False)
        so = np.zeros(sample.size + 1, np.int64)
        np.cumsum(np.diff(off)[sample], out=so[1:])
        sids = np.concatenate([clicks[off[u]:off[u + 1]] for u in sample])
        Do, Io = fo.knn_fast(xq[sample], xb, K + int(np.diff(off).max()), 0)
        Dx, Ix = xo.exclude_topk(Do, Io, None, so, sids, 0, K, np.empty((sample.size, K), np.float32),
                                 np.empty((sample.size, K), np.int64))
        rep = compare_topk(Dd.cpu().numpy()[sample], Ih[sample], Dx, Ix, 0)
        r["oracle_sample_4096"] = dict(ok=bool(rep["ok"]), **{k: v for k, v in rep.items() if k != "ok"
                                                               and isinstance(v, (int, float, bool))})
        r["plain_top50_clicked"] = clicked_share(flat.search(xq_d, K)[1].cpu().numpy(), off, clicks, n)
    res["flat_config1_ip"] = r
    del flat
    # the same catalog id-carrying: lists of external ids
    ext = np.arange(n, dtype=np.int64) * 3 + 2 ** 33
    m = ShardedIndexFlat(D, 0)
    m.add_with_ids(xb, ext)
    clicks_ext = torch.from_numpy(ext).to(dev)[clicks_d]
    exm = (off_d, clicks_ext)
    r = alternate(lambda: m.search(xq_d, K), lambda: m.search(xq_d, K, exclude=exm), 7)
    r["ranks"] = gathered(per_rank(m, xq_d, exm, (off, clicks_ext), 5))
    _, I = m.search(xq_d, K, exclude=exm)
    Im = I.cpu().numpy()
    r["no_clicked_article_returned"] = no_clicked(np.where(Im >= 0, (Im - 2 ** 33) // 3, -1), off, clicks, n)
    res["idmap_config1_ip"] = r
    del m
    torch.cuda.empty_cache()
    # config 2, IVF (plain: stored global positions)
    big, (boff, bclicks) = synth.user_profiles(xb, topics, 250_000, 44, return_clicks=True)
    big_d, boff_d, bclicks_d = (torch.from_numpy(a).to(dev) for a in (big, boff, bclicks))
    ivf = ShardedIndexIVFFlat(D, 250, 0)
    ivf.train_global(xb)
    ivf.add_global(xb)
    ivf.nprobe = 16
    exb = (boff_d, bclicks_d)
    r = dict(nq=int(big.shape[0]), nlist=250, nprobe=16)
    r.update(alternate(lambda: ivf.search(big_d, K), lambda: ivf.search(big_d, K, exclude=exb), 5))
    r["ranks"] = gathered(per_rank(ivf, big_d, exb, (boff, bclicks_d - ivf.id_base), 3))
    _, I = ivf.search(big_d, K, exclude=exb)
    r["no_clicked_article_returned"] = no_clicked(I.cpu().numpy(), boff, bclicks, n)
    res["ivf_config2_ip"] = r
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(dict(world=world, card=res["cards"][0], written=out_path,
                              **{w: [res[w]["plain_ms"], res[w]["excluded_ms"], res[w]["no_clicked_article_returned"]]
                                 for w in ("flat_config1_ip", "idmap_config1_ip", "ivf_config2_ip")})))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
