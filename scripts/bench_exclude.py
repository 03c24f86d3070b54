"""Per-query exclusion lists on one B200 (search(..., exclude=(offsets, ids))) with the synthetic click
histories. Writes profiles/exclude_bench.json (or the path given) with the card name and power limit
read in the same run. Device-resident inputs, CUDA-event timing, plain and excluded calls alternated:
  - config-1 flat IP (364,047 x 250, 50,000 users, k = 50), and the same catalog behind IndexIDMap;
  - config-2 IVF (nlist 250, nprobe 16, IP, 250,000 users, k = 50);
  - per group: query count and k'; the time of nrb_exclude_topk alone on the group's over-fetched
    result; nrb_fallback_query_count of a plain search at k' against k = 50 (the fp16 filter's margin
    slots shrink as k' approaches 112);
  - the share of plain top-50 slots that held an article the user had clicked, over all users.

  python scripts/bench_exclude.py [out.json]
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import newsrecommend_b200.faiss as nf  # noqa: E402
from newsrecommend_b200 import _lib, synth  # noqa: E402

K, D = 50, 250
REPS = 7


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, mhz = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=mhz)
    except Exception as e:  # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def event_ms(fn, launches=1):
    """Device time of `launches` calls of fn between two CUDA events, per call."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(launches):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / launches


def alternate(plain, excluded, reps=REPS):
    """Both calls warmed up, then timed in turn: medians and every run."""
    plain()
    excluded()
    tp, te = [], []
    for _ in range(reps):
        tp.append(event_ms(plain))
        te.append(event_ms(excluded))
    return dict(plain_ms=float(np.median(tp)), excluded_ms=float(np.median(te)),
                plain_ms_all=[round(t, 3) for t in tp], excluded_ms_all=[round(t, 3) for t in te])


def groups(off, k):
    need = k + np.diff(off)
    out = {}
    for name, m in (("filter", need <= 112), ("wide", (need > 112) & (need <= _lib.MAX_K)), ("long", need > _lib.MAX_K)):
        rows = np.nonzero(m)[0]
        out[name] = dict(nq=int(rows.size), k_prime=int(need[rows].max()) if rows.size and name != "long" else None,
                         rows=rows)
    return out


def kernel_part(search, x_d, off, off_d, ids_d, grp, metric):
    """nrb_exclude_topk alone on each group's over-fetched result, and the filter fallbacks at k'."""
    res = {}
    nq = x_d.shape[0]
    Dout = torch.empty((nq, K), dtype=torch.float32, device=x_d.device)
    Iout = torch.empty((nq, K), dtype=torch.int64, device=x_d.device)
    for name in ("filter", "wide"):
        g = grp[name]
        if not g["nq"]:
            continue
        rows = torch.from_numpy(g["rows"].astype(np.int64)).to(x_d.device)
        xg = x_d.index_select(0, rows)
        kq = g["k_prime"]
        f0 = _lib.lib.nrb_fallback_query_count()
        Dg, Ig = search(xg, kq)
        torch.cuda.synchronize()
        f1 = _lib.lib.nrb_fallback_query_count()
        search(xg, K)
        torch.cuda.synchronize()
        f2 = _lib.lib.nrb_fallback_query_count()
        st = torch.cuda.current_stream().cuda_stream

        def run():
            nf.check(_lib.lib.nrb_exclude_topk(Dg.data_ptr(), Ig.data_ptr(), g["nq"], kq, rows.data_ptr(),
                                               off_d.data_ptr(), ids_d.data_ptr(), metric, K, Dout.data_ptr(),
                                               Iout.data_ptr(), st), "exclude_topk")
        run()
        res[name] = dict(nq=g["nq"], k_prime=kq, exclude_kernel_ms=event_ms(run, 50),
                         fallback_queries_at_k_prime=int(f1 - f0), fallback_queries_at_k50=int(f2 - f1),
                         group_search_at_k_prime_ms=event_ms(lambda: search(xg, kq)),
                         group_search_at_k50_ms=event_ms(lambda: search(xg, K)))
    res["long"] = dict(nq=grp["long"]["nq"])
    return res


def clicked_share(I, off, clicks, n):
    """Share of the top-k slots holding a row the user clicked."""
    owner = np.repeat(np.arange(off.size - 1), np.diff(off))
    ret = I.astype(np.int64) + np.arange(I.shape[0])[:, None] * np.int64(n)
    hit = np.isin(ret, np.unique(clicks + owner * np.int64(n)))
    return dict(share_of_slots=float(hit.mean()), users_with_a_clicked_slot=float(hit.any(1).mean()),
                mean_clicked_slots_per_user=float(hit.sum(1).mean()))


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "exclude_bench.json")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    xb, topics = synth.g_skew(synth.N_ARTICLES, D, 42, return_topics=True)
    n = xb.shape[0]
    xq, (off, clicks) = synth.user_profiles(xb, topics, synth.N_TEST_USERS, 43, return_clicks=True)
    xb_d, xq_d = torch.from_numpy(xb).to(dev), torch.from_numpy(xq).to(dev)
    off_d, clicks_d = torch.from_numpy(off).to(dev), torch.from_numpy(clicks).to(dev)
    res = dict(bench="exclude", card=card(), catalog=[n, D], k=K,
               timing="CUDA events around each call (device-resident queries, lists and results); median of the "
                      "listed runs, plain and excluded calls alternated",
               lists="synth.user_profiles(..., return_clicks=True): each user's clicked rows, duplicates kept")
    # config 1, flat IP
    flat = nf.IndexFlatIP(D)
    flat.add(xb_d)
    grp = groups(off, K)
    r = dict(nq=int(xq.shape[0]), list_len_mean=float(np.diff(off).mean()), list_len_max=int(np.diff(off).max()),
             groups={k: dict(nq=v["nq"], k_prime=v["k_prime"]) for k, v in grp.items()})
    r.update(alternate(lambda: flat.search(xq_d, K), lambda: flat.search(xq_d, K, exclude=(off_d, clicks_d))))
    r["kernel"] = kernel_part(lambda x, k: flat.search(x, k), xq_d, off, off_d, clicks_d, grp, 0)
    _, I = flat.search(xq_d, K)
    r["plain_top50_clicked"] = clicked_share(I.cpu().numpy(), off, clicks, n)
    _, Ix = flat.search(xq_d, K, exclude=(off_d, clicks_d))
    r["excluded_top50_clicked"] = clicked_share(Ix.cpu().numpy(), off, clicks, n)
    res["flat_config1_ip"] = r
    # the same catalog behind IndexIDMap (ids >= 2^32), lists of external ids
    ext = torch.arange(n, dtype=torch.int64, device=dev) * 3 + 2 ** 33
    m = nf.IndexIDMap(nf.IndexFlatIP(D))
    m.add_with_ids(xb_d, ext)
    clicks_ext = ext[clicks_d]
    res["idmap_config1_ip"] = alternate(lambda: m.search(xq_d, K), lambda: m.search(xq_d, K, exclude=(off_d, clicks_ext)))
    del flat, m
    torch.cuda.empty_cache()
    # config 2, IVF
    big, (boff, bclicks) = synth.user_profiles(xb, topics, 250_000, 44, return_clicks=True)
    big_d, boff_d, bclicks_d = (torch.from_numpy(a).to(dev) for a in (big, boff, bclicks))
    ivf = nf.IndexIVFFlat(nf.IndexFlatIP(D), D, 250, nf.METRIC_INNER_PRODUCT)
    ivf.train(xb_d)
    ivf.add(xb_d)
    ivf.nprobe = 16
    bgrp = groups(boff, K)
    r = dict(nq=int(big.shape[0]), nlist=250, nprobe=16,
             groups={k: dict(nq=v["nq"], k_prime=v["k_prime"]) for k, v in bgrp.items()})
    r.update(alternate(lambda: ivf.search(big_d, K), lambda: ivf.search(big_d, K, exclude=(boff_d, bclicks_d)), 5))
    r["kernel"] = kernel_part(lambda x, k: ivf.search(x, k), big_d, boff, boff_d, bclicks_d, bgrp, 0)
    _, I = ivf.search(big_d, K)
    r["plain_top50_clicked"] = clicked_share(I.cpu().numpy(), boff, bclicks, n)
    res["ivf_config2_ip"] = r
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(card=res["card"], written=out_path,
                          flat=[res["flat_config1_ip"]["plain_ms"], res["flat_config1_ip"]["excluded_ms"]],
                          idmap=[res["idmap_config1_ip"]["plain_ms"], res["idmap_config1_ip"]["excluded_ms"]],
                          ivf=[res["ivf_config2_ip"]["plain_ms"], res["ivf_config2_ip"]["excluded_ms"]])))


if __name__ == "__main__":
    main()
