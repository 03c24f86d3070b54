"""Search-time ID selectors on one B200 (SearchParameters(sel=...)). Writes profiles/filtered_bench.json
(or the path given) with the card name and power limit read in the same run:
  - config-1 flat (364,047 x 250, 50,000 CUDA-tensor queries, k = 50, IP and L2): IDSelectorRange keeping
    the newest 100 / 50 / 10 / 1 % and IDSelectorNot(IDSelectorBatch) of 1,000 ids. Selection plus
    compaction, the search of the compacted subset and the whole filtered call, beside the
    unfiltered search;
  - nq = 1 numpy latency (the masked single-call route) at 100 / 10 / 1 % against the unfiltered call;
  - IVF nlist 250, nprobe 16, IP: 250,000 queries and nq = 16, at 100 % and 10 %;
  - a parity sample of the filtered results against numpy brute force over the selected rows.

  python scripts/bench_filtered.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import newsrecommend_b200.faiss as nf  # noqa: E402
from newsrecommend_b200 import synth  # noqa: E402
from newsrecommend_b200.parity import compare_topk  # noqa: E402

NQ, K, D = 50_000, 50, 250
REPS = 5
FRACS = (1.0, 0.5, 0.1, 0.01)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, mhz = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=mhz)
    except Exception as e:  # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def med(fn, reps=REPS):
    ts = [host_ms(fn)[0] for _ in range(reps)]
    return float(np.median(ts)), [round(t, 3) for t in ts]


def brute(xq, xb, labels, k, metric):
    """fp64 top-k over the rows xb (labelled `labels`), ties by position."""
    sc = xq.astype(np.float64) @ xb.astype(np.float64).T
    if metric == nf.METRIC_L2:
        sc = (xq.astype(np.float64) ** 2).sum(1)[:, None] - 2 * sc + (xb.astype(np.float64) ** 2).sum(1)[None]
    o = np.argsort(-sc if metric == 0 else sc, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(sc, o, 1), labels[o]


def flat_part(xb, xb_d, xq, xq_d, n):
    out = {}
    rng = np.random.default_rng(7)
    block = rng.choice(n, 1000, replace=False).astype(np.int64)
    sels = {f"range_{int(f * 100)}pct": nf.IDSelectorRange(n - int(round(f * n)), n) for f in FRACS}
    sels["not_batch_1000"] = nf.IDSelectorNot(nf.IDSelectorBatch(block))
    for metric in (nf.METRIC_INNER_PRODUCT, nf.METRIC_L2):
        idx = nf.IndexFlat(D, metric)
        idx.add(xb_d)
        idx.search(xq_d, K)
        unf, unf_all = med(lambda: idx.search(xq_d, K))
        res = dict(unfiltered_ms=unf, unfiltered_ms_all=unf_all)
        for name, sel in sels.items():
            p = nf.SearchParameters(sel=sel)
            idx.search(xq_d, K, params=p)

            def compact():
                rows = nf._selected_rows(sel, None, n, xb_d.device)
                sub = nf._gather_packed(idx._xb, rows) if 0 < rows.shape[0] < n else None
                return rows, sub
            c_ms, c_all = med(compact)
            rows, packed = compact()
            kept = int(rows.shape[0])
            sub = idx
            if packed is not None:
                sub = nf.IndexFlat(D, metric)
                sub._xb = packed
            s_ms, s_all = med(lambda: sub.search(xq_d, K))
            t_ms, t_all = med(lambda: idx.search(xq_d, K, params=p))
            res[name] = dict(kept_rows=kept, select_compact_ms=c_ms, subset_search_ms=s_ms, filtered_total_ms=t_ms,
                             select_compact_ms_all=c_all, subset_search_ms_all=s_all, filtered_total_ms_all=t_all,
                             compaction_bytes=compaction_bytes(n, kept, idx._xb.kp) if packed is not None else 0)
        # parity sample: 10 % window and the blocklist, 64 queries, against numpy brute force
        par = {}
        for name in ("range_10pct", "not_batch_1000"):
            sel = sels[name]
            keep = np.arange(n) >= sel.imin if name == "range_10pct" else ~np.isin(np.arange(n), block)
            Dg, Ig = idx.search(xq[:64], K, params=nf.SearchParameters(sel=sel))
            Dt, It = brute(xq[:64], xb[keep], np.nonzero(keep)[0], K, metric)
            rep = compare_topk(Dg, Ig, Dt, It, metric)
            par[name] = dict(ok=bool(rep["ok"]), recall=float(rep.get("recall", float("nan"))))
        res["parity_sample"] = par
        out["ip" if metric == 0 else "l2"] = res
        del idx
        torch.cuda.empty_cache()
    return out


def compaction_bytes(n, nkeep, kp):
    """HBM bytes of selection + compaction from shapes: id_select writes member (8 B a row), the
    two-bucket counting sort reads member twice and writes order (8 + 8 + 4), the kept raw rows are
    gathered (read + write kp * 4) and re-packed as one add() (read d * 4; write raw, hi, lo at
    kp * 4, norms 4; the fp16 plane re-reads raw and writes kp * 2), and the labels are gathered."""
    return n * 28 + nkeep * (2 * kp * 4 + D * 4 + 3 * kp * 4 + 4 + kp * 4 + kp * 2 + 12)


def single_query_part(xb_d, xq, n):
    idx = nf.IndexFlatIP(D)
    idx.add(xb_d)
    q = xq[:1]
    res = {}
    for _ in range(20):
        idx.search(q, K)
    calls = 200

    def loop(p):
        def run():
            for i in range(calls):
                idx.search(xq[i:i + 1], K, params=p) if p is not None else idx.search(xq[i:i + 1], K)
        return run
    ms, all_ = med(loop(None))
    res["unfiltered_ms_per_call"] = ms / calls
    for f in (1.0, 0.1, 0.01):
        p = nf.SearchParameters(sel=nf.IDSelectorRange(n - int(round(f * n)), n))
        loop(p)()
        ms, all_ = med(loop(p))
        res[f"range_{int(f * 100)}pct_ms_per_call"] = ms / calls
    res["calls_per_timing"] = calls
    return res


def ivf_part(xb_d, xq_big_d, n):
    quant = nf.IndexFlatIP(D)
    ivf = nf.IndexIVFFlat(quant, D, 250, nf.METRIC_INNER_PRODUCT)
    ivf.train(xb_d)
    ivf.add(xb_d)
    ivf.nprobe = 16
    res = {}
    for nq in (xq_big_d.shape[0], 16):
        x = xq_big_d[:nq]
        ivf.search(x, K)
        unf, unf_all = med(lambda: ivf.search(x, K), 3)
        r = dict(unfiltered_ms=unf, unfiltered_ms_all=unf_all)
        for f in (1.0, 0.1):
            p = nf.SearchParametersIVF(sel=nf.IDSelectorRange(n - int(round(f * n)), n))
            ivf.search(x, K, params=p)
            ms, all_ = med(lambda: ivf.search(x, K, params=p), 3)
            r[f"range_{int(f * 100)}pct_ms"] = ms
            r[f"range_{int(f * 100)}pct_ms_all"] = all_
        res[f"nq_{nq}"] = r
    return res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "filtered_bench.json")
    torch.cuda.set_device(0)
    xb, topics = synth.g_skew(synth.N_ARTICLES, D, 42, return_topics=True)
    xq = synth.user_profiles(xb, topics, NQ, 43)
    n = xb.shape[0]
    xb_d, xq_d = torch.from_numpy(xb).cuda(), torch.from_numpy(xq).cuda()
    res = dict(bench="filtered", card=card(), catalog=[n, D], nq=NQ, k=K,
               timing="host clock around each call, ending in a device synchronise; median of the listed runs",
               selectors="positions on a plain IndexFlat; range_P = the newest P % of rows")
    res["flat_config1"] = flat_part(xb, xb_d, xq, xq_d, n)
    res["flat_nq1_numpy"] = single_query_part(xb_d, xq, n)
    big = synth.user_profiles(xb, topics, 250_000, 44)
    res["ivf_nlist250_nprobe16_ip"] = ivf_part(xb_d, torch.from_numpy(big).cuda(), n)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(card=res["card"], written=out_path)))


if __name__ == "__main__":
    main()
