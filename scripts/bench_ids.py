"""External ids on one B200: what IndexIDMap's label translation adds to the config-1 search, and
what remove_ids costs on the full catalog (flat by range and by batch, IVF nlist 250 plus the list
rebuild on the next search). Prints one JSON line with the card name and power limit.

  python scripts/bench_ids.py
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import newsrecommend_b200.faiss as nf  # noqa: E402
from newsrecommend_b200 import synth  # noqa: E402

HBM_TBPS = 7.7  # HGX B200 data sheet, one GPU
NQ, K, D = 50_000, 50, 250
REPS = 10


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, mhz = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=mhz)
    except Exception as e:  # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def removal_bytes(n, nkeep, kp, idmap):
    """HBM bytes the removal moves, from shapes: id_select reads the ids and writes member (8 + 8 B
    a row; rows are positions for a plain IndexFlat), the two-bucket counting sort reads member
    twice and writes order (8 + 8 + 4), the survivors' raw rows are gathered (read + write kp * 4
    each) and re-packed (read d * 4; write raw, hi, lo at kp * 4, norms 4, fp16 plane kp * 2 after
    re-reading raw), and the id map is gathered (read order 4 + id 8, write 8)."""
    b = n * (16 if idmap else 8) + n * 20
    b += nkeep * (2 * kp * 4 + D * 4 + 3 * kp * 4 + 4 + kp * 4 + kp * 2)
    if idmap:
        b += nkeep * 20
    return b


def main():
    torch.cuda.set_device(0)
    xb, topics = synth.g_skew(synth.N_ARTICLES, D, 42, return_topics=True)
    xq = synth.user_profiles(xb, topics, NQ, 43)
    n = xb.shape[0]
    ids = 100_000 + np.arange(n, dtype=np.int64) * 3  # synthetic article ids in publication order
    xb_d, xq_d = torch.from_numpy(xb).cuda(), torch.from_numpy(xq).cuda()
    res = dict(bench="ids", card=card(), catalog=[n, D], nq=NQ, k=K)

    # --- config-1 search: plain IndexFlatIP vs IndexIDMap over the same rows, alternating
    plain = nf.IndexFlatIP(D)
    plain.add(xb_d)
    m = nf.IndexIDMap(nf.IndexFlatIP(D))
    m.add_with_ids(xb_d, ids)
    for f in (plain, m):
        f.search(xq_d, K)
        f.search(xq, K)
    t = {"plain_dev": [], "idmap_dev": [], "plain_host": [], "idmap_host": []}
    same = True
    for _ in range(REPS):
        ms, (Dp, Ip) = event_ms(lambda: plain.search(xq_d, K))
        t["plain_dev"].append(ms)
        ms, (Dm, Im) = event_ms(lambda: m.search(xq_d, K))
        t["idmap_dev"].append(ms)
        same &= bool(torch.equal(Dp, Dm)) and bool(torch.equal(torch.from_numpy(ids).cuda()[Ip], Im))
        t["plain_host"].append(host_ms(lambda: plain.search(xq, K))[0])
        t["idmap_host"].append(host_ms(lambda: m.search(xq, K))[0])
    med = {key: float(np.median(v)) for key, v in t.items()}
    lab0 = torch.empty(NQ * K, dtype=torch.int64, device="cuda").random_(0, n)  # row labels of one search
    lab = torch.empty_like(lab0)
    map_ms = []
    for _ in range(REPS):
        lab.copy_(lab0)  # the translation is in place: every timed call starts from row labels
        map_ms.append(event_ms(lambda: nf._map_ids(m.id_map, lab))[0])
    map_ms = np.median(map_ms)
    res["search"] = dict(
        ms_median=med, ms_all={key: [round(x, 3) for x in v] for key, v in t.items()},
        added_ms_device_tensors=med["idmap_dev"] - med["plain_dev"], added_ms_numpy=med["idmap_host"] - med["plain_host"],
        map_ids_kernel_ms=float(map_ms), map_ids_bytes=NQ * K * (8 + 8 + 8), same_D_and_translated_I=same)

    # --- remove_ids of 10 % of the catalog from an IndexIDMap (flat) by range and by batch
    cut = int(ids[n // 10])
    sels = {"range": lambda: nf.IDSelectorRange(0, cut), "batch": lambda: nf.IDSelectorBatch(ids[: n // 10])}
    rem = {}
    for name, mk in sels.items():
        ms = []
        for _ in range(5):
            mm = nf.IndexIDMap(nf.IndexFlatIP(D))
            mm.add_with_ids(xb_d, ids)
            sel = mk()
            t_ms, r = host_ms(lambda: mm.remove_ids(sel))
            assert r == n // 10
            ms.append(t_ms)
        by = removal_bytes(n, n - n // 10, 256, True)
        rem[name] = dict(ms_median=float(np.median(ms)), ms_all=[round(x, 3) for x in ms], removed=n // 10, bytes=by,
                         tb_per_s=by / (np.median(ms) * 1e-3) / 1e12,
                         frac_of_hbm_peak=by / (np.median(ms) * 1e-3) / 1e12 / HBM_TBPS)
    res["remove_idmap_flat_10pct"] = rem

    # --- IVF nlist 250: remove_ids by range, then the list rebuild the next search performs
    quant = nf.IndexFlatIP(D)
    ivf = nf.IndexIVFFlat(quant, D, 250, nf.METRIC_INNER_PRODUCT)
    ivf.train(xb_d)
    ivf.nprobe = 16
    rm, rb, srch = [], [], []
    for _ in range(5):
        ivf.reset()
        ivf.add_with_ids(xb_d, ids)
        ivf._build_lists()
        t_ms, r = host_ms(lambda: ivf.remove_ids(nf.IDSelectorRange(0, cut)))
        assert r == n // 10
        rm.append(t_ms)
        rb.append(host_ms(ivf._build_lists)[0])
        srch.append(event_ms(lambda: ivf.search(xq_d, K))[0])
    res["ivf_nlist250_remove_10pct_range"] = dict(
        remove_ms_median=float(np.median(rm)), list_rebuild_ms_median=float(np.median(rb)),
        remove_plus_rebuild_ms=float(np.median(rm) + np.median(rb)), search_after_ms_median=float(np.median(srch)),
        remove_ms_all=[round(x, 3) for x in rm], rebuild_ms_all=[round(x, 3) for x in rb])
    print(json.dumps(res))


if __name__ == "__main__":
    main()
