"""Robustness of the default fp16 filter outside the benchmark distribution (VERDICT r1 weak #7): queries that
the filter flags are recomputed by the 3xTF32 pipeline at ~4x the cost, so the fallback RATE decides the
throughput. Config-1 shape (364,047 x 250, 50,000 queries, top-50 IP), device-resident, per case:
queries/s, fallback queries, parity sample vs the oracle.
  * g_skew        the benchmark data (topic mixture, Zipf weights)
  * g_iso         isotropic Gaussian items and queries: the worst-case-gap variant of SURVEY 8d
  * dup x m       near-duplicate-heavy catalog (news reposts): 364,047 / m base articles, each present m
                  times with relative noise 1e-4 -- inside the filter's error margin (2 * 1.07e-3 * |q| * max|x|),
                  so every copy of an article near the k-th rank lands in the margin set
One JSON line."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import newsrecommend_b200.faiss as nf
from newsrecommend_b200 import _lib, synth
from newsrecommend_b200.parity import compare_topk
from oracle import faiss_oracle as fo

fo.build()
NB, D, NQ, K = synth.N_ARTICLES, 250, 50_000, 50


def run(name, xb, xq):
    index = nf.IndexFlatIP(D)
    index.add(torch.from_numpy(xb).cuda())
    xq_d = torch.from_numpy(xq).cuda()
    planes = index._query_planes(K)

    def step():
        q = nf.PackedMatrix.from_tensor(xq_d, planes=planes)
        return index.search_packed(q, K)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    f0 = int(_lib.lib.nrb_fallback_query_count())
    _lib.profile_enable(True)
    _lib.profile_read()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        Dd, Id = step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    kms, kn = _lib.profile_read()
    _lib.profile_enable(False)
    fb = (int(_lib.lib.nrb_fallback_query_count()) - f0) // reps
    ns = 1024
    pick = np.linspace(0, NQ - 1, ns).astype(np.int64)
    Do, Io = fo.knn_fast(xq[pick], xb, K, 0)
    rep = compare_topk(Dd[pick].cpu().numpy(), Id[pick].cpu().numpy(), Do, Io, 0)
    return dict(case=name, qps=NQ / dt, ms=dt * 1e3, k2_kernel_ms=kms / reps, k2_launches_per_search=kn / reps,
                fallback_queries=fb, fallback_rate=fb / NQ,
                parity_ok=bool(rep["ok"]), recall=rep["recall"], max_rel_score_err=rep["max_rel_score_err"])


out = []
xb, topics = synth.g_skew(NB, D, 42, return_topics=True)
xq = synth.user_profiles(xb, topics, NQ, 43)
out.append(run("g_skew (benchmark data)", xb, xq))
out.append(run("g_iso (isotropic Gaussian)", synth.g_iso(NB, D, 1234), synth.g_iso(NQ, D, 1235)))
rng = np.random.default_rng(7)
for m in [int(a) for a in os.environ.get("NRB_DUPS", "4,16,64").split(",")]:
    nbase = NB // m
    base = xb[:nbase]
    rep_rows = np.tile(np.arange(nbase), m + 1)[:NB]
    xd = base[rep_rows] * (1.0 + 1e-4 * rng.standard_normal((NB, 1), dtype=np.float32)) \
        + 1e-4 * np.linalg.norm(base[rep_rows], axis=1, keepdims=True) / np.sqrt(D) * rng.standard_normal((NB, D), dtype=np.float32)
    xd = np.ascontiguousarray(xd.astype(np.float32))
    out.append(run("dup x %d (relative noise 1e-4)" % m, xd, xq))
print(json.dumps(dict(shape=[NB, D, NQ, K], cases=out)))
