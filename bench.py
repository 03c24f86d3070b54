#!/usr/bin/env python
"""bench.py -- the headline benchmark of BASELINE.json: queries/s of exact top-50 inner-product
search over the Tianchi-news-shaped catalog (364,047 items x 250-d fp32), 50,000 user queries
per step (the search Retrieval.py:32 performs per user, in its north-star IndexFlatIP form).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

* our arm: one process per GPU (torchrun for N > 1). N = 1: the whole catalog on one B200.
  N > 1 ("strong" scaling: the job is fixed, value = queries of one step x steps /
  max-over-ranks device time): the N ranks form N/S replica groups of S catalog shards each
  (--shards S; default: shards of at least 180,000 rows and at least 2 of them, i.e. S = 2 for this
  364,047-row catalog -- north_star item 4 with the shard size a deployment would pick; S = N and
  S = 1 are timed beside it as `other_decompositions`). Inside a group the catalog rows are sharded,
  every rank searches the group's queries on its shard, the per-shard results travel as 8-byte
  (score, local row) words in an NCCL all-to-all BY QUERY RANGE and each rank merges its own
  query range (K4). The query batch is split over the replica groups. --shards 1 is the
  degenerate layout with no collective (catalog replicated on every GPU, queries split); it
  is timed as `other_decomposition`. Parity against the oracle is asserted on every rank for
  the decomposition that is timed.
* --impl reference: the reference's CPU path for the same search. faiss (the library the
  reference calls) is not installable in this image, so this times the faiss-equivalent oracle
  port (oracle/faiss_oracle.py: OpenBLAS sgemm blocks + heap handler, all host threads) on a
  bounded query sample per step.

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NB, D, NQ, K = 364_047, 250, 50_000, 50
MIN_SHARD_ROWS = 180_000  # default layout: catalog shards are not cut smaller than this (see run_ours)
METRIC = "queries/s, top-50 IP over 364k x 250 items (flat exact search)"
WORKLOAD = "flat_ip_top50: 50,000 queries x 364,047 items x 250-d fp32 (BASELINE configs[0], the config the metric is quoted on)"
ALG_FLOP = 2.0 * NQ * NB * D  # 9.101e12 per step (SURVEY 8d): padding and the 3x TF32 passes not counted


def _synth():
    """newsrecommend_b200/synth.py loaded as a stand-alone module: importing the package would
    dlopen libnrb200.so, and the reference arm must not map the product library."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_nrb_synth", os.path.join(ROOT, "newsrecommend_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def job_config():
    """The job both arms run -- identical keys and values in both JSON lines."""
    return {"workload": WORKLOAD, "k": K,
            "l2": "inputs larger than L2: every step streams the 364,047-row catalog (186 MB fp16 plane + gathers from "
                  "the 373 MB fp32 plane on the GPU, 364 MB fp32 on the CPU; B200 L2 is 126 MB)"}


def default_shards(world: int, nb: int) -> int:
    """Catalog shards per replica group when --shards is not given: shards keep at least MIN_SHARD_ROWS
    rows, but a multi-GPU run always has at least 2 (its timed path contains the exchange + K4 merge);
    the count divides the world size."""
    if world <= 1:
        return 1
    s = max(2, min(world, nb // MIN_SHARD_ROWS))
    while world % s:
        s -= 1
    return max(1, s)


def make_data():
    synth = _synth()
    xb, topics = synth.g_skew(NB, D, 42, return_topics=True)
    xq = synth.user_profiles(xb, topics, NQ, 43)
    return xb, xq


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16": 1590.0, "bf16_sustained": 1400.0, "src": "fallback"}
    try:
        m = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        p = {"hbm_gbs": m["hbm_gbs"], "bf16": m["bf16_tflops"], "bf16_sustained": m["bf16_tflops_sustained"],
             "src": "measured"}
    except Exception:  # noqa: BLE001
        pass
    # TF32 cuBLAS peak measured on this pool by scripts/gpu_probe.py (same method as the bf16
    # figure; profiles/r01_probe.json): 740.7 burst / 604.0 sustained TFLOP/s.
    p["tf32"], p["tf32_sustained"] = 740.7, 604.0
    return p


def ncu_traffic(path_name):
    """(bytes per launch, source) of the dominant kernel from the committed ncu capture listed in
    profiles/ncu_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum, `ncu --set full`)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[path_name]
        return float(t["bytes"]), t["source"]
    except Exception:  # noqa: BLE001
        return None, None


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML polled every ~2 ms from a
    thread (nvidia-smi -lms 100 as the fallback; the timed region is only ~0.1-0.2 s long)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.nvml, self.h, self.samples, self.run = None, None, [], False

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:  # noqa: BLE001
                self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nvml = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.run = True
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:  # noqa: BLE001
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while self.run:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    reasons = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:  # noqa: BLE001
                    reasons = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                util = int(nv.nvmlDeviceGetUtilizationRates(self.h).gpu)
                self.samples.append((mhz, reasons, util))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.run = False
            self.th.join(timeout=1.0)
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
            sm = [m for m, _, _ in self.samples]
            reasons = sorted({n for _, r, _ in self.samples for n, b in bits.items() if r & b})
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                    "sm_max_mhz": self.max_mhz, "samples": len(sm), "reasons": reasons, "source": "nvml, 2 ms poll"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


def dump_outputs(path, arrays, rank=0, world=1):
    """--dump-outputs: the arrays the last timed step returned, as DIR/<name>.npy; scores stay
    float32, ids and query rows become float64 (exact below 2**53). The inputs are seeded, so two
    builds run with the same arguments can be compared array for array. With N > 1 GPUs every rank
    writes the rows it owns, as <name>.rank<r>.npy."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        np.save(os.path.join(path, (name if world == 1 else f"{name}.rank{rank}") + ".npy"), a)


def use_all_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs must use every host core they can."""
    cores = len(os.sched_getaffinity(0))
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)  # OpenBLAS behind numpy (the sgemm blocks)
    except Exception:  # noqa: BLE001
        pass
    try:
        import ctypes
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(cores)  # the oracle's OpenMP loops
    except Exception:  # noqa: BLE001
        pass
    return cores


def cpu_baseline(xb, xq, budget_s=12.0):
    """faiss-equivalent oracle port on the host cores, bounded sample of the same workload."""
    from oracle import faiss_oracle as fo
    fo.build()
    cores = use_all_host_threads()
    fo.knn_fast(xq[:512], xb, K, 0)  # warm-up (thread pools, page-in)
    t0 = time.perf_counter()
    fo.knn_fast(xq[:2048], xb, K, 0)
    rate = 2048 / (time.perf_counter() - t0)
    n = int(min(NQ, max(4096, rate * budget_s)))
    n = n // 4096 * 4096 or 4096
    t0 = time.perf_counter()
    fo.knn_fast(xq[:n], xb, K, 0)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"first {n} of the {NQ} queries against the full 364,047-item catalog, {dt:.1f} s, "
                      f"oracle port (OpenBLAS sgemm blocks 4096 x 16384 + faiss heap handler, OpenMP)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import faiss_oracle as fo
    fo.build()
    xb, xq = make_data()
    cores = use_all_host_threads()
    fo.knn_fast(xq[:512], xb, K, 0)
    t0 = time.perf_counter()
    fo.knn_fast(xq[:2048], xb, K, 0)
    rate = 2048 / (time.perf_counter() - t0)
    steps, warm = args.steps, args.warmup
    budget = float(os.environ.get("NRB_REF_BUDGET_S", "150")) / max(1, steps + warm)  # whole run within a few minutes
    n = int(min(NQ, max(2048, rate * budget)))
    n = max(2048, n // 2048 * 2048)
    for _ in range(warm):
        fo.knn_fast(xq[:n], xb, K, 0)
    t0 = time.perf_counter()
    for _ in range(steps):
        Dr, Ir = fo.knn_fast(xq[:n], xb, K, 0)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"D": Dr, "I": Ir})
    v = n * steps / dt
    sample = (f"each step = first {n} of {NQ} queries against the full catalog; faiss is not installable here, "
              f"this is the faiss-equivalent oracle port on all {cores} host threads")
    args.out.emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": job_config(),
        "cpu_baseline": {"value": v, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import newsrecommend_b200.faiss as nf
    from newsrecommend_b200 import _lib
    from newsrecommend_b200.parity import compare_topk
    from newsrecommend_b200.sharded import ShardedIndexFlat

    xb, xq = make_data()
    path_id = {"auto": _lib.PATH_AUTO, "tc": _lib.PATH_TC, "tc1": _lib.PATH_TC1, "tc16": _lib.PATH_TC16}[args.path]
    one_pass = args.path in ("auto", "tc1", "tc16")
    f16 = args.path in ("auto", "tc16")

    # Layout for N > 1 (the job stays config 1: 50,000 queries x 364,047 items): N / S replica
    # groups of S catalog shards. Replica group g answers queries [g*NQ/R, (g+1)*NQ/R).
    groups = {}

    def layout(S):
        S = max(1, min(S, world))
        while world % S:
            S -= 1
        R = world // S
        g = rank // S
        if S > 1 and S not in groups:
            groups[S] = [dist.new_group(ranks=list(range(i * S, (i + 1) * S))) for i in range(R)] if R > 1 else [None]
        per = (NQ + R - 1) // R
        return S, R, g, min(NQ, g * per), min(NQ, (g + 1) * per)

    def build(S_req):
        S, R, g, lo, hi = layout(S_req)
        xq_dev = torch.from_numpy(xq[lo:hi]).cuda()
        # host side of the end-to-end leg: page-locked query batch and result arrays, handed to
        # the public API as numpy arrays (faiss's search(x, k, D, I) convention)
        xq_pin = torch.from_numpy(xq[lo:hi]).pin_memory().numpy()
        D_pin = torch.empty((hi - lo, K), dtype=torch.float32, pin_memory=True).numpy()
        I_pin = torch.empty((hi - lo, K), dtype=torch.int64, pin_memory=True).numpy()
        if S > 1:
            idx = ShardedIndexFlat(D, nf.METRIC_INNER_PRODUCT, group=groups[S][g], exchange=args.exchange)
            idx.add_global(xb)
            idx.local.path = path_id
            rows = idx.local.ntotal

            def step_device():  # results stay partitioned by query range: (D, I, spans) of this rank's rows
                return idx.search(xq_dev, K, gather=False)

            def step_e2e():  # each rank: H2D of its own rows, NVLink all-gather of the query rows, D2H of its rows
                spans = idx.search_host(xq_pin, K, D_pin, I_pin)
                return D_pin, I_pin, spans
        else:
            idx = nf.IndexFlatIP(D)
            idx.add(xb)
            idx.path = path_id
            planes = idx._query_planes(K)
            rows = idx.ntotal

            def step_device():
                q = nf.PackedMatrix.from_tensor(xq_dev, planes=planes)  # K0 on the fresh query batch
                return idx.search_packed(q, K)

            def step_e2e():
                idx.search(xq_pin, K, D=D_pin, I=I_pin)  # the call a user makes: numpy in, numpy out
                return D_pin, I_pin, [(0, hi - lo)]

        nq_rank = hi - lo  # queries whose scores this rank computes (against `rows` catalog rows)
        return dict(step_device=step_device, step_e2e=step_e2e, lo=lo, hi=hi, rows=rows, S=S, R=R, nq_rank=nq_rank)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def measure(run, sampler=None, keep_outputs=False):
        for _ in range(args.warmup):
            run["step_device"]()
        sync_all()
        if sampler is not None:
            sampler.start()
        _lib.profile_enable(True)
        _lib.profile_read()
        n0 = _lib.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        # results are dropped at once so that every step reuses the same output blocks; only the
        # last step's are kept (for --dump-outputs)
        for _ in range(args.steps - 1):
            run["step_device"]()
        last = run["step_device"]()
        ev1.record()
        sync_all()
        ms = ev0.elapsed_time(ev1)
        launches = _lib.launch_count() - n0
        kern_ms, kern_n = _lib.profile_read()
        _lib.profile_enable(False)
        clocks = sampler.stop() if sampler is not None else None
        outputs = None
        if keep_outputs:  # copied before the end-to-end leg reuses the index
            outputs = {"D": last[0].cpu().numpy(), "I": last[1].cpu().numpy()}
            if world > 1:  # the rows of the batch this rank returns, as query indices
                spans = last[2] if len(last) > 2 else [(0, run["hi"] - run["lo"])]
                rows = [np.arange(a, b) for a, b in spans] or [np.empty(0, np.int64)]
                outputs["query_rows"] = run["lo"] + np.concatenate(rows)
        t = torch.tensor([ms], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        # end to end through the public API with host buffers
        for _ in range(max(1, min(args.warmup, 3))):
            run["step_e2e"]()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            Dh, Ih, spans = run["step_e2e"]()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # parity of THIS decomposition, on every rank: a sample of the rows this rank owns against the oracle
        from oracle import faiss_oracle as fo
        fo.build()
        if world == 1:
            use_all_host_threads()
        rows_own = np.concatenate([np.arange(a, b) for a, b in spans]) if spans else np.empty(0, np.int64)
        ns = min(args.parity_queries if world == 1 else max(64, args.parity_queries // world), rows_own.size)
        pick = rows_own[np.linspace(0, rows_own.size - 1, ns).astype(np.int64)] if ns else rows_own
        rep = dict(ok=True, recall=1.0, exact_ordered=1.0, max_rel_score_err=0.0)
        if ns:
            Do, Io = fo.knn_fast(xq[run["lo"] + pick], xb, K, 0)
            rep = compare_topk(Dh[pick], Ih[pick], Do, Io, 0)
        flags = torch.tensor([1.0 if rep["ok"] else 0.0, float(ns), rep["recall"] * ns, rep["exact_ordered"] * ns],
                             device="cuda", dtype=torch.float64)
        worst = torch.tensor([rep["max_rel_score_err"]], device="cuda", dtype=torch.float64)
        if world > 1:
            ok_t = flags[:1].clone()
            dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
            dist.all_reduce(flags, op=dist.ReduceOp.SUM)
            dist.all_reduce(worst, op=dist.ReduceOp.MAX)
            flags[0] = ok_t[0]
        f = flags.tolist()
        parity = {"queries": int(f[1]), "ok": bool(f[0] >= 1.0), "recall_at_50": f[2] / max(1.0, f[1]),
                  "exact_ordered": f[3] / max(1.0, f[1]), "max_rel_score_err": float(worst.item()),
                  "checked_on": "every rank, rows it owns, vs the oracle port"}
        return dict(ms=ms, launches=launches, kern_ms=kern_ms, kern_n=kern_n, clocks=clocks,
                    e2e_s=float(t.item()), parity=parity, outputs=outputs)

    def describe(run):
        if world == 1:
            return "single GPU"
        if run["S"] == 1:
            return f"queries split over {world} GPUs, packed catalog (1.3 GB) replicated, no data-path collective"
        s = (f"catalog row-sharded {run['S']} ways, per-shard top-k, NCCL {args.exchange} of 8-byte (score, row) words "
             f"by query range, K4 merge of each rank's own query range")
        if run["R"] > 1:
            s += f"; {run['R']} replica groups of {run['S']} shards, the query batch split over the groups"
        return s

    # Default layout: shard the catalog only as far as a shard keeps MIN_SHARD_ROWS rows. A shard search
    # re-discovers every query's top-k threshold from scratch, and that warm-up costs about as much
    # as scanning 250 tiles at the steady rate: a 364k-row catalog cut 8 ways (178-tile units) never
    # leaves it (measured: profiles/r02_bench_n8.json). Config 1 -> replica groups of 2 shards at every
    # N > 1 (N = 2: the box is one group); a 10M-row catalog -> one group of N shards.
    S_main = args.shards if args.shards > 0 else default_shards(world, NB)
    run = build(S_main)
    res = measure(run, ClockSampler(local) if rank == 0 else None, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res["outputs"], rank, world)
    ms, launches, kern_ms, kern_n, clocks, e2e_s = (res[k] for k in ("ms", "launches", "kern_ms", "kern_n", "clocks", "e2e_s"))
    main_desc = describe(run)
    run = {k: v for k, v in run.items() if not callable(v)}  # drop the index (frees HBM)
    alts = []
    if world > 1 and args.alt:
        for alt_S in sorted({1, world} - {run["S"]}):
            torch.cuda.empty_cache()
            run2 = build(alt_S)
            r2 = measure(run2)
            alts.append({"decomposition": describe(run2), "shards": run2["S"], "value": NQ * args.steps / (r2["ms"] / 1e3),
                         "ms_per_step": r2["ms"] / args.steps, "e2e": NQ * args.steps / r2["e2e_s"],
                         "kernel_ms_avg": r2["kern_ms"] / max(1, r2["kern_n"]), "parity_sample": r2["parity"]})
            del run2
    alt = alts[0] if alts else None

    if rank == 0:
        pk = peaks()
        value = NQ * args.steps / (ms / 1e3)
        # roofline of the dominant kernel: algorithmic flops of this rank's share of the job
        alg = 2.0 * run["nq_rank"] * run["rows"] * D
        launches_per_step = max(1.0, kern_n / args.steps)
        kavg_s = kern_ms / max(1, kern_n) / 1e3
        alg_per_launch = alg / launches_per_step
        achieved = alg_per_launch / kavg_s / 1e12 if kavg_s > 0 else 0.0
        # the timed region is steps x ~9 ms (well under a second): the burst figure is the denominator
        timed_s = ms / 1e3
        burst = timed_s < 2.0
        passes = 1.0 if one_pass else 3.0
        if f16:
            peak = pk["bf16"] if burst else pk["bf16_sustained"]
            kname = ("topk_tc3_kernel<IP, fp16> (tcgen05 kind::f16 filter on power-of-two scaled fp16 planes "
                     "with error margin; exact fp32 refine follows)")
            note = ("peak = MEASURED_PEAKS (%s) dense bf16/fp16 %s %.1f TFLOP/s (burst %.1f, sustained %.1f; the timed "
                    "region is %.2f s)" % (pk["src"], "burst" if burst else "sustained", peak, pk["bf16"],
                                           pk["bf16_sustained"], timed_s))
            pipe_frac = achieved * 256.0 / 250.0 / peak
        else:
            tf32_peak = pk["tf32"] if burst else pk["tf32_sustained"]
            peak = tf32_peak / passes
            kname = ("topk_tc3_kernel<IP> (tcgen05 1xTF32 filter with error margin; exact fp32 refine follows)"
                     if one_pass else "topk_tc2_kernel<IP> (tcgen05 3xTF32 + fused selection)")
            note = ("peak = cuBLAS TF32 %s %.1f TFLOP/s (scripts/gpu_probe.py, same method as MEASURED_PEAKS.json; "
                    "profiles/r01_probe.json) / %d TF32 pass(es) per product"
                    % ("burst" if burst else "sustained", tf32_peak, int(passes)))
            pipe_frac = achieved * passes * 256.0 / 250.0 / tf32_peak
        traffic, traffic_src = ncu_traffic("tc16" if f16 else "tc1" if one_pass else "tc") if world == 1 else (None, None)
        roof = {
            "bound": "tensor",
            "kernel": kname,
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "peak_note": note,
            "tensor_pipe_frac": pipe_frac,
            "frac_of_sustained_peak": achieved / (pk["bf16_sustained"] if f16 else pk["tf32_sustained"] / passes),
            "kernel_ms_avg": kavg_s * 1e3, "kernel_launches_timed": kern_n,
            "alg_flop_per_launch": alg_per_launch,
            # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel at N = 1, from the
            # committed `ncu --set full` capture named in traffic_source (offline, not measured in this run)
            "traffic": traffic, "traffic_source": traffic_src,
        }
        cfg = job_config()
        out = {
            "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": ("f32 (fp16 tcgen05 filter with a proven error margin + exact fp32 rescoring)" if f16 else
                      "f32 (1xTF32 tcgen05 filter + exact fp32 rescoring)" if one_pass
                      else "f32 (3xTF32 tcgen05, fp32 accumulate)"),
            "data": "synthetic",
            "config": cfg,
            "detail": {"parallelism": main_desc, "path": args.path,
                       "fallback_queries": int(_lib.lib.nrb_fallback_query_count()),
                       "timed": "K0 query pack + K2 tcgen05 distance/selection + select" +
                                (" + exact refine" if one_pass else "") +
                                (" + pack + NCCL exchange + K4 merge" if run["S"] > 1 else "")},
            "roofline": roof,
            "e2e": {"value": NQ * args.steps / e2e_s, "unit": "queries/s",
                    "h2d_bytes_per_step": NQ * D * 4, "d2h_bytes_per_step": NQ * K * 12},
            "gpu_launches": int(launches), "clocks": clocks, "other_decomposition": alt,
            "other_decompositions": alts,
            "parity_sample": res["parity"],
        }
        if world == 1 and not os.environ.get("NRB_BENCH_SKIP_CPU"):  # skipped only for ncu captures
            out["cpu_baseline"] = cpu_baseline(xb, xq)
        args.out.emit(out)
    ok = res["parity"]["ok"] and all(a["parity_sample"]["ok"] for a in alts) if rank == 0 else True
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        raise SystemExit("bench.py: parity against the oracle FAILED for the timed decomposition")


class _StdoutGuard:
    """Libraries (NCCL's version banner, torchrun notices) write to fd 1; the contract is ONE JSON
    line on stdout. Route fd 1 to stderr for the whole run and emit the JSON on the saved fd."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, obj):
        sys.stdout.flush()
        os.write(self.real, (json.dumps(obj) + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shards", type=int, default=0,
                    help="N > 1: catalog shards per replica group (default 0 = shards of >= 180,000 rows, at least 2: "
                         "config 1 -> N/2 replica groups of 2 shards; N = the whole box is one group of N catalog "
                         "shards; 1 = catalog replicated, queries split, no collective)")
    ap.add_argument("--exchange", default="alltoall", choices=["alltoall", "allgather"],
                    help="exchange step of the catalog-sharded search (all-to-all by query range, or the all-gather "
                         "north_star names literally)")
    ap.add_argument("--parity-queries", type=int, default=2048,
                    help="queries checked against the oracle after the timed runs (spread over the batch)")
    ap.add_argument("--no-alt", dest="alt", action="store_false",
                    help="N > 1: do not also time the other decomposition")
    ap.add_argument("--path", default="auto", choices=["auto", "tc", "tc1", "tc16"],
                    help="auto/tc16 = fp16 filter + exact fp32 refine (default), tc1 = the same with the 1xTF32 "
                         "filter, tc = 3xTF32")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the (D, I) results of the last timed step as DIR/<name>.npy "
                         "(30 MB for the default job)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.out = _StdoutGuard()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
