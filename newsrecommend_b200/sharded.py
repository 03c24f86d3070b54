"""Catalog sharding across the GPUs of one box (BASELINE.json north_star item 4, SURVEY 8e).

One process per GPU (torch.distributed, NCCL over NVLink / NVSwitch). The catalog rows are split
into contiguous ranges -- rank r owns ids [nb*r/G, nb*(r+1)/G) -- every rank sees all queries and
runs the exact top-k kernel on its shard. The exchange step comes in two forms:

* ``exchange="alltoall"`` (default): all-to-all BY QUERY RANGE. Every rank packs its per-shard
  results as 8-byte (score bits, local row) words (nrb_pack_topk), sends to rank j the rows of the
  queries rank j owns, and merges only its own nq/G queries (nrb_merge_topk_packed, K4). Per rank
  this moves and merges 1/G of what the all-gather does. The batch is processed in chunks; the
  exchange of chunk i runs on NCCL's stream while chunk i+1 is being searched, and every chunk is
  split G ways, so all ranks merge all the time.
* ``exchange="allgather"``: the contract north_star names literally -- all-gather of the packed
  per-shard results and a k-way merge of all queries on every rank.

The merged result equals the single-index answer up to the order of exact ties. The reference has
no distributed code at all (SURVEY 2.2); this is the north star's extension of IndexFlat.search.

Host logic only; `make_index` (per-rank index) and `codec` (pack / merge) are injectable so that
the same code runs under gloo on CPU with the oracle index and numpy stand-ins (tests/).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

CHUNK_WAVES = 7  # queries per chunk = CHUNK_WAVES full waves of the search kernel (7 x 18,944)


def shard_range(nb: int, world: int, rank: int) -> tuple[int, int]:
    """Balanced contiguous row ranges: shard sizes differ by at most one row and no shard is empty
    while nb >= world (ceil-sized ranges leave trailing shards empty, e.g. nb = 9, world = 8)."""
    return nb * rank // world, nb * (rank + 1) // world


def chunk_slices(nq: int, world: int, chunk: int) -> list[tuple[int, int, int]]:
    """[(c0, c1, per)]: the batch in chunks of `chunk` queries; inside a chunk rank r owns rows
    [c0 + r*per, min(c1, c0 + (r+1)*per)) -- ceil-sized slices, so that the concatenation of the
    (padded) slices in rank order is the chunk itself (what all_gather_into_tensor produces)."""
    out = []
    for c0 in range(0, nq, chunk):
        c1 = min(nq, c0 + chunk)
        out.append((c0, c1, -(-(c1 - c0) // world)))
    return out


def owned_rows(nq: int, world: int, rank: int, chunk: int) -> list[tuple[int, int]]:
    """Query rows whose final result lands on `rank`, as (lo, hi) spans in batch order."""
    spans = []
    for c0, c1, per in chunk_slices(nq, world, chunk):
        lo, hi = min(c1, c0 + rank * per), min(c1, c0 + (rank + 1) * per)
        spans.append((lo, hi))
    return spans


class GpuCodec:
    """Wire format + K4 merge on the device (libnrb200)."""

    @staticmethod
    def pack(D: torch.Tensor, I: torch.Tensor, id_base: int) -> torch.Tensor:
        from ._lib import check, lib
        P = torch.empty(D.shape, dtype=torch.int64, device=D.device)
        check(lib.nrb_pack_topk(D.data_ptr(), I.data_ptr(), id_base, D.numel(), P.data_ptr(),
                                torch.cuda.current_stream().cuda_stream), "pack_topk")
        return P

    @staticmethod
    def merge(P: torch.Tensor, bases: torch.Tensor, metric: int):
        from ._lib import check, lib
        G, nq, k = P.shape
        D = torch.empty((nq, k), dtype=torch.float32, device=P.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=P.device)
        check(lib.nrb_merge_topk_packed(P.data_ptr(), bases.data_ptr(), G, nq, k, metric, D.data_ptr(), I.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream), "merge_topk_packed")
        return D, I


class _ShardedSearch:
    """The exchange machinery shared by the sharded indexes: chunking, packing, all-to-all by query
    range (or all-gather), K4 merge, final gather, host-array entry point. A subclass provides
    `search_local` (per-shard top-k of one query chunk) and the shard's first global id."""

    def _init_sharding(self, metric: int, group, codec, exchange: str, chunk_queries, cuda_index: bool):
        assert exchange in ("alltoall", "allgather")
        self.metric_type, self.group, self.exchange_mode = metric, group, exchange
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._cuda_index = cuda_index
        self.codec = codec or GpuCodec
        self.ntotal = 0
        self.id_base = 0
        self.bases = None  # i64[G]: first global id of every shard
        self._bases_host = [0]
        self.chunk_queries = chunk_queries

    def _set_bases_global(self, nb: int):
        self._bases_host = [shard_range(nb, self.world, r)[0] for r in range(self.world)]
        self.bases = None

    def _set_bases_gathered(self):
        if self.world > 1:
            t = torch.tensor([self.id_base], dtype=torch.int64, device=self._dev())
            out = torch.empty(self.world, dtype=torch.int64, device=self._dev())
            dist.all_gather_into_tensor(out, t, group=self.group)
            self._bases_host = out.cpu().tolist()
        else:
            self._bases_host = [self.id_base]
        self.bases = None

    def _dev(self):
        if self._cuda_index:
            return torch.device("cuda", torch.cuda.current_device())
        return torch.device("cpu")

    def _bases(self):
        if self.bases is None:
            self.bases = torch.tensor(self._bases_host, dtype=torch.int64, device=self._dev())
        return self.bases

    def _chunk(self) -> int:
        if self.chunk_queries:
            return int(self.chunk_queries)
        if self._cuda_index:
            from .faiss import _wave_rows
            return CHUNK_WAVES * _wave_rows()
        return 1 << 17

    # ------------------------------------------------------------------ search pieces
    def search_local(self, xq, k: int):
        """Per-shard top-k of a raw query chunk with GLOBAL ids: (D f32[n,k], I i64[n,k]) tensors."""
        raise NotImplementedError

    def _exchange_start(self, P: torch.Tensor, per: int):
        """Starts the exchange of one chunk's packed per-shard results P i64[cn, k]. Returns
        (recv i64[G, rows, k], work handle or None): alltoall -> rows = this rank's slice of the
        chunk, allgather -> rows = the whole chunk."""
        cn, k = P.shape
        G, r = self.world, self.rank
        if G == 1:
            return P.unsqueeze(0), None
        if self.exchange_mode == "allgather":
            recv = torch.empty((G * cn, k), dtype=P.dtype, device=P.device)
            work = dist.all_gather_into_tensor(recv, P, group=self.group, async_op=True)
            return recv.view(G, cn, k), work
        in_rows = [max(0, min(cn, (j + 1) * per) - min(cn, j * per)) for j in range(G)]
        mine = in_rows[r]
        recv = torch.empty((G * mine, k), dtype=P.dtype, device=P.device)
        work = dist.all_to_all_single(recv, P, [mine] * G, in_rows, group=self.group, async_op=True)
        return recv.view(G, mine, k), work

    def search(self, xq, k: int, gather: bool = True):
        """xq: the FULL query batch on every rank (CUDA tensor fp32 [nq, d]; ndarray on the CPU test
        path). gather=True: (D, I) of all queries on every rank (a final all-gather of the merged
        slices). gather=False: the merged results of this rank's own rows only, as
        (D, I, spans) with spans = owned_rows(nq, ...)."""
        nq = xq.shape[0]
        G = self.world
        chunk = self._chunk()
        pending = None
        parts = []

        def finish(p):
            recv, work = p
            if work is not None:
                work.wait()
            parts.append(self.codec.merge(recv, self._bases(), self.metric_type))

        for c0, c1, per in chunk_slices(nq, G, chunk):
            D, I = self.search_local(xq[c0:c1], k)
            P = self.codec.pack(D, I, self.id_base)
            nxt = self._exchange_start(P, per)
            if pending is not None:
                finish(pending[:2])  # merged after the NEXT chunk's search was queued: its exchange overlaps that search
            pending = nxt + (P,)  # P stays referenced until its exchange has been waited for
        if pending is not None:
            finish(pending[:2])
        if self.exchange_mode == "allgather" or G == 1:
            D = torch.cat([p[0] for p in parts]) if len(parts) != 1 else parts[0][0]
            I = torch.cat([p[1] for p in parts]) if len(parts) != 1 else parts[0][1]
            if gather:
                return D, I
            spans = owned_rows(nq, G, self.rank, chunk)
            if G == 1:
                return D, I, spans
            sel = torch.cat([torch.arange(lo, hi) for lo, hi in spans]).to(D.device)
            return D[sel], I[sel], spans
        spans = owned_rows(nq, G, self.rank, chunk)
        if not gather:
            D = torch.cat([p[0] for p in parts]) if len(parts) != 1 else parts[0][0]
            I = torch.cat([p[1] for p in parts]) if len(parts) != 1 else parts[0][1]
            return D, I, spans
        return self._gather_all(parts, nq, k, chunk)

    def _gather_all(self, parts, nq: int, k: int, chunk: int):
        """All-gather of the merged per-rank slices, chunk by chunk, back into batch order."""
        G = self.world
        dev = parts[0][0].device
        D = torch.empty((nq, k), dtype=torch.float32, device=dev)
        I = torch.empty((nq, k), dtype=torch.int64, device=dev)
        for (c0, c1, per), (Dm, Im) in zip(chunk_slices(nq, G, chunk), parts):
            Dp = torch.zeros((per, k), dtype=torch.float32, device=dev)
            Ip = torch.zeros((per, k), dtype=torch.int64, device=dev)
            Dp[: Dm.shape[0]] = Dm
            Ip[: Im.shape[0]] = Im
            Dg = torch.empty((G * per, k), dtype=torch.float32, device=dev)
            Ig = torch.empty((G * per, k), dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(Dg, Dp, group=self.group)
            dist.all_gather_into_tensor(Ig, Ip, group=self.group)
            D[c0:c1] = Dg[: c1 - c0]
            I[c0:c1] = Ig[: c1 - c0]
        return D, I

    # ------------------------------------------------------------------ end to end from host memory
    def search_host(self, xq_host: np.ndarray, k: int, D_out: np.ndarray, I_out: np.ndarray):
        """The call a user of the sharded index makes with HOST arrays: every rank passes the same
        page-locked fp32 [nq, d] batch and the same-shaped output arrays; each rank copies only ITS
        rows host-to-device (1/G of the batch), the ranks all-gather the query rows over NVLink,
        search, exchange, merge, and each rank copies the results of its own rows back into
        D_out / I_out (rows owned by other ranks are left untouched). Returns the owned spans."""
        assert self._cuda_index, "search_host is the CUDA path"
        nq, d = xq_host.shape
        G, r = self.world, self.rank
        dev = self._dev()
        chunk = self._chunk()
        src = torch.from_numpy(xq_host)
        Dt, It = torch.from_numpy(D_out), torch.from_numpy(I_out)
        pending = None
        spans = []

        def finish(p):
            recv, work, lo, hi, c0 = p
            if work is not None:
                work.wait()
            if self.exchange_mode == "allgather" and G > 1:
                recv = recv[:, lo - c0:hi - c0].contiguous()  # merge (and return) only the owned rows
            Dm, Im = self.codec.merge(recv, self._bases(), self.metric_type)
            if hi > lo:
                Dt[lo:hi].copy_(Dm, non_blocking=True)
                It[lo:hi].copy_(Im, non_blocking=True)
            spans.append((lo, hi))
            return Dm, Im

        keep = []
        for c0, c1, per in chunk_slices(nq, G, chunk):
            lo, hi = min(c1, c0 + r * per), min(c1, c0 + (r + 1) * per)
            mine = torch.zeros((per, d), dtype=torch.float32, device=dev) if hi - lo < per else \
                torch.empty((per, d), dtype=torch.float32, device=dev)
            if hi > lo:
                mine[: hi - lo].copy_(src[lo:hi], non_blocking=True)  # H2D of this rank's rows only
            if G > 1:
                full = torch.empty((G * per, d), dtype=torch.float32, device=dev)
                dist.all_gather_into_tensor(full, mine, group=self.group)
            else:
                full = mine
            D, I = self.search_local(full[: c1 - c0], k)
            P = self.codec.pack(D, I, self.id_base)
            recv, work = self._exchange_start(P, per)
            if pending is not None:
                keep.append(finish(pending[:5]))
            pending = (recv, work, lo, hi, c0, P)
        if pending is not None:
            keep.append(finish(pending[:5]))
        torch.cuda.current_stream().synchronize()
        return spans


class ShardedIndexFlat(_ShardedSearch):
    """Row-sharded exact index (IndexFlatIP / IndexFlatL2 semantics over the whole catalog)."""

    def __init__(self, d: int, metric: int = 1, group=None, make_index=None, codec=None, exchange: str = "alltoall",
                 chunk_queries: int | None = None):
        self._init_sharding(metric, group, codec, exchange, chunk_queries, cuda_index=make_index is None)
        self.d = d
        if make_index is None:
            from .faiss import IndexFlat
            make_index = IndexFlat
        self.local = make_index(d, metric)

    # ------------------------------------------------------------------ build
    def add_global(self, x):
        """Every rank passes the SAME full matrix; each keeps only its own row range."""
        nb = x.shape[0]
        assert self.ntotal == 0, "add_global is a one-shot build"
        lo, hi = shard_range(nb, self.world, self.rank)
        self.id_base = lo
        self.local.add(x[lo:hi])
        self.ntotal = nb
        self._set_bases_global(nb)

    def add_local(self, x_local, id_base: int, ntotal: int):
        """Each rank passes only ITS rows (global ids id_base ... id_base + len - 1): for catalogs
        that no single process ever holds whole (10M x 256 sharded: BASELINE configs[4])."""
        assert self.ntotal == 0, "add_local is a one-shot build"
        self.id_base = int(id_base)
        self.local.add(x_local)
        self.ntotal = int(ntotal)
        self._set_bases_gathered()

    def search_local(self, xq, k: int):
        if self._cuda_index:
            from .faiss import PackedMatrix
            q = PackedMatrix.from_tensor(xq, planes=self.local._query_planes(k))  # K0 on the fresh chunk
            return self.local.search_packed(q, k, self.id_base)
        D, I = self.local.search(np.ascontiguousarray(xq), k)
        I = torch.as_tensor(I)
        return torch.as_tensor(D), torch.where(I >= 0, I + self.id_base, I)


# ------------------------------------------------------------------------------------ sharded IVF
class GpuKMeansOps:
    """Device pieces of one data-parallel Lloyd iteration (libnrb200): exact nearest-centroid
    assignment of this rank's rows (K2, k = 1), fp64 partial sums | counts (K1b without the
    division), means from the all-reduced table, device split_clusters."""

    def __init__(self, d: int, k: int, metric: int):
        from . import faiss as nf
        self.nf, self.d, self.k, self.metric = nf, d, k, metric
        self.index = nf.IndexFlat(d, metric)
        self.xs = None

    def device(self):
        return torch.device("cuda", torch.cuda.current_device())

    def to_device(self, x):
        return self.nf._to_device_f32(x)[0]

    def set_rows(self, x: torch.Tensor):
        self.n = x.shape[0]
        self.xs = self.nf.PackedMatrix.from_tensor(x, planes=("raw", "hi", "lo", "norms", "h16")) if self.n else None

    def assign(self, cent: torch.Tensor):
        """(assign i64[n], objective f64 scalar tensor) of this rank's rows against cent f32[k, d]."""
        self.index.reset()
        self.index.add(cent)
        if not self.n:
            return None, torch.zeros((), dtype=torch.float64, device=self.device())
        D, I = self.index.search_packed(self.xs, 1)
        return I.reshape(-1), D.sum(dtype=torch.float64)

    def partial_sums(self, assign, table: torch.Tensor):
        """table f64[k * (d + 1) + 1]: sums | counts of this rank's rows (the last slot is the caller's)."""
        from ._lib import check, lib
        table[: self.k * (self.d + 1)].zero_()
        if not self.n:
            return
        wsb = lib.nrb_kmeans_update_workspace(self.n, self.k, self.xs.kp)
        ws = torch.empty(wsb, dtype=torch.uint8, device=table.device)
        check(lib.nrb_kmeans_partial_sums(self.xs.raw.data_ptr(), self.n, self.d, self.xs.kp, assign.data_ptr(), self.k,
                                          table.data_ptr(), ws.data_ptr(), wsb, torch.cuda.current_stream().cuda_stream),
              "kmeans_partial_sums")

    def means_and_split(self, table: torch.Tensor, n_total: int, spherical: bool):
        """(centroids f32[k, d], imbalance, nsplit) from the all-reduced table."""
        from ._lib import check, lib
        st = torch.cuda.current_stream().cuda_stream
        cent = torch.empty((self.k, self.d), dtype=torch.float32, device=table.device)
        hassign = torch.empty(self.k, dtype=torch.float32, device=table.device)
        stats = torch.zeros(3, dtype=torch.float64, device=table.device)
        check(lib.nrb_kmeans_means(table.data_ptr(), self.k, self.d, cent.data_ptr(), hassign.data_ptr(), st), "kmeans_means")
        check(lib.nrb_split_clusters(self.d, self.k, n_total, hassign.data_ptr(), cent.data_ptr(), stats.data_ptr(), st),
              "split_clusters")
        if spherical:
            check(lib.nrb_normalize_l2(cent.data_ptr(), self.k, self.d, self.d, st), "normalize_l2")
        s = stats.cpu()
        if s[2] < 0:
            raise RuntimeError("split_clusters: no cluster to split")
        return cent, float(s[1]), int(s[2])


def _rand_perm(n: int, seed: int) -> np.ndarray:
    """faiss::rand_perm (std::mt19937) through the C-ABI host helper; no GPU needed."""
    import ctypes as C
    from ._lib import check, lib
    perm = np.empty(n, dtype=np.int32)
    check(lib.nrb_rand_perm_host(C.c_void_p(perm.ctypes.data), n, seed), "rand_perm")
    return perm


def _gather_rows_by_position(x_local, id_base: int, ids: np.ndarray, group, world: int, to_device, device):
    """rows[j] = catalog row ids[j], assembled from the shards: every rank fills the rows it owns into
    a zero matrix and the ranks add their matrices (x + 0 is exact), so every rank ends up with
    the same [len(ids), d] matrix. Used for the k-means subsample and the initial centroids."""
    n_local, d = x_local.shape
    mine = np.nonzero((ids >= id_base) & (ids < id_base + n_local))[0]
    out = torch.zeros((len(ids), d), dtype=torch.float32, device=device)
    if len(mine):
        src = to_device(x_local)
        sel = torch.from_numpy((ids[mine] - id_base).astype(np.int64)).to(device)
        out[torch.from_numpy(mine).to(device)] = src.index_select(0, sel)
    if world > 1:
        dist.all_reduce(out, group=group)
    return out


def train_kmeans_data_parallel(x_local, id_base: int, ntotal: int, k: int, cp, metric: int, group=None, ops=None,
                               verbose: bool = False):
    """Lloyd k-means over a ROW-SHARDED training set with one shared set of centroids (SURVEY 8e):
    every rank assigns its own rows, the ranks all-reduce ONE fp64 table per iteration
    (k x (d + 1) sums | counts + the objective: <= 0.65 MB at nlist 325, d 250) and every rank
    derives the same centroids and the same split_clusters decisions from it. faiss's sampling is
    kept: the training set is rand_perm(ntotal, seed)[: k * max_points_per_centroid] of the GLOBAL
    rows (each rank keeps the part it owns, in permutation order), the initial centroids are rows
    rand_perm(n_train, seed + 1)[:k] of that set. With one rank this is Clustering.train up to the
    association of the fp64 sums. Returns (centroids f32[k, d] tensor, [ClusteringIterationStats])."""
    from .faiss import ClusteringIterationStats
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    n_local, d = x_local.shape
    if ntotal < k:
        raise RuntimeError("Number of training points (%d) should be at least as large as number of "
                           "clusters (%d)" % (ntotal, k))
    ops = ops or GpuKMeansOps(d, k, metric)
    dev = ops.device()
    if ntotal > k * cp.max_points_per_centroid:
        ids = _rand_perm(ntotal, cp.seed)[: k * cp.max_points_per_centroid].astype(np.int64)
    else:
        ids = np.arange(ntotal, dtype=np.int64)
    n_train = len(ids)
    mine = np.nonzero((ids >= id_base) & (ids < id_base + n_local))[0]
    xl = ops.to_device(x_local)
    rows = xl.index_select(0, torch.from_numpy((ids[mine] - id_base).astype(np.int64)).to(dev)) if len(mine) else \
        torch.empty((0, d), dtype=torch.float32, device=dev)
    ops.set_rows(rows)
    init_pos = _rand_perm(n_train, cp.seed + 1)[:k].astype(np.int64)
    cent = _gather_rows_by_position(x_local, id_base, ids[init_pos], group, world, ops.to_device, dev)
    if n_train == k:
        return cent, []
    table = torch.zeros(k * (d + 1) + 1, dtype=torch.float64, device=dev)
    stats = []
    for it in range(cp.niter):
        assign, obj = ops.assign(cent)
        ops.partial_sums(assign, table)
        table[-1] = obj
        if world > 1:
            dist.all_reduce(table, group=group)
        obj_all = float(table[-1])
        cent, imb, nsplit = ops.means_and_split(table, n_train, cp.spherical)
        stats.append(ClusteringIterationStats(float(np.float32(obj_all)), imb, nsplit))
        if verbose:
            print("  Iteration %d objective=%g imbalance=%.3f nsplit=%d" % (it, obj_all, imb, nsplit))
    return cent, stats


class ShardedIndexIVFFlat(_ShardedSearch):
    """IndexIVFFlat over a row-sharded catalog (SURVEY 8e, "Partitioning (IVF)"): ONE shared coarse
    quantizer (the same nlist centroids on every rank), every inverted list's rows split across
    the ranks by catalog row range (row-sharding WITHIN lists: a skewed list is spread over all
    GPUs), so the merged result equals the single-index answer -- unlike faiss's IndexShards of
    independently trained IVFs, which changes the results. train: "gather" = the k-means subsample
    (faiss's rand_perm rows) is assembled on every rank and every rank runs the identical
    deterministic trainer (bit-equal to single-index training); "data_parallel" = each rank keeps
    its rows and the ranks all-reduce one fp64 table per iteration (train_kmeans_data_parallel).
    search: every rank sees all queries, runs coarse search + list scan on its part of the probed
    lists, then the same exchange + K4 merge as ShardedIndexFlat."""

    def __init__(self, d: int, nlist: int, metric: int = 1, group=None, make_index=None, make_ivf=None, codec=None,
                 kmeans_ops=None, exchange: str = "alltoall", chunk_queries: int | None = None):
        cuda = make_ivf is None
        self._init_sharding(metric, group, codec, exchange, chunk_queries, cuda_index=cuda)
        self.d, self.nlist, self.nprobe = d, nlist, 1
        if cuda:
            from .faiss import IndexFlat, IndexIVFFlat
            make_index, make_ivf = IndexFlat, IndexIVFFlat
        self.quantizer = make_index(d, metric)
        self.local = make_ivf(self.quantizer, d, nlist, metric)
        self.cp = self.local.cp
        self._kmeans_ops = kmeans_ops
        self.iteration_stats = []

    @property
    def is_trained(self) -> bool:
        return self.local.is_trained

    def _to_local_device(self, x):
        if self._cuda_index:
            from .faiss import _to_device_f32
            return _to_device_f32(x)[0]
        return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32))

    def _set_centroids(self, cent):
        """Rank 0's centroids on every rank (they are equal already; the broadcast pins it)."""
        cent = cent.contiguous()
        if self.world > 1:
            dist.broadcast(cent, src=dist.get_global_rank(self.group, 0) if self.group is not None else 0, group=self.group)
        self.quantizer.reset()
        self.quantizer.add(cent if self._cuda_index else cent.numpy())
        self.local.is_trained = True

    def train_local(self, x_local, id_base: int, ntotal: int, mode: str = "gather"):
        """x_local: this rank's catalog rows (global ids id_base ...). See the class docstring."""
        assert mode in ("gather", "data_parallel")
        k, cp = self.nlist, self.cp
        if mode == "data_parallel":
            cent, stats = train_kmeans_data_parallel(x_local, id_base, ntotal, k, cp, self.metric_type, self.group,
                                                     self._kmeans_ops)
            self.iteration_stats = stats
            self._set_centroids(cent)
            return
        if ntotal > k * cp.max_points_per_centroid:
            ids = _rand_perm(ntotal, cp.seed)[: k * cp.max_points_per_centroid].astype(np.int64)
        else:
            ids = np.arange(ntotal, dtype=np.int64)
        sub = _gather_rows_by_position(x_local, id_base, ids, self.group, self.world, self._to_local_device, self._dev())
        # the subsample is exactly what Clustering.train would have drawn from the whole catalog;
        # training on it (n == k * max_points: no second subsampling) continues with seed + 1
        self.quantizer.reset()
        self.local.is_trained = False
        self.local.train(sub if self._cuda_index else sub.numpy())
        self.iteration_stats = self.local.clustering.iteration_stats
        cent = self.quantizer.reconstruct_n() if self._cuda_index else self.quantizer.xb
        self._set_centroids(torch.as_tensor(np.ascontiguousarray(cent)).to(self._dev()))

    def train_global(self, x, mode: str = "gather"):
        """Every rank passes the SAME full matrix."""
        lo, hi = shard_range(x.shape[0], self.world, self.rank)
        self.train_local(x[lo:hi], lo, x.shape[0], mode)

    def add_global(self, x):
        nb = x.shape[0]
        assert self.ntotal == 0, "add_global is a one-shot build"
        lo, hi = shard_range(nb, self.world, self.rank)
        self.id_base = lo
        self.local.add(x[lo:hi])
        self.ntotal = nb
        self._set_bases_global(nb)

    def add_local(self, x_local, id_base: int, ntotal: int):
        assert self.ntotal == 0, "add_local is a one-shot build"
        self.id_base = int(id_base)
        self.local.add(x_local)
        self.ntotal = int(ntotal)
        self._set_bases_gathered()

    def search_local(self, xq, k: int):
        self.local.nprobe = self.nprobe
        if self._cuda_index:
            D, I = self.local.search(xq, k)  # ids = local insertion rows
            return D, torch.where(I >= 0, I + self.id_base, I)
        D, I = self.local.search(np.ascontiguousarray(xq), k)
        I = torch.as_tensor(I)
        return torch.as_tensor(D), torch.where(I >= 0, I + self.id_base, I)
