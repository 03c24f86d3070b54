"""`faiss`-compatible surface of the B200 candidate-retrieval path.

Mirrors exactly the symbols /root/reference/Retrieval.py uses (Retrieval.py:12-32: Clustering,
IndexHNSWFlat, IndexFlatL2, vector_float_to_array, index.search) plus the index surface
BASELINE.json's north_star names (IndexFlatIP, IndexIVFFlat with train/add/search, nlist /
nprobe / k semantics, METRIC_*, normalize_L2). Semantics follow SURVEY.md section 8b. External
ids (IndexIDMap, IndexIVFFlat.add_with_ids, remove_ids with IDSelectorBatch / IDSelectorRange /
IDSelectorNot) stand in for the article-id array that Retrieval.py:7,23 keeps beside the index.

Search-time selectors follow faiss: `index.search(x, k, params=SearchParameters(sel=...))` on the flat
indexes and IndexIDMap, `SearchParametersIVF(sel=..., nprobe=...)` on IndexIVFFlat. The selector
tests row positions on a plain flat index, external ids on IndexIDMap and stored ids on IndexIVFFlat
(whose coarse search still ranks every centroid; only the list scan skips unselected rows). Rows
that are not selected never appear in a result; when fewer than k rows qualify the tail is padded
with I = -1 as for k > ntotal. Small batches (the HBM-regime kernels) scan with a row mask; larger
ones search a compacted copy of the selected rows, built like one add() of those rows, and map the
labels back on the device, so such a search returns what the same search of an index built from
only the selected rows returns.

Per-query exclusion lists: `search(x, k, exclude=(offsets, ids))` on the same three index types keeps
query q from returning any label in ids[offsets[q]:offsets[q+1]] (labels as for selectors; combines
with params). Each query is searched at k plus its list length and the listed labels are dropped on
the device by nrb_exclude_topk (_search_excluded).

Host code only: every array lives in HBM as torch tensors and all arithmetic is done by
libnrb200.so (hand-written sm_100a CUDA) through the C-ABI in include/nrb200.h. numpy in ->
numpy out (synchronous, like faiss); CUDA torch tensors in -> CUDA torch tensors out
(asynchronous on the current stream). No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import sys

import math

import numpy as np
import torch

from . import _lib
from ._lib import (METRIC_INNER_PRODUCT, METRIC_L2, PATH_AUTO, PATH_SIMT, PATH_TC, PATH_TC1, PATH_TC16, Matrix,
                   check, lib)

__all__ = [
    "METRIC_INNER_PRODUCT", "METRIC_L2", "IndexFlat", "IndexFlatL2", "IndexFlatIP", "IndexHNSWFlat",
    "IndexIVFFlat", "IndexIDMap", "IDSelectorBatch", "IDSelectorRange", "IDSelectorNot", "SearchParameters",
    "SearchParametersIVF", "Clustering", "ClusteringParameters", "vector_float_to_array", "normalize_L2",
]

_FLT_MAX = 3.4028234663852886e38
SMALL_NQ = 20  # faiss's distance_compute_blas_threshold: below it faiss itself leaves the GEMM route (SURVEY 3.2)
IVF_SMALL_NQ = 64  # IVF batches up to this size take the HBM-regime list scan (nrb_ivf_scan_small)
IVF_QUERY_BATCH = 262144  # queries per nrb_ivf_search call (bounds the regrouped query planes and partial rows: ~16 GB at nprobe 16, k 50)


# ------------------------------------------------------------------------------------ helpers
def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("newsrecommend_b200 needs a CUDA (sm_100) device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def _round_kp(d: int) -> int:
    return (d + 31) // 32 * 32


def _to_device_f32(x):
    """Returns (2-D fp32 CUDA tensor with unit column stride, came_from_numpy)."""
    if isinstance(x, torch.Tensor):
        t = x
        if t.dtype != torch.float32:
            t = t.float()
        if not t.is_cuda:
            t = t.to(_device(), non_blocking=True)
        from_np = False
    else:
        a = np.ascontiguousarray(x, dtype=np.float32)
        t = torch.from_numpy(a).to(_device(), non_blocking=True)
        from_np = True
    assert t.dim() == 2, "expected a 2-D array"
    if t.stride(1) != 1:
        t = t.contiguous()
    return t, from_np


def _to_host(t: torch.Tensor, out: np.ndarray | None = None) -> np.ndarray:
    """Device -> host. `out`: caller-provided array (faiss's search(x, k, D=None, I=None)
    convention); page-locked memory makes the copy a single async DMA."""
    if out is not None:
        assert out.shape == tuple(t.shape) and out.flags.c_contiguous, "bad output array"
        torch.from_numpy(out).copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out
    buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    buf.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return buf.numpy()


def _to_host_pair(D: torch.Tensor, I: torch.Tensor, Do=None, Io=None):
    """Both result arrays with one synchronisation."""
    if Do is None:
        Do = torch.empty(D.shape, dtype=D.dtype, pin_memory=True).numpy()
    if Io is None:
        Io = torch.empty(I.shape, dtype=I.dtype, pin_memory=True).numpy()
    assert Do.shape == tuple(D.shape) and Io.shape == tuple(I.shape) and Do.dtype == np.float32 and Io.dtype == np.int64
    torch.from_numpy(Do).copy_(D, non_blocking=True)
    torch.from_numpy(Io).copy_(I, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return Do, Io


_COPY_STREAMS: dict = {}


def _copy_streams():
    """(host-to-device, device-to-host) side streams of the current device."""
    dev = torch.cuda.current_device()
    if dev not in _COPY_STREAMS:
        _COPY_STREAMS[dev] = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
    return _COPY_STREAMS[dev]


_WAVE_ROWS: dict = {}


def _wave_rows() -> int:
    """Query rows of one full wave of the tcgen05 kernels: 256 per CTA pair."""
    dev = torch.cuda.current_device()
    if dev not in _WAVE_ROWS:
        n = C.c_int(0)
        ok = lib.nrb_device_info(C.byref(n), None, None) == 0 and n.value >= 2
        _WAVE_ROWS[dev] = (n.value if ok else 148) // 2 * 256
    return _WAVE_ROWS[dev]


def _h16_scale_for(max_norm: float) -> float:
    """Power of two s with max_norm * s in [2^14, 2^15): no element of a row can overflow fp16."""
    if not (max_norm > 0.0) or not math.isfinite(max_norm):
        return 1.0
    e = min(max(math.frexp(max_norm)[1] - 1, -60), 60)  # floor(log2(max_norm))
    return float(2.0 ** (14 - e))


class PackedMatrix:
    """Device form of a row-major fp32 matrix (struct nrb_matrix): zero-padded raw rows, tf32
    hi / lo planes, squared norms and the scaled fp16 plane of the fp16 filter. Grows
    geometrically on append. The fp16 plane carries ONE power-of-two scale for index storage
    (track_max_norm=True; re-packed from the raw plane if a later append outgrows it) and one
    scale per row for query batches."""

    def __init__(self, d: int, device=None, planes=("raw", "hi", "lo", "norms"), track_max_norm=False):
        self.d = d
        self.kp = _round_kp(d)
        self.n = 0
        self.device = device or _device()
        self.planes = tuple(planes)
        self._cap = 0
        self.raw = self.hi = self.lo = self.norms = self.h16 = self.row_scale = None
        # max row norm: the item side of the filter paths needs it; costs one small reduction +
        # sync per append, so only index storage tracks it
        self.track_max_norm = track_max_norm and "norms" in planes
        self.max_norm = 0.0
        self.h16_scale = 0.0
        if "h16" in self.planes and not self.track_max_norm:
            self.planes = self.planes + ("row_scale",)
        if "h16" in self.planes and self.track_max_norm:
            assert "raw" in self.planes, "the uniform-scale fp16 plane is (re)built from the raw plane"

    def _reserve(self, n: int):
        if n <= self._cap:
            return
        cap = max(n, int(self._cap * 1.5), 128)
        for name in self.planes:
            shape = (cap,) if name in ("norms", "row_scale") else (cap, self.kp)
            dtype = torch.float16 if name == "h16" else torch.float32
            new = torch.empty(shape, dtype=dtype, device=self.device)
            old = getattr(self, name)
            if old is not None and self.n:
                new[: self.n].copy_(old[: self.n])
            setattr(self, name, new)
        self._cap = cap

    def append(self, x: torch.Tensor):
        """x: fp32 CUDA [m, d] (row stride arbitrary)."""
        m = x.shape[0]
        assert x.shape[1] == self.d
        self._reserve(self.n + m)
        if m:
            off = self.n
            if any(p is not None for p in (self.raw, self.hi, self.lo, self.norms)):
                check(lib.nrb_pack_rows(
                    x.data_ptr(), m, self.d, x.stride(0), self.kp,
                    _ptr(self.raw[off:]) if self.raw is not None else 0,
                    _ptr(self.hi[off:]) if self.hi is not None else 0,
                    _ptr(self.lo[off:]) if self.lo is not None else 0,
                    _ptr(self.norms[off:]) if self.norms is not None else 0, _stream()), "pack_rows")
            if self.track_max_norm:
                self.max_norm = max(self.max_norm, float(self.norms[off:off + m].max().sqrt()))
            if self.h16 is not None:
                if self.track_max_norm:
                    # keep the current scale while the largest row still fits fp16 with headroom
                    if self.h16_scale > 0.0 and self.max_norm * self.h16_scale <= 60000.0:
                        lo_row, rows = off, m
                    else:
                        self.h16_scale = _h16_scale_for(self.max_norm)
                        lo_row, rows = 0, off + m
                    check(lib.nrb_pack_rows_h16(_ptr(self.raw[lo_row:]), rows, self.d, self.kp, self.kp,
                                                self.h16_scale, _ptr(self.h16[lo_row:]), 0, _stream()), "pack_rows_h16")
                else:
                    check(lib.nrb_pack_rows_h16(x.data_ptr(), m, self.d, x.stride(0), self.kp, 0.0,
                                                _ptr(self.h16[off:]), _ptr(self.row_scale[off:]), _stream()),
                          "pack_rows_h16")
        self.n += m

    def clear(self):
        self.n = 0
        self.max_norm = 0.0
        self.h16_scale = 0.0

    def struct(self) -> Matrix:
        m = Matrix()
        m.raw = _ptr(self.raw) if self.raw is not None else None
        m.hi = _ptr(self.hi) if self.hi is not None else None
        m.lo = _ptr(self.lo) if self.lo is not None else None
        m.norms = _ptr(self.norms) if self.norms is not None else None
        m.h16 = _ptr(self.h16) if self.h16 is not None else None
        m.h16_row_scale = _ptr(self.row_scale) if self.row_scale is not None else None
        m.h16_scale = self.h16_scale if self.h16 is not None else 0.0
        m.n, m.d, m.kp = self.n, self.d, self.kp
        m.max_norm = self.max_norm if self.track_max_norm else 0.0
        return m

    @classmethod
    def from_tensor(cls, x: torch.Tensor, planes=("raw", "hi", "lo", "norms")):
        p = cls(x.shape[1], x.device, planes)
        p.append(x)
        return p


def _search_flat_dev(q: PackedMatrix, b: PackedMatrix, metric: int, k: int, id_base: int = 0,
                     path: int = PATH_AUTO):
    """nrb_search_flat on packed matrices -> (D f32[nq,k], I i64[nq,k]) CUDA tensors."""
    nq = q.n
    D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    if nq == 0:
        return D, I
    wsb = lib.nrb_search_flat_workspace(nq, b.n, k, q.kp)
    ws = torch.empty(wsb, dtype=torch.uint8, device=q.device)
    qs, bs = q.struct(), b.struct()
    check(lib.nrb_search_flat(C.byref(qs), C.byref(bs), metric, k, id_base, D.data_ptr(), I.data_ptr(),
                              ws.data_ptr(), wsb, path, _stream()), "search_flat")
    return D, I


_INDEX_PLANES = ("raw", "hi", "lo", "norms", "h16")


# ------------------------------------------------------------------------------------ ids
class IDSelectorRange:
    """faiss.IDSelectorRange: selects imin <= id < imax. A host-side description that remove_ids
    hands to nrb_id_select; assume_sorted is accepted for faiss compatibility and changes nothing."""

    def __init__(self, imin: int, imax: int, assume_sorted: bool = False):
        self.imin, self.imax, self.assume_sorted = int(imin), int(imax), bool(assume_sorted)

    def is_member(self, i: int) -> bool:
        return self.imin <= i < self.imax


class IDSelectorBatch:
    """faiss.IDSelectorBatch: selects the ids of a set (duplicates allowed). IDSelectorBatch(ids),
    or faiss's SWIG form IDSelectorBatch(n, ids) with a numpy array in place of the pointer (the
    first n entries count)."""

    def __init__(self, *args):
        if len(args) == 2:
            n, ids = int(args[0]), _int64_ids(args[1], "IDSelectorBatch")
            if not 0 <= n <= ids.shape[0]:
                raise ValueError(f"IDSelectorBatch: n={n} but {ids.shape[0]} ids given")
            ids = ids[:n]
        elif len(args) == 1:
            ids = _int64_ids(args[0], "IDSelectorBatch")
        else:
            raise TypeError("IDSelectorBatch(ids) or IDSelectorBatch(n, ids)")
        self.ids = np.ascontiguousarray(ids)

    def is_member(self, i: int) -> bool:
        return bool(np.any(self.ids == i))


class IDSelectorNot:
    """faiss.IDSelectorNot: selects the ids `sel` does not. Evaluated as sel's own test with the keep
    sense flipped (nrb_id_select marks sel's members, the search keeps the others): no extra pass."""

    def __init__(self, sel):
        if not isinstance(sel, (IDSelectorRange, IDSelectorBatch, IDSelectorNot)):
            raise TypeError(f"IDSelectorNot wraps an IDSelectorRange, IDSelectorBatch or IDSelectorNot, not {type(sel)}")
        self.sel = sel

    def is_member(self, i: int) -> bool:
        return not self.sel.is_member(i)


class SearchParameters:
    """faiss.SearchParameters: per-call search options. sel (an IDSelector, or None) restricts the
    search to the rows it selects."""

    def __init__(self, sel=None, **fields):
        if fields:
            raise TypeError(f"{type(self).__name__}: unsupported field(s) {sorted(fields)}")
        if sel is not None and not isinstance(sel, (IDSelectorRange, IDSelectorBatch, IDSelectorNot)):
            raise TypeError(f"sel must be an IDSelectorRange, IDSelectorBatch or IDSelectorNot, not {type(sel)}")
        self.sel = sel


class SearchParametersIVF(SearchParameters):
    """faiss.SearchParametersIVF: sel as SearchParameters; nprobe, when set, replaces index.nprobe for
    the call. max_codes (a cap on scanned rows) is not supported: anything but 0 raises."""

    def __init__(self, sel=None, nprobe=None, max_codes=0, **fields):
        super().__init__(sel, **fields)
        if max_codes:
            raise NotImplementedError("SearchParametersIVF.max_codes is not supported (the scan is exhaustive)")
        self.nprobe = None if nprobe is None else int(nprobe)
        self.max_codes = 0


def _search_sel(params, ivf: bool):
    """(selector or None, nprobe override or None) of a search's params argument."""
    if params is None:
        return None, None
    if ivf and not isinstance(params, SearchParametersIVF):
        raise RuntimeError("IndexIVF params have incorrect type")
    if not isinstance(params, SearchParameters):
        raise TypeError(f"params must be a SearchParameters, not {type(params)}")
    return params.sel, getattr(params, "nprobe", None)


def _int64_ids(a, what: str) -> np.ndarray:
    """A 1-D host array of integer ids as int64 (floats are refused, not truncated)."""
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    a = np.asarray(a)
    if a.ndim != 1 or not (np.issubdtype(a.dtype, np.integer) or a.size == 0):
        raise TypeError(f"{what}: expected a 1-D integer id array, got {a.dtype} of shape {a.shape}")
    return a.astype(np.int64, copy=False)


def _selector(sel):
    """remove_ids' argument: an IDSelector, or an id array wrapped in IDSelectorBatch (faiss's
    Python layer does the same)."""
    if isinstance(sel, (IDSelectorBatch, IDSelectorRange, IDSelectorNot)):
        return sel
    if isinstance(sel, (np.ndarray, torch.Tensor)):
        return IDSelectorBatch(sel)
    raise TypeError("remove_ids takes an IDSelectorBatch, an IDSelectorRange, an IDSelectorNot or an int64 id array, "
                    f"not {type(sel)}")


def _unwrap_not(sel):
    """(innermost Range / Batch selector, keep): a row is selected when nrb_id_select's member value
    for that inner selector equals keep (1, or 0 under an odd number of IDSelectorNot)."""
    keep = 1
    while isinstance(sel, IDSelectorNot):
        sel, keep = sel.sel, 1 - keep
    if not isinstance(sel, (IDSelectorRange, IDSelectorBatch)):
        raise TypeError(f"expected an IDSelectorRange, IDSelectorBatch or IDSelectorNot, not {type(sel)}")
    return sel, keep


def _select(sel, ids, n: int, dev):
    """Row mask of a selector over n rows whose ids are ids (i64 CUDA tensor) or, when ids is None,
    the row positions: (member i64 CUDA tensor from nrb_id_select, keep); row i is selected when
    member[i] == keep. Queued on the current stream, no synchronisation."""
    base, keep = _unwrap_not(sel)
    member = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    if isinstance(base, IDSelectorRange):
        batch, nb, imin, imax = None, 0, base.imin, base.imax
    else:
        batch = torch.from_numpy(base.ids).to(dev) if base.ids.size else None
        nb, imin, imax = base.ids.size, 0, 0
    wsb = lib.nrb_id_select_workspace(nb)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=dev)
    check(lib.nrb_id_select(_ptr(ids), n, _ptr(batch), nb, imin, imax, member.data_ptr(), ws.data_ptr(), wsb,
                            _stream()), "id_select")
    return member, keep


def _selected_rows(sel, ids, n: int, dev, selected: bool = True) -> torch.Tensor:
    """The rows a selector picks (selected=True) or leaves (False), in their old order, as an i32
    CUDA tensor: nrb_id_select marks the rows, nrb_ivf_build_lists with two buckets partitions them
    stably (member 0 first). Reads one count back, so it synchronises the stream."""
    member, keep = _select(sel, ids, n, dev)
    offsets = torch.empty(3, dtype=torch.int32, device=dev)
    order = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    wsb = lib.nrb_ivf_build_lists_workspace(n, 2)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    check(lib.nrb_ivf_build_lists(member.data_ptr(), n, 2, offsets.data_ptr(), order.data_ptr(), ws.data_ptr(), wsb,
                                  _stream()), "ivf_build_lists")
    n0 = int(_to_host(offsets[1:2])[0])
    return order[:n0] if (keep if selected else 1 - keep) == 0 else order[n0:n]


def _keep_partition(sel, ids, n: int, dev):
    """remove_ids' stable partition: (order i32 CUDA tensor of the rows sel does not select, number
    of rows it selects); synchronises the stream once."""
    order = _selected_rows(sel, ids, n, dev, selected=False)
    return order, n - order.shape[0]


def _positions_kept(sel, n: int):
    """Number of row positions 0..n-1 a selector keeps, worked out on the host (no device work)."""
    base, keep = _unwrap_not(sel)
    if isinstance(base, IDSelectorRange):
        c = max(0, min(base.imax, n) - max(base.imin, 0))
    else:
        c = np.unique(base.ids[(base.ids >= 0) & (base.ids < n)]).size
    return c if keep else n - c


def _padding(nq: int, k: int, metric: int, dev):
    """The result of a search with no row to return: I = -1, D = -FLT_MAX (IP) / +FLT_MAX (L2)."""
    D = torch.full((nq, k), _FLT_MAX if metric == METRIC_L2 else -_FLT_MAX, dtype=torch.float32, device=dev)
    return D, torch.full((nq, k), -1, dtype=torch.int64, device=dev)


def _gather_i64(src: torch.Tensor, order: torch.Tensor) -> torch.Tensor:
    dst = torch.empty(order.shape[0], dtype=torch.int64, device=src.device)
    check(lib.nrb_gather_i64(src.data_ptr(), order.data_ptr(), order.shape[0], dst.data_ptr(), _stream()),
          "gather_i64")
    return dst


def _gather_packed(p: PackedMatrix, order: torch.Tensor) -> PackedMatrix:
    """The rows order[:] of p's raw plane appended to a fresh PackedMatrix with p's planes: every
    plane, max_norm and h16_scale come out as if those rows had been added in one call."""
    n = order.shape[0]
    raw = torch.empty((n, p.kp), dtype=torch.float32, device=p.device)
    check(lib.nrb_gather_rows(p.raw.data_ptr(), p.kp, order.data_ptr(), n, raw.data_ptr(), _stream()), "gather_rows")
    out = PackedMatrix(p.d, p.device, planes=p.planes, track_max_norm=p.track_max_norm)
    out.append(raw[:, : p.d])
    return out


def _ids_arg(ids, n: int, dev) -> torch.Tensor:
    """add_with_ids' ids: an int64 numpy array or torch tensor of length n -> i64 CUDA tensor."""
    if isinstance(ids, np.ndarray):
        ok = ids.dtype == np.int64
        t = torch.from_numpy(np.ascontiguousarray(ids)) if ok else None
    elif isinstance(ids, torch.Tensor):
        ok, t = ids.dtype == torch.int64, ids
    else:
        ok = False
    if not ok or t.dim() != 1 or t.shape[0] != n:
        raise TypeError(f"add_with_ids: ids must be an int64 numpy array or tensor of length {n}")
    return t.to(dev, non_blocking=True).contiguous()


def _map_ids(id_map: torch.Tensor | None, I: torch.Tensor):
    """IndexIDMap's label translation on the current stream, in place: I = id_map[I] where I >= 0."""
    if id_map is not None and id_map.numel():
        check(lib.nrb_map_ids(id_map.data_ptr(), I.data_ptr(), I.numel(), _stream()), "map_ids")


# ------------------------------------------------------------------------------------ exclusion lists
_FILTER_MAX_K = 112  # the fp16 filter's k bound (_query_planes, IndexIVFFlat.search's eligibility check)


def _exclude_arg(exclude, nq: int):
    """search()'s exclude=(offsets, ids): a CSR pair of int64 numpy arrays or tensors, checked before any
    device work. Returns (offsets as a host int64 array, offsets, ids)."""
    if not isinstance(exclude, (tuple, list)) or len(exclude) != 2:
        raise TypeError("exclude must be a pair (offsets, ids) of int64 arrays")
    arrs = []
    for a, what in zip(exclude, ("offsets", "ids")):
        if isinstance(a, torch.Tensor):
            ok = a.dtype == torch.int64
        elif isinstance(a, np.ndarray):
            ok = a.dtype == np.int64
        else:
            ok = False
        if not ok:
            raise TypeError(f"exclude: {what} must be an int64 numpy array or tensor, not {getattr(a, 'dtype', type(a))}")
        if a.ndim != 1:
            raise ValueError(f"exclude: {what} must be 1-D, got shape {tuple(a.shape)}")
        arrs.append(a)
    off, ids = arrs
    off_h = off.detach().cpu().numpy() if isinstance(off, torch.Tensor) else off
    if off_h.shape[0] != nq + 1:
        raise ValueError(f"exclude: offsets has {off_h.shape[0]} entries for {nq} queries (needs nq + 1)")
    if off_h[0] != 0 or off_h[-1] != ids.shape[0]:
        raise ValueError(f"exclude: offsets must run from 0 to len(ids) = {ids.shape[0]}, "
                         f"not {int(off_h[0])} .. {int(off_h[-1])}")
    if (np.diff(off_h) < 0).any():
        raise ValueError("exclude: offsets decrease")
    return off_h, off, ids


def _exclude_to_device(off_h, off, ids, dev):
    """The checked CSR pair as i64 CUDA tensors (offsets, ids)."""
    off_d = off.to(dev) if isinstance(off, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(off_h)).to(dev)
    ids_d = ids.to(dev) if isinstance(ids, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(ids)).to(dev)
    if ids_d.numel() == 0:
        ids_d = torch.empty(1, dtype=torch.int64, device=dev)  # never read; keeps the pointer valid
    return off_d.contiguous(), ids_d.contiguous()


def _list_member(row_ids, n: int, ids_d: torch.Tensor, lo: int, hi: int, sel_mask, dev):
    """Row mask of one query's exclusion list ids_d[lo:hi] over n rows whose labels are row_ids (i64
    CUDA tensor, or None for row positions), ANDed with a selector's mask sel_mask = _select(...) or None:
    (member, keep = 0) in the form the masked kernels take. The AND is nrb_sel_keys with the list's
    member as key and 1 as the drop value: a row scans when the selector keeps it and the list misses it."""
    nb = hi - lo
    member = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    wsb = lib.nrb_id_select_workspace(nb)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=dev)
    check(lib.nrb_id_select(_ptr(row_ids), n, ids_d.data_ptr() + 8 * lo if nb else None, nb, 0, 0, member.data_ptr(),
                            ws.data_ptr(), wsb, _stream()), "id_select")
    if sel_mask is not None:
        both = torch.empty_like(member)
        check(lib.nrb_sel_keys(sel_mask[0].data_ptr(), sel_mask[1], member.data_ptr(), n, 1, both.data_ptr(),
                               _stream()), "sel_keys")
        member = both
    return member, 0


def _search_excluded(t: torch.Tensor, k: int, metric: int, exclude, group_search, long_search):
    """search(..., exclude=(offsets, ids)) over the CUDA query batch t -> (D, I) CUDA tensors; exclude is
    what _exclude_arg returned.

    Query q's list holds E_q = offsets[q+1] - offsets[q] labels (duplicates counted). At most E_q of its
    top k + E_q rows are excluded, so the survivors hold the exact top k of the rows it may see. The
    queries with k + E_q <= 112 (the fp16 filter's bound) form one group and those with 112 < k + E_q <=
    128 another; each group is gathered and searched once by group_search(x, k') at k' = k + its longest
    list, and nrb_exclude_topk drops the listed labels and scatters the group's first k survivors into
    its rows of D, I. A query with k + E_q > 128 (MAX_K) cannot over-fetch: long_search(x_q, lo, hi)
    scans it alone with its list as a row mask."""
    nq, dev = t.shape[0], t.device
    off_h = exclude[0]
    off_d, ids_d = _exclude_to_device(*exclude, dev)
    D = torch.empty((nq, k), dtype=torch.float32, device=dev)
    I = torch.empty((nq, k), dtype=torch.int64, device=dev)
    need = k + np.diff(off_h)
    for group in (need <= _FILTER_MAX_K, (need > _FILTER_MAX_K) & (need <= _lib.MAX_K)):
        rows = np.nonzero(group)[0]
        if rows.size == 0:
            continue
        kq = int(need[rows].max())
        if rows.size == nq:
            qidx, xg = None, t
        else:
            qidx = torch.from_numpy(rows.astype(np.int64)).to(dev)
            xg = t.index_select(0, qidx)
        Dg, Ig = group_search(xg, kq)
        check(lib.nrb_exclude_topk(Dg.data_ptr(), Ig.data_ptr(), rows.size, kq, _ptr(qidx), off_d.data_ptr(),
                                   ids_d.data_ptr(), metric, k, D.data_ptr(), I.data_ptr(), _stream()), "exclude_topk")
    for q in np.nonzero(need > _lib.MAX_K)[0]:
        Dq, Iq = long_search(t[q:q + 1], int(off_h[q]), int(off_h[q + 1]), ids_d)
        D[q].copy_(Dq[0])
        I[q].copy_(Iq[0])
    return D, I


# ------------------------------------------------------------------------------------ flat
class IndexFlat:
    """IndexFlatL2 / IndexFlatIP (Retrieval.py:25-26,32; SURVEY 8b). add() copies into HBM."""

    def __init__(self, d: int, metric: int = METRIC_L2):
        self.d = int(d)
        self.metric_type = metric
        self.is_trained = True
        self.verbose = False
        # PATH_AUTO: fp16 filter + exact fp32 refine (PATH_TC16) when eligible (d <= 256, k <= 112),
        # else 3xTF32 (PATH_TC); PATH_TC1 = the same filter on the tf32 hi planes, PATH_TC forces
        # 3xTF32, PATH_SIMT the fp32 CUDA-core kernels
        self.path = PATH_AUTO
        self.small_nq = SMALL_NQ  # batches below this take the low-latency exact path (0 disables it)
        self._xb: PackedMatrix | None = None
        self._struct_cache = None

    @property
    def ntotal(self) -> int:
        return 0 if self._xb is None else self._xb.n

    def train(self, x):
        pass

    def add(self, x):
        t, _ = _to_device_f32(x)
        assert t.shape[1] == self.d
        if self._xb is None:
            self._xb = PackedMatrix(self.d, t.device, planes=_INDEX_PLANES, track_max_norm=True)
        self._xb.append(t)
        self._struct_cache = None

    def reset(self):
        if self._xb is not None:
            self._xb.clear()
        self._struct_cache = None

    def _struct(self) -> Matrix:
        """struct nrb_matrix of the stored rows, cached between add() calls (the per-call cost of
        the low-latency path is a handful of microseconds; rebuilding six tensor views is not)."""
        if self._struct_cache is None:
            self._struct_cache = self._packed().struct()
        return self._struct_cache

    def _search_small_host(self, a: np.ndarray, k: int, D=None, I=None, member=None, keep: int = 1):
        """nq < 20, numpy in / numpy out (the call Retrieval.py:32 makes 50,000 times with nq = 1):
        ONE C-ABI call -- staged H2D, the row-per-warp fp32 kernels, D2H, one sync. member / keep:
        the row mask of a selector (_select), scanned by the masked kernels."""
        nq = a.shape[0]
        if D is None:
            D = np.empty((nq, k), dtype=np.float32)
        if I is None:
            I = np.empty((nq, k), dtype=np.int64)
        assert D.shape == (nq, k) and I.shape == (nq, k) and D.dtype == np.float32 and I.dtype == np.int64
        assert D.flags.c_contiguous and I.flags.c_contiguous, "bad output array"
        if member is None:
            check(lib.nrb_search_small_host(C.byref(self._struct()), a.ctypes.data, nq, self.d, self.metric_type, k, 0,
                                            D.ctypes.data, I.ctypes.data, _stream()), "search_small_host")
        else:
            check(lib.nrb_search_small_host_sel(C.byref(self._struct()), a.ctypes.data, nq, self.d, self.metric_type, k,
                                                0, D.ctypes.data, I.ctypes.data, _stream(), member.data_ptr(), keep),
                  "search_small_host_sel")
        return D, I

    def _search_small_dev(self, t: torch.Tensor, k: int, id_base: int = 0, member=None, keep: int = 1):
        """The same route for a CUDA tensor batch: asynchronous on the current stream."""
        nq = t.shape[0]
        D = torch.empty((nq, k), dtype=torch.float32, device=t.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=t.device)
        wsb = lib.nrb_search_small_workspace(nq, self.ntotal, k)
        ws = torch.empty(wsb, dtype=torch.uint8, device=t.device)
        if member is None:
            check(lib.nrb_search_small(t.data_ptr(), t.stride(0), nq, self.d, C.byref(self._struct()), self.metric_type,
                                       k, id_base, D.data_ptr(), I.data_ptr(), ws.data_ptr(), wsb, _stream()),
                  "search_small")
        else:
            check(lib.nrb_search_small_sel(t.data_ptr(), t.stride(0), nq, self.d, C.byref(self._struct()),
                                           self.metric_type, k, id_base, D.data_ptr(), I.data_ptr(), ws.data_ptr(), wsb,
                                           _stream(), member.data_ptr(), keep), "search_small_sel")
        return D, I

    def _packed(self) -> PackedMatrix:
        if self._xb is None:
            self._xb = PackedMatrix(self.d, planes=_INDEX_PLANES, track_max_norm=True)
        return self._xb

    def search_packed(self, q: PackedMatrix, k: int, id_base: int = 0):
        if self.ntotal == 0:
            # faiss on an empty index: I = -1, D = +/-FLT_MAX (also what an empty catalog shard returns)
            nq = q.n
            D = torch.full((nq, k), _FLT_MAX if self.metric_type == METRIC_L2 else -_FLT_MAX,
                           dtype=torch.float32, device=q.device)
            return D, torch.full((nq, k), -1, dtype=torch.int64, device=q.device)
        return _search_flat_dev(q, self._packed(), self.metric_type, k, id_base, self.path)

    def add_with_ids(self, x, ids):
        raise RuntimeError("add_with_ids not implemented for this type of index")

    def remove_ids(self, sel) -> int:
        """faiss IndexFlatCodes::remove_ids: `sel` selects row positions. The rows after each removed
        row move up (a stable compaction), and the storage is rebuilt as one add() of the survivors,
        so max_norm and the fp16 scale shrink with them. Returns the number of rows removed."""
        n = self.ntotal
        if n == 0:
            _selector(sel)
            return 0
        order, removed = _keep_partition(_selector(sel), None, n, self._xb.device)
        if removed:
            self._keep_rows(order)
        return removed

    def _keep_rows(self, order: torch.Tensor):
        self._xb = _gather_packed(self._xb, order)
        self._struct_cache = None

    def search(self, x, k: int, D=None, I=None, *, params=None, exclude=None):
        """(D, I) = search(x, k). Like faiss, optional preallocated numpy outputs D f32[nq,k],
        I i64[nq,k] are filled and returned (page-locked buffers avoid a staging copy).
        params: SearchParameters (or SearchParametersIVF) whose sel selects row positions.
        exclude: (offsets i64[nq+1], ids i64) CSR lists, numpy or tensors; query q returns no row
        position in ids[offsets[q]:offsets[q+1]] (a -1 or an absent id excludes nothing)."""
        sel, _ = _search_sel(params, False)
        if exclude is not None:
            return self._search_exclude(x, k, D, I, None, sel, exclude)
        if sel is not None:
            return self._search_filtered(x, k, D, I, None, sel)
        return self._search(x, k, D, I, None)

    def _search_exclude(self, x, k: int, D, I, id_map: torch.Tensor | None, sel, exclude):
        """search() with per-query exclusion lists (_search_excluded): the lists and sel test
        id_map[row] (IndexIDMap) or the row position. Numpy batches take one copy in and one copy back;
        the pipelined host route is not used."""
        assert k > 0
        if k > _lib.MAX_K:
            raise RuntimeError(f"k={k} > {_lib.MAX_K} is not supported by the selection stage")
        k, n = int(k), self.ntotal
        nq = x.shape[0] if isinstance(x, torch.Tensor) else np.asarray(x).shape[0]
        ex = _exclude_arg(exclude, nq)
        if n == 0 or nq == 0:
            return self._search_filtered(x, k, D, I, id_map, sel) if sel is not None else self._search(x, k, D, I, id_map)
        t, from_np = _to_device_f32(x)
        assert t.shape[1] == self.d
        dev = t.device
        sel_mask = []

        def group_search(xg, kq):
            if sel is not None:
                return self._search_filtered(xg, kq, None, None, id_map, sel)
            return self._search(xg, kq, None, None, id_map)

        def long_search(xq, lo, hi, ids_d):
            if sel is not None and not sel_mask:
                sel_mask.append(_select(sel, id_map, n, dev))
            member, keep = _list_member(id_map, n, ids_d, lo, hi, sel_mask[0] if sel_mask else None, dev)
            Dq, Iq = self._search_small_dev(xq, k, member=member, keep=keep)
            _map_ids(id_map, Iq)
            return Dq, Iq

        Dd, Id = _search_excluded(t, k, self.metric_type, ex, group_search, long_search)
        if from_np or D is not None or I is not None:
            return _to_host_pair(Dd, Id, D, I)
        return Dd, Id

    def _search_filtered(self, x, k: int, D, I, id_map: torch.Tensor | None, sel):
        """search() over the rows sel selects; sel tests id_map[row] (IndexIDMap) or the row position.
        Batches that would take the low-latency route (nq < small_nq) scan the whole index with the
        row mask (the masked HBM-regime kernels). Every other batch searches a compacted subset: the
        selected rows in their order, re-packed as one add() of those rows (own max_norm and fp16
        scale), on the unchanged route, and its labels go back through one nrb_map_ids."""
        assert k > 0
        if k > _lib.MAX_K:
            raise RuntimeError(f"k={k} > {_lib.MAX_K} is not supported by the selection stage")
        k, n = int(k), self.ntotal
        nq = x.shape[0] if isinstance(x, torch.Tensor) else np.asarray(x).shape[0]
        if n == 0 or nq == 0:
            _unwrap_not(sel)
            return self._search(x, k, D, I, id_map)
        dev = self._xb.device
        if self.small_nq and self.path == PATH_AUTO and nq < self.small_nq:
            if id_map is None and _positions_kept(sel, n) == 0:
                subset, labels = None, None
            else:
                member, keep = _select(sel, id_map, n, dev)
                if not isinstance(x, torch.Tensor) and id_map is None:
                    a = np.ascontiguousarray(x, dtype=np.float32)
                    assert a.ndim == 2 and a.shape[1] == self.d
                    return self._search_small_host(a, k, D, I, member, keep)
                t, from_np = _to_device_f32(x)
                assert t.shape[1] == self.d
                Dd, Id = self._search_small_dev(t, k, member=member, keep=keep)
                _map_ids(id_map, Id)
                if from_np or D is not None or I is not None:
                    return _to_host_pair(Dd, Id, D, I)
                return Dd, Id
        else:
            rows = _selected_rows(sel, id_map, n, dev)
            if rows.shape[0] == n:  # every row: the index itself
                subset, labels = self, id_map
            elif rows.shape[0] == 0:
                subset, labels = None, None
            else:
                subset = IndexFlat(self.d, self.metric_type)
                subset.path, subset.small_nq = self.path, self.small_nq
                subset._xb = _gather_packed(self._xb, rows)
                labels = rows.long() if id_map is None else _gather_i64(id_map, rows)
        if subset is not None:
            return subset._search(x, k, D, I, labels)
        # no row selected: no search
        Dd, Id = _padding(nq, k, self.metric_type, dev)
        if not isinstance(x, torch.Tensor) or D is not None or I is not None:
            return _to_host_pair(Dd, Id, D, I)
        return Dd, Id

    def _search(self, x, k: int, D, I, id_map: torch.Tensor | None):
        """search(); id_map (IndexIDMap): labels are translated on the device before any copy back."""
        assert k > 0
        if k > _lib.MAX_K:
            raise RuntimeError(f"k={k} > {_lib.MAX_K} is not supported by the selection stage")
        small = self.small_nq and self.path == PATH_AUTO and 0 < self.ntotal
        if not isinstance(x, torch.Tensor) and torch.cuda.is_available():
            a = np.ascontiguousarray(x, dtype=np.float32)
            assert a.ndim == 2 and a.shape[1] == self.d
            if small and 0 < a.shape[0] < self.small_nq and id_map is None:
                return self._search_small_host(a, int(k), D, I)
            if a.shape[0] >= 2 * _wave_rows():
                return self._search_host_pipelined(a, int(k), D, I, id_map)
        t, from_np = _to_device_f32(x)
        assert t.shape[1] == self.d
        if small and 0 < t.shape[0] < self.small_nq:
            Dd, Id = self._search_small_dev(t, int(k))
            _map_ids(id_map, Id)
            if from_np or D is not None or I is not None:
                return _to_host_pair(Dd, Id, D, I)
            return Dd, Id
        q = PackedMatrix.from_tensor(t, planes=self._query_planes(int(k)))
        Dd, Id = self.search_packed(q, int(k))
        _map_ids(id_map, Id)
        if from_np or D is not None or I is not None:
            return _to_host_pair(Dd, Id, D, I)
        return Dd, Id

    def _search_host_pipelined(self, a: np.ndarray, k: int, D=None, I=None, id_map=None):
        """Host arrays in, host arrays out, for batches of at least two waves: the batch is cut at
        wave boundaries (one wave = one 256-query unit pair per CTA pair, so the cuts cost the
        kernel nothing), all host-to-device copies are queued on a copy stream up front, and each
        chunk's results travel back on a third stream while the next chunk is being searched."""
        nq = a.shape[0]
        dev = _device()
        if D is None:
            D = torch.empty((nq, k), dtype=torch.float32, pin_memory=True).numpy()
        if I is None:
            I = torch.empty((nq, k), dtype=torch.int64, pin_memory=True).numpy()
        assert D.shape == (nq, k) and I.shape == (nq, k) and D.dtype == np.float32 and I.dtype == np.int64
        assert D.flags.c_contiguous and I.flags.c_contiguous, "bad output array"
        step = _wave_rows()
        cuts = list(range(0, nq, step))
        if len(cuts) > 1 and nq - cuts[-1] < step // 4:
            cuts.pop()  # a sliver at the end rides with the previous chunk
        bounds = [(lo, cuts[i + 1] if i + 1 < len(cuts) else nq) for i, lo in enumerate(cuts)]
        cur = torch.cuda.current_stream()
        h2d, d2h = _copy_streams()
        h2d.wait_stream(cur)
        src = torch.from_numpy(a)
        staged, keep = [], []
        with torch.cuda.stream(h2d):
            for lo, hi in bounds:
                xd = torch.empty((hi - lo, self.d), dtype=torch.float32, device=dev)
                xd.copy_(src[lo:hi], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(h2d)
                staged.append((xd, ev))
        Dt, It = torch.from_numpy(D), torch.from_numpy(I)
        planes = self._query_planes(k)
        for (lo, hi), (xd, ev) in zip(bounds, staged):
            cur.wait_event(ev)
            xd.record_stream(cur)
            q = PackedMatrix.from_tensor(xd, planes=planes)
            Dd, Id = self.search_packed(q, k)
            _map_ids(id_map, Id)
            done = torch.cuda.Event()
            done.record(cur)
            with torch.cuda.stream(d2h):
                d2h.wait_event(done)
                Dt[lo:hi].copy_(Dd, non_blocking=True)
                It[lo:hi].copy_(Id, non_blocking=True)
            Dd.record_stream(d2h)
            Id.record_stream(d2h)
            keep.append((q, Dd, Id))
        d2h.synchronize()
        cur.wait_stream(d2h)
        return D, I

    def _query_planes(self, k: int = 1):
        """Planes the chosen path reads on the query side (mirrors the eligibility rule of
        nrb_search_flat; queries flagged by a filter are re-split from the raw plane)."""
        filt_ok = _round_kp(self.d) <= 256 and k <= 112 and self._packed().max_norm > 0.0  # empty / all-zero index
        if self.path == PATH_TC16 or (self.path == PATH_AUTO and filt_ok):
            return ("raw", "norms", "h16")
        if self.path == PATH_TC1:
            return ("raw", "hi", "norms")
        need = ("raw",) if self.path == PATH_SIMT else ("hi", "lo")
        return need + (("norms",) if self.metric_type == METRIC_L2 else ())

    def assign(self, x, k: int = 1):
        return self.search(x, k)[1]

    def reconstruct_n(self, i0: int = 0, n: int | None = None) -> np.ndarray:
        n = self.ntotal - i0 if n is None else n
        return _to_host(self._packed().raw[i0:i0 + n, : self.d].contiguous())


class IndexFlatL2(IndexFlat):
    def __init__(self, d: int):
        super().__init__(d, METRIC_L2)


class IndexFlatIP(IndexFlat):
    def __init__(self, d: int):
        super().__init__(d, METRIC_INNER_PRODUCT)


class IndexIDMap:
    """faiss.IndexIDMap over an empty IndexFlat (or subclass): rows carry caller-given int64 ids, such
    as the article ids that Retrieval.py:7 splits off the embedding table and Retrieval.py:23 maps
    rows back to by hand. The ids live on the device beside the rows; search() runs the inner
    index's own route (the same D on every path) and translates labels with nrb_map_ids on the
    current stream before any copy back; -1 stays -1. Numpy batches of fewer than 20 queries cannot
    take the single-call host route (its kernels write straight into host memory), so they run the
    device route, the translation and one copy back: a few microseconds more per call than the plain
    index. IndexIVFFlat carries ids of its own (add_with_ids) and is not wrapped."""

    def __init__(self, index):
        if not isinstance(index, IndexFlat):
            raise TypeError(f"IndexIDMap wraps an IndexFlat (IndexFlatIP, IndexFlatL2); {type(index).__name__} "
                            "is not supported (IndexIVFFlat has add_with_ids of its own)")
        if index.ntotal != 0:
            raise RuntimeError("index must be empty on input")
        self.index = index
        self.id_map: torch.Tensor | None = None  # i64[ntotal] on the device, row order

    ntotal = property(lambda self: self.index.ntotal)
    d = property(lambda self: self.index.d)
    metric_type = property(lambda self: self.index.metric_type)
    is_trained = property(lambda self: self.index.is_trained)

    def train(self, x):
        self.index.train(x)

    def add(self, x):
        raise RuntimeError("add does not make sense with IndexIDMap, use add_with_ids")

    def add_with_ids(self, x, ids):
        t, _ = _to_device_f32(x)
        assert t.shape[1] == self.d
        ids_d = _ids_arg(ids, t.shape[0], t.device)
        self.index.add(t)
        self.id_map = ids_d if self.id_map is None or self.id_map.numel() == 0 else torch.cat([self.id_map, ids_d])

    def search(self, x, k: int, D=None, I=None, *, params=None, exclude=None):
        """params: SearchParameters whose sel selects external ids (faiss's IDSelectorTranslated).
        exclude: (offsets, ids) CSR lists of external ids, as IndexFlat.search takes them."""
        sel, _ = _search_sel(params, False)
        if exclude is not None:
            return self.index._search_exclude(x, k, D, I, self.id_map if self.ntotal else None, sel, exclude)
        if sel is not None:
            return self.index._search_filtered(x, k, D, I, self.id_map if self.ntotal else None, sel)
        return self.index._search(x, k, D, I, self.id_map if self.ntotal else None)

    def remove_ids(self, sel) -> int:
        """faiss IndexIDMapTemplate::remove_ids: selects on the external ids, compacts the inner
        index and the id map with the same stable partition. Returns the number of rows removed."""
        sel = _selector(sel)
        n = self.ntotal
        if n == 0:
            return 0
        order, removed = _keep_partition(sel, self.id_map, n, self.id_map.device)
        if removed:
            self.index._keep_rows(order)
            self.id_map = _gather_i64(self.id_map, order)
        return removed

    def reset(self):
        self.index.reset()
        self.id_map = None


class IndexHNSWFlat(IndexFlatL2):
    """Accepted for Retrieval.py:16. The reference uses HNSW(M=32) only as the k-means assigner
    over <= 325 centroids; its parallel graph build is nondeterministic, so it cannot be
    reproduced bit for bit even by faiss itself. Here it is an EXACT L2 index (what
    IndexIVFFlat.train uses); documented divergence, SURVEY 8a row a3."""

    def __init__(self, d: int, M: int = 32):
        super().__init__(d)
        self.M = M


# ------------------------------------------------------------------------------------ k-means
class ClusteringParameters:
    def __init__(self):
        self.niter = 25
        self.nredo = 1
        self.verbose = False
        self.spherical = False
        self.int_centroids = False
        self.update_index = False
        self.frozen_centroids = False
        self.min_points_per_centroid = 39
        self.max_points_per_centroid = 256
        self.seed = 1234
        self.decode_block_size = 32768


class ClusteringIterationStats:
    def __init__(self, obj, imbalance_factor, nsplit):
        self.obj = obj
        self.imbalance_factor = imbalance_factor
        self.nsplit = nsplit


def rand_perm(n: int, seed: int) -> np.ndarray:
    """faiss::rand_perm through the C-ABI host helper (std::mt19937)."""
    perm = np.empty(n, dtype=np.int32)
    check(lib.nrb_rand_perm_host(perm.ctypes.data, n, seed), "rand_perm")
    return perm


def kmeans_update(x: PackedMatrix, assign: torch.Tensor, k: int):
    """One centroid update (K1b): returns (centroids f32[k,d], hassign f32[k]) CUDA tensors."""
    cent = torch.empty((k, x.d), dtype=torch.float32, device=x.device)
    hassign = torch.empty((k,), dtype=torch.float32, device=x.device)
    wsb = lib.nrb_kmeans_update_workspace(x.n, k, x.kp)
    ws = torch.empty(wsb, dtype=torch.uint8, device=x.device)
    check(lib.nrb_kmeans_update(x.raw.data_ptr(), x.n, x.d, x.kp, assign.data_ptr(), k, cent.data_ptr(),
                                hassign.data_ptr(), ws.data_ptr(), wsb, _stream()), "kmeans_update")
    return cent, hassign


class Clustering(ClusteringParameters):
    """faiss.Clustering(d, k) as used at Retrieval.py:12-19: Lloyd k-means with faiss's
    subsampling (256*k rows, rand_perm seed), random-row init (seed+1), mean update and
    empty-cluster split. Assignment = exact search on `index` (K2 with k=1), update = K1b."""

    def __init__(self, d: int, k: int, cp: ClusteringParameters | None = None):
        super().__init__()
        if cp is not None:
            self.__dict__.update(cp.__dict__)
        self.d = int(d)
        self.k = int(k)
        self.centroids = np.empty(0, dtype=np.float32)
        self.iteration_stats = []
        self.trace = None  # hook(it, centroids_in, assign, centroids_out) with numpy arrays

    def train(self, x, index):
        t, _ = _to_device_f32(x)
        n, d = t.shape
        k = self.k
        assert d == self.d
        if n < k:
            raise RuntimeError("Number of training points (%d) should be at least as large as number of "
                               "clusters (%d)" % (n, k))
        if not bool(torch.isfinite(t).all()):
            raise RuntimeError("input contains NaN's or Inf's")
        dev = t.device
        if n > k * self.max_points_per_centroid:
            perm = rand_perm(n, self.seed)[: k * self.max_points_per_centroid]
            sel = torch.from_numpy(perm.astype(np.int64)).to(dev)
            t = t.index_select(0, sel)
            n = t.shape[0]
        elif n < k * self.min_points_per_centroid:
            print("WARNING clustering %d points to %d centroids: please provide at least %d training points"
                  % (n, k, k * self.min_points_per_centroid), file=sys.stderr)
        if n == k:
            self.centroids = _to_host(t.contiguous()).reshape(-1)
            index.reset()
            index.add(t)
            return
        # rows for the assignment kernel: scaled fp16 plane (fp16 filter + exact refine) when d <= 256,
        # else tf32 hi / lo planes (3xTF32)
        xs = PackedMatrix.from_tensor(t, planes=("raw", "norms", "h16") if _round_kp(d) <= 256 else ("raw", "hi", "lo", "norms"))
        x_max_norm = float(xs.norms[:n].max().sqrt())  # the one host read before the loop: sizes the filter margin
        best = None
        for redo in range(self.nredo):
            perm = rand_perm(n, self.seed + 1 + redo * 15486557)[:k]
            cent = t.index_select(0, torch.from_numpy(perm.astype(np.int64)).to(dev)).contiguous()
            if self.spherical:
                check(lib.nrb_normalize_l2(cent.data_ptr(), k, d, d, _stream()), "normalize_l2")
            # the whole iteration loop is ONE C-ABI call queued on the stream (nrb_kmeans_train): pack
            # centroids, K2 assignment (k = 1), objective, K1b update, device split_clusters; the only
            # host synchronisation is the read of the per-iteration statistics at the end. A trace hook
            # (teacher-forced parity tests) runs the same call one iteration at a time.
            metric = index.metric_type
            wsb = lib.nrb_kmeans_train_workspace(n, k, xs.kp)
            ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
            st_dev = torch.zeros((max(self.niter, 1), 4), dtype=torch.float64, device=dev)
            xs_struct = xs.struct()
            xs_struct.max_norm = x_max_norm
            assign = torch.empty(n, dtype=torch.int64, device=dev) if self.trace is not None else None

            def run(it0, its):
                check(lib.nrb_kmeans_train(C.byref(xs_struct), k, its, metric, 1 if self.spherical else 0,
                                           cent.data_ptr(), _ptr(assign), st_dev[it0:].data_ptr(), ws.data_ptr(), wsb,
                                           _stream()), "kmeans_train")

            if self.trace is None:
                run(0, self.niter)
            else:
                for it in range(self.niter):
                    cent_in = _to_host(cent)
                    run(it, 1)
                    self.trace(it, cent_in, _to_host(assign), _to_host(cent))
            sh = _to_host(st_dev)
            if (sh[: self.niter, 2] < 0).any():
                raise RuntimeError("split_clusters: no cluster to split")
            stats = [ClusteringIterationStats(float(np.float32(sh[it, 0])), float(sh[it, 1]), int(sh[it, 2]))
                     for it in range(self.niter)]
            obj = stats[-1].obj if stats else 0.0
            if self.verbose:
                for it, s_ in enumerate(stats):
                    print("  Iteration %d objective=%g imbalance=%.3f nsplit=%d" % (it, s_.obj, s_.imbalance_factor, s_.nsplit))
            index.reset()
            index.add(cent)
            if self.nredo > 1:
                better = best is None or (obj > best[0] if index.metric_type == METRIC_INNER_PRODUCT
                                          else obj < best[0])
                if better:
                    best = (obj, cent.clone(), stats)
            else:
                best = (obj, cent, stats)
        _, cent, stats = best
        if self.nredo > 1:
            index.reset()
            index.add(cent)
        self.centroids = _to_host(cent).reshape(-1)
        self.iteration_stats = stats


def vector_float_to_array(v) -> np.ndarray:
    """Retrieval.py:19 -- copy of the centroid vector as a numpy array."""
    return np.array(v, dtype=np.float32, copy=True)


def normalize_L2(x):
    """faiss.normalize_L2: in place on a numpy array or CUDA tensor; zero rows untouched."""
    if isinstance(x, torch.Tensor) and x.is_cuda:
        assert x.dim() == 2 and x.stride(1) == 1 and x.dtype == torch.float32
        check(lib.nrb_normalize_l2(x.data_ptr(), x.shape[0], x.shape[1], x.stride(0), _stream()), "normalize_l2")
        return
    assert isinstance(x, np.ndarray) and x.dtype == np.float32 and x.ndim == 2
    t = torch.from_numpy(np.ascontiguousarray(x)).to(_device())
    check(lib.nrb_normalize_l2(t.data_ptr(), t.shape[0], t.shape[1], t.stride(0), _stream()), "normalize_l2")
    x[...] = _to_host(t)


# ------------------------------------------------------------------------------------ IVF
class IndexIVFFlat:
    """IndexIVFFlat(quantizer, d, nlist, metric): train = k-means on the quantizer (cp.niter =
    10), add = nearest centroid + list-contiguous layout, search = coarse top-nprobe + list
    scan (SURVEY 3.3). In the reference this is the hand-rolled k-means -> cluster_to_articles
    -> nearest-centroid pipeline of Retrieval.py:11-34.

    Every row carries an int64 id: add() numbers rows ntotal, ntotal+1, ... as faiss does (also after
    removals), add_with_ids() stores the ids given, remove_ids() drops rows by id. The lists keep
    rows in insertion order, so with arbitrary ids exact score ties come out in list-position
    order, where faiss orders them by id."""

    def __init__(self, quantizer: IndexFlat, d: int, nlist: int, metric: int = METRIC_L2):
        self.quantizer = quantizer
        self.d = int(d)
        self.nlist = int(nlist)
        self.metric_type = metric
        self.nprobe = 1
        self.is_trained = False
        self.verbose = False
        self.path = PATH_AUTO
        self.cp = ClusteringParameters()
        self.cp.niter = 10
        self.clustering = None
        self._x: PackedMatrix | None = None   # rows in insertion order (raw plane only)
        self._assign = None                   # i64[ntotal] list of every row
        self._ids = None                      # i64[ntotal] id of every row
        self._lists = None                    # dict built lazily: packed planes in list order

    @property
    def ntotal(self) -> int:
        return 0 if self._x is None else self._x.n

    def train(self, x):
        if self.quantizer.is_trained and self.quantizer.ntotal == self.nlist:
            self.is_trained = True
            return
        clus = Clustering(self.d, self.nlist, self.cp)
        clus.verbose = self.verbose or self.cp.verbose
        self.quantizer.reset()
        clus.train(x, self.quantizer)
        self.clustering = clus
        self.is_trained = True

    def add(self, x):
        self.add_with_ids(x, None)

    def add_with_ids(self, x, ids):
        """ids: int64 numpy array or tensor of length n; None numbers the rows from ntotal."""
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        t, _ = _to_device_f32(x)
        assert t.shape[1] == self.d
        n0 = self.ntotal
        ids = torch.arange(n0, n0 + t.shape[0], dtype=torch.int64, device=t.device) if ids is None else \
            _ids_arg(ids, t.shape[0], t.device)
        if self._x is None:
            self._x = PackedMatrix(self.d, t.device, planes=("raw",))
        q = PackedMatrix.from_tensor(t, planes=self.quantizer._query_planes(1))
        _, a = self.quantizer.search_packed(q, 1)
        a = a.reshape(-1)
        self._assign = a if self._assign is None or n0 == 0 else torch.cat([self._assign, a])
        self._ids = ids if self._ids is None or n0 == 0 else torch.cat([self._ids, ids])
        self._x.append(t)
        self._lists = None

    def remove_ids(self, sel) -> int:
        """faiss IndexIVF::remove_ids: selects on the row ids; the rows, their lists and their ids are
        compacted with one stable partition and the lists are rebuilt on the next search, as after
        add(). Returns the number of rows removed."""
        sel = _selector(sel)
        n = self.ntotal
        if n == 0:
            return 0
        order, removed = _keep_partition(sel, self._ids, n, self._x.device)
        if removed:
            self._x = _gather_packed(self._x, order)
            self._assign = _gather_i64(self._assign, order)
            self._ids = _gather_i64(self._ids, order)
            self._lists = None
        return removed

    def reset(self):
        if self._x is not None:
            self._x.clear()
        self._assign = None
        self._ids = None
        self._lists = None

    def _build_lists(self):
        if self._lists is None:
            self._lists = self._pack_lists(self._assign, self.nlist)
        return self._lists

    def _filtered_lists(self, sel):
        """The lists of the rows sel selects (by stored id), not cached: nrb_sel_keys sends every
        other row to an extra bucket nlist that is never packed. The counting sort is stable, so
        each list holds its selected rows in the order of the unfiltered list, and the planes come
        out as those of an index built from the selected rows alone."""
        n, dev = self.ntotal, self._x.device
        member, keep = _select(sel, self._ids, n, dev)
        key = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        check(lib.nrb_sel_keys(member.data_ptr(), keep, self._assign.data_ptr(), n, self.nlist, key.data_ptr(),
                               _stream()), "sel_keys")
        return self._pack_lists(key, self.nlist + 1)

    def _pack_lists(self, key: torch.Tensor, nbuckets: int):
        """List-contiguous planes of the rows whose key (i64[ntotal], in [0, nbuckets)) is below
        nlist: a stable counting sort by key, a gather of those rows, hi / lo / norms and the
        scaled fp16 plane. nbuckets > nlist: the rows of the extra buckets are left out."""
        n, dev = self.ntotal, self._x.device
        offsets = torch.empty(nbuckets + 1, dtype=torch.int32, device=dev)
        order = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        wsb = lib.nrb_ivf_build_lists_workspace(n, nbuckets)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        check(lib.nrb_ivf_build_lists(key.data_ptr(), n, nbuckets, offsets.data_ptr(),
                                      order.data_ptr(), ws.data_ptr(), wsb, _stream()), "ivf_build_lists")
        off_h = _to_host(offsets[: self.nlist + 1]).astype(np.int64)
        n = int(off_h[-1])  # rows in lists 0 .. nlist-1
        kp = self._x.kp
        raw = torch.empty((max(n, 1), kp), dtype=torch.float32, device=dev)
        check(lib.nrb_gather_rows(self._x.raw.data_ptr(), kp, order.data_ptr(), n, raw.data_ptr(), _stream()),
              "gather_rows")
        packed = PackedMatrix(self.d, dev)
        packed._reserve(max(n, 1))  # a filter may keep no row
        packed.raw = raw  # already list-ordered and padded; derive hi / lo / norms from it
        check(lib.nrb_pack_rows(raw.data_ptr(), n, self.d, kp, kp, 0, packed.hi.data_ptr(), packed.lo.data_ptr(),
                                packed.norms.data_ptr(), _stream()), "pack_rows")
        packed.n = n
        # scaled fp16 plane + max norm: the fp16 filter of the list scan (NRB_PATH_TC16)
        if n:
            packed.track_max_norm = True
            packed.max_norm = float(packed.norms[:n].max().sqrt())
            if packed.max_norm > 0.0:
                packed.h16 = torch.empty((n, kp), dtype=torch.float16, device=dev)
                packed.h16_scale = _h16_scale_for(packed.max_norm)
                check(lib.nrb_pack_rows_h16(raw.data_ptr(), n, self.d, kp, kp, packed.h16_scale,
                                            packed.h16.data_ptr(), 0, _stream()), "pack_rows_h16")
        ids = _gather_i64(self._ids, order[:n])
        sizes = np.diff(off_h)
        return dict(packed=packed, ids=ids, offsets=offsets[: self.nlist + 1], offsets_host=off_h,
                    max_len=int(sizes.max()) if sizes.size else 0)

    def list_sizes(self) -> np.ndarray:
        return np.diff(self._build_lists()["offsets_host"])

    def search(self, x, k: int, *, params=None, exclude=None):
        """params: SearchParametersIVF. Its sel selects stored ids: the coarse search still ranks
        every centroid, and the scan of the nprobe lists skips the rows sel does not select. Its
        nprobe, when set, replaces index.nprobe for this call.
        exclude: (offsets, ids) CSR lists of stored ids, as IndexFlat.search takes them."""
        sel, nprobe_p = _search_sel(params, True)
        if exclude is not None:
            return self._search_exclude(x, k, params, sel, nprobe_p, exclude)
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        t, from_np = _to_device_f32(x)
        assert t.shape[1] == self.d
        assert k > 0
        nprobe = min(int(self.nprobe if nprobe_p is None else nprobe_p), self.nlist)
        if k > _lib.MAX_K or nprobe > _lib.MAX_K:
            raise RuntimeError(f"k / nprobe > {_lib.MAX_K} is not supported by the selection stage")
        nq, dev = t.shape[0], t.device
        D = torch.empty((nq, k), dtype=torch.float32, device=dev)
        I = torch.empty((nq, k), dtype=torch.int64, device=dev)
        if self.ntotal == 0:
            D.fill_(3.4028234663852886e38 if self.metric_type == METRIC_L2 else -3.4028234663852886e38)
            I.fill_(-1)
        elif nq:
            small = self.path == PATH_AUTO and nq <= IVF_SMALL_NQ and nq * nprobe <= 65535 and self.quantizer.ntotal
            # a selector: the small route masks the cached lists, the batch route scans lists of the
            # selected rows only
            L = self._build_lists() if sel is None or small else self._filtered_lists(sel)
            if L["packed"].n == 0:  # the selector keeps no row: no search
                D.fill_(3.4028234663852886e38 if self.metric_type == METRIC_L2 else -3.4028234663852886e38)
                I.fill_(-1)
                nq = 0
            # PATH_AUTO: fp16 filter + exact refine over the lists when eligible (raw, norms, h16 for
            # the filter; hi, lo for the queries it flags), else the 3xTF32 scan
            filt = self.path in (PATH_AUTO, PATH_TC16) and L["packed"].h16 is not None and k <= 112 and \
                _round_kp(self.d) <= 256
            planes = ("raw",) if self.path == PATH_SIMT else ("hi", "lo")
            planes = tuple(dict.fromkeys(planes + self.quantizer._query_planes(nprobe) +
                                         (("raw", "norms", "h16") if filt else ()) +
                                         (("norms",) if self.metric_type == METRIC_L2 else ())))
            ls = L["packed"].struct()
            if small and nq:
                self._scan_small(t, int(k), nprobe, L, D, I,
                                 None if sel is None else _select(sel, L["ids"], self.ntotal, dev))  # list order
                nq = 0  # done
            for q0 in range(0, nq, IVF_QUERY_BATCH):
                q1 = min(nq, q0 + IVF_QUERY_BATCH)
                q = PackedMatrix.from_tensor(t[q0:q1], planes=planes)
                _, coarse = self.quantizer.search_packed(q, nprobe)
                wsb = lib.nrb_ivf_search_workspace(q.n, nprobe, k, q.kp, self.nlist, L["max_len"])
                ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
                qs = q.struct()
                check(lib.nrb_ivf_search(C.byref(qs), C.byref(ls), L["offsets"].data_ptr(), self.nlist,
                                         L["max_len"], L["ids"].data_ptr(), coarse.data_ptr(), nprobe,
                                         self.metric_type, int(k), D[q0:q1].data_ptr(), I[q0:q1].data_ptr(),
                                         ws.data_ptr(), wsb, self.path, _stream()), "ivf_search")
        if from_np:
            return _to_host_pair(D, I)
        return D, I

    def _scan_small(self, t: torch.Tensor, k: int, nprobe: int, L, D: torch.Tensor, I: torch.Tensor, mask=None):
        """HBM-regime route for small batches: exact fp32 coarse search + row-per-warp list scan of the
        lists L into D, I. mask: (member, keep) over the packed list rows, or None (every row)."""
        nq = t.shape[0]
        _, coarse = self.quantizer._search_small_dev(t, nprobe) if nq < SMALL_NQ else self.quantizer.search(t, nprobe)
        wsb = lib.nrb_ivf_scan_small_workspace(nq, nprobe, L["max_len"], self.ntotal, k)
        ws = torch.empty(wsb, dtype=torch.uint8, device=t.device)
        ls = L["packed"].struct()
        args = (t.data_ptr(), t.stride(0), nq, self.d, C.byref(ls), L["offsets"].data_ptr(), self.nlist,
                L["max_len"], L["ids"].data_ptr(), coarse.data_ptr(), nprobe, self.metric_type, k,
                D.data_ptr(), I.data_ptr(), ws.data_ptr(), wsb, _stream())
        if mask is None:
            check(lib.nrb_ivf_scan_small(*args), "ivf_scan_small")
        else:
            check(lib.nrb_ivf_scan_small_sel(*args, mask[0].data_ptr(), mask[1]), "ivf_scan_small_sel")

    def _search_exclude(self, x, k: int, params, sel, nprobe_p, exclude):
        """search() with per-query exclusion lists (_search_excluded) of stored ids. The long group
        scans the cached lists with the list's row mask (and sel's) on the small route."""
        nq = x.shape[0] if isinstance(x, torch.Tensor) else np.asarray(x).shape[0]
        ex = _exclude_arg(exclude, nq)
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        assert k > 0
        k = int(k)
        nprobe = min(int(self.nprobe if nprobe_p is None else nprobe_p), self.nlist)
        if k > _lib.MAX_K or nprobe > _lib.MAX_K:
            raise RuntimeError(f"k / nprobe > {_lib.MAX_K} is not supported by the selection stage")
        t, from_np = _to_device_f32(x)
        assert t.shape[1] == self.d
        dev = t.device
        if self.ntotal == 0 or nq == 0:
            D, I = self.search(t, k, params=params)
        else:
            sel_mask = []

            def long_search(xq, lo, hi, ids_d):
                L = self._build_lists()
                if sel is not None and not sel_mask:
                    sel_mask.append(_select(sel, L["ids"], self.ntotal, dev))
                mask = _list_member(L["ids"], self.ntotal, ids_d, lo, hi, sel_mask[0] if sel_mask else None, dev)
                Dq = torch.empty((1, k), dtype=torch.float32, device=dev)
                Iq = torch.empty((1, k), dtype=torch.int64, device=dev)
                self._scan_small(xq, k, nprobe, L, Dq, Iq, mask)
                return Dq, Iq

            D, I = _search_excluded(t, k, self.metric_type, ex,
                                    lambda xg, kq: self.search(xg, kq, params=params), long_search)
        if from_np:
            return _to_host_pair(D, I)
        return D, I
