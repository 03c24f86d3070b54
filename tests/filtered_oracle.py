"""faiss's search-time selector semantics (SearchParameters::sel) restated in numpy on top of the
CPU oracle (test infrastructure only). IDSelectorNot, and filtered search of the flat, IndexIDMap
and IndexIVFFlat oracle indexes of tests/ids_oracle.py:
  - flat: the selector tests row positions, every unselected row is skipped;
  - IndexIDMap: it tests the external ids (faiss wraps it in IDSelectorTranslated);
  - IndexIVFFlat: it tests the stored ids; the coarse search ranks every centroid, only the scan of
    the probed lists skips unselected rows.
Fewer than k selected rows: the tail is padded with I = -1, D = -FLT_MAX (IP) / +FLT_MAX (L2)."""
import copy

import numpy as np

import ids_oracle as io
from oracle import faiss_oracle as fo


class IDSelectorNot:
    """IDSelectorNot: the ids `sel` does not select."""

    def __init__(self, sel):
        self.sel = sel

    def members(self, ids):
        return ~self.sel.members(ids)


def search_flat(index, x, k, sel):
    """IndexFlat::search with SearchParameters(sel=sel): sel tests positions 0 .. ntotal-1."""
    pos = np.nonzero(sel.members(np.arange(index.ntotal, dtype=np.int64)))[0]
    sub = fo.IndexFlat(index.d, index.metric_type)
    sub.add(index.xb[pos] if pos.size else np.empty((0, index.d), np.float32))
    D, I = sub.search(x, k) if pos.size else _padded(np.asarray(x).shape[0], k, index.metric_type)
    return D, np.where(I < 0, -1, pos[np.maximum(I, 0)] if pos.size else -1)


def search_idmap(index, x, k, sel):
    """IndexIDMap::search with sel on the external ids (IDSelectorTranslated)."""
    D, I = search_flat(index.index, x, k, io._IDSelectorTranslated(index.id_map, sel))
    return D, np.where(I < 0, -1, index.id_map[np.maximum(I, 0)] if index.id_map.size else -1)


def filtered_ivf(index, sel):
    """A view of an oracle IndexIVFFlat whose lists hold only the rows sel selects (list order kept)
    and whose quantizer is the original: its search() is IndexIVF::search with sel, and it can be
    handed to code that reads the lists (_build_csr)."""
    off, ids, rows = index._build_csr()
    keep = sel.members(ids)
    sizes = np.array([keep[off[l]:off[l + 1]].sum() for l in range(index.nlist)], dtype=np.int64)
    foff = np.zeros(index.nlist + 1, dtype=np.int64)
    np.cumsum(sizes, out=foff[1:])
    view = copy.copy(index)
    view._csr = (foff, np.ascontiguousarray(ids[keep]), np.ascontiguousarray(rows[keep]))
    view._build_csr = lambda: view._csr
    view.ntotal = int(keep.sum())
    return view


def search_ivf(index, x, k, sel, nprobe=None):
    view = filtered_ivf(index, sel)
    if nprobe is not None:
        view.nprobe = nprobe
    return view.search(x, k)


def _padded(nq, k, metric):
    return (np.full((nq, k), -3.4028235e38 if metric == 0 else 3.4028235e38, dtype=np.float32),
            np.full((nq, k), -1, dtype=np.int64))
