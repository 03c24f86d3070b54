"""faiss's external-id semantics restated in numpy on top of the CPU oracle (test infrastructure
only): IndexFlat.remove_ids, IndexIVFFlat.add_with_ids / remove_ids, IndexIDMap, IDSelectorBatch /
IDSelectorRange. Everything else is oracle.faiss_oracle's, re-exported unchanged, so the module
stands in for the oracle in the id tests."""
import numpy as np

from oracle import faiss_oracle as fo
from oracle.faiss_oracle import *  # noqa: F401,F403


class IDSelectorRange:
    """IDSelectorRange: imin <= id < imax."""

    def __init__(self, imin, imax, assume_sorted=False):
        self.imin, self.imax = int(imin), int(imax)

    def members(self, ids):
        ids = np.asarray(ids, dtype=np.int64)
        return (ids >= self.imin) & (ids < self.imax)


class IDSelectorBatch:
    """IDSelectorBatch(ids) or the SWIG form IDSelectorBatch(n, ids): membership in a set of ids
    (faiss adds a Bloom filter in front of the set; it changes no answer)."""

    def __init__(self, *args):
        ids = np.asarray(args[-1], dtype=np.int64).reshape(-1)
        if len(args) == 2:
            ids = ids[:int(args[0])]
        self.ids = ids

    def members(self, ids):
        return np.isin(np.asarray(ids, dtype=np.int64), self.ids)


class _IDSelectorTranslated:
    """IDSelectorTranslated: position i is selected when id_map[i] is."""

    def __init__(self, id_map, sel):
        self.id_map, self.sel = id_map, sel

    def members(self, pos):
        return self.sel.members(self.id_map[np.asarray(pos, dtype=np.int64)])


def _as_selector(sel):
    """faiss's Python layer wraps a plain id array in IDSelectorBatch."""
    if hasattr(sel, "members"):
        return sel
    sel = np.asarray(sel)
    assert sel.ndim == 1
    return IDSelectorBatch(sel.size, sel)


class IndexFlat(fo.IndexFlat):
    def add_with_ids(self, x, ids):
        raise RuntimeError("add_with_ids not implemented for this type of index")

    def remove_ids(self, sel):
        """IndexFlatCodes::remove_ids: sel selects row POSITIONS; the survivors move up in order
        (stable compaction), so rows are renumbered. Returns the number removed."""
        keep = ~_as_selector(sel).members(np.arange(self.ntotal, dtype=np.int64))
        nremove = int(self.ntotal - keep.sum())
        self.xb = np.ascontiguousarray(self.xb[keep])
        return nremove


class IndexFlatL2(IndexFlat):
    def __init__(self, d):
        super().__init__(d, fo.METRIC_L2)


class IndexFlatIP(IndexFlat):
    def __init__(self, d):
        super().__init__(d, fo.METRIC_INNER_PRODUCT)


class IndexIDMap:
    """IndexIDMapTemplate<Index>: the wrapped index holds the rows, id_map[i] the id of row i."""

    def __init__(self, index):
        if index.ntotal != 0:
            raise RuntimeError("index must be empty on input")
        self.index = index
        self.id_map = np.empty(0, dtype=np.int64)

    @property
    def ntotal(self):
        return self.index.ntotal

    def add(self, x):
        raise RuntimeError("add does not make sense with IndexIDMap, use add_with_ids")

    def add_with_ids(self, x, ids):
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        assert ids.shape[0] == np.asarray(x).shape[0]
        self.index.add(x)
        self.id_map = np.concatenate([self.id_map, ids])

    def search(self, x, k):
        D, I = self.index.search(x, k)
        if self.id_map.size:
            I = np.where(I < 0, I, self.id_map[np.maximum(I, 0)])
        return D, I

    def remove_ids(self, sel):
        sel = _as_selector(sel)
        nremove = self.index.remove_ids(_IDSelectorTranslated(self.id_map, sel))
        self.id_map = self.id_map[~sel.members(self.id_map)]
        return nremove

    def reset(self):
        self.index.reset()
        self.id_map = np.empty(0, dtype=np.int64)


class IndexIVFFlat(fo.IndexIVFFlat):
    def add_with_ids(self, x, ids):
        """IndexIVF::add_with_ids: add() with the ids given instead of ntotal, ntotal + 1, ..."""
        if not self.is_trained:
            raise RuntimeError("Error: 'is_trained' failed")
        x = fo._as_f32(x)
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        assert ids.shape[0] == x.shape[0]
        assign = self.quantizer.assign(x, 1).reshape(-1)
        order = np.argsort(assign, kind="stable")
        bounds = np.searchsorted(assign[order], np.arange(self.nlist + 1))
        for l in range(self.nlist):
            sel = order[bounds[l]:bounds[l + 1]]
            if sel.size:
                self._lists[l].append((ids[sel], x[sel]))
        self.ntotal += x.shape[0]
        self._csr = None

    def remove_ids(self, sel):
        """IndexIVF::remove_ids, literally: in each list, an entry whose id is selected is
        overwritten by the list's last entry and the list shrinks by one, so list order is NOT
        preserved. Returns the number removed."""
        sel = _as_selector(sel)
        nremove = 0
        for l in range(self.nlist):
            if not self._lists[l]:
                continue
            ids = np.concatenate([c[0] for c in self._lists[l]])
            rows = np.concatenate([c[1] for c in self._lists[l]])
            hit = sel.members(ids)
            size, j = ids.shape[0], 0
            while j < size:
                if hit[j]:
                    size -= 1
                    ids[j], rows[j], hit[j] = ids[size], rows[size], hit[size]
                else:
                    j += 1
            nremove += ids.shape[0] - size
            self._lists[l] = [(ids[:size].copy(), rows[:size].copy())] if size else []
        self.ntotal -= nremove
        self._csr = None
        return nremove
