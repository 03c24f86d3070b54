"""Per-query exclusion lists (search(..., exclude=(offsets, ids))) restated in numpy on top of the CPU
oracle (test infrastructure only).

exclude_topk restates nrb_exclude_topk: row r of an over-fetched result (query qidx[r], or r) drops
every entry whose label is >= 0 and in the query's list, and keeps its first k survivors in order; the
rest is padding (I = -1, D = -FLT_MAX for IP, +FLT_MAX for L2).

search_excluded restates the whole feature: query q is searched at k + E_q (E_q = its list length,
duplicates counted), its listed labels are dropped and the first k survivors kept. At most E_q of the
top k + E_q are excluded, so this is the top k of the rows the query may see."""
import numpy as np

FLT_MAX = np.float32(3.4028234663852886e38)


def exclude_topk(Din, Iin, qidx, off, ids, metric, k, D, I):
    """nrb_exclude_topk into D, I (f32 / i64 [nq, k], written in the rows the qidx entries name)."""
    pad = FLT_MAX if metric == 1 else -FLT_MAX
    for r in range(Din.shape[0]):
        q = r if qidx is None else int(qidx[r])
        lst = ids[off[q]:off[q + 1]]
        keep = ~((Iin[r] >= 0) & np.isin(Iin[r], lst))
        d, i = Din[r][keep][:k], Iin[r][keep][:k]
        D[q], I[q] = pad, -1
        D[q, :d.size], I[q, :i.size] = d, i
    return D, I


def search_excluded(search, x, k, off, ids, metric):
    """search(x, k) -> (D, I) of an oracle index (padding past its rows); every query over-fetches by
    its own list length, in one call per distinct k + E_q."""
    nq = x.shape[0]
    need = k + np.diff(off)
    D = np.empty((nq, k), dtype=np.float32)
    I = np.empty((nq, k), dtype=np.int64)
    for kq in np.unique(need):
        rows = np.nonzero(need == kq)[0]
        Dg, Ig = search(x[rows], int(kq))
        exclude_topk(np.asarray(Dg), np.asarray(Ig), rows, off, ids, metric, k, D, I)
    return D, I


def csr(lists):
    """(offsets, ids) int64 CSR of a list of id lists."""
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(l) for l in lists], out=off[1:])
    ids = np.concatenate([np.asarray(l, dtype=np.int64) for l in lists]) if lists else np.empty(0, np.int64)
    return off, ids.astype(np.int64)
