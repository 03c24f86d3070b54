"""Synthetic data of the Tianchi-news shape (SURVEY.md section 8d). The reference ships no data
(`news/` is git-ignored, /root/reference/.gitignore:1-2), so every test and benchmark uses
these seeded generators; the same numpy arrays go to the oracle and to the GPU path.

G-skew reproduces the list-size skew of the README centroid table (readme.md:17-22); plain
Gaussian data makes faiss-style k-means degenerate (SURVEY Appendix B-E2).
"""
from __future__ import annotations

import numpy as np

N_ARTICLES = 364_047   # Retrieval.py:7
N_TEST_USERS = 50_000  # utils.py:17
D_RAW = 250            # articles_emb.csv width


def g_iso(n: int, d: int, seed: int) -> np.ndarray:
    return np.random.default_rng(seed).standard_normal((n, d), dtype=np.float32)


def g_skew(n: int, d: int, seed: int, n_topics: int = 461, r: int = 16, zipf: float = 0.8,
           within: float = 0.7, noise: float = 0.02, return_topics: bool = False):
    """Low-rank (r latent dims) mixture of `n_topics` topics with Zipf(zipf) weights."""
    rng = np.random.default_rng(seed)
    w = 1.0 / np.arange(1, n_topics + 1) ** zipf
    w /= w.sum()
    comp = rng.choice(n_topics, size=n, p=w)
    centers = rng.standard_normal((n_topics, r)).astype(np.float32)
    z = centers[comp] + within * rng.standard_normal((n, r), dtype=np.float32)
    q, _ = np.linalg.qr(rng.standard_normal((d, r)))
    W = q.T.astype(np.float32)  # r x d, orthonormal rows
    x = z @ W + noise * rng.standard_normal((n, d), dtype=np.float32)
    x = np.ascontiguousarray(x, dtype=np.float32)
    return (x, comp) if return_topics else x


def user_profiles(items: np.ndarray, topics: np.ndarray | None, n_users: int, seed: int,
                  mean_clicks: float = 6.5, max_clicks: int = 64, return_clicks: bool = False):
    """Mean of L clicked item rows, L ~ clip(Geometric(1/mean_clicks), 1, max_clicks); 70 % of a
    user's clicks come from one topic, 30 % uniformly (the dataset has ~6.5 clicks per user,
    others/data_analysis.ipynb:1868,1981). return_clicks: also return the click history as CSR,
    (offsets i64[n_users+1], clicked rows i64), user u's clicks being rows[offsets[u]:offsets[u+1]]
    (a row clicked twice appears twice); the profiles are the same either way."""
    rng = np.random.default_rng(seed)
    n = items.shape[0]
    L = np.clip(rng.geometric(1.0 / mean_clicks, size=n_users), 1, max_clicks)
    total = int(L.sum())
    owner = np.repeat(np.arange(n_users), L)
    picks = rng.integers(0, n, size=total)
    if topics is not None:
        order = np.argsort(topics, kind="stable")
        st = topics[order]
        n_topics = int(topics.max()) + 1
        bounds = np.searchsorted(st, np.arange(n_topics + 1))
        sizes = np.maximum(np.diff(bounds), 1)
        fav = topics[rng.integers(0, n, size=n_users)]  # favourite topic ~ topic popularity
        in_topic = rng.random(total) < 0.7
        ft = fav[owner]
        local = (rng.random(total) * sizes[ft]).astype(np.int64)
        tpick = order[np.minimum(bounds[ft] + local, n - 1)]
        picks = np.where(in_topic, tpick, picks)
    out = np.zeros((n_users, items.shape[1]), dtype=np.float32)
    np.add.at(out, owner, items[picks])
    out /= L[:, None].astype(np.float32)
    if return_clicks:
        offsets = np.zeros(n_users + 1, dtype=np.int64)
        np.cumsum(L, out=offsets[1:])
        return out, (offsets, picks.astype(np.int64, copy=False))
    return out
