"""Inputs of the golden fixtures in tests/golden/, rebuilt from their seeds.

The .npz files hold the oracle's answers and the sha256 of the inputs they were computed from, not
the inputs themselves (random float32 matrices do not compress, and each fixture would exceed 1 MB).
load() regenerates the inputs, refuses them if their digest differs from the recorded one, and
returns inputs and answers in one dict keyed like the fixture. Every generator here uses numpy's
seeded Generator and elementwise float32 arithmetic only: no BLAS or LAPACK call, whose rounding
depends on the CPU kernel it dispatches to, so the inputs are the same bits on every machine."""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def skew(n, d, seed, n_topics=40, r=8, within=0.7, noise=0.02):
    """Low-rank (r latent dims) mixture of Zipf-weighted topics, like synth.g_skew, with a random
    Gaussian basis instead of g_skew's QR and the projection done as r elementwise updates."""
    rng = np.random.default_rng(seed)
    w = 1.0 / np.arange(1, n_topics + 1)
    comp = rng.choice(n_topics, size=n, p=w / w.sum())
    centers = rng.standard_normal((n_topics, r), dtype=np.float32)
    z = centers[comp] + within * rng.standard_normal((n, r), dtype=np.float32)
    basis = rng.standard_normal((r, d), dtype=np.float32) / np.float32(np.sqrt(d))
    x = noise * rng.standard_normal((n, d), dtype=np.float32)
    for j in range(r):
        x += z[:, j, None] * basis[j]
    return x, comp


def flat_small():
    rng = np.random.default_rng(20261018)
    xb = rng.standard_normal((2000, 250), dtype=np.float32)
    xq = rng.standard_normal((48, 250), dtype=np.float32)
    return dict(xb=xb, xq=xq)


def kmeans_small():
    """x, and xs: the rows k-means iterates on (20 centroids x 256 points < 6000 rows -> faiss's
    rand_perm(1234) subsample)."""
    from oracle import faiss_oracle as fo
    x, _ = skew(6000, 64, 7)
    return dict(x=x, xs=x[fo.rand_perm(x.shape[0], 1234)[:20 * 256]])


def ivf_small():
    from newsrecommend_b200 import synth
    xb, topics = skew(8000, 64, 11)
    return dict(xb=xb, xq=synth.user_profiles(xb, topics, 64, 12))


INPUTS = {"flat_small": flat_small, "kmeans_small": kmeans_small, "ivf_small": ivf_small}


def digest(inputs):
    h = hashlib.sha256()
    for name in sorted(inputs):
        a = np.ascontiguousarray(inputs[name])
        h.update(f"{name}:{a.dtype.str}:{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def load(name):
    inputs = INPUTS[name]()
    with np.load(os.path.join(GOLDEN, name + ".npz")) as f:
        out = {k: f[k] for k in f.files}
    want = str(out.pop("inputs_sha256"))
    assert digest(inputs) == want, f"{name}: regenerated inputs differ from the ones the fixture was computed on"
    out.update(inputs)
    return out
