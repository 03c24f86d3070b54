"""Generates the committed golden fixtures from the oracle and fp64 brute force. faiss itself is
not importable in this image (SURVEY.md section 8c), so the fixtures pin the ORACLE (a later edit
that changes its answers fails tests/test_oracle.py::test_golden_*), and the GPU tests compare
against the same files. The inputs are not stored: tests/golden_inputs.py rebuilds them from their
seeds and checks them against the digest recorded here. Run: python tests/golden/make_golden.py"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import golden_inputs  # noqa: E402
from oracle import faiss_oracle as fo  # noqa: E402


def save(name, inputs, **answers):
    np.savez_compressed(os.path.join(HERE, name + ".npz"), inputs_sha256=golden_inputs.digest(inputs), **answers)


g = golden_inputs.flat_small()
out = {}
for metric in (0, 1):
    D, I = fo.knn(g["xq"], g["xb"], 10, metric)
    Dt, It = fo.truth_topk(g["xq"], g["xb"], 10, metric)
    out[f"D{metric}"], out[f"I{metric}"], out[f"Dt{metric}"], out[f"It{metric}"] = D, I, Dt, It
save("flat_small", g, **out)
np.savez(os.path.join(HERE, "rand_perm.npz"), perm20_seed1234=fo.rand_perm(20, 1234))

# k-means: 3 teacher-forced iterations on a small skewed mixture
g = golden_inputs.kmeans_small()
clus = fo.Clustering(64, 20)
clus.niter = 3
trace = []
clus.trace = lambda it, cin, a, cout: trace.append((cin.copy(), a.copy(), cout.copy()))
clus.train(g["x"], fo.IndexFlatL2(64))
assert np.array_equal(clus.subsample(g["x"]), g["xs"])  # the iterations ran on the subsample
save("kmeans_small", g, cin=np.stack([t[0] for t in trace]), assign=np.stack([t[1] for t in trace]),
     cout=np.stack([t[2] for t in trace]), centroids=clus.centroids)
# IVF-Flat: trained centroids, list sizes and nprobe = 4 results for both metrics
g = golden_inputs.ivf_small()
ivf_out = {}
for metric, qcls in ((0, fo.IndexFlatIP), (1, fo.IndexFlatL2)):
    quant = qcls(64)
    ivf = fo.IndexIVFFlat(quant, 64, 16, metric)
    ivf.train(g["xb"])
    ivf.add(g["xb"])
    ivf.nprobe = 4
    D, I = ivf.search(g["xq"], 10)
    ivf_out[f"cent{metric}"] = quant.xb.copy()
    ivf_out[f"sizes{metric}"] = ivf.list_sizes()
    ivf_out[f"D{metric}"], ivf_out[f"I{metric}"] = D, I
save("ivf_small", g, **ivf_out)
print("golden fixtures written")
