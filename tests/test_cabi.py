"""CPU-side checks of the C-ABI library: it loads without a GPU, exports every symbol that
include/nrb200.h declares, its host helpers agree with the oracle, and the compute entry points
fail loudly (no CPU fallback) when there is no device."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from newsrecommend_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "nrb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nrb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    syms = _declared_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(_lib.lib, s), f"libnrb200.so does not export {s}"
    assert sorted(_lib.SYMBOLS) == syms


def test_library_has_no_torch_or_libcuda_link_dependency():
    import subprocess
    out = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "libtorch" not in out and "libcuda.so" not in out and "libc10" not in out


def test_version_and_error_buffer():
    assert _lib.lib.nrb_version() >= 100
    assert isinstance(_lib.last_error(), str)


def test_rand_perm_host_matches_oracle(oracle):
    for n, seed in ((1, 1), (17, 1234), (5000, 1235)):
        perm = np.empty(n, dtype=np.int32)
        assert _lib.lib.nrb_rand_perm_host(perm.ctypes.data, n, seed) == 0
        assert np.array_equal(perm, oracle.rand_perm(n, seed))


def test_split_clusters_host_matches_oracle(oracle):
    rng = np.random.default_rng(0)
    k, d, n = 12, 10, 500
    cent = rng.standard_normal((k, d)).astype(np.float32)
    h = rng.integers(5, 80, size=k).astype(np.float32)
    h[[2, 7, 11]] = 0
    c1, h1 = cent.copy(), h.copy()
    c2, h2 = cent.copy(), h.copy()
    ns1 = oracle.split_clusters(c1, h1, n)
    ns2 = _lib.lib.nrb_split_clusters_host(d, k, n, h2.ctypes.data, c2.ctypes.data)
    assert ns1 == ns2 == 3
    assert np.array_equal(c1, c2) and np.array_equal(h1, h2)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_compute_fails_loudly_without_gpu():
    q = _lib.Matrix()
    b = _lib.Matrix()
    q.n, q.d, q.kp = 4, 32, 32
    b.n, b.d, b.kp = 4, 32, 32
    D = np.zeros((4, 1), dtype=np.float32)
    I = np.zeros((4, 1), dtype=np.int64)
    rc = _lib.lib.nrb_search_flat(C.byref(q), C.byref(b), 0, 1, 0, D.ctypes.data, I.ctypes.data, None, 0, 0, None)
    assert rc == -3  # NRB_ERR_NO_DEVICE
    with pytest.raises(RuntimeError, match="no CPU fallback|no CUDA device"):
        _lib.check(rc, "search_flat")
    import newsrecommend_b200.faiss as nf
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        nf.IndexFlatIP(8).add(np.zeros((2, 8), dtype=np.float32))


def test_argument_validation():
    q = _lib.Matrix()
    b = _lib.Matrix()
    q.n, q.d, q.kp = 4, 32, 32
    b.n, b.d, b.kp = 4, 16, 32
    D = np.zeros((4, 1), dtype=np.float32)
    I = np.zeros((4, 1), dtype=np.int64)
    rc = _lib.lib.nrb_search_flat(C.byref(q), C.byref(b), 0, 1, 0, D.ctypes.data, I.ctypes.data, None, 0, 0, None)
    assert rc == -1 and "dimension mismatch" in _lib.last_error()
    b.d = 32
    rc = _lib.lib.nrb_search_flat(C.byref(q), C.byref(b), 0, 1000, 0, D.ctypes.data, I.ctypes.data, None, 0, 0, None)
    assert rc == -1 and "out of range" in _lib.last_error()


def test_shim_exposes_reference_surface():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "shim"))
    try:
        import faiss  # the shim
        for name in ("Clustering", "IndexHNSWFlat", "IndexFlatL2", "IndexFlatIP", "IndexIVFFlat",
                     "vector_float_to_array", "normalize_L2", "METRIC_L2", "METRIC_INNER_PRODUCT"):
            assert hasattr(faiss, name), name
        c = faiss.Clustering(256, 300)  # Retrieval.py:12-14
        c.niter = 80
        c.verbose = True
        assert (c.seed, c.max_points_per_centroid, c.min_points_per_centroid, c.nredo) == (1234, 256, 39, 1)
        ivf_cp = faiss.IndexIVFFlat(faiss.IndexFlatL2(8), 8, 4).cp
        assert ivf_cp.niter == 10
        v = faiss.vector_float_to_array([1.0, 2.0])
        assert v.dtype == np.float32
    finally:
        sys.path.pop(0)
        sys.modules.pop("faiss", None)


def test_matrix_struct_layout_matches_header(tmp_path):
    """struct nrb_matrix as bound by ctypes has the size and field offsets gcc gives the header."""
    import subprocess
    src = tmp_path / "layout.c"
    fields = [f[0] for f in _lib.Matrix._fields_]
    body = "".join(f'printf("%zu\\n", offsetof(nrb_matrix, {f}));' for f in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "nrb200.h"\n'
                   'int main(void){printf("%zu\\n", sizeof(nrb_matrix));' + body + "return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert out[0] == C.sizeof(_lib.Matrix)
    assert out[1:] == [getattr(_lib.Matrix, f).offset for f in fields]


def test_h16_scale_is_a_power_of_two_with_headroom():
    import math
    import newsrecommend_b200.faiss as nf
    for mx in (1e-30, 3e-5, 0.75, 1.0, 15.8, 16.0, 1234.5, 6.0e4, 1e20):
        s = nf._h16_scale_for(mx)
        assert math.log2(s) == round(math.log2(s))
        assert 2.0 ** 14 <= mx * s < 2.0 ** 15 or mx < 2.0 ** -60 or mx > 2.0 ** 60
    assert nf._h16_scale_for(0.0) == 1.0 and nf._h16_scale_for(float("inf")) == 1.0


def _plan(nq, nb, k, path):
    out = (C.c_int32 * 10)()
    assert _lib.lib.nrb_plan_flat_describe(nq, nb, k, path, out) == 0, _lib.last_error()
    names = ("nqt", "npairs", "full_pairs", "tail_pairs", "tsplit", "chunk_rows", "n_units", "S", "grid", "single")
    return dict(zip(names, list(out)))


@pytest.mark.skipif(torch.cuda.is_available() and torch.cuda.get_device_properties(0).multi_processor_count != 148,
                    reason="expectations are written for 148 SMs")
def test_flat_planner_invariants_and_known_plans():
    """Host logic of the flat search plan (csrc/api.cu plan_flat), checked without a device."""
    TC, TC16, SIMT = _lib.PATH_TC, _lib.PATH_TC16, _lib.PATH_SIMT
    # config 1: 50,000 queries = 391 tiles = 196 pairs = 2 full waves of 74 + 48 tail pairs cut 2..4 ways
    p = _plan(50000, 364047, 50, TC16)
    assert (p["nqt"], p["npairs"], p["full_pairs"], p["tail_pairs"], p["single"]) == (391, 196, 148, 48, 0)
    assert 2 <= p["tsplit"] <= 4 and p["grid"] == 148 and p["n_units"] == 2 * (148 + 48 * p["tsplit"])
    # 6,250 queries per GPU (N = 8): 49 tiles; CTA pairs stop at 2 chunks, single CTAs take 3 (147 of 148 SMs)
    p = _plan(6250, 364047, 50, TC16)
    assert (p["nqt"], p["single"], p["tsplit"], p["n_units"], p["grid"]) == (49, 1, 3, 147, 147)
    assert _plan(6250, 364047, 50, TC)["single"] == 0  # the 3xTF32 kernels have no single-CTA form
    # invariants over a sweep
    for path in (TC, TC16, SIMT):
        for nq in (1, 127, 128, 129, 1000, 6250, 18944, 18945, 50000, 250000):
            for nb in (1, 255, 256, 5000, 364047):
                p = _plan(nq, nb, 10, path)
                assert p["nqt"] == (nq + 127) // 128 and p["npairs"] == (p["nqt"] + 1) // 2
                assert p["chunk_rows"] % 256 == 0 and p["chunk_rows"] * p["tsplit"] >= nb
                assert p["chunk_rows"] * (p["tsplit"] - 1) < max(nb, 1)  # no empty chunk
                assert p["S"] == p["tsplit"] * (1 if path == SIMT else 2)
                if p["single"]:
                    assert path == TC16 and p["full_pairs"] == 0 and p["n_units"] == p["nqt"] * p["tsplit"]
                    assert 1 <= p["grid"] <= 148
                else:
                    assert p["full_pairs"] + p["tail_pairs"] == p["npairs"]
                    assert p["n_units"] == 2 * (p["full_pairs"] + p["tail_pairs"] * p["tsplit"])
                    assert p["grid"] >= 1 and (path == SIMT or p["grid"] % 2 == 0)
                if p["full_pairs"]:
                    assert p["full_pairs"] % (148 if path == SIMT else 74) == 0
    bad = (C.c_int32 * 10)()
    assert _lib.lib.nrb_plan_flat_describe(10, 10, 5, _lib.PATH_AUTO, bad) == -1


def test_reference_script_fixtures_are_byte_identical():
    """tests/fixtures/reference_scripts holds test DATA: copies of three reference scripts that the
    GPU suite runs unmodified. They must match the sha256 and size recorded from the originals."""
    import hashlib
    import json
    d = os.path.join(ROOT, "tests", "fixtures", "reference_scripts")
    prov = json.load(open(os.path.join(d, "PROVENANCE.json")))
    assert sorted(prov["files"]) == ["Retrieval.py", "finialize_retrieval.py", "utils.py"]
    for name, meta in prov["files"].items():
        b = open(os.path.join(d, name), "rb").read()
        assert hashlib.sha256(b).hexdigest() == meta["sha256"] and len(b) == meta["bytes"]
