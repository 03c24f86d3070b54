"""Drop-in `faiss` module: put /root/repo/shim on PYTHONPATH and the unmodified reference
script (`import faiss`, Retrieval.py:2) runs on the B200 path. Kept outside the package so it
can never shadow a real faiss that is used as an oracle."""
from newsrecommend_b200.faiss import *  # noqa: F401,F403
from newsrecommend_b200.faiss import (METRIC_INNER_PRODUCT, METRIC_L2, Clustering,  # noqa: F401
                                      ClusteringParameters, IndexFlat, IndexFlatIP, IndexFlatL2,
                                      IndexHNSWFlat, IndexIDMap, IndexIVFFlat, IDSelectorBatch, IDSelectorRange,
                                      normalize_L2, vector_float_to_array)
