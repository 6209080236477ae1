"""Drop-in module named `faiss` for luzbetak/rag-faiss-embedding.

Put this directory (rag-faiss-embedding_b200/shim) ahead of site-packages on sys.path / PYTHONPATH and
the reference's `import faiss` (faiss_store.py:4, rag_datastore_manager.py:8) resolves here, so
faiss_store.py, rag_datastore_manager.py, query.py, 2-cli-rag-search.py and initialize_rag.py run
unchanged on the B200 engine.  Only the surface those files use is provided; everything is backed by
the sm_100a C-ABI library -- there is no CPU implementation behind this module.
"""
import importlib.util as _ilu
import os as _os
import sys as _sys

_root = _os.path.dirname(_os.path.dirname(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__)))))
if "rag_faiss_embedding_b200" not in _sys.modules and _ilu.find_spec("rag_faiss_embedding_b200") is None:
    _sys.path.insert(0, _root)

from rag_faiss_embedding_b200 import (  # noqa: E402,F401
    METRIC_INNER_PRODUCT,
    METRIC_L2,
    IDSelectorBatch,
    IDSelectorRange,
    IndexFlat,
    IndexFlatIP,
    IndexFlatL2,
    read_index,
    write_index,
)

__version__ = "b200flat-1"


def omp_set_num_threads(n):  # the reference pins OMP threads for faiss-cpu; meaningless here
    return None


def get_num_gpus():
    from rag_faiss_embedding_b200 import device_count

    return device_count()
