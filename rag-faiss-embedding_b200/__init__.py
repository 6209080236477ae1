"""B200-native exact vector search for the hot path of luzbetak/rag-faiss-embedding.

Python host above the C-ABI library (include/b200flat.h, csrc/*.cu).  Importing this package loads
(building if necessary) the CUDA extension; it fails loudly if that is impossible.
"""
from . import _capi
from ._capi import (  # noqa: F401
    ALGO_AUTO,
    ALGO_SCAN,
    ALGO_TENSOR,
    STORE_BF16,
    STORE_F32,
    B200FlatError,
    SearchParams,
)
from .index import (  # noqa: F401
    METRIC_INNER_PRODUCT,
    METRIC_L2,
    IDSelectorAnd,
    IDSelectorArray,
    IDSelectorBatch,
    IDSelectorBitmap,
    IDSelectorNot,
    IDSelectorOr,
    IDSelectorRange,
    IDSelectorXor,
    IndexFlat,
    IndexFlatIP,
    IndexFlatL2,
    SearchParameters,
    read_index,
    write_index,
)
from .store import FAISSVectorStore  # noqa: F401
from .sharded import ShardedIndexFlat, merge_range, merge_topk  # noqa: F401

_capi.load()


def device_count() -> int:
    """Usable sm_100 devices (0 on a CPU-only box)."""
    return int(_capi.load().b2f_device_count())


def library_path() -> str:
    return _capi.LIB_PATH
