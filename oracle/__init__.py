"""CPU oracle for the flat-search hot path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this package.  The product (rag-faiss-embedding_b200/) never does.  See flat_oracle.c for the parity
status ("parity unpinned" for search results; on-disk layout pinned by the reference's own file).
"""
from .flat_oracle import (  # noqa: F401
    METRIC_INNER_PRODUCT,
    METRIC_L2,
    CENTRE_ROWS,
    build,
    c_search,
    c_synth_rows,
    c_read_index,
    c_write_index,
    c_max_threads,
    np_search_f64,
    np_search_blas,
    torch_search_blas,
    np_synth_rows,
    np_centre,
    np_bf16_rne,
    np_bf16_rows,
    np_read_index,
    np_write_index,
    recall_and_errors,
)
