"""CPU tier: the shapes of tests/test_gpu_edges.py reach every tensor-path kernel variant.

The planner (b2f_plan_describe, host code of the library) decides which K2 kernel a search runs; this checks, without a
GPU, that the GPU edge tests still reach each one -- so a planner change cannot quietly move them all onto one path."""
import ctypes

from tests import test_gpu_edges as edges

QRES_MAX_KB = 6   # gemm_topk_sm100.cu: the query tile stays resident in shared memory up to 6 k-blocks of 64 (d <= 384)


def _variants(lib, nq, n, d, k, slack):
    out = (ctypes.c_int32 * 12)()
    assert lib.b2f_plan_describe(nq, n, d, k, slack, out) == 0
    kp, chunk, passes, list_mode, pair = list(out)[:5]
    if kp == 0:
        return {"tensor unavailable"}
    assert chunk * passes >= nq
    found = {f"k'={kp}"}
    if passes >= 2:
        found.add("multi-pass")
    if not list_mode:
        found.add(f"heap k'={kp}")
    elif pair:
        assert (d + 63) // 64 <= QRES_MAX_KB
        found.add("pair")
    elif (d + 63) // 64 <= QRES_MAX_KB:
        found.add("Q-resident list")
    else:
        found.add("streamed list")
    return found


def test_gpu_edge_shapes_reach_every_tensor_kernel():
    from rag_faiss_embedding_b200 import _capi

    lib = _capi.load()
    reached = set()
    for nq, n, d, k, slack in edges.plan_shapes():
        reached |= _variants(lib, nq, n, d, k, slack)
    required = {"pair", "Q-resident list", "streamed list", "heap k'=32", "heap k'=64", "multi-pass", "tensor unavailable"}
    required |= {f"k'={kp}" for kp in (32, 64, 72, 192, 256)}
    assert required <= reached, sorted(required - reached)
    # ... and every one of them under both metrics
    assert set(edges.METRICS) == {0, 1}


def test_kprime_table_matches_planner():
    """The k' table the GPU test asserts against is the planner's own mapping (k + max(22, ceil(0.9 k)), rounded up to
    32 / 64 / a multiple of 8, 0 above 256), steps included."""
    from rag_faiss_embedding_b200 import _capi

    lib = _capi.load()
    n, d, nq = edges.KPRIME_DATA
    out = (ctypes.c_int32 * 12)()
    for k, kp in edges.KPRIME.items():
        assert lib.b2f_plan_describe(nq, n, d, k, 0, out) == 0 and out[0] == kp, (k, out[0])
    for (k, slack), kp in edges.KPRIME_SLACK.items():
        assert lib.b2f_plan_describe(nq, n, d, k, slack, out) == 0 and out[0] == kp, (k, slack, out[0])
    for k in range(1, 300):   # the documented rule, restated
        want = k + max(22, -(-9 * k // 10))
        want = 32 if want <= 32 else 64 if want <= 64 else (want + 7) // 8 * 8
        assert lib.b2f_plan_describe(nq, n, d, k, 0, out) == 0 and out[0] == (want if want <= 256 else 0), k
