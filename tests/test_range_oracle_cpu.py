"""CPU tier: the float64 range-search restatement (tests/range_reference.py) against scikit-learn's brute-force radius
neighbours, its RangeSearchResult layout and edge cases, and the argument checks of the C-ABI range search that need no GPU."""
import ctypes
import math

import numpy as np
import pytest

import oracle as orc
from tests.range_reference import np_range_search_f64


def _data(n=3000, d=48, nq=21, seed=5):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, d)).astype(np.float32), rng.standard_normal((nq, d)).astype(np.float32)


def _gap_radius(keys, m):
    """A radius midway between the m-th and (m+1)-th smallest of `keys`, moved to the next gap wider than 1e-4 relative
    so that < and <= cannot differ."""
    s = np.sort(keys)
    while m < len(s) - 1 and s[m] - s[m - 1] <= 1e-4 * abs(s[m]):
        m += 1
    return 0.5 * (s[m - 1] + s[m])


def _check_layout(lims, D, I, nq):
    assert lims.dtype == np.int64 and lims.shape == (nq + 1,) and lims[0] == 0
    assert np.all(np.diff(lims) >= 0) and lims[-1] == len(D) == len(I)
    for q in range(nq):
        ids = I[lims[q]:lims[q + 1]]
        assert np.all(np.diff(ids) > 0)   # ascending, no duplicates


@pytest.mark.parametrize("metric", [orc.METRIC_L2, orc.METRIC_INNER_PRODUCT])
@pytest.mark.parametrize("m", [1, 10, 100, 1000])
def test_range_oracle_vs_sklearn(metric, m):
    """Restatement against an implementation this repo did not write.  L2: scikit-learn's radius is on euclidean
    distances, so it gets sqrt(radius).  IP: cosine distance on unit rows, 1 - ip, ranks identically."""
    sk = pytest.importorskip("sklearn.neighbors")
    xb, xq = _data()
    if metric == orc.METRIC_INNER_PRODUCT:
        xb = (xb / np.linalg.norm(xb, axis=1, keepdims=True)).astype(np.float32)
        xq = (xq / np.linalg.norm(xq, axis=1, keepdims=True)).astype(np.float32)
    x64, q64 = xb.astype(np.float64), xq.astype(np.float64)
    keys0 = ((x64 - q64[0]) ** 2).sum(1) if metric == orc.METRIC_L2 else -(x64 @ q64[0])
    r = _gap_radius(keys0, m)
    radius = r if metric == orc.METRIC_L2 else -r
    lims, D, I = np_range_search_f64(xb, xq, radius, metric)
    _check_layout(lims, D, I, len(xq))
    assert lims[1] - lims[0] >= m
    if metric == orc.METRIC_L2:
        nn = sk.NearestNeighbors(algorithm="brute", metric="euclidean").fit(x64)
        d_sk, i_sk = nn.radius_neighbors(q64, radius=math.sqrt(radius), sort_results=False)
    else:
        nn = sk.NearestNeighbors(algorithm="brute", metric="cosine").fit(x64)
        d_sk, i_sk = nn.radius_neighbors(q64, radius=1.0 - radius, sort_results=False)
    for q in range(len(xq)):
        got_i = I[lims[q]:lims[q + 1]]
        got_d = D[lims[q]:lims[q + 1]]
        order = np.argsort(i_sk[q])
        want_i, want_d = i_sk[q][order], d_sk[q][order]
        want_d = want_d ** 2 if metric == orc.METRIC_L2 else 1.0 - want_d
        # rows that sit within 1e-6 relative of the radius may fall either way: scikit-learn normalises the float32 unit
        # rows once more for the cosine, and takes a square root for the euclidean distance
        edge = np.abs((((x64 - q64[q]) ** 2).sum(1) if metric == orc.METRIC_L2 else x64 @ q64[q]) - radius) <= 1e-6 * abs(radius)
        assert set(got_i.tolist()) ^ set(want_i.tolist()) <= set(np.nonzero(edge)[0].tolist())
        common = np.intersect1d(got_i, want_i)
        assert np.allclose(got_d[np.searchsorted(got_i, common)], want_d[np.searchsorted(want_i, common)], rtol=1e-6, atol=1e-6)


def test_range_oracle_strict_and_empty():
    xb = np.array([[0.0], [1.0], [2.0], [np.nan], [np.inf]], np.float32)
    xq = np.array([[0.0], [np.nan]], np.float32)
    lims, D, I = np_range_search_f64(xb, xq, 1.0, orc.METRIC_L2)   # dist 1 is not < 1
    assert lims.tolist() == [0, 1, 1] and I.tolist() == [0] and D.tolist() == [0.0]
    lims, D, I = np_range_search_f64(xb, xq, 4.0 + 1e-9, orc.METRIC_L2)
    assert lims.tolist() == [0, 3, 3] and I.tolist() == [0, 1, 2]      # NaN / inf distances are never hits
    for r in (0.0, -1.0):                                              # an L2 radius <= 0 returns nothing
        lims, D, I = np_range_search_f64(xb, xq, r, orc.METRIC_L2)
        assert lims.tolist() == [0, 0, 0] and len(D) == len(I) == 0
    lims, D, I = np_range_search_f64(xb, xq[:1] + 1, 1.0, orc.METRIC_INNER_PRODUCT)   # ip > 1 (strict), NaN never
    assert I.tolist() == [2, 4] and D[0] == 2.0 and np.isinf(D[1])
    lims, D, I = np_range_search_f64(xb, xq[:0], 1.0, orc.METRIC_L2)
    assert lims.tolist() == [0] and len(I) == 0
    lims, D, I = np_range_search_f64(xb, xq, np.nan, orc.METRIC_L2)   # nothing compares true with a NaN radius
    assert lims.tolist() == [0, 0, 0]


def test_capi_range_search_rejects_bad_arguments():
    """The argument checks run before the index or a device is touched (NULL index, nq < 0, NaN radius, NULL out)."""
    from rag_faiss_embedding_b200 import _capi

    lib = _capi.load()
    out = ctypes.c_void_p()
    q = np.zeros((1, 4), np.float32)
    P = _capi.SearchParams()
    dummy = ctypes.create_string_buffer(64)   # never dereferenced: the arguments are rejected first
    cases = [
        (None, 1, q.ctypes.data, 1.0, ctypes.byref(out), "index is NULL"),
        (ctypes.addressof(dummy), -1, q.ctypes.data, 1.0, ctypes.byref(out), "nq=-1"),
        (ctypes.addressof(dummy), 1, None, 1.0, ctypes.byref(out), "bad arguments"),
        (ctypes.addressof(dummy), 1, q.ctypes.data, float("nan"), ctypes.byref(out), "radius is NaN"),
        (ctypes.addressof(dummy), 1, q.ctypes.data, 1.0, None, "out is NULL"),
    ]
    for ix, nq, qp, radius, outp, msg in cases:
        rc = lib.b2f_index_range_search(ix, nq, qp, ctypes.c_float(radius), _capi.MEM_HOST, None, ctypes.byref(P), outp)
        assert rc == _capi.EINVAL and msg in _capi.last_error(), (msg, rc, _capi.last_error())
        assert out.value is None
    info = (ctypes.c_int64 * 5)()
    lims = (ctypes.c_int64 * 2)()
    assert lib.b2f_range_result_lims(None, lims) == _capi.EINVAL
    assert lib.b2f_range_result_info(None, info) == _capi.EINVAL
    assert lib.b2f_range_result_fetch(None, None, None, _capi.MEM_HOST, None) == _capi.EINVAL
    assert lib.b2f_range_result_destroy(None) == _capi.OK
