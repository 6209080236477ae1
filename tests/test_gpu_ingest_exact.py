"""GPU tier (-m gpu): bf16-storage ingest, bit for bit against the numpy restatement (oracle.np_centre / np_bf16_rows).

With bf16 storage the ingest decides the data itself: the stored row is r = fl32(mu + bf16(x - mu)), and every search
measures distances to r.  mu is the mean of the first min(n, 65536) rows of the FIRST add call, whatever route that call
takes and however the route stages it (host chunks, pooling chunks, generator chunks, file chunks).  So the same rows
must give the same index bit for bit on every route: numpy add, CUDA-tensor add, add_synthetic, add_pooled and
read_index into bf16 storage.  The first-call sizes sit on both sides of every staging chunk (64 MB host / pooling, 256 MB
generator, 32 MB file chunks), the widths reach both the float4 (d % 4 == 0) and the scalar ingest path."""
import numpy as np
import pytest

import oracle as orc
from tests.exact_checks import check_structure

pytestmark = pytest.mark.gpu

SEED = 2024


def _chunk_rows(mb, d):
    return (mb << 20) // (4 * d)


# (n, d) of the first add.  d = 384: around 64 rows, 65536 rows and the file (32 MB) / host (64 MB) chunks;
# d = 1536: around the file, host and generator (256 MB) chunks; then every ingest width class.
ROUTE_CASES = ([(n, 384) for n in (1, 63, 64, 65, 4097, 65535, 65536, 65537, 100000)]
               + [(_chunk_rows(mb, 384) + e, 384) for mb in (32, 64) for e in (-1, 0, 1)]
               + [(_chunk_rows(mb, 1536) + e, 1536) for mb in (32, 64, 256) for e in (-1, 0, 1)]
               + [(65537, 1536), (70000, 1), (70000, 7), (70000, 96), (20000, 1030), (17000, 4096)])


@pytest.fixture(scope="module")
def m():
    import rag_faiss_embedding_b200 as mod

    assert mod.device_count() > 0, "no B200 visible"
    return mod


def _same(got, want, what):
    """Bit for bit; NaN positions compared separately (the device's NaN payload is not pinned)."""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN positions differ"
    g, w = got[~nan].view(np.uint32), want[~nan].view(np.uint32)
    bad = np.flatnonzero(g != w)
    if bad.size:
        i = bad[0]
        raise AssertionError(f"{what}: {bad.size} of {g.size} values differ, e.g. {got[~nan][i]!r} vs {want[~nan][i]!r}")


def _restated(first, *later):
    mu = orc.np_centre(first)
    return np.concatenate([orc.np_bf16_rows(x, mu) for x in (first,) + later]) if later else orc.np_bf16_rows(first, mu)


def _build(m, route, x, tmp_path, metric=1, seed=None):
    """A bf16-storage index whose first add call receives the rows x through `route`."""
    import torch

    n, d = x.shape
    if route == "read":
        path = tmp_path / "in.bin"
        orc.np_write_index(path, x, metric)
        ix = m.read_index(str(path), storage=m.STORE_BF16)
        path.unlink()
        return ix
    ix = m.IndexFlat(d, metric, storage=m.STORE_BF16)
    if route == "numpy":
        ix.add(x)
    elif route == "tensor":
        ix.add(torch.from_numpy(x).cuda())
    elif route == "pooled":   # CLS over one token: the pooled row is the token itself, bit for bit
        ix.add_pooled(torch.from_numpy(x).cuda()[:, None, :], None, pool="cls")
    elif route == "synth":
        ix.add_synthetic(seed, 0, n)
    else:
        raise ValueError(route)
    torch.cuda.synchronize()
    return ix


def _check_search(D, I, D_ref, I_ref, metric, min_recall=1.0):
    check_structure(D, I, metric)
    r = orc.recall_and_errors(D, I, D_ref, I_ref, metric, rel_tol=1e-5)
    assert r["recall"] >= min_recall and r["id_mismatch"] == 0 and r["padding_ok"] and r["max_rel_err"] <= 1e-5, r


# ---- every route, every first-call size ------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", ROUTE_CASES)
def test_routes_store_the_restated_rows(m, n, d, tmp_path):
    x = orc.c_synth_rows(SEED, 0, n, d)
    want = _restated(x)
    want_file = tmp_path / "want.bin"
    orc.np_write_index(want_file, want)
    want_bytes = want_file.read_bytes()
    for route in ("numpy", "tensor", "synth", "pooled", "read"):
        ix = _build(m, route, x, tmp_path, seed=SEED)
        assert ix.ntotal == n
        _same(ix.reconstruct_n(), want, f"{route} n={n} d={d}")
        got_file = tmp_path / f"{route}.bin"
        m.write_index(ix, str(got_file))
        assert got_file.read_bytes() == want_bytes, (route, n, d)
        got_file.unlink()
        del ix


@pytest.mark.parametrize("n,d,normalize", [(65537, 384, False), (_chunk_rows(64, 384) + 1, 384, True),
                                           (_chunk_rows(64, 1536) + 1, 1536, False)])
def test_add_pooled_mean_stores_the_restated_pooled_rows(m, n, d, normalize):
    """Masked-mean pooling (vectorised path at d = 384, scalar at d = 1536): the index holds the restatement of exactly
    the rows pool_normalize returns for the same input."""
    import torch

    from rag_faiss_embedding_b200.encoder import pool_normalize

    g = torch.Generator().manual_seed(n)
    h = (torch.randn(n, 2, d, generator=g) * 0.3 + torch.randn(d, generator=g)).cuda()
    mask = (torch.rand(n, 2, generator=g) < 0.6).to(torch.int64)
    mask[:, 0] = 1
    mask = mask.cuda()
    rows = pool_normalize(h, mask, "mean", normalize).cpu().numpy()
    ix = m.IndexFlat(d, 1, storage=m.STORE_BF16)
    ix.add_pooled(h, mask, pool="mean", normalize=normalize)
    torch.cuda.synchronize()
    _same(ix.reconstruct_n(), _restated(rows), f"pooled mean n={n} d={d}")


# ---- several adds: the first call fixes the centre --------------------------------------------------------------
@pytest.mark.parametrize("first", (1, 10, 65537))
def test_later_adds_round_around_the_first_centre(m, first):
    import torch

    d = 384
    rng = np.random.default_rng(first)
    off = rng.standard_normal(d).astype(np.float32) * 3
    x = (rng.standard_normal((first + 70000, d)) + off).astype(np.float32)
    ix = m.IndexFlat(d, 1, storage=m.STORE_BF16)
    ix.add(x[:first])
    ix.add(x[first:first + 50000])
    ix.add(torch.from_numpy(x[first + 50000:]).cuda())
    ix.add_synthetic(SEED, 0, 5000)
    torch.cuda.synchronize()
    s = orc.c_synth_rows(SEED, 0, 5000, d)
    _same(ix.reconstruct_n(), _restated(x[:first], x[first:], s), f"first call {first}")
    # reset: the next first call takes a new centre
    ix.reset()
    y = (x[:first + 3000] * 0.5 - 1).astype(np.float32)
    ix.add(y)
    _same(ix.reconstruct_n(), _restated(y), f"after reset, first call {first + 3000}")


# ---- magnitudes --------------------------------------------------------------------------------------------------
MAGNITUDES = ("subnormal", "tiny", "huge", "overflow", "mixed")


def _magnitude_rows(kind, d):
    rng = np.random.default_rng([MAGNITUDES.index(kind), d])
    g = lambda n: rng.standard_normal((n, d))   # noqa: E731
    if kind == "subnormal":       # rows and centred differences below 2^-126
        return (g(5000) * 3e-39 + 1e-39).astype(np.float32)
    if kind == "tiny":            # around the smallest normal
        return ((1 + 0.3 * g(5000)) * 1e-38).astype(np.float32)
    if kind == "huge":
        return (1e30 + g(70000) * 1e28).astype(np.float32)
    if kind == "overflow":        # 64-row float32 block sums overflow: those blocks are skipped; the partial last one is not
        x = ((1 + 0.01 * g(4100)) * 1e37).astype(np.float32)
        x[:, ::2] *= np.where(rng.random((4100, 1)) < 0.5, -1, 1).astype(np.float32)   # random signs: sums stay finite
        return x
    if kind == "mixed":           # columns of mixed scale: 1e20, 1e-20, constant, zero
        x = (g(70000) + 5).astype(np.float32)
        x[:, 0] = (g(70000)[:, 0] + 2) * 1e20
        x[:, 1] = (g(70000)[:, 1] + 2) * 1e-20
        x[:, 2] = np.float32(0.1)
        x[:, 3] = 0
        return x
    raise ValueError(kind)


@pytest.mark.parametrize("d", (7, 96))
@pytest.mark.parametrize("kind", MAGNITUDES)
def test_magnitudes(m, kind, d, tmp_path):
    x = _magnitude_rows(kind, d)
    assert np.isfinite(x).all()
    want = _restated(x)
    if kind == "overflow":
        with np.errstate(over="ignore"):
            assert np.isinf(np.cumsum(x[:64, 1::2], 0, np.float32)[-1]).all()   # (the case really overflows)
    for route in ("numpy", "tensor", "pooled", "read"):
        _same(_build(m, route, x, tmp_path).reconstruct_n(), want, f"{kind} d={d} {route}")


# ---- non-finite values -------------------------------------------------------------------------------------------
NAN_AT = ((3, 5), (40000, 1), (66000, 3))       # first block, a later block within the first 65536 rows, after them
INF_AT = ((10, 6), (20, 0), (40001, 2), (69000, 4))


def _nonfinite_rows(d, inf):
    rng = np.random.default_rng(d)
    x = (rng.standard_normal((70000, d)) * 0.5 + rng.standard_normal(d) * 4).astype(np.float32)
    for r, c in NAN_AT:
        x[r, c % d] = np.nan
    if inf:
        for i, (r, c) in enumerate(INF_AT):
            x[r, c % d] = np.inf if i % 2 == 0 else -np.inf
    return x


@pytest.mark.parametrize("d", (7, 96))
@pytest.mark.parametrize("inf", (False, True))
def test_non_finite_entries(m, d, inf, tmp_path):
    x = _nonfinite_rows(d, inf)
    want = _restated(x)
    assert np.isfinite(orc.np_centre(x)).all()
    for route in ("numpy", "tensor", "pooled", "read"):
        _same(_build(m, route, x, tmp_path).reconstruct_n(), want, f"d={d} inf={inf} {route}")


@pytest.mark.parametrize("metric", (1, 0))
@pytest.mark.parametrize("storage", ("bf16", "fp32"))
def test_search_skips_nan_rows(m, storage, metric):
    """NaN rows (in the first block, within the first 65536 rows, after them) never come back, on either path; the rest
    is the float64 answer over the finite rows."""
    d, nq, k = 96, 64, 10
    x = _nonfinite_rows(d, inf=False)
    ix = m.IndexFlat(d, metric, storage=m.STORE_BF16 if storage == "bf16" else m.STORE_F32)
    ix.add(x)
    rows = ix.reconstruct_n()
    ok = np.isfinite(rows).all(1)
    assert (~ok).sum() == len(NAN_AT)
    keep = np.flatnonzero(ok)
    rng = np.random.default_rng(5)
    q = (x[keep[rng.integers(0, keep.size, nq)]] + rng.standard_normal((nq, d)).astype(np.float32) * 0.1).astype(np.float32)
    q[0] = x[3]                                  # a NaN row's finite entries as a query
    q[0, 5] = 0
    D_ref, I_ref = orc.np_search_f64(rows[keep], q, k, metric)
    I_ref = np.where(I_ref >= 0, keep[np.maximum(I_ref, 0)], -1)
    for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
        D, I = ix.set_search_params(algo=algo).search(q, k)
        assert not np.isin(I, np.flatnonzero(~ok)).any(), (algo, storage, metric)
        _check_search(D, I, D_ref, I_ref, metric)
    print(f"NaN rows, {storage} metric {metric}: {ix.stats()['fallback_queries']} exact-scan queries")


def test_search_with_inf_rows_is_exact(m):
    """Rows with an infinite entry: their L2 distance is infinite, they never enter; the rest is exact.  (Such a row makes
    the certification bound infinite, so every tensor-path query goes to the exact scan: printed, not asserted.)"""
    d, nq, k = 96, 64, 10
    x = _nonfinite_rows(d, inf=True)
    ix = m.IndexFlat(d, 1, storage=m.STORE_BF16)
    ix.add(x)
    rows = ix.reconstruct_n()
    keep = np.flatnonzero(np.isfinite(rows).all(1))
    rng = np.random.default_rng(6)
    q = (x[keep[rng.integers(0, keep.size, nq)]] + rng.standard_normal((nq, d)).astype(np.float32) * 0.1).astype(np.float32)
    D_ref, I_ref = orc.np_search_f64(rows[keep], q, k, 1)
    I_ref = np.where(I_ref >= 0, keep[np.maximum(I_ref, 0)], -1)
    for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
        D, I = ix.set_search_params(algo=algo).search(q, k)
        _check_search(D, I, D_ref, I_ref, 1)
    print(f"inf rows, bf16 L2: {ix.stats()['fallback_queries']} of {nq} tensor-path queries went to the exact scan")


# ---- search agreement across routes ------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", (1, 0))
@pytest.mark.parametrize("n,d", [(_chunk_rows(64, 384) + 1, 384), (_chunk_rows(64, 1536) + 1, 1536)])
def test_routes_search_alike(m, n, d, metric, tmp_path):
    """Each row's arithmetic is deterministic, so the exact scan gives the same bits on every route; the tensor path
    matches float64 over the restated rows."""
    nq, k = 50, 10
    x = orc.c_synth_rows(SEED, 0, n, d)
    rows = _restated(x)
    q = (x[np.random.default_rng(n).integers(0, n, nq)] + np.float32(0.05)).astype(np.float32)
    D_ref, I_ref = orc.np_search_f64(rows, q, k, metric)
    scan = None
    for route in ("numpy", "tensor", "synth", "pooled", "read"):
        ix = _build(m, route, x, tmp_path, metric=metric, seed=SEED)
        D, I = ix.set_search_params(algo=m.ALGO_SCAN).search(q, k)
        if scan is None:
            scan = (D, I)
            _check_search(D, I, D_ref, I_ref, metric)
        assert np.array_equal(I, scan[1]) and np.array_equal(D.view(np.uint32), scan[0].view(np.uint32)), route
        D, I = ix.set_search_params(algo=m.ALGO_TENSOR).search(q, k)
        assert ix.stats()["last_algo"] == m.ALGO_TENSOR
        _check_search(D, I, D_ref, I_ref, metric)


# ---- a bf16 file read back -----------------------------------------------------------------------------------------
def test_bf16_file_round_trip(m, tmp_path):
    """A bf16 index writes its rows r1 in fp32.  Read into fp32 storage they come back exactly; read into bf16 storage they
    are a new first add: a new centre from r1, and r1 rounded again around it."""
    n, d = 70000, 384
    rng = np.random.default_rng(77)
    x = (rng.standard_normal((n, d)) * 0.2 + rng.standard_normal(d) * 2).astype(np.float32)
    ix = m.IndexFlat(d, 1, storage=m.STORE_BF16)
    ix.add(x)
    path = tmp_path / "bf16.bin"
    m.write_index(ix, str(path))
    r1, metric = orc.np_read_index(path)
    _same(r1, _restated(x), "written rows")
    _same(m.read_index(str(path), storage=m.STORE_F32).reconstruct_n(), r1, "read into fp32 storage")
    r2 = m.read_index(str(path), storage=m.STORE_BF16).reconstruct_n()
    _same(r2, _restated(r1), "read into bf16 storage")
    diff = np.abs(r2.astype(np.float64) - r1)
    rel = (diff / np.maximum(np.abs(r1), 1e-30)).max()
    print(f"bf16 file read back into bf16 storage: {np.count_nonzero(diff)} of {diff.size} values changed, "
          f"largest change {diff.max():.3g} ({rel:.3g} relative to the row value), mean |x| {np.abs(x).mean():.3g}")
