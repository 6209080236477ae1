"""GPU tier (-m gpu): the CUDA path, called through the C-ABI, against the CPU oracle and the golden
fixtures.  Tolerances (BASELINE.json north_star): ids identical except among exact-distance ties;
distances within 1e-5 relative (1e-4 absolute floor near zero) -- both search paths end in fp32
exact-difference arithmetic, like faiss's fvec_L2sqr."""
import os

import numpy as np
import pytest

import oracle as orc
from tests.exact_checks import check_structure

pytestmark = pytest.mark.gpu

FLT_MAX = np.finfo(np.float32).max
REL = 1e-5


@pytest.fixture(scope="module")
def m():
    import rag_faiss_embedding_b200 as mod

    assert mod.device_count() > 0, "no B200 visible"
    return mod


def _check(D, I, D_ref, I_ref, metric, rel=REL, min_recall=1.0):
    check_structure(D, I, metric)
    r = orc.recall_and_errors(D, I, D_ref, I_ref, metric, rel_tol=rel)
    # min_recall < 1 only where fp32 keys of neighbouring rows differ by less than an ulp, so that the k-th and the
    # (k+1)-th neighbour of a float64 oracle are a tie in the reference's own fp32 arithmetic (id_mismatch still
    # requires every position to agree in id or -- within `rel` -- in distance)
    assert r["recall"] >= min_recall, r
    assert r["id_mismatch"] == 0, r
    assert r["padding_ok"], r
    assert r["max_rel_err"] <= rel, r
    return r


def _make(m, xb, metric, **kw):
    ix = m.IndexFlat(xb.shape[1], metric, **kw)
    if xb.shape[0]:
        ix.add(xb)
    return ix


# ---- golden fixture: the reference's own FAISS-written index ------------------------------------------
def test_fixture_read_search_write(m, golden, tmp_path):
    ix = m.read_index(golden["index_path"])
    assert (ix.d, ix.ntotal, ix.metric_type, ix.is_trained) == (384, 23, 1, True)
    xb, _ = orc.np_read_index(golden["index_path"])
    assert np.array_equal(ix.reconstruct_n(0, 23), xb)
    assert np.array_equal(ix.reconstruct(7), xb[7])
    for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
        ix.set_search_params(algo=algo)
        for case in golden["cases"]:
            if case["metric"] != 1 or (algo == m.ALGO_TENSOR and case["k"] > 10):
                continue
            q = xb if case["queries"] == "self" else golden["perturbed"]
            D, I = ix.search(q, case["k"])
            _check(D, I, np.asarray(case["dists"]), np.asarray(case["ids"], np.int64), 1)
    out = tmp_path / "roundtrip.bin"
    m.write_index(ix, out)
    assert open(out, "rb").read() == open(golden["index_path"], "rb").read()
    # inner-product twin of the same rows
    ip = _make(m, xb, 0)
    for case in golden["cases"]:
        if case["metric"] != 0:
            continue
        q = xb if case["queries"] == "self" else golden["perturbed"]
        D, I = ip.search(q, case["k"])
        _check(D, I, np.asarray(case["dists"]), np.asarray(case["ids"], np.int64), 0)
    out2 = tmp_path / "ip.bin"
    m.write_index(ip, out2)
    assert open(out2, "rb").read()[:4] == b"IxFI"
    back = m.read_index(out2)
    assert back.metric_type == 0 and np.array_equal(back.reconstruct_n(), xb)


def test_reference_wrapper_on_fixture(m, golden):
    """The FAISSVectorStore surface (faiss_store.py) over the real index: row -> doc id mapping."""
    s = m.FAISSVectorStore(dimension=384, index_path=golden["index_path"])
    assert s.doc_ids == golden["mapping"]
    xb, _ = orc.np_read_index(golden["index_path"])
    case = next(c for c in golden["cases"] if c["metric"] == 1 and c["k"] == 5 and c["queries"] == "self")
    for row in (0, 1, 2, 7, 22):
        d, ids = s.search(xb[row], k=5)
        assert ids == [golden["mapping"][i] for i in case["ids"][row]]
        assert np.allclose(d, case["dists"][row], rtol=1e-5, atol=1e-4)
    d, ids = s.search(xb[0], k=40)
    assert len(ids) == 23


# ---- K1 streaming scan vs oracle -----------------------------------------------------------------------
@pytest.mark.parametrize("metric", [1, 0])
@pytest.mark.parametrize("n,d,nq,k", [
    (1, 384, 1, 1), (23, 384, 1, 5), (1000, 384, 3, 10), (5000, 768, 8, 10), (4097, 96, 5, 100),
    (3000, 100, 2, 7), (777, 1, 4, 3), (2500, 30, 9, 128), (50000, 384, 1, 10), (20000, 64, 17, 1024),
    (300, 1026, 2, 10),
])
def test_scan_vs_oracle(m, metric, n, d, nq, k):
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, nq, d)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_SCAN)
    D, I = ix.search(xq, k)
    D_ref, I_ref = orc.np_search_f64(xb, xq, k, metric)
    _check(D, I, D_ref, I_ref, metric)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_SCAN and st["last_launches"] == 1   # scan + merge + formatting: one cooperative launch


def test_edge_cases(m):
    xb = orc.c_synth_rows(1, 0, 10, 8)
    ix = _make(m, xb, 1)
    D, I = ix.search(xb[:2], 16)           # k > ntotal
    assert (I[:, 10:] == -1).all() and (D[:, 10:] == FLT_MAX).all() and I[:, 0].tolist() == [0, 1]
    e = m.IndexFlatL2(8)                   # empty index
    D, I = e.search(xb[:2], 3)
    assert (I == -1).all() and (D == FLT_MAX).all()
    e = m.IndexFlatIP(8)
    D, I = e.search(xb[:2], 3)
    assert (I == -1).all() and (D == -FLT_MAX).all()
    dup = _make(m, np.repeat(xb[:1], 5, 0), 1)   # exact ties -> ascending label
    D, I = dup.search(xb[:1], 3)
    assert I.tolist() == [[0, 1, 2]] and (D == 0).all()
    bad = xb.copy()
    bad[3] = np.nan                        # NaN rows never enter
    D, I = _make(m, bad, 1).search(xb[:1], 10)
    assert 3 not in I[0].tolist() and I[0, -1] == -1
    with pytest.raises(AssertionError):
        ix.search(xb[:1], 0)
    with pytest.raises(AssertionError):
        ix.search(np.zeros((1, 9), np.float32), 1)
    with pytest.raises(AssertionError):
        ix.add(np.zeros((1, 9), np.float32))
    with pytest.raises(RuntimeError):
        m.read_index("/nonexistent/index.bin")
    with pytest.raises(RuntimeError):
        ix.reconstruct(10)
    ix.reset()
    assert ix.ntotal == 0
    ix.add(xb[:3])
    assert ix.ntotal == 3 and ix.search(xb[:1], 1)[1][0, 0] == 0
    D, I = ix.search(np.zeros((0, 8), np.float32), 3)   # empty query batch
    assert D.shape == (0, 3) and I.shape == (0, 3)


def test_incremental_add_and_growth(m):
    d = 48
    xb = orc.c_synth_rows(9, 0, 5000, d)
    ix = m.IndexFlatL2(d)
    for a, b in ((0, 1), (1, 700), (700, 1500), (1500, 5000)):   # crosses the initial capacity
        ix.add(xb[a:b])
    assert ix.ntotal == 5000 and np.array_equal(ix.reconstruct_n(), xb)
    xq = orc.c_synth_rows(10, 0, 4, d)
    D, I = ix.search(xq, 10)
    _check(D, I, *orc.np_search_f64(xb, xq, 10, 1), 1)


# ---- K2 tensor path (tcgen05 + fused top-k + exact re-rank + certification) vs oracle --------------------
@pytest.mark.parametrize("metric", [1, 0])
@pytest.mark.parametrize("n,d,nq,k", [
    (300, 384, 1, 10), (5000, 384, 33, 10), (20000, 384, 128, 10), (100000, 384, 200, 10),
    (7000, 768, 64, 10), (9000, 100, 130, 5), (70000, 64, 1024, 10), (4000, 384, 16, 20),
    (256, 384, 9, 1), (257, 128, 300, 10), (100000, 64, 2400, 10),
])
def test_tensor_vs_oracle(m, metric, n, d, nq, k):
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, nq, d)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    D_ref, I_ref = orc.np_search_f64(xb, xq, k, metric)
    _check(D, I, D_ref, I_ref, metric)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_TENSOR and st["last_kprime"] in (32, 64)
    if n >= 5000:   # random data: the fused filter must not overflow its candidate lists
        assert st["overflow_queries"] == 0, st


@pytest.mark.parametrize("metric,normalize,n,d,nq,k", [
    (0, True, 60000, 768, 70, 100),     # config 3's shape in small: normalised inner product, k = 100 (k' = 192)
    (1, False, 40000, 384, 300, 100),
    (1, False, 30000, 64, 4096, 100),   # big batch x big k': processed in query chunks
    (0, False, 20000, 128, 33, 128),    # largest k served by the tensor path (k' = 256)
])
def test_tensor_large_k(m, metric, normalize, n, d, nq, k):
    xb = orc.c_synth_rows(1234, 0, n, d, normalize)
    xq = orc.c_synth_rows(5678, 0, nq, d, normalize)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb, xq, k, metric), metric)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_TENSOR and st["last_kprime"] >= k + 22 and st["overflow_queries"] == 0, st


def test_tensor_hard_inputs(m):
    """Near-duplicates and mean-shifted rows (the fixture's distribution: norm ~7.7, tiny relative gaps)
    stress the bf16 coarse pass; certification + exact fallback must keep results exact."""
    rng = np.random.default_rng(7)
    d, n = 384, 30000
    base = (rng.standard_normal((n, d)) * 0.25 + 0.4).astype(np.float32)
    base[1000:1100] = base[999] + rng.standard_normal((100, d)).astype(np.float32) * 1e-3  # a tight cluster
    xq = np.concatenate([base[995:1005] + 1e-4, (rng.standard_normal((30, d)) * 0.25 + 0.4).astype(np.float32)])
    for metric in (1, 0):
        ix = _make(m, base, metric).set_search_params(algo=m.ALGO_TENSOR)
        D, I = ix.search(xq, 10)
        _check(D, I, *orc.np_search_f64(base, xq, 10, metric), metric)
        st = ix.stats()
        # the tight cluster defeats the k'-candidate bound: those queries are answered either from the complete
        # candidate lists (extended certification, no database pass) or by the exact scan
        assert st["rescued_queries"] + st["fallback_queries"] > 0, st
    # with certification off the same call may miss, but must still return sorted, valid rows
    ix.set_search_params(certify=False)
    D, I = ix.search(xq, 10)
    assert (I >= 0).all() and (np.diff(D, axis=1) <= 1e-6).all()


def test_tensor_list_overflow_falls_back(m):
    """Adversarial order: every later row is closer to the queries than all earlier ones, so every row
    passes the running threshold and the per-(query, split) candidate lists overflow.  The overflow
    must be detected and those queries answered by the exact scan."""
    rng = np.random.default_rng(11)
    n, d, nq, k = 40000, 128, 20, 10
    q0 = rng.standard_normal(d).astype(np.float32)
    dirs = rng.standard_normal((n, d)).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    radius = np.linspace(30.0, 1.0, n, dtype=np.float32)[:, None]     # strictly shrinking distance to q0
    xb = (q0[None, :] + dirs * radius).astype(np.float32)
    xq = (q0[None, :] + rng.standard_normal((nq, d)).astype(np.float32) * 1e-3).astype(np.float32)
    ix = _make(m, xb, 1).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb, xq, k, 1), 1)
    assert ix.stats()["fallback_queries"] > 0


def test_random_shapes_both_paths(m):
    """Seeded sweep over ragged shapes (d not a multiple of 8 / 64, n around tile boundaries, k from 1 to 100,
    batches around the 128-query tile), three data distributions (N(0,1); mean-shifted fixture-like rows with
    tiny relative gaps; heavy duplicates = exact-distance ties), L2 and IP, both GPU paths against the oracle."""
    rng = np.random.default_rng(2024)
    for case in range(18):
        d = int(rng.choice([1, 7, 30, 64, 100, 128, 250, 384, 520]))
        n = int(rng.choice([1, 33, 255, 256, 257, 1000, 4099, 20000, 70001]))
        nq = int(rng.choice([1, 2, 9, 31, 127, 128, 129, 300]))
        k = int(rng.choice([1, 3, 10, 37, 100]))
        metric = int(rng.integers(0, 2))
        kind = case % 3
        if kind == 0:
            xb = rng.standard_normal((n, d)).astype(np.float32)
            xq = rng.standard_normal((nq, d)).astype(np.float32)
        elif kind == 1:
            xb = (rng.standard_normal((n, d)) * 0.2 + 0.4).astype(np.float32)
            xq = (rng.standard_normal((nq, d)) * 0.2 + 0.4).astype(np.float32)
        else:
            base = rng.standard_normal((max(n // 7, 1), d)).astype(np.float32)
            xb = base[rng.integers(0, base.shape[0], n)]
            xq = base[rng.integers(0, base.shape[0], nq)] + (rng.standard_normal((nq, d)) * 1e-3).astype(np.float32)
        D_ref, I_ref = orc.np_search_f64(xb, xq, k, metric)
        ix = _make(m, xb, metric)
        for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
            if algo == m.ALGO_TENSOR and k > 100:
                continue
            D, I = ix.set_search_params(algo=algo).search(xq, k)
            r = orc.recall_and_errors(D, I, D_ref, I_ref, metric, rel_tol=REL)
            assert r["recall"] == 1.0 and r["id_mismatch"] == 0 and r["padding_ok"] and r["max_rel_err"] <= REL, \
                (case, dict(n=n, d=d, nq=nq, k=k, metric=metric, kind=kind, algo=algo), r)


def test_many_fallbacks_with_query_chunks(m):
    """Adversarial row order (every later row closer to the queries than all earlier ones: every candidate list
    overflows) in a batch big enough to be processed in more than one tensor pass (k' = 192 caps a pass at 3072
    queries): the closing exact scan must pick up the failures of every pass -- thousands of queries, walked in
    groups inside one launch -- and scatter them to the right rows."""
    rng = np.random.default_rng(11)
    n, d, nq, k = 20000, 64, 3300, 100
    q0 = rng.standard_normal(d).astype(np.float32)
    dirs = rng.standard_normal((n, d)).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    radius = np.linspace(30.0, 1.0, n, dtype=np.float32)[:, None]
    xb = (q0[None, :] + dirs * radius).astype(np.float32)
    xq = (q0[None, :] + rng.standard_normal((nq, d)).astype(np.float32) * 1e-3).astype(np.float32)
    ix = _make(m, xb, 1).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb, xq, k, 1), 1)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_TENSOR and st["fallback_queries"] > nq // 2, st


def test_centred_scan_copy_certifies_embedding_like_data(m):
    """Rows that share a large common component (sentence embeddings; the reference's own index has |x| ~ 7.7
    and relative neighbour gaps of 1e-4): the scan copy is taken around the mean of the first rows, so the bf16
    pass stays decisive and (nearly) every query is certified without the exact scan -- L2 and IP, and the
    results stay exact either way."""
    rng = np.random.default_rng(21)
    n, d, nq, k = 50000, 384, 256, 10
    common = rng.standard_normal(d).astype(np.float32) * 0.4
    xb = (common[None, :] + rng.standard_normal((n, d)).astype(np.float32) * 0.02).astype(np.float32)
    xq = (common[None, :] + rng.standard_normal((nq, d)).astype(np.float32) * 0.02).astype(np.float32)
    # inner product: unit vectors with cosines around 0.94 (wider noise than the L2 case: at cosines of 0.997 fp32
    # inner products of neighbouring rows differ by less than one ulp and even the reference's own fp32 scan would
    # order them differently from a float64 oracle)
    xbn = common[None, :] + rng.standard_normal((n, d)).astype(np.float32) * 0.1
    xqn = common[None, :] + rng.standard_normal((nq, d)).astype(np.float32) * 0.1
    xbn = (xbn / np.linalg.norm(xbn, axis=1, keepdims=True)).astype(np.float32)
    xqn = (xqn / np.linalg.norm(xqn, axis=1, keepdims=True)).astype(np.float32)
    for metric, b, q in ((1, xb, xq), (0, xbn, xqn)):
        ix = _make(m, b, metric).set_search_params(algo=m.ALGO_TENSOR)
        D, I = ix.search(q, k)
        _check(D, I, *orc.np_search_f64(b, q, k, metric), metric)
        st = ix.stats()
        assert st["last_algo"] == m.ALGO_TENSOR and st["fallback_queries"] <= nq // 20, (metric, st)
    # rows added later (another batch, same centre) and a search after reset (new centre) stay exact
    ix = _make(m, xb[:1000], 1).set_search_params(algo=m.ALGO_TENSOR)
    ix.add(xb[1000:30000] + 0.5)          # far from the first batch's mean
    both = np.concatenate([xb[:1000], xb[1000:30000] + 0.5])
    D, I = ix.search(xq[:64], k)
    _check(D, I, *orc.np_search_f64(both, xq[:64], k, 1), 1)
    ix.reset()
    ix.add(xb[:5000] - 3.0)
    D, I = ix.search(xq[:64] - 3.0, k)
    _check(D, I, *orc.np_search_f64(xb[:5000] - 3.0, xq[:64] - 3.0, k, 1), 1)


def test_bf16_storage_is_reproducible(m):
    """The same vectors give the same index, bit for bit: bf16 storage rounds the rows around the centre (the mean of the
    first rows), so the centre must not depend on the order in which thread blocks finish (it is summed in 64-bit fixed
    point).  With float atomics two indexes built from the same rows differed by a bf16 ulp in a few coordinates."""
    rng = np.random.default_rng(31)
    n, d = 70000, 96
    xb = (rng.standard_normal((n, d)) + rng.standard_normal(d)[None, :] * 3).astype(np.float32)
    first = None
    for rep in range(4):
        ix = m.IndexFlat(d, m.METRIC_L2, storage=m.STORE_BF16)
        ix.add(xb[:40000])
        ix.add(xb[40000:])
        rows = ix.reconstruct_n()
        if first is None:
            first = rows
            plain = np.abs(rows - xb).max()
            assert plain < 0.05          # (rows are bf16-close to the input)
        else:
            assert np.array_equal(rows.view(np.uint32), first.view(np.uint32)), rep


@pytest.mark.parametrize("metric", [1, 0])
def test_centred_bf16_storage_certifies_embedding_like_data(m, metric, tmp_path):
    """The bf16-storage twin of the test above (BASELINE configs[3] stores bf16): rows sharing a large common
    component are stored as bf16(x - mu), so the tensor pass stays decisive and certifies (nearly) every query; the
    stored rows are also CLOSER to the fp32 input than a plain bf16 cast; results are exact on the authoritative rows,
    through add in two batches, write_index / read_index and the exact scan."""
    import torch

    rng = np.random.default_rng(22)
    n, d, nq, k = 50000, 384, 256, 10
    common = rng.standard_normal(d).astype(np.float32) * 0.4
    scale = 0.02 if metric == 1 else 0.1
    xb = (common[None, :] + rng.standard_normal((n, d)).astype(np.float32) * scale).astype(np.float32)
    xq = (common[None, :] + rng.standard_normal((nq, d)).astype(np.float32) * scale).astype(np.float32)
    if metric == 0:
        xb = (xb / np.linalg.norm(xb, axis=1, keepdims=True)).astype(np.float32)
        xq = (xq / np.linalg.norm(xq, axis=1, keepdims=True)).astype(np.float32)
    ix = m.IndexFlat(d, metric, storage=m.STORE_BF16)
    ix.add(xb[:30000])
    ix.add(xb[30000:])
    rows = ix.reconstruct_n()
    plain = torch.from_numpy(xb).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.abs(rows - xb).mean() < 0.5 * np.abs(plain - xb).mean()    # centred rounding is several times finer
    # (unit vectors with cosines ~0.95 stored at bf16 resolution: a few fp32 inner products at the k-th boundary are
    # exact ties in fp32 arithmetic while the float64 oracle still orders them)
    tie_ok = 0.999 if metric == 0 else 1.0
    ix.set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(rows, xq, k, metric), metric, min_recall=tie_ok)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_TENSOR and st["fallback_queries"] <= nq // 20, (metric, st)
    Ds, Is = ix.set_search_params(algo=m.ALGO_SCAN).search(xq[:9], k)
    _check(Ds, Is, *orc.np_search_f64(rows, xq[:9], k, metric), metric, min_recall=tie_ok)
    # the file holds the authoritative rows in fp32 (FAISS layout); an fp32-storage index read from it answers alike
    path = tmp_path / "bf16.bin"
    m.write_index(ix, path)
    back = m.read_index(path)
    assert np.array_equal(back.reconstruct_n(), rows)
    D2, I2 = back.set_search_params(algo=m.ALGO_TENSOR).search(xq, k)
    _check(D2, I2, D, I, metric, min_recall=tie_ok)


@pytest.mark.parametrize("metric", [1, 0])
def test_big_batch_warp_merge(m, metric):
    """Batches of >= 8192 queries take the warp-per-query list merge; queries it cannot hold are passed on to the block
    kernel.  Exact on benign data, and on data where the k' best cannot certify (near-duplicate rows: dozens of rows
    within the bf16 band of the k-th neighbour), so that the re-rank of every list entry and the exact scan must answer."""
    n, d, nq, k = 60000, 128, 8192, 10
    xb = orc.c_synth_rows(1234, 0, n, d, metric == 0)
    xq = orc.c_synth_rows(5678, 0, nq, d, metric == 0)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb, xq, k, metric), metric)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_TENSOR and st["fallback_queries"] == 0, st
    # clusters of 40 near-duplicates around 600 centres: the neighbours of a query near a centre are separated by far less
    # than the bf16 rounding band, so the k' stage often fails and the later stages must answer
    rng = np.random.default_rng(5)
    centres = rng.standard_normal((600, d)).astype(np.float32)
    xb2 = (np.repeat(centres, 40, axis=0) + rng.standard_normal((24000, d)).astype(np.float32) * 2e-3).astype(np.float32)
    xq2 = (centres[rng.integers(0, 600, nq)] + rng.standard_normal((nq, d)).astype(np.float32) * 2e-3).astype(np.float32)
    if metric == 0:
        xb2 /= np.linalg.norm(xb2, axis=1, keepdims=True)
        xq2 /= np.linalg.norm(xq2, axis=1, keepdims=True)
    ix2 = _make(m, xb2, metric).set_search_params(algo=m.ALGO_TENSOR)
    D2, I2 = ix2.search(xq2, k)
    # (normalised near-duplicates: most of the 40 inner products of a cluster are EQUAL in fp32, so which ids fill the
    # k slots is a tie -- every position must still agree in id or in distance)
    _check(D2, I2, *orc.np_search_f64(xb2, xq2, k, metric), metric, min_recall=0.999 if metric == 1 else 0.0)


def _near_duplicates(nc, dup, nq, metric, ordered=False, seed=9, d=128):
    """nc clusters of `dup` near-duplicates (noise 1e-3: far inside the bf16 rounding band), rows in random order unless
    `ordered`; queries next to randomly chosen cluster centres."""
    rng = np.random.default_rng(seed)
    centres = rng.standard_normal((nc, d)).astype(np.float32)
    xb = (np.repeat(centres, dup, axis=0) + rng.standard_normal((nc * dup, d)).astype(np.float32) * 1e-3).astype(np.float32)
    if not ordered:
        xb = xb[rng.permutation(len(xb))]
    xq = (centres[rng.integers(0, nc, nq)] + rng.standard_normal((nq, d)).astype(np.float32) * 1e-3).astype(np.float32)
    if metric == 0:
        xb /= np.linalg.norm(xb, axis=1, keepdims=True)
        xq /= np.linalg.norm(xq, axis=1, keepdims=True)
    return xb, xq


@pytest.mark.parametrize("metric", [1, 0])
def test_range_pass_serves_uncertified_queries(m, metric):
    """Data denser than the bf16 band (clusters of 400 near-duplicates): the candidate lists cut INSIDE a cluster, so neither
    the k' best nor the extended stage can certify and the first search re-runs every query through the exact scan, four
    per database pass.  The index notices and from the next search on serves them with the range pass -- ONE more tensor
    pass with a fixed threshold per query (every row whose coarse key can belong to a true top-k row is listed and
    re-ranked).  Results are exact both ways; the second search must leave (almost) nothing to the exact scan."""
    import time

    import torch

    d, k, nq = 128, 10, 512
    xb, xq = _near_duplicates(60, 400, nq, metric)
    ref = orc.np_search_f64(xb, xq, k, metric)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_TENSOR)
    tie_ok = 0.999 if metric == 1 else 0.0   # (normalised near-duplicates: fp32 inner products tie, see the test above)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    D, I = ix.search(xq, k)
    t_first = time.perf_counter() - t0
    _check(D, I, *ref, metric, min_recall=tie_ok)
    st1 = ix.stats()
    assert st1["fallback_queries"] > nq // 2 and st1["overflow_queries"] == 0, st1
    t0 = time.perf_counter()
    D2, I2 = ix.search(xq, k)
    t_second = time.perf_counter() - t0
    _check(D2, I2, *ref, metric, min_recall=tie_ok)
    st2 = ix.stats()
    served = st2["range_queries"] - st1["range_queries"]
    left = st2["fallback_queries"] - st1["fallback_queries"]
    print(f"range pass: first search {st1['fallback_queries']} exact-scan queries in {t_first * 1e3:.2f} ms; second search "
          f"{served} range queries, {left} exact-scan queries in {t_second * 1e3:.2f} ms")
    assert served == st1["fallback_queries"], (st1, st2)
    assert left <= 4, (st1, st2)
    # ... and a third search with other queries, device tensors, stays exact
    xq3 = torch.from_numpy(xq[::-1].copy()).cuda()
    D3, I3 = ix.search(xq3, k)
    torch.cuda.synchronize()
    _check(D3.cpu().numpy(), I3.cpu().numpy(), ref[0][::-1], ref[1][::-1], metric, min_recall=tie_ok)
    assert ix.stats()["fallback_queries"] - st2["fallback_queries"] <= 4


@pytest.mark.parametrize("layout", ["huge", "ordered"])
def test_neighbourhoods_beyond_every_list_fall_back_exactly(m, layout):
    """Two shapes no candidate list can hold.  "huge": 4000 near-duplicates per cluster in random row order -- every list
    stays within its capacity but a query has more entries than the merge stages; it selects the k' best straight from
    the lists (no overflow is counted), fails certification WITH a k-th distance, and the range pass that is then tried
    overflows as well, so it switches itself off again: exact scans, slow, exact.  "ordered": clusters of 80 stored
    contiguously -- a query's best rows all sit in one or two lists, the shared thresholds (which need good rows in MANY
    lists) never tighten and the lists overflow: the first search is answered by the exact scan, and the index switches
    to its order-robust mode -- per-thread heaps in the first pass (exact top-k' of every split whatever the order) plus
    the range pass for the near-duplicates the heaps cannot certify -- which leaves nothing to the exact scan."""
    metric, k, nq = 1, 10, 256
    xb, xq = _near_duplicates(6, 4000, nq, metric) if layout == "huge" else _near_duplicates(300, 80, nq, metric, ordered=True)
    ref = orc.np_search_f64(xb, xq, k, metric)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_TENSOR)
    seen = []
    for it in range(5):
        D, I = ix.search(xq, k)
        _check(D, I, *ref, metric, min_recall=0.999)
        seen.append(ix.stats())
    assert seen[0]["fallback_queries"] == nq, seen[0]
    if layout == "huge":
        assert seen[0]["overflow_queries"] == 0, seen[0]          # the merge worked from the lists in global memory
        assert seen[2]["range_queries"] > 0, seen[2]               # the range pass was tried ...
        assert seen[4]["range_queries"] == seen[3]["range_queries"], seen   # ... and gave up
    else:
        assert seen[0]["overflow_queries"] == nq, seen[0]
        assert seen[4]["overflow_queries"] == nq, seen[4]                      # no list overflowed again ...
        assert seen[4]["fallback_queries"] - seen[1]["fallback_queries"] <= 4, seen   # ... and from the third search on nothing needs the exact scan
        assert seen[4]["range_queries"] > 0, seen[4]


def test_very_large_batch_is_cut_into_list_passes(m):
    """20000 queries are far more than one wave of query tiles: the planner cuts the batch into LIST-mode passes
    (not the multi-wave HEAP selection); results must be exact and independent of the cut."""
    n, d, nq, k = 30000, 64, 20000, 10
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, nq, d)
    ix = _make(m, xb, 1).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb, xq, k, 1), 1)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_TENSOR and st["overflow_queries"] == 0, st
    D2, I2 = ix.search(xq[7000:7300], k)
    assert np.array_equal(I2, I[7000:7300]) and np.allclose(D2, D[7000:7300], rtol=1e-6)


def test_random_operation_sequence(m, tmp_path):
    """Seeded fuzz over the index life cycle: adds (host arrays and device tensors, growing the storage several
    times), searches (host / device buffers, both paths, changing batch sizes and k, so the workspace is
    re-carved and re-allocated while earlier device-buffer searches may still be in flight), reset, reconstruct,
    write + read.  Every search is checked against the oracle on a host mirror of the rows."""
    import torch

    rng = np.random.default_rng(77)
    for metric in (1, 0):
        d = 96
        ix = m.IndexFlat(d, metric)
        mirror = np.zeros((0, d), np.float32)
        pending = []   # device-buffer results checked later (they are produced asynchronously)
        for step in range(70):
            op = rng.choice(["add", "add_dev", "search", "search", "search_dev", "search_dev", "reset", "io", "recon"],
                            p=[0.14, 0.1, 0.24, 0.0, 0.3, 0.0, 0.04, 0.06, 0.12])
            if op in ("add", "add_dev") or mirror.shape[0] == 0:
                n = int(rng.choice([1, 5, 100, 1500, 9000]))
                x = (rng.standard_normal((n, d)) + 0.3).astype(np.float32)
                ix.add(torch.from_numpy(x).cuda() if op == "add_dev" else x)
                mirror = np.concatenate([mirror, x])
                assert ix.ntotal == mirror.shape[0]
            elif op in ("search", "search_dev"):
                nq = int(rng.choice([1, 3, 40, 130, 600]))
                k = int(rng.choice([1, 10, 50]))
                algo = int(rng.choice([m.ALGO_AUTO, m.ALGO_SCAN, m.ALGO_TENSOR]))
                xq = (rng.standard_normal((nq, d)) + 0.3).astype(np.float32)
                ix.set_search_params(algo=algo)
                ref = orc.np_search_f64(mirror, xq, k, metric)
                if op == "search_dev":
                    pending.append((ix.search(torch.from_numpy(xq).cuda(), k), ref, (step, nq, k, algo)))
                else:
                    D, I = ix.search(xq, k)
                    _check(D, I, *ref, metric)
            elif op == "reset":
                torch.cuda.synchronize()
                for (D, I), ref, tag in pending:
                    _check(D.cpu().numpy(), I.cpu().numpy(), *ref, metric)
                pending = []
                ix.reset()
                mirror = np.zeros((0, d), np.float32)
            elif op == "io":
                path = tmp_path / f"fuzz_{metric}_{step}.bin"
                m.write_index(ix, path)
                back = m.read_index(path)
                assert back.ntotal == ix.ntotal and back.metric_type == metric
                assert np.array_equal(back.reconstruct_n(), mirror)
                ix = back
            else:
                i = int(rng.integers(0, mirror.shape[0]))
                assert np.array_equal(ix.reconstruct(i), mirror[i])
        torch.cuda.synchronize()
        for (D, I), ref, tag in pending:
            r = orc.recall_and_errors(D.cpu().numpy(), I.cpu().numpy(), *ref, metric)
            assert r["recall"] == 1.0 and r["id_mismatch"] == 0 and r["padding_ok"] and r["max_rel_err"] <= REL, (tag, r)


def test_async_device_searches_back_to_back(m):
    """Device-buffer searches return without synchronising (the uncertified-query count never visits the
    host): several searches queued back to back on one stream, then on another stream, must all be right."""
    import torch

    n, d, k = 60000, 128, 10
    xb = orc.c_synth_rows(1234, 0, n, d)
    ix = _make(m, xb, 1).set_search_params(algo=m.ALGO_TENSOR)
    batches = [orc.c_synth_rows(100 + i, 0, nq, d) for i, nq in enumerate((200, 64, 300, 1, 129))]
    outs = [ix.search(torch.from_numpy(b).cuda(), k) for b in batches]
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        side.wait_stream(torch.cuda.current_stream())
        outs2 = [ix.search(torch.from_numpy(b).cuda(), k) for b in batches[:2]]
    torch.cuda.synchronize()
    for b, (D, I) in zip(batches + batches[:2], outs + outs2):
        _check(D.cpu().numpy(), I.cpu().numpy(), *orc.np_search_f64(xb, b, k, 1), 1)
    st = ix.stats()
    assert st["searches"] == 7 and st["overflow_queries"] == 0, st


def test_auto_dispatch(m):
    xb = orc.c_synth_rows(1, 0, 4000, 128)
    ix = _make(m, xb, 1)
    ix.search(orc.c_synth_rows(2, 0, 1, 128), 10)     # the reference's batch size -> exact fp32 scan
    assert ix.stats()["last_algo"] == m.ALGO_SCAN
    ix.set_search_params(scan_max_nq=8)
    ix.search(orc.c_synth_rows(2, 0, 8, 128), 10)
    assert ix.stats()["last_algo"] == m.ALGO_SCAN
    ix.set_search_params(scan_max_nq=1)
    ix.search(orc.c_synth_rows(2, 0, 64, 128), 10)
    assert ix.stats()["last_algo"] == m.ALGO_TENSOR
    D, I = ix.search(orc.c_synth_rows(2, 0, 64, 128), 200)   # k' > 64: falls back to the exact scan
    assert ix.stats()["last_algo"] == m.ALGO_SCAN
    _check(D, I, *orc.np_search_f64(xb, orc.c_synth_rows(2, 0, 64, 128), 200, 1), 1)


# ---- bf16 storage: the oracle runs on the authoritative (rounded) rows ----------------------------------
@pytest.mark.parametrize("algo_name", ["scan", "tensor"])
def test_bf16_storage(m, algo_name):
    """bf16 storage keeps ONE copy: bf16(x - mu) around the index's centre mu (mean of the first rows); the
    authoritative row is fl32(mu + bf16(x - mu)), which is what reconstruct / write_index return and what both
    search paths measure distances to."""
    n, d, nq, k = 20000, 384, 40, 10
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, nq, d)
    ix = m.IndexFlat(d, 1, storage=m.STORE_BF16)
    ix.add(xb)
    xb_r = ix.reconstruct_n()
    mu = xb.mean(0)
    # within the bf16 rounding of the CENTRED value (2^-9 relative), plus slack for the centre being an fp32 mean
    assert np.all(np.abs(xb_r - xb) <= 2.0 ** -8 * np.abs(xb - mu) + 1e-3)
    assert np.array_equal(ix.reconstruct(7), xb_r[7]) and np.array_equal(ix.reconstruct_n(100, 50), xb_r[100:150])
    ix.set_search_params(algo=m.ALGO_SCAN if algo_name == "scan" else m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb_r, xq, k, 1), 1)
    # AUTO on bf16 storage: every batch size (the reference's nq = 1 included) goes to the tensor path
    ix.set_search_params(algo=m.ALGO_AUTO)
    D1, I1 = ix.search(xq[:1], k)
    _check(D1, I1, *orc.np_search_f64(xb_r, xq[:1], k, 1), 1)
    assert ix.stats()["last_algo"] == m.ALGO_TENSOR


# ---- torch tensor handoff, pooling kernel, synthetic generator, merge kernel ---------------------------
def test_torch_device_pointers(m):
    import torch

    d = 384
    xb = orc.c_synth_rows(1234, 0, 3000, d)
    xq = orc.c_synth_rows(5678, 0, 20, d)
    ix = m.IndexFlatL2(d)
    ix.add(torch.from_numpy(xb).cuda())
    Dt, It = ix.search(torch.from_numpy(xq).cuda(), 10)
    assert Dt.is_cuda and It.dtype == torch.int64
    torch.cuda.synchronize()
    _check(Dt.cpu().numpy(), It.cpu().numpy(), *orc.np_search_f64(xb, xq, 10, 1), 1)


def test_pool_normalize_and_add_pooled(m):
    import torch

    from rag_faiss_embedding_b200.encoder import pool_normalize

    torch.manual_seed(0)
    B, T, d = 37, 19, 384
    h = torch.randn(B, T, d, device="cuda") * 2 + 0.5
    lens = torch.randint(1, T + 1, (B,), device="cuda")
    mask = (torch.arange(T, device="cuda")[None, :] < lens[:, None]).to(torch.int64)
    cls = pool_normalize(h, mask, "cls", False)
    assert torch.equal(cls, h[:, 0])                      # reference semantics: raw CLS token, bit exact
    mean_ref = (h * mask[..., None]).sum(1) / mask.sum(1, keepdim=True).clamp(min=1e-9)
    mean = pool_normalize(h, mask, "mean", False)
    assert torch.allclose(mean, mean_ref, rtol=1e-5, atol=1e-6)
    nrm = pool_normalize(h, mask, "mean", True)
    assert torch.allclose(nrm, torch.nn.functional.normalize(mean_ref, dim=1), rtol=1e-5, atol=1e-6)
    ix = m.IndexFlatIP(d)
    ix.add_pooled(h, mask, pool="mean", normalize=True)
    ix.add_pooled(h, None, pool="cls", normalize=False)
    torch.cuda.synchronize()
    assert ix.ntotal == 2 * B
    rows = ix.reconstruct_n()
    assert np.allclose(rows[:B], nrm.cpu().numpy(), rtol=1e-6, atol=1e-7)
    assert np.array_equal(rows[B:], h[:, 0].cpu().numpy())
    D, I = ix.search(nrm.cpu().numpy()[:5], 1)
    assert I[:, 0].tolist() == [0, 1, 2, 3, 4] or (D[:, 0] >= 1 - 1e-4).all()
    # query side of the hand-off: pool + normalise + search in one call == pooling first, then searching
    Dp, Ip = ix.search_pooled(h, mask, 3, pool="mean", normalize=True)
    Dr, Ir = ix.search(nrm, 3)
    torch.cuda.synchronize()
    assert torch.equal(Ip, Ir) and torch.allclose(Dp, Dr, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("normalize", [False, True])
def test_add_pooled_bf16_storage_both_metrics(m, metric, normalize):
    """add_pooled into a bf16-storage index, inner product included: the per-row bias of the tensor pass must come
    from the ingest kernel (IP: -mu.x, not |x|^2), so the tensor path -- where AUTO sends every batch on bf16
    storage -- finds the true neighbours of the rounded rows."""
    import torch

    from rag_faiss_embedding_b200.encoder import pool_normalize

    torch.manual_seed(3)
    B, T, d, k = 3000, 5, 128, 10
    h = torch.randn(B, T, d, device="cuda") + 0.25
    mask = torch.ones(B, T, dtype=torch.int64, device="cuda")
    ix = m.IndexFlat(d, metric, storage=m.STORE_BF16)
    ix.add_pooled(h[:2000], mask[:2000], pool="mean", normalize=normalize)
    ix.add_pooled(h[2000:], mask[2000:], pool="mean", normalize=normalize)
    rows = ix.reconstruct_n()   # the authoritative (rounded) rows
    pooled = pool_normalize(h, mask, "mean", normalize)
    assert np.allclose(rows, pooled.cpu().numpy(), rtol=1e-2, atol=1e-2)
    xq = pooled[:64].cpu().numpy() + 0.01
    for algo in (m.ALGO_AUTO, m.ALGO_TENSOR, m.ALGO_SCAN):
        D, I = ix.set_search_params(algo=algo).search(xq, k)
        _check(D, I, *orc.np_search_f64(rows, xq, k, metric), metric)
        if algo != m.ALGO_SCAN:
            assert ix.stats()["last_algo"] == m.ALGO_TENSOR


def test_add_on_side_stream_is_ordered_before_search(m):
    """A device-tensor add enqueued on a caller stream behind a long-running kernel, immediately followed by a numpy
    search (the index's own non-blocking stream), a growth re-allocation and a write: every consumer must wait for
    the ingest (no torch.cuda.synchronize() anywhere in between)."""
    import torch

    d, k = 128, 5
    xb = orc.c_synth_rows(1234, 0, 6000, d)
    xq = orc.c_synth_rows(5678, 0, 8, d)
    side = torch.cuda.Stream()
    ix = m.IndexFlatL2(d)
    ix.add(xb[:1000])                       # capacity 1024: the next add must grow the storage
    big = torch.empty(64 << 20, device="cuda")
    with torch.cuda.stream(side):
        for _ in range(20):
            big.normal_()                   # keeps the side stream busy for a while
        xt = torch.from_numpy(xb[1000:1020]).cuda(non_blocking=False)
        ix.add(xt)                          # enqueued behind the busy work on `side`
        for _ in range(20):
            big.normal_()
        ix.add(torch.from_numpy(xb[1020:6000]).cuda())   # grows: copies the old rows (incl. the pending 20) first
    D, I = ix.search(xq, k)                 # numpy search: index stream
    _check(D, I, *orc.np_search_f64(xb, xq, k, 1), 1)
    assert np.array_equal(ix.reconstruct_n(990, 40), xb[990:1030])
    torch.cuda.synchronize()


def test_tensor_on_other_device_is_rejected(m):
    import torch

    ix = m.IndexFlatL2(16)
    ix.add(np.zeros((4, 16), np.float32))
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    x = torch.zeros(2, 16, device="cuda:1")
    for fn in (lambda: ix.search(x, 1), lambda: ix.add(x),
               lambda: ix.search_tensors_into(x, 1, torch.empty(2, 1, device="cuda:1"),
                                              torch.empty(2, 1, dtype=torch.int64, device="cuda:1"))):
        with pytest.raises(AssertionError):
            fn()


def test_synth_bit_identical(m):
    from rag_faiss_embedding_b200.encoder import synth_rows

    for norm in (False, True):
        a = synth_rows(1234, 999_983, 257, 384, norm).cpu().numpy()
        b = orc.c_synth_rows(1234, 999_983, 257, 384, norm)
        assert np.array_equal(a, b)
    ix = m.IndexFlatL2(96)
    ix.add_synthetic(77, 5, 1000)
    assert np.array_equal(ix.reconstruct_n(), orc.c_synth_rows(77, 5, 1000, 96))


def test_merge_topk_kernel(m):
    import torch

    from tests.helpers import np_merge

    rng = np.random.default_rng(3)
    for metric in (1, 0):
        G, nq, k = 8, 50, 10
        D = np.sort(rng.random((G, nq, k)).astype(np.float32), axis=2)
        if metric == 0:
            D = D[:, :, ::-1].copy()
        I = rng.permutation(G * nq * k).reshape(G, nq, k).astype(np.int64)
        D[3, :, 7:] = FLT_MAX if metric == 1 else -FLT_MAX   # a short shard
        I[3, :, 7:] = -1
        D[5] = D[2]                                           # exact ties across shards -> lower label first
        Dm, Im = m.merge_topk(metric, torch.from_numpy(D).cuda(), torch.from_numpy(I).cuda())
        D_ref, I_ref = np_merge(metric, D, I)
        assert np.array_equal(Im.cpu().numpy(), I_ref) and np.array_equal(Dm.cpu().numpy(), D_ref)


# ---- full-size properties at the BASELINE config (1M x 384, fp32, L2, k=10) -----------------------------
def test_full_size_properties(m):
    n, d, k = 1_000_000, 384, 10
    ix = m.IndexFlatL2(d)
    ix.add_synthetic(1234, 0, n)
    assert ix.ntotal == n
    # self-queries: every row's nearest neighbour is itself at distance exactly 0 (exact-difference form)
    rows = np.array([0, 1, 255, 256, 499_999, 777_777, 999_999])
    q_self = np.stack([orc.c_synth_rows(1234, int(r), 1, d)[0] for r in rows])
    for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
        D, I = ix.set_search_params(algo=algo).search(q_self, k)
        assert I[:, 0].tolist() == rows.tolist() and (D[:, 0] == 0).all()
        assert (np.diff(D, axis=1) >= 0).all()
    # sampled parity against the oracle's own exhaustive scan (8 queries x 1M rows on the host)
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, 1024, d)
    D_ref, I_ref = orc.c_search(xb, xq[:8], k, 1, algo=1)
    D8, I8 = ix.set_search_params(algo=m.ALGO_SCAN).search(xq[:8], k)
    _check(D8, I8, D_ref, I_ref, 1)
    # the two GPU paths must agree with each other on the whole 1024-query batch
    Dt, It = ix.set_search_params(algo=m.ALGO_TENSOR).search(xq, k)
    _check(Dt[:8], It[:8], D_ref, I_ref, 1)
    Ds, Is = ix.set_search_params(algo=m.ALGO_SCAN).search(xq[:64], k)
    _check(Dt[:64], It[:64], Ds, Is, 1)
    # idempotence and batch-independence: a query's answer does not depend on its batch
    D1, I1 = ix.set_search_params(algo=m.ALGO_TENSOR).search(xq[100:101], k)
    assert np.array_equal(I1[0], It[100]) and np.allclose(D1[0], Dt[100], rtol=1e-6)


def test_large_bf16_index_properties(m):
    """> 4 GiB of bf16 rows (6M x 384) and long per-split streams: exercises 64-bit addressing, the adaptive
    candidate-list capacity and the overflow path.  Checked through size-independent properties: self
    queries return themselves at distance 0, and the tensor path agrees with the exact scan."""
    n, d, k = 6_000_000, 384, 10
    ix = m.IndexFlat(d, 1, storage=m.STORE_BF16)
    ix.reserve(n)
    ix.add_synthetic(1234, 0, n)
    rows = [0, 1, n // 2, n - 1]
    q_self = np.stack([ix.reconstruct(r) for r in rows])   # the stored (authoritative, rounded) rows
    assert np.allclose(q_self, np.stack([orc.c_synth_rows(1234, r, 1, d)[0] for r in rows]), rtol=2.0 ** -7, atol=1e-2)
    xq = np.concatenate([q_self, orc.c_synth_rows(5678, 0, 1020, d)])
    Dt, It = ix.set_search_params(algo=m.ALGO_TENSOR).search(xq, k)
    assert It[:4, 0].tolist() == rows and (Dt[:4, 0] == 0).all()
    assert (np.diff(Dt, axis=1) >= 0).all() and (It >= 0).all() and (It < n).all()
    Ds, Is = ix.set_search_params(algo=m.ALGO_SCAN).search(xq[:16], k)
    _check(Dt[:16], It[:16], Ds, Is, 1)
