"""GPU tier (-m gpu): every search kernel variant at its shape and scale edges, against float64 brute force.

test_gpu_parity.py covers data distributions; this file covers shapes and magnitudes: the streamed K2 kernel at common
embedding widths (d up to 4096), the streaming scan up to d = 16384 (one query per group), the k' steps of the tensor
path, bf16 storage at ragged d, power-of-two scale invariance, a centre far from the origin, the pooling kernel and the
shard merge.  The shapes are module constants so that tests/test_edges_plan_cpu.py can check, without a GPU, which
tensor-path kernels they reach."""
import ctypes

import numpy as np
import pytest

import oracle as orc
from tests.exact_checks import check_structure

pytestmark = pytest.mark.gpu

FLT_MAX = np.finfo(np.float32).max
REL = 1e-5
METRICS = (1, 0)   # every tensor-path shape below runs under L2 and inner product

# (n, d, nq, k) for ALGO_TENSOR.  d > 384 (more than QRES_MAX_KB = 6 k-blocks): the streamed LIST kernel, 7 to 64 k-blocks;
# n = 256 t + 1 / 256 t - 1 put one row in a last database tile / leave it one short; d <= 384 cases reach the pair kernel
# (an odd count of 7 query tiles), the Q-resident LIST kernel, HEAP mode with k' = 32 and 64 (a single database tile) and
# a batch the planner cuts into several passes (k' = 192).
TENSOR_SHAPES = [
    (30000, 385, 129, 10),
    (25601, 449, 1000, 10),
    (20000, 1024, 1, 10),
    (20000, 1536, 129, 100),
    (20479, 3072, 129, 10),
    (12000, 4096, 33, 10),
    (30000, 384, 833, 10),
    (30000, 384, 300, 10),
    (200, 128, 64, 10),
    (200, 128, 64, 20),
    (8000, 449, 4096, 100),
]
EMBED_SHAPE = (30000, 1536, 256, 10)   # normalised-embedding-like data at a common encoder width

# k -> k' = k + max(22, ceil(0.9 k)) rounded up to 32 / 64 / a multiple of 8; 0 = beyond 256, served by the exact scan
KPRIME = {10: 32, 11: 64, 20: 64, 33: 64, 34: 72, 42: 80, 43: 88, 100: 192, 134: 256, 135: 0}
# (k, slack) -> k' when the caller sets the slack
KPRIME_SLACK = {(10, 5): 32, (10, 30): 64, (10, 70): 80, (20, 100): 120, (100, 156): 256, (100, 157): 0}
KPRIME_DATA = (20000, 128, 64)   # (n, d, nq)

SCAN_D = (2049, 4096, 8193, 16384)
SCAN_K = (1, 100, 1024)
SCAN_NQ = (1, 3, 9)
SCAN_N = 2000

BF16_RAGGED_D = (1, 7, 30, 100, 130, 1030)
SCALES = (-40, -20, -6, 6, 20, 40)


def plan_shapes():
    """Every (nq, n, d, k, slack) the tensor-path tests below search with."""
    shapes = [(nq, n, d, k, 0) for n, d, nq, k in TENSOR_SHAPES]
    n, d, nq, k = EMBED_SHAPE
    shapes.append((nq, n, d, k, 0))
    n, d, nq = KPRIME_DATA
    shapes += [(nq, n, d, k, 0) for k in KPRIME]
    shapes += [(nq, n, d, k, s) for k, s in KPRIME_SLACK]
    return shapes


@pytest.fixture(scope="module")
def m():
    import rag_faiss_embedding_b200 as mod

    assert mod.device_count() > 0, "no B200 visible"
    return mod


def _check(D, I, D_ref, I_ref, metric, rel=REL, min_recall=1.0, abs_floor=1e-4):
    check_structure(D, I, metric)
    r = orc.recall_and_errors(D, I, D_ref, I_ref, metric, rel_tol=rel, abs_floor=abs_floor)
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


def _plan(m, nq, n, d, k, slack=0):
    out = (ctypes.c_int32 * 12)()
    assert m._capi.load().b2f_plan_describe(nq, n, d, k, slack, out) == 0
    return dict(zip(["kp", "chunk", "passes", "list", "pair"], list(out)[:5]))


# ---- K2 tensor path at large d -------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("n,d,nq,k", TENSOR_SHAPES)
def test_tensor_shapes_vs_oracle(m, metric, n, d, nq, k):
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, nq, d)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb, xq, k, metric), metric)
    st = ix.stats()
    assert st["last_algo"] == m.ALGO_TENSOR and st["last_kprime"] == KPRIME[k], st
    assert st["last_kprime"] == _plan(m, nq, n, d, k)["kp"]
    if n >= 5000:   # random data: the fused filter must not overflow its candidate lists
        assert st["overflow_queries"] == 0, st


@pytest.mark.parametrize("metric", METRICS)
def test_tensor_embedding_like_large_d_certifies(m, metric):
    """Rows sharing a large common component at d = 1536: the certification slack gam = 4 (d + 16) u grows with d, and the
    bound must still certify (nearly) every query -- the results are exact either way."""
    n, d, nq, k = EMBED_SHAPE
    rng = np.random.default_rng(41)
    common = rng.standard_normal(d).astype(np.float32) * 0.4
    noise = 0.02 if metric == 1 else 0.1
    xb = (common[None, :] + rng.standard_normal((n, d)).astype(np.float32) * noise).astype(np.float32)
    xq = (common[None, :] + rng.standard_normal((nq, d)).astype(np.float32) * noise).astype(np.float32)
    if metric == 0:
        xb = (xb / np.linalg.norm(xb, axis=1, keepdims=True)).astype(np.float32)
        xq = (xq / np.linalg.norm(xq, axis=1, keepdims=True)).astype(np.float32)
    ix = _make(m, xb, metric).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    st = ix.stats()
    print(f"d = {d} metric {metric}: {st['fallback_queries']} exact-scan, {st['range_queries']} range-pass, "
          f"{st['rescued_queries']} rescued of {nq} queries")
    assert st["last_algo"] == m.ALGO_TENSOR and st["fallback_queries"] <= nq // 20, st
    # (unit vectors with cosines ~0.94 at d = 1536: the fp32 inner products of a few rows at the k-th boundary differ by
    # less than their own rounding, a tie in fp32 arithmetic that the float64 oracle still orders; every position must
    # still agree in id or in distance)
    _check(D, I, *orc.np_search_f64(xb, xq, k, metric), metric, min_recall=0.999 if metric == 0 else 1.0)


# ---- K1 streaming scan at large d: one, two or four queries per group ------------------------------------
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("d", SCAN_D)
@pytest.mark.parametrize("storage", ["fp32", "bf16"])
def test_scan_large_d_vs_oracle(m, storage, d, metric):
    rng = np.random.default_rng(d)
    xb = (rng.standard_normal((SCAN_N, d)) + 0.3).astype(np.float32)
    xq = (rng.standard_normal((max(SCAN_NQ), d)) + 0.3).astype(np.float32)
    ix = m.IndexFlat(d, metric, storage=m.STORE_BF16 if storage == "bf16" else m.STORE_F32)
    ix.add(xb)
    rows = ix.reconstruct_n()
    if storage == "fp32":
        assert np.array_equal(rows, xb)
    else:
        assert np.abs(rows - xb).max() < 0.05
    D_ref, I_ref = orc.np_search_f64(rows, xq, max(SCAN_K), metric)
    ix.set_search_params(algo=m.ALGO_SCAN)
    for k in SCAN_K:
        for nq in SCAN_NQ:
            D, I = ix.search(xq[:nq], k)
            _check(D, I, D_ref[:nq, :k], I_ref[:nq, :k], metric)
            st = ix.stats()
            assert st["last_algo"] == m.ALGO_SCAN and st["last_launches"] == 1, (k, nq, st)


# ---- k' steps of the tensor path -------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_kprime_steps(m, metric):
    n, d, nq = KPRIME_DATA
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, nq, d)
    kmax = max(max(KPRIME), max(k for k, _ in KPRIME_SLACK))
    D_ref, I_ref = orc.np_search_f64(xb, xq, kmax, metric)
    ix = _make(m, xb, metric)
    cases = [(k, 0, kp) for k, kp in KPRIME.items()] + [(k, s, kp) for (k, s), kp in KPRIME_SLACK.items()]
    for k, slack, kp in cases:
        p = m.SearchParams()
        p.algo, p.slack = m.ALGO_TENSOR, slack
        D, I = ix.search(xq, k, params=p)
        _check(D, I, D_ref[:, :k], I_ref[:, :k], metric)
        st = ix.stats()
        assert _plan(m, nq, n, d, k, slack)["kp"] == kp, (k, slack)
        if kp:
            assert st["last_algo"] == m.ALGO_TENSOR and st["last_kprime"] == kp, (k, slack, st)
        else:   # k' > 256: an explicit TENSOR request is served by the exact scan
            assert st["last_algo"] == m.ALGO_SCAN and st["last_kprime"] == 0, (k, slack, st)


# ---- bf16 storage at ragged d: scalar ingest / re-rank branches, padded query and centre tiles in K1 --------
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("d", BF16_RAGGED_D)
def test_bf16_storage_ragged_d(m, d, metric):
    rng = np.random.default_rng(100 + d)
    n, nq, k = 6000, 40, 10
    xb = (rng.standard_normal((n, d)) * 0.5 + rng.standard_normal(d)[None, :] * 2).astype(np.float32)
    xq = (xb[rng.integers(0, n, nq)] + rng.standard_normal((nq, d)).astype(np.float32) * 0.1).astype(np.float32)
    ix = m.IndexFlat(d, metric, storage=m.STORE_BF16)
    ix.add(xb[:4000])
    ix.add(xb[4000:])
    rows = ix.reconstruct_n()
    # within the bf16 rounding of the CENTRED value (2^-9 relative; the centre is the mean of the first add), plus slack for
    # the centre being an fp32 mean and for the fp32 addition that forms the authoritative row
    mu = xb[:4000].astype(np.float64).mean(0)
    assert np.all(np.abs(rows - xb) <= 2.0 ** -8 * np.abs(xb - mu) + 1e-3)
    assert np.abs(rows - xb).max() > 0    # (the rows really are rounded)
    D_ref, I_ref = orc.np_search_f64(rows, xq, k, metric)
    # (d = 1: thousands of rows share one rounded value, and two different float64 distances can round to the same fp32
    # one -- a tie in fp32 arithmetic that the oracle still orders; every position must still agree in id or distance)
    tie_ok = 0.99 if d == 1 else 1.0
    for algo in (m.ALGO_SCAN, m.ALGO_TENSOR, m.ALGO_AUTO):
        D, I = ix.set_search_params(algo=algo).search(xq, k)
        _check(D, I, D_ref, I_ref, metric, min_recall=tie_ok)
        assert ix.stats()["last_algo"] == (m.ALGO_SCAN if algo == m.ALGO_SCAN else m.ALGO_TENSOR)


# ---- scale invariance (metamorphic) --------------------------------------------------------------------
def _near_duplicates(nc, dup, nq, metric, seed=9, d=128):
    """nc clusters of `dup` near-duplicates (noise 1e-3: far inside the bf16 rounding band) in random row order; queries next
    to randomly chosen cluster centres (as in test_gpu_parity.py)."""
    rng = np.random.default_rng(seed)
    centres = rng.standard_normal((nc, d)).astype(np.float32)
    xb = (np.repeat(centres, dup, axis=0) + rng.standard_normal((nc * dup, d)).astype(np.float32) * 1e-3).astype(np.float32)
    xb = xb[rng.permutation(len(xb))]
    xq = (centres[rng.integers(0, nc, nq)] + rng.standard_normal((nq, d)).astype(np.float32) * 1e-3).astype(np.float32)
    if metric == 0:
        xb /= np.linalg.norm(xb, axis=1, keepdims=True)
        xq /= np.linalg.norm(xq, axis=1, keepdims=True)
    return xb, xq


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("data", ["random", "near_duplicates"])
def test_scale_invariance(m, data, metric):
    """Rows and queries scaled by 2^s are exact in fp32 over this range, and both paths end in the fp32 exact re-rank /
    exact scan, whose arithmetic commutes with a power-of-two scale.  So every scaled search must return the SAME ids
    and exactly 2^(2 s) times the distances of the unscaled one, bit for bit -- on the first search and on the second,
    which (near-duplicates) runs the range pass.  An absolute constant anywhere in the centring, the certification or
    the range thresholds that changed a decision would show up here."""
    k = 10
    if data == "random":
        rng = np.random.default_rng(17)
        xb = rng.standard_normal((20000, 128)).astype(np.float32)
        xq = rng.standard_normal((200, 128)).astype(np.float32)
        tie_ok = 1.0
    else:
        xb, xq = _near_duplicates(60, 400, 512, metric)
        tie_ok = 0.999 if metric == 1 else 0.0   # normalised near-duplicates: fp32 inner products tie
    runs = {}
    for s in (0,) + SCALES:
        f = np.float32(2.0 ** s)
        b, q = xb * f, xq * f
        assert np.array_equal(b / f, xb) and np.array_equal(q / f, xq)
        ref = orc.np_search_f64(b, q, k, metric)
        ix = _make(m, b, metric)
        out = []
        for algo in (m.ALGO_SCAN, m.ALGO_TENSOR, m.ALGO_TENSOR):
            D, I = ix.set_search_params(algo=algo).search(q, k)
            _check(D, I, *ref, metric, min_recall=tie_ok, abs_floor=1e-4 * 2.0 ** (2 * s))
            out.append((D, I, ix.stats()))
        runs[s] = out
    for s in SCALES:
        f2 = np.float32(2.0 ** (2 * s))
        for (D0, I0, st0), (D, I, st) in zip(runs[0], runs[s]):
            assert np.array_equal(I, I0), s
            assert np.array_equal(D.view(np.uint32), (D0 * f2).view(np.uint32)), s
            for key in ("fallback_queries", "range_queries", "rescued_queries", "overflow_queries"):
                assert st[key] == st0[key], (s, key, st0, st)
    st_lo, st_hi = runs[SCALES[0]][-1][2], runs[SCALES[-1]][-1][2]
    print(f"{data} metric {metric}: after two tensor searches at s = {SCALES[0]} / {SCALES[-1]}: "
          f"exact-scan {st_lo['fallback_queries']} / {st_hi['fallback_queries']}, "
          f"range-pass {st_lo['range_queries']} / {st_hi['range_queries']}")
    if data == "near_duplicates":
        assert runs[0][-1][2]["range_queries"] > 0   # the second tensor search did run the range pass


# ---- a centre far from the origin ----------------------------------------------------------------------
def test_centre_of_rows_far_from_origin(m):
    """Rows around a per-coordinate mean of ~4e8 (70000 rows, more than the 65536 the centre is taken from): the 64-bit
    fixed-point sum of the first rows is ~2.6e13 per column, far past what a fixed 2^24 scale holds.  The centre must
    still be the mean: bf16 storage keeps rows several times closer to the input than a plain bf16 cast, and fp32
    storage certifies (nearly) every query instead of handing them to the exact scan.  Results are exact either way."""
    import torch

    rng = np.random.default_rng(51)
    n, d, nq, k = 70000, 64, 64, 10
    mean = (4e8 * (1 + 0.1 * rng.standard_normal(d))).astype(np.float32)
    xb = (mean[None, :] + rng.standard_normal((n, d)).astype(np.float32) * 2.0 ** 20).astype(np.float32)
    xq = (mean[None, :] + rng.standard_normal((nq, d)).astype(np.float32) * 2.0 ** 20).astype(np.float32)
    ix = _make(m, xb, 1).set_search_params(algo=m.ALGO_TENSOR)
    D, I = ix.search(xq, k)
    _check(D, I, *orc.np_search_f64(xb, xq, k, 1), 1)
    st = ix.stats()
    print(f"centre ~4e8, fp32 storage: {st['fallback_queries']} exact-scan of {nq} queries")
    assert st["last_algo"] == m.ALGO_TENSOR and st["fallback_queries"] <= nq // 20, st
    ix = m.IndexFlat(d, 1, storage=m.STORE_BF16)
    ix.add(xb)
    rows = ix.reconstruct_n()
    plain = torch.from_numpy(xb).to(torch.bfloat16).to(torch.float32).numpy()
    err, err_plain = np.abs(rows - xb).mean(), np.abs(plain - xb).mean()
    print(f"centre ~4e8, bf16 storage: mean |row - x| {err:.4g}, plain bf16 cast {err_plain:.4g}")
    assert err < 0.1 * err_plain
    for algo in (m.ALGO_TENSOR, m.ALGO_SCAN):
        D, I = ix.set_search_params(algo=algo).search(xq, k)
        _check(D, I, *orc.np_search_f64(rows, xq, k, 1), 1)


# ---- K7 pooling ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", (7, 100, 384, 1030, 2048))
def test_pool_normalize_vs_float64(m, d):
    """CLS / masked mean, normalised or not, over masks with holes, an all-zero mask row and an all-zero hidden row, on both
    the vectorised (d % 4 == 0, d / 4 <= 256) and the scalar mean path, T from 1 to 513 (not a multiple of the token
    stride).  Reference: torch in float64.  Bound: the fp32 rounding of a T-term sum and of a d-term norm."""
    import torch

    from rag_faiss_embedding_b200.encoder import pool_normalize

    g = torch.Generator().manual_seed(d)
    u = 2.0 ** -24
    for T in (1, 5, 37, 513):
        B = 9
        h = torch.randn(B, T, d, generator=g) * 2 + 0.5
        h[1] = 0.0                                             # a zero row: normalising it must give 0, not NaN
        mask = (torch.rand(B, T, generator=g) < 0.7).to(torch.int64)
        mask[:, 0] = 1
        mask[0] = 0                                            # an all-zero mask row: mean = 0 / 1e-9 = 0
        if T > 2:
            mask[2, 1::2] = 0                                  # holes
        hd, md = h.double(), mask.double()
        cnt = md.sum(1, keepdim=True).clamp(min=1e-9)
        for pool in ("cls", "mean"):
            if pool == "cls":
                v, mag = hd[:, 0], hd[:, 0].abs()
            else:
                v = (hd * md[..., None]).sum(1) / cnt
                mag = (hd.abs() * md[..., None]).sum(1) / cnt   # the sum of |terms| the fp32 rounding scales with
            for normalize in (False, True):
                ref, tol = v, (T + 4) * u * mag
                if normalize:
                    nrm = v.norm(dim=1, keepdim=True).clamp(min=1e-12)
                    ref = v / nrm
                    tol = tol / nrm + (d + 8) * u * ref.abs() + 1e-30
                got = pool_normalize(h.cuda(), mask.cuda(), pool, normalize).cpu().double()
                assert torch.isfinite(got).all(), (T, pool, normalize)
                err = (got - ref).abs()
                assert (err <= 2 * tol).all(), (T, pool, normalize, float(err.max()), float((err / (2 * tol + 1e-300)).max()))
                assert (got[1] == 0).all() and (pool == "cls" or (got[0] == 0).all())
                if pool == "cls" and not normalize:
                    assert torch.equal(got.float(), h[:, 0])   # reference semantics: the raw CLS token, bit exact
    # the query side of the hand-off: pooling + normalising + searching in one call == pooling first, then searching
    rng = np.random.default_rng(d)
    xb = rng.standard_normal((500, d)).astype(np.float32)
    for metric in METRICS:
        ix = _make(m, xb, metric)
        hc, mc = h.cuda(), mask.cuda()
        for pool, normalize in (("mean", True), ("cls", False)):
            Dp, Ip = ix.search_pooled(hc, mc, 5, pool=pool, normalize=normalize)
            Dr, Ir = ix.search(pool_normalize(hc, mc, pool, normalize), 5)
            torch.cuda.synchronize()
            assert torch.equal(Ip, Ir) and torch.equal(Dp, Dr), (metric, pool)
            pooled = pool_normalize(hc, mc, pool, normalize).cpu().numpy()
            _check(Dp.cpu().numpy(), Ip.cpu().numpy(), *orc.np_search_f64(xb, pooled, 5, metric), metric)


# ---- shard merge -----------------------------------------------------------------------------------------
def _parts(rng, G, nq, k, metric):
    """G sorted per-shard lists [G, nq, k] with distances from a small set (exact ties across parts), labels unique, each
    list ordered by (distance, label) as a shard search returns it, every third part short (padded with -1)."""
    keys = rng.integers(0, 40, (G, nq, k)).astype(np.float32) / np.float32(8)
    if G > 2:
        keys[1] = keys[0]                                     # whole-list ties across parts: the lower label first
    ids = rng.permutation(G * nq * k * 2)[: G * nq * k].reshape(G, nq, k).astype(np.int64)
    order = np.lexsort((ids, keys), axis=2)
    keys = np.take_along_axis(keys, order, 2)
    ids = np.take_along_axis(ids, order, 2)
    for g in range(0, G, 3):
        short = int(rng.integers(0, k))
        keys[g, :, short:] = np.inf
        ids[g, :, short:] = -1
    D = keys if metric == 1 else -keys
    D = np.where(ids < 0, FLT_MAX if metric == 1 else -FLT_MAX, D).astype(np.float32)
    return D, ids


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("G", (1, 31, 32, 33, 200))
def test_merge_topk_parts_and_k(m, G, metric):
    """merge_topk and the packed-message form the sharded search uses ([D | pad | I] per part, one stride), against the
    numpy restatement, bit for bit.  The kernel merges up to 32 parts (one lane per part); more is refused, not merged
    wrongly."""
    import torch

    from rag_faiss_embedding_b200 import _capi as C
    from tests.helpers import np_merge

    rng = np.random.default_rng(G * 10 + metric)
    nq = 5
    for k in (1, 10, 257, 1024):
        D, I = _parts(rng, G, nq, k, metric)
        Dt, It = torch.from_numpy(D).cuda(), torch.from_numpy(I).cuda()
        off_i = (nq * k * 4 + 15) // 16 * 16
        part = (off_i + nq * k * 8 + 15) // 16 * 16
        recv = torch.zeros(G * part, dtype=torch.uint8, device="cuda")
        for g in range(G):
            recv[g * part: g * part + nq * k * 4].view(torch.float32).copy_(Dt[g].reshape(-1))
            recv[g * part + off_i: g * part + off_i + nq * k * 8].view(torch.int64).copy_(It[g].reshape(-1))
        Ds = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        Is = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        stream = ctypes.c_void_p(int(torch.cuda.current_stream().cuda_stream) or 1)
        rc = C.load().b2f_merge_topk_strided(metric, nq, k, G, recv.data_ptr(), recv.data_ptr() + off_i, part,
                                             Ds.data_ptr(), Is.data_ptr(), 0, stream)
        if G > 32:
            assert rc == C.EINVAL and "nparts" in C.last_error()
            with pytest.raises(RuntimeError):
                m.merge_topk(metric, Dt, It)
            continue
        assert rc == C.OK, C.last_error()
        Dm, Im = m.merge_topk(metric, Dt, It)
        torch.cuda.synchronize()
        D_ref, I_ref = np_merge(metric, D, I)
        for got_D, got_I in ((Dm, Im), (Ds, Is)):
            assert np.array_equal(got_I.cpu().numpy(), I_ref), (G, k)
            assert np.array_equal(got_D.cpu().numpy().view(np.uint32), D_ref.view(np.uint32)), (G, k)
