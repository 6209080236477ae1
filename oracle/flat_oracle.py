"""numpy twin of oracle/flat_oracle.c plus its ctypes loader.  TEST INFRASTRUCTURE ONLY.

Restates what the reference delegates to faiss-cpu IndexFlat (faiss_store.py:29,46,64,91,106;
rag_datastore_manager.py:138,173,186,205,218).  faiss itself is absent here: "parity unpinned" for
search results; the on-disk layout is pinned by the reference's data/faiss_index.bin.

  np_search_f64   float64 brute force, the arbiter of "which ids are the true top-k"
  np_search_blas  faiss's nq>=20 path on real BLAS (numpy matmul): 4096 x 1024 blocks, expanded form,
                  clamp at 0 -- used as the all-cores CPU baseline in bench.py
  c_search        the C restatement (seq path for nq<20, blocked sgemm path otherwise, heap/reservoir)
"""
from __future__ import annotations

import ctypes
import os
import struct
import subprocess

import numpy as np

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
_FLT_MAX = np.finfo(np.float32).max

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "liborc.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile flat_oracle.c (gcc + OpenMP) into oracle/_build/liborc.so."""
    src = os.path.join(_HERE, "flat_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    return _LIB_PATH


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = ctypes.CDLL(_LIB_PATH)
        fp = ctypes.POINTER(ctypes.c_float)
        ip = ctypes.POINTER(ctypes.c_int64)
        L.orc_search.argtypes = [fp, ctypes.c_int64, ctypes.c_int, ctypes.c_int, fp, ctypes.c_int64,
                                 ctypes.c_int64, fp, ip, ctypes.c_int, ctypes.c_int]
        L.orc_search.restype = ctypes.c_int
        L.orc_synth_rows.argtypes = [ctypes.c_uint64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int,
                                     ctypes.c_int, fp]
        L.orc_synth_rows.restype = None
        L.orc_write_index.argtypes = [ctypes.c_char_p, fp, ctypes.c_int64, ctypes.c_int, ctypes.c_int]
        L.orc_write_index.restype = ctypes.c_int
        L.orc_read_index_header.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int),
                                            ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int)]
        L.orc_read_index_header.restype = ctypes.c_int
        L.orc_read_index_rows.argtypes = [ctypes.c_char_p, fp, ctypes.c_int64]
        L.orc_read_index_rows.restype = ctypes.c_int
        L.orc_max_threads.restype = ctypes.c_int
        _lib = L
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _fp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def c_max_threads() -> int:
    return int(_load().orc_max_threads())


def c_search(xb, xq, k, metric=METRIC_L2, algo=0, nthreads=0):
    """IndexFlat.search restated in C.  algo 0 = faiss's choice, 1 = seq, 2 = blas."""
    xb, xq = _f32(xb), _f32(xq)
    nb, d = xb.shape if xb.ndim == 2 else (0, xq.shape[1])
    nq = xq.shape[0]
    assert xq.shape[1] == d
    D = np.empty((nq, k), np.float32)
    I = np.empty((nq, k), np.int64)
    rc = _load().orc_search(_fp(xb), nb, d, metric, _fp(xq), nq, k, _fp(D),
                            I.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), algo, nthreads)
    if rc != 0:
        raise AssertionError("orc_search: bad arguments (k must be > 0)")
    return D, I


def c_synth_rows(seed, row0, nrows, d, normalize=False):
    out = np.empty((nrows, d), np.float32)
    _load().orc_synth_rows(seed, row0, nrows, d, int(bool(normalize)), _fp(out))
    return out


def c_write_index(path, xb, metric=METRIC_L2):
    xb = _f32(xb)
    rc = _load().orc_write_index(os.fsencode(path), _fp(xb), xb.shape[0], xb.shape[1], metric)
    if rc != 0:
        raise RuntimeError(f"orc_write_index({path!r}) failed: {rc}")


def c_read_index(path):
    d, nt, mt = ctypes.c_int(), ctypes.c_int64(), ctypes.c_int()
    rc = _load().orc_read_index_header(os.fsencode(path), ctypes.byref(d), ctypes.byref(nt), ctypes.byref(mt))
    if rc != 0:
        raise RuntimeError(f"orc_read_index_header({path!r}) failed: {rc}")
    x = np.empty((nt.value, d.value), np.float32)
    rc = _load().orc_read_index_rows(os.fsencode(path), _fp(x), x.size)
    if rc != 0:
        raise RuntimeError(f"orc_read_index_rows({path!r}) failed: {rc}")
    return x, mt.value


# ------------------------------------------------------------------------------------------------
# numpy twins
# ------------------------------------------------------------------------------------------------
def _finish(keys, ids, k, metric):
    """keys: smaller is better, [nq, m]; ids [nq, m] -> faiss-shaped (D, I), ties by ascending id."""
    nq, m = keys.shape
    D = np.full((nq, k), _FLT_MAX if metric == METRIC_L2 else -_FLT_MAX, np.float32)
    I = np.full((nq, k), -1, np.int64)
    kk = min(k, m)
    if kk:
        order = np.lexsort((ids, keys), axis=1)[:, :kk]
        ks = np.take_along_axis(keys, order, 1)
        D[:, :kk] = (ks if metric == METRIC_L2 else -ks).astype(np.float32)
        I[:, :kk] = np.take_along_axis(ids, order, 1)
        bad = ~np.isfinite(ks) | np.isnan(ks)
        if bad.any():  # NaN / inf never enter faiss's heap
            D[:, :kk][bad] = _FLT_MAX if metric == METRIC_L2 else -_FLT_MAX
            I[:, :kk][bad] = -1
    return D, I


def np_search_f64(xb, xq, k, metric=METRIC_L2, block=2048):
    """float64 exact-difference brute force; distances returned as float64-accurate fp32."""
    xb = np.asarray(xb, np.float64)
    xq = np.asarray(xq, np.float64)
    nb = xb.shape[0]
    nq = xq.shape[0]
    best_k = np.empty((nq, 0), np.float64)
    best_i = np.empty((nq, 0), np.int64)
    for j0 in range(0, nb, block):
        xs = xb[j0:j0 + block]
        if metric == METRIC_L2:
            # exact difference form in float64 (no cancellation issue at this precision)
            keys = (xq * xq).sum(1)[:, None] + (xs * xs).sum(1)[None, :] - 2.0 * (xq @ xs.T)
            # recompute small values exactly to avoid cancellation around 0
            small = keys < 1e-6 * ((xq * xq).sum(1)[:, None] + 1e-300)
            if small.any():
                qi, xi = np.nonzero(small)
                keys[qi, xi] = ((xq[qi] - xs[xi]) ** 2).sum(1)
        else:
            keys = -(xq @ xs.T)
        ids = np.broadcast_to(np.arange(j0, j0 + xs.shape[0], dtype=np.int64), keys.shape)
        best_k = np.concatenate([best_k, keys], 1)
        best_i = np.concatenate([best_i, ids], 1)
        if best_k.shape[1] > 4 * k + block:
            order = np.lexsort((best_i, best_k), axis=1)[:, :k]
            best_k = np.take_along_axis(best_k, order, 1)
            best_i = np.take_along_axis(best_i, order, 1)
    return _finish(best_k, best_i, k, metric)


def np_search_blas(xb, xq, k, metric=METRIC_L2, bs_q=4096, bs_b=1024 * 16):
    """faiss exhaustive_*_blas restated on numpy's BLAS (fp32 sgemm, expanded form, clamp at 0).

    bs_b defaults to 16 x faiss's 1024 so the Python loop overhead does not dominate the timing;
    the arithmetic per (query,row) is unchanged.
    """
    xb, xq = _f32(xb), _f32(xq)
    nb, nq = xb.shape[0], xq.shape[0]
    D = np.empty((nq, k), np.float32)
    I = np.empty((nq, k), np.int64)
    xn = np.einsum("ij,ij->i", xb, xb) if metric == METRIC_L2 else None
    for i0 in range(0, nq, bs_q):
        q = xq[i0:i0 + bs_q]
        qn = np.einsum("ij,ij->i", q, q) if metric == METRIC_L2 else None
        bk = np.empty((q.shape[0], 0), np.float32)
        bi = np.empty((q.shape[0], 0), np.int64)
        for j0 in range(0, nb, bs_b):
            xs = xb[j0:j0 + bs_b]
            ip = q @ xs.T
            if metric == METRIC_L2:
                keys = qn[:, None] + xn[None, j0:j0 + bs_b] - 2.0 * ip
                np.maximum(keys, 0, out=keys)
            else:
                keys = -ip
            kk = min(k, keys.shape[1])
            part = np.argpartition(keys, kk - 1, axis=1)[:, :kk] if kk < keys.shape[1] else \
                np.broadcast_to(np.arange(keys.shape[1]), keys.shape)
            bk = np.concatenate([bk, np.take_along_axis(keys, part, 1)], 1)
            bi = np.concatenate([bi, part.astype(np.int64) + j0], 1)
            if bk.shape[1] > 8 * k:
                order = np.lexsort((bi, bk), axis=1)[:, :k]
                bk = np.take_along_axis(bk, order, 1)
                bi = np.take_along_axis(bi, order, 1)
        D[i0:i0 + bs_q], I[i0:i0 + bs_q] = _finish(bk, bi, k, metric)
    return D, I


def torch_search_blas(xb, xq, k, metric=METRIC_L2, bs_q=4096, bs_b=16384, nthreads=0):
    """Same restatement as np_search_blas with the sgemm done by torch's CPU BLAS (MKL, the library
    faiss-cpu wheels link) and selection by torch.topk; the fastest CPU form available here, used as
    the all-cores baseline in bench.py.  xb / xq: numpy fp32."""
    import torch

    if nthreads > 0:
        torch.set_num_threads(nthreads)
    xb_t = torch.from_numpy(_f32(xb))
    xq_t = torch.from_numpy(_f32(xq))
    nb, nq = xb_t.shape[0], xq_t.shape[0]
    l2 = metric == METRIC_L2
    xn = (xb_t * xb_t).sum(1) if l2 else None
    D = np.empty((nq, k), np.float32)
    I = np.empty((nq, k), np.int64)
    for i0 in range(0, nq, bs_q):
        q = xq_t[i0:i0 + bs_q]
        qn = (q * q).sum(1) if l2 else None
        bk = torch.empty((q.shape[0], 0), dtype=torch.float32)
        bi = torch.empty((q.shape[0], 0), dtype=torch.int64)
        for j0 in range(0, nb, bs_b):
            xs = xb_t[j0:j0 + bs_b]
            ip = q @ xs.T
            if l2:
                keys = ip.mul_(-2.0).add_(qn[:, None]).add_(xn[None, j0:j0 + bs_b]).clamp_(min=0)
            else:
                keys = ip.neg_()
            kk = min(k, keys.shape[1])
            v, idx = torch.topk(keys, kk, dim=1, largest=False)
            bk = torch.cat([bk, v], 1)
            bi = torch.cat([bi, idx + j0], 1)
            if bk.shape[1] > 16 * k:
                v, o = torch.topk(bk, min(k, bk.shape[1]), dim=1, largest=False)
                bk, bi = v, torch.gather(bi, 1, o)
        D[i0:i0 + bs_q], I[i0:i0 + bs_q] = _finish(bk.numpy(), bi.numpy(), k, metric)
    return D, I


_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)


def _mix64(z):
    z = z ^ (z >> np.uint64(30))
    z = z * _M1
    z = z ^ (z >> np.uint64(27))
    z = z * _M2
    return z ^ (z >> np.uint64(31))


def _synth_int(seed, idx):
    with np.errstate(over="ignore"):
        a = _mix64(np.uint64(seed) + np.uint64(0x9E3779B97F4A7C15) * (np.uint64(2) * idx + np.uint64(1)))
        b = _mix64(a ^ np.uint64(0xD1B54A32D192ED03))
        c = _mix64(b + idx)
        s = np.zeros(idx.shape, np.int64)
        for w in (a, b, c):
            for i in range(4):
                s += ((w >> np.uint64(16 * i)) & np.uint64(0xFFFF)).astype(np.int64)
    return s - 393210


def np_synth_rows(seed, row0, nrows, d, normalize=False):
    """Same bits as orc_synth_rows / the CUDA generator."""
    idx = (np.arange(row0, row0 + nrows, dtype=np.uint64)[:, None] * np.uint64(d)
           + np.arange(d, dtype=np.uint64)[None, :])
    v = _synth_int(seed, idx)
    if not normalize:
        return (v.astype(np.float32) * np.float32(1.0 / 65536.0)).astype(np.float32)
    ss = (v * v).sum(1)
    nrm = np.sqrt(ss.astype(np.float64))
    out = np.where(ss[:, None] > 0, v.astype(np.float64) / np.where(nrm == 0, 1, nrm)[:, None], 0.0)
    return out.astype(np.float32)


CENTRE_ROWS = 65536   # the centre is the mean of the first min(n, CENTRE_ROWS) rows of the first add


def np_centre(first_rows):
    """Same bits as the device centre (ingest.cu mean_rows_kernel + mean_finish_kernel) of an index whose first add
    call receives `first_rows`.  m = min(n, 65536) rows in 64-row blocks (the last may be partial); each block sums its
    column in float32, row after row from 0; a block whose sum is not finite is skipped but still counts in m.  The
    finite block sums go into a 64-bit fixed-point accumulator at 2^e(c), e = 62 - exponent(max |block sum| * nblocks),
    each rounded half to even (__double2ll_rn); mu = fl32(acc * 2^-e / m) in float64."""
    x = _f32(first_rows)
    m = min(x.shape[0], CENTRE_ROWS)
    d = x.shape[1]
    if m == 0:
        return np.zeros(d, np.float32)
    x = x[:m]
    nblocks = (m + 63) // 64
    pad = np.zeros((nblocks * 64, d), np.float32)   # a partial last block is padded with zeros: a + 0 == a
    pad[:m] = x
    sums = np.empty((nblocks, d), np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        for b0 in range(0, nblocks, 64):
            # np.cumsum adds sequentially (np.sum would add pairwise); the kernel's leading 0 + x0 only turns -0 into +0
            sums[b0:b0 + 64] = np.cumsum(pad[64 * b0:64 * (b0 + 64)].reshape(-1, 64, d), 1, np.float32)[:, -1]
    fin = np.isfinite(sums)
    a = np.where(fin, sums, np.float32(0)).astype(np.float64)
    colmax = np.abs(a).max(0)
    _, ex = np.frexp(colmax * nblocks)
    e = np.where(colmax > 0, 62 - ex, 0).astype(np.int64)
    terms = np.rint(np.ldexp(a, e[None, :])).astype(np.int64)   # rint: half to even; |term| <= 2^62 / nblocks
    acc = terms.sum(0)
    return (np.ldexp(acc.astype(np.float64), -e) / np.float64(m)).astype(np.float32)


def np_bf16_rne(x):
    """float32 -> bfloat16 (round to nearest even, subnormals kept, overflow to inf) -> float32.  NaN stays NaN."""
    u = _f32(x).view(np.uint32).astype(np.uint64)
    r = ((u + np.uint64(0x7FFF) + ((u >> np.uint64(16)) & np.uint64(1))) & np.uint64(0xFFFF0000)).astype(np.uint32)
    out = r.view(np.float32)
    return np.where(np.isnan(x), np.float32(np.nan), out).astype(np.float32)


def np_bf16_rows(x, mu):
    """The authoritative rows of a bf16-storage index: r = fl32(mu + bf16_rne(fl32(x - mu)))."""
    x, mu = _f32(x), _f32(mu)
    with np.errstate(over="ignore", invalid="ignore"):
        return (mu[None, :] + np_bf16_rne(x - mu[None, :])).astype(np.float32)


def np_write_index(path, xb, metric=METRIC_L2):
    xb = _f32(xb)
    n, d = xb.shape
    with open(path, "wb") as f:
        f.write(b"IxF2" if metric == METRIC_L2 else b"IxFI")
        f.write(struct.pack("<iqqqBiQ", d, n, 1 << 20, 1 << 20, 1, metric, n * d))
        f.write(xb.astype("<f4").tobytes())


def np_read_index(path):
    with open(path, "rb") as f:
        b = f.read()
    if b[:4] not in (b"IxF2", b"IxFI", b"IxFl"):
        raise RuntimeError(f"not an IndexFlat file: fourcc {b[:4]!r}")
    d, n, _, _, trained, metric = struct.unpack("<iqqqBi", b[4:37])
    off = 37 + (4 if metric > 1 else 0)
    (sz,) = struct.unpack("<Q", b[off:off + 8])
    if sz != n * d:
        raise RuntimeError("corrupt IndexFlat file: size field != ntotal*d")
    x = np.frombuffer(b, "<f4", sz, off + 8).reshape(n, d).copy()
    return x, metric


def recall_and_errors(D, I, D_ref, I_ref, metric=METRIC_L2, rel_tol=1e-5, abs_floor=1e-4):
    """Compare (D, I) against the oracle's (D_ref, I_ref).

    ids must be identical except among exact-distance ties (BASELINE.json north_star): a position
    passes if the ids match, or if the distances at that position agree within tolerance (a tie or
    near-tie swap).  Returns dict(recall, id_mismatch, max_rel_err).
    """
    D = np.asarray(D, np.float64)
    D_ref = np.asarray(D_ref, np.float64)
    nq, k = I.shape
    hits = 0
    total = 0
    for q in range(nq):
        ref = set(int(i) for i in I_ref[q] if i >= 0)
        got = set(int(i) for i in I[q] if i >= 0)
        total += len(ref)
        hits += len(ref & got)
    valid = (I_ref >= 0)
    denom = np.maximum(np.abs(D_ref), abs_floor / rel_tol)
    rel = np.where(valid, np.abs(D - D_ref) / denom, 0.0)
    mism = valid & (I != I_ref) & (rel > rel_tol)
    pad_ok = np.array_equal(I[~valid], I_ref[~valid])
    return {
        "recall": hits / max(total, 1),
        "id_mismatch": int(mism.sum()),
        "max_rel_err": float(rel.max()) if rel.size else 0.0,
        "padding_ok": bool(pad_ok),
    }
