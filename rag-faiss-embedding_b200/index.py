"""IndexFlat / IndexFlatL2 / IndexFlatIP, read_index, write_index -- the slice of the `faiss`
Python API that the reference uses (faiss_store.py:29,46,64,91,106,126;
rag_datastore_manager.py:138,173,186,205,218), backed by the sm_100a C-ABI library.

numpy in -> numpy out (host buffers, synchronous, faiss semantics).
torch CUDA tensors in -> torch CUDA tensors out (device pointers handed over with data_ptr(); the
work is enqueued on the current torch stream; PyTorch is only the tensor handoff).
Errors follow faiss's Python wrapper: AssertionError for a dimension mismatch or k <= 0,
RuntimeError (B200FlatError) for I/O / format / CUDA failures.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np

from . import _capi as C

METRIC_INNER_PRODUCT = C.METRIC_INNER_PRODUCT
METRIC_L2 = C.METRIC_L2


def _assert(cond, msg: str):
    """faiss's Python wrapper signals bad shapes / k with AssertionError; keep that under python -O too."""
    if not cond:
        raise AssertionError(msg)


def _is_torch(x) -> bool:
    return type(x).__module__.split(".")[0] == "torch" and hasattr(x, "data_ptr")


def _default_device() -> int:
    env = os.environ.get("B200FLAT_DEVICE")
    if env is not None:
        return int(env)
    return int(os.environ.get("LOCAL_RANK", "0")) if os.environ.get("B200FLAT_USE_LOCAL_RANK") else 0


def _default_storage() -> int:
    return C.STORE_BF16 if os.environ.get("B200FLAT_STORAGE", "fp32").lower() in ("bf16", "bfloat16") else C.STORE_F32


def _torch_stream(t) -> int:
    """cudaStream_t of torch's current stream.  torch's default stream is the legacy default stream, whose
    handle is 0 -- which the C-ABI reads as "use the index's own stream" -- so it is passed as
    cudaStreamLegacy (0x1) to keep the work ordered with the caller's other torch ops."""
    import torch

    h = int(torch.cuda.current_stream(t.device).cuda_stream)
    return h if h != 0 else 1


def _id_array(x) -> np.ndarray:
    """A 1-D array of ids as faiss's wrapper takes it: any integer (or numeric) array, coerced to int64."""
    if _is_torch(x):
        x = x.detach().cpu().numpy()
    x = np.asarray(x)
    _assert(x.ndim == 1, f"expected a 1-D array of ids, got shape {x.shape}")
    return np.ascontiguousarray(x, dtype=np.int64)


class IDSelectorRange:
    """faiss.IDSelectorRange(imin, imax): the ids imin <= i < imax."""

    def __init__(self, imin: int, imax: int):
        self.imin = int(imin)
        self.imax = int(imax)


class IDSelectorBatch:
    """faiss.IDSelectorBatch(ids) or IDSelectorBatch(n, ids): the first n of ids (any order; duplicates allowed)."""

    def __init__(self, *args):
        if len(args) == 1:
            self.ids = _id_array(args[0])
        elif len(args) == 2:
            n, ids = int(args[0]), _id_array(args[1])
            _assert(0 <= n <= ids.shape[0], f"IDSelectorBatch: n={n} but {ids.shape[0]} ids given")
            self.ids = ids[:n]
        else:
            raise TypeError("IDSelectorBatch(ids) or IDSelectorBatch(n, ids)")


class IndexFlat:
    """Exact (brute-force) index with faiss.IndexFlat's surface."""

    def __init__(self, d: int, metric: int = METRIC_L2, *, storage: Optional[int] = None,
                 device: Optional[int] = None, _handle=None):
        self._lib = C.load()
        self.is_trained = True
        self.verbose = False
        self._params = C.SearchParams()
        if _handle is not None:
            self._h = _handle
            return
        h = ctypes.c_void_p()
        C.check(self._lib.b2f_index_create(int(d), int(metric),
                                           _default_storage() if storage is None else int(storage),
                                           _default_device() if device is None else int(device),
                                           ctypes.byref(h)))
        self._h = h

    # ---- attributes ------------------------------------------------------------------------
    @property
    def d(self) -> int:
        return int(self._lib.b2f_index_d(self._h))

    @property
    def ntotal(self) -> int:
        return int(self._lib.b2f_index_ntotal(self._h))

    @property
    def metric_type(self) -> int:
        return int(self._lib.b2f_index_metric(self._h))

    @property
    def device(self) -> int:
        return int(self._lib.b2f_index_device(self._h))

    @property
    def storage(self) -> int:
        return int(self._lib.b2f_index_storage(self._h))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and getattr(self, "_lib", None) is not None:
            try:
                self._lib.b2f_index_destroy(h)
            except Exception:  # interpreter shutdown
                pass
            self._h = None

    # ---- tuning knobs (no reference counterpart; defaults reproduce IndexFlat results) ---------
    def set_search_params(self, *, algo: Optional[int] = None, scan_max_nq: Optional[int] = None,
                          slack: Optional[int] = None, certify: Optional[bool] = None,
                          id_offset: Optional[int] = None, profile: Optional[bool] = None):
        p = self._params
        if algo is not None:
            p.algo = int(algo)
        if scan_max_nq is not None:
            p.scan_max_nq = int(scan_max_nq)
        if slack is not None:
            p.slack = int(slack)
        if certify is not None:
            p.certify = 1 if certify else -1
        if id_offset is not None:
            p.id_offset = int(id_offset)
        if profile is not None:
            p.profile = 1 if profile else 0
        return self

    def _check_tensor(self, t, what: str):
        # a CUDA pointer of another GPU would be dereferenced on the index's device (illegal address, sticky error)
        _assert(t.is_cuda and t.device.index == self.device,
                f"{what} must be a CUDA tensor on the index's GPU (cuda:{self.device}), got {t.device}")

    def stats(self) -> dict:
        s = C.Stats()
        C.check(self._lib.b2f_index_stats(self._h, ctypes.byref(s)))
        return s.as_dict()

    def reserve(self, nrows: int):
        C.check(self._lib.b2f_index_reserve(self._h, int(nrows)))

    # ---- faiss surface ----------------------------------------------------------------------
    def _coerce_host(self, x) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32)
        _assert(x.ndim == 2, "expected a 2-D array [n, d]")
        n, d = x.shape
        _assert(d == self.d, f"dimension mismatch: got {d}, index has d={self.d}")
        return x

    def add(self, x):
        """index.add(x): faiss_store.py:46, rag_datastore_manager.py:173."""
        if _is_torch(x) and x.is_cuda:
            import torch

            _assert(x.dim() == 2 and x.shape[1] == self.d, f"dimension mismatch: got {tuple(x.shape)}, d={self.d}")
            self._check_tensor(x, "x")
            x = x.to(torch.float32).contiguous()
            C.check(self._lib.b2f_index_add(self._h, x.shape[0], x.data_ptr(), C.MEM_DEVICE, _torch_stream(x)))
            return
        if _is_torch(x):
            x = x.detach().cpu().numpy()
        x = self._coerce_host(x)
        C.check(self._lib.b2f_index_add(self._h, x.shape[0], x.ctypes.data, C.MEM_HOST, None))

    def add_synthetic(self, seed: int, row0: int, nrows: int, normalize: bool = False):
        """Append rows of the counter-based synthetic matrix, generated on the device."""
        C.check(self._lib.b2f_index_add_synth(self._h, int(seed), int(row0), int(nrows), int(bool(normalize))))

    def add_pooled(self, hidden, attention_mask=None, pool: str = "cls", normalize: bool = False):
        """Fused encoder epilogue (replaces vectorization.py:44-47): hidden [B,T,d] CUDA fp32 tensor."""
        import torch

        _assert(_is_torch(hidden) and hidden.is_cuda and hidden.dim() == 3 and hidden.shape[2] == self.d,
                "add_pooled expects a CUDA tensor [B, T, d]")
        self._check_tensor(hidden, "hidden")
        hidden = hidden.to(torch.float32).contiguous()
        mptr = None
        if attention_mask is not None:
            attention_mask = attention_mask.to(device=hidden.device, dtype=torch.int64).contiguous()
            mptr = attention_mask.data_ptr()
        C.check(self._lib.b2f_index_add_pooled(self._h, hidden.data_ptr(), mptr, hidden.shape[0], hidden.shape[1],
                                               C.POOL_MEAN if pool == "mean" else C.POOL_CLS, int(bool(normalize)),
                                               _torch_stream(hidden)))

    def search_pooled(self, hidden, attention_mask, k: int, pool: str = "cls", normalize: bool = False):
        """Query side of the encoder hand-off: hidden [B,T,d] CUDA fp32 -> pooled (+ normalised) on the device ->
        search; returns CUDA tensors (D [B,k] float32, I [B,k] int64) on the current torch stream."""
        import torch

        _assert(k > 0, "k must be > 0")
        _assert(_is_torch(hidden) and hidden.is_cuda and hidden.dim() == 3 and hidden.shape[2] == self.d,
                "search_pooled expects a CUDA tensor [B, T, d]")
        self._check_tensor(hidden, "hidden")
        hidden = hidden.to(torch.float32).contiguous()
        mptr = None
        if attention_mask is not None:
            attention_mask = attention_mask.to(device=hidden.device, dtype=torch.int64).contiguous()
            mptr = attention_mask.data_ptr()
        B = hidden.shape[0]
        D = torch.empty((B, k), dtype=torch.float32, device=hidden.device)
        I = torch.empty((B, k), dtype=torch.int64, device=hidden.device)
        C.check(self._lib.b2f_index_search_pooled(self._h, hidden.data_ptr(), mptr, B, hidden.shape[1],
                                                  C.POOL_MEAN if pool == "mean" else C.POOL_CLS, int(bool(normalize)), k,
                                                  D.data_ptr(), I.data_ptr(), _torch_stream(hidden), ctypes.byref(self._params)))
        return D, I

    def search(self, x, k: int, *, params: Optional[C.SearchParams] = None):
        """index.search(x, k) -> (D float32 [n,k], I int64 [n,k]): faiss_store.py:64,
        rag_datastore_manager.py:218."""
        _assert(k > 0, "k must be > 0")
        p = params if params is not None else self._params
        if _is_torch(x) and x.is_cuda:
            import torch

            _assert(x.dim() == 2 and x.shape[1] == self.d, f"dimension mismatch: got {tuple(x.shape)}, d={self.d}")
            self._check_tensor(x, "x")
            x = x.to(torch.float32).contiguous()
            D = torch.empty((x.shape[0], k), dtype=torch.float32, device=x.device)
            I = torch.empty((x.shape[0], k), dtype=torch.int64, device=x.device)
            C.check(self._lib.b2f_index_search(self._h, x.shape[0], x.data_ptr(), k, D.data_ptr(), I.data_ptr(),
                                               C.MEM_DEVICE, _torch_stream(x), ctypes.byref(p)))
            return D, I
        if _is_torch(x):
            x = x.detach().cpu().numpy()
        x = self._coerce_host(x)
        n = x.shape[0]
        D = np.empty((n, k), dtype=np.float32)
        I = np.empty((n, k), dtype=np.int64)
        C.check(self._lib.b2f_index_search(self._h, n, x.ctypes.data, k, D.ctypes.data, I.ctypes.data,
                                           C.MEM_HOST, None, ctypes.byref(p)))
        return D, I

    def search_tensors_into(self, x, k: int, D, I, *, params: Optional[C.SearchParams] = None):
        """Device-buffer search into caller-owned CUDA tensors D [n,k] float32 / I [n,k] int64 (contiguous); lets a
        caller place both results inside one message buffer.  Enqueued on the current torch stream."""
        import torch

        _assert(k > 0, "k must be > 0")
        _assert(x.is_cuda and x.dim() == 2 and x.shape[1] == self.d, f"dimension mismatch: got {tuple(x.shape)}, d={self.d}")
        _assert(D.is_cuda and I.is_cuda and D.dtype == torch.float32 and I.dtype == torch.int64
                and D.is_contiguous() and I.is_contiguous() and tuple(D.shape) == (x.shape[0], k) == tuple(I.shape),
                "D / I must be contiguous CUDA tensors [n, k] of float32 / int64")
        for t, what in ((x, "x"), (D, "D"), (I, "I")):
            self._check_tensor(t, what)
        x = x.to(torch.float32).contiguous()
        p = params if params is not None else self._params
        C.check(self._lib.b2f_index_search(self._h, x.shape[0], x.data_ptr(), k, D.data_ptr(), I.data_ptr(),
                                           C.MEM_DEVICE, _torch_stream(x), ctypes.byref(p)))

    def range_search(self, x, radius: float, *, params: Optional[C.SearchParams] = None):
        """index.range_search(x, radius) -> (lims, D, I), faiss's RangeSearchResult: query i owns
        D[lims[i]:lims[i+1]] / I[lims[i]:lims[i+1]], ids ascending.  L2: squared distance < radius; IP: ip > radius.
        numpy in: lims uint64, D float32, I int64 numpy arrays.  CUDA tensor in: int64 / float32 / int64 CUDA tensors
        on the current torch stream.  The five numbers of b2f_range_result_info go to self.last_range_info."""
        p = params if params is not None else self._params
        dev = _is_torch(x) and x.is_cuda
        if dev:
            import torch

            _assert(x.dim() == 2 and x.shape[1] == self.d, f"dimension mismatch: got {tuple(x.shape)}, d={self.d}")
            self._check_tensor(x, "x")
            x = x.to(torch.float32).contiguous()
            stream = _torch_stream(x)
            qptr, mem = x.data_ptr(), C.MEM_DEVICE
        else:
            if _is_torch(x):
                x = x.detach().cpu().numpy()
            x = self._coerce_host(x)
            stream = None
            qptr, mem = x.ctypes.data, C.MEM_HOST
        n = x.shape[0]
        h = ctypes.c_void_p()
        C.check(self._lib.b2f_index_range_search(self._h, n, qptr, ctypes.c_float(radius), mem, stream, ctypes.byref(p),
                                                 ctypes.byref(h)))
        try:
            lims = np.empty(n + 1, dtype=np.int64)
            C.check(self._lib.b2f_range_result_lims(h, lims.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
            total = int(lims[-1])
            if dev:
                D = torch.empty(total, dtype=torch.float32, device=x.device)
                I = torch.empty(total, dtype=torch.int64, device=x.device)
                C.check(self._lib.b2f_range_result_fetch(h, D.data_ptr(), I.data_ptr(), C.MEM_DEVICE, stream))
                lims_out = torch.from_numpy(lims).to(x.device)
            else:
                D = np.empty(total, dtype=np.float32)
                I = np.empty(total, dtype=np.int64)
                C.check(self._lib.b2f_range_result_fetch(h, D.ctypes.data, I.ctypes.data, C.MEM_HOST, None))
                lims_out = lims.astype(np.uint64)
            info = (ctypes.c_int64 * 5)()
            C.check(self._lib.b2f_range_result_info(h, info))
            self.last_range_info = dict(zip(("hits", "tensor_queries", "scan_queries", "launches", "host_syncs"), list(info)))
        finally:
            self._lib.b2f_range_result_destroy(h)
        return lims_out, D, I

    def search_into(self, x: np.ndarray, k: int, D: np.ndarray, I: np.ndarray):
        """Host-buffer search into caller-owned (ideally pinned) arrays: the raw C-ABI call."""
        C.check(self._lib.b2f_index_search(self._h, x.shape[0], x.ctypes.data, k, D.ctypes.data, I.ctypes.data,
                                           C.MEM_HOST, None, ctypes.byref(self._params)))

    def reset(self):
        C.check(self._lib.b2f_index_reset(self._h))

    def remove_ids(self, x) -> int:
        """index.remove_ids(sel) (faiss IndexFlat::remove_ids): x is an IDSelectorRange, an IDSelectorBatch or a 1-D
        integer array (numpy or torch).  The survivors keep their order and are renumbered from 0, so every label above
        a removed row shifts down; ids outside [0, ntotal) are ignored.  Returns the number of rows removed."""
        n = ctypes.c_int64(0)
        if isinstance(x, IDSelectorRange):
            C.check(self._lib.b2f_index_remove_range(self._h, x.imin, x.imax, ctypes.byref(n)))
        else:
            ids = x.ids if isinstance(x, IDSelectorBatch) else _id_array(x)
            C.check(self._lib.b2f_index_remove_ids(self._h, ids.shape[0], ids.ctypes.data, ctypes.byref(n)))
        return int(n.value)

    def reconstruct(self, key: int) -> np.ndarray:
        out = np.empty((self.d,), np.float32)
        rc = self._lib.b2f_index_reconstruct(self._h, int(key), 1, out.ctypes.data, C.MEM_HOST, None)
        C.check(rc)
        return out

    def reconstruct_n(self, n0: int = 0, ni: int = -1) -> np.ndarray:
        if ni < 0:
            ni = self.ntotal - n0
        out = np.empty((ni, self.d), np.float32)
        C.check(self._lib.b2f_index_reconstruct(self._h, int(n0), int(ni), out.ctypes.data, C.MEM_HOST, None))
        return out


class IndexFlatL2(IndexFlat):
    def __init__(self, d: int, **kw):
        super().__init__(d, METRIC_L2, **kw)


class IndexFlatIP(IndexFlat):
    def __init__(self, d: int, **kw):
        super().__init__(d, METRIC_INNER_PRODUCT, **kw)


def write_index(index: IndexFlat, path) -> None:
    """faiss.write_index: faiss_store.py:91, rag_datastore_manager.py:186."""
    C.check(index._lib.b2f_index_write(index._h, os.fsencode(os.fspath(path))))


def read_index(path, *, storage: Optional[int] = None, device: Optional[int] = None) -> IndexFlat:
    """faiss.read_index: faiss_store.py:106, rag_datastore_manager.py:205."""
    lib = C.load()
    h = ctypes.c_void_p()
    C.check(lib.b2f_index_read(os.fsencode(os.fspath(path)), _default_storage() if storage is None else int(storage),
                               _default_device() if device is None else int(device), ctypes.byref(h)))
    metric = int(lib.b2f_index_metric(h))
    cls = IndexFlatL2 if metric == METRIC_L2 else IndexFlatIP
    obj = cls.__new__(cls)
    IndexFlat.__init__(obj, 0, metric, _handle=h)
    return obj
