"""Row-sharded exact search across the GPUs of one box (SURVEY 8e; BASELINE config 4).

One process per GPU (torch.distributed for the plumbing: ranks, the one-time exchange of IPC handles, barriers).
Every rank holds a contiguous range of the database rows in its own single-GPU IndexFlat; queries are
replicated; each rank searches its shard (global label = shard offset + local row) straight into a message
buffer, and ONE kernel per rank pushes the message into every peer's receive buffer over NVLink peer memory,
flags, waits for the peers' flags and merges the world parts (csrc/exchange.cu; the whole step is one C call,
b2f_exchange_search).  B200FLAT_EXCHANGE=nccl (or a failed IPC set-up) selects the NCCL form of the same step:
one all_gather_into_tensor of the packed messages + the CUDA merge kernel (b2f_merge_topk_strided).
Exact top-k over a partition = merge of per-part exact top-k, so results equal the single-GPU index.

The reference has no multi-process code; its file order / .mapping list stay valid because global
labels are plain row numbers of the concatenated database.
"""
from __future__ import annotations

import ctypes
from typing import Callable, List, Optional, Tuple

import numpy as np

from . import _capi as C
from .index import METRIC_L2, IDSelectorBatch, IDSelectorRange, IndexFlat, _assert, _id_array, _is_torch


def partition_rows(n: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous ranges [start, stop) per rank: rank r gets rows [r*ceil(n/G), min(n, (r+1)*ceil(n/G)))."""
    per = -(-n // world) if n > 0 else 0
    return [(min(n, r * per), min(n, (r + 1) * per)) for r in range(world)]


class SegmentMap:
    """local row -> global label for a shard filled by several add() calls (piecewise offsets)."""

    def __init__(self):
        self.local_starts: List[int] = []
        self.global_starts: List[int] = []
        self.nlocal = 0

    def append(self, global_start: int, count: int):
        if count <= 0:
            return
        if self.local_starts and self.global_starts[-1] + (self.nlocal - self.local_starts[-1]) == global_start:
            self.nlocal += count  # contiguous with the previous segment
            return
        self.local_starts.append(self.nlocal)
        self.global_starts.append(global_start)
        self.nlocal += count

    def single_offset(self) -> Optional[int]:
        if not self.local_starts:
            return 0
        return self.global_starts[0] if len(self.local_starts) == 1 else None

    def remove(self, labels: np.ndarray) -> np.ndarray:
        """Takes the sorted unique global labels `labels` out: returns the local rows of this shard that hold them, and
        renumbers what is left as remove_ids does -- each segment's global start moves down by the labels removed below
        it, its local start by the local rows removed below it; empty segments go, contiguous ones merge."""
        starts = self.local_starts + [self.nlocal]
        local = []
        kept = SegmentMap()
        for i, (ls, gs) in enumerate(zip(self.local_starts, self.global_starts)):
            cnt = starts[i + 1] - ls
            lo, hi = np.searchsorted(labels, [gs, gs + cnt])
            local.append(labels[lo:hi] - gs + ls)
            kept.append(gs - int(lo), cnt - int(hi - lo))
        self.local_starts, self.global_starts, self.nlocal = kept.local_starts, kept.global_starts, kept.nlocal
        return np.concatenate(local) if local else np.zeros(0, np.int64)

    def monotone(self) -> bool:
        """True when local row order is global label order (each segment's labels above the previous segment's): then
        mapping a label-sorted list of local rows gives a label-sorted list of global labels.  add, add_synthetic and
        remove_ids keep it; add_local with a lower global_start than an earlier segment breaks it."""
        ends = self.local_starts[1:] + [self.nlocal]
        return all(self.global_starts[i] + (ends[i] - self.local_starts[i]) <= self.global_starts[i + 1]
                   for i in range(len(self.local_starts) - 1))

    def to_global_numpy(self, local_ids: np.ndarray) -> np.ndarray:
        out = local_ids.astype(np.int64, copy=True)
        if not self.local_starts:
            return out
        ls = np.asarray(self.local_starts, np.int64)
        gs = np.asarray(self.global_starts, np.int64)
        valid = out >= 0
        seg = np.searchsorted(ls, out[valid], side="right") - 1
        out[valid] = out[valid] - ls[seg] + gs[seg]
        return out

    def to_global_torch(self, local_ids):
        import torch

        if not self.local_starts:
            return local_ids
        ls = torch.tensor(self.local_starts, dtype=torch.int64, device=local_ids.device)
        gs = torch.tensor(self.global_starts, dtype=torch.int64, device=local_ids.device)
        seg = (torch.bucketize(local_ids.clamp(min=0), ls, right=True) - 1).clamp(min=0)
        return torch.where(local_ids >= 0, local_ids - ls[seg] + gs[seg], local_ids)


def merge_topk(metric: int, D_parts, I_parts):
    """[G, nq, k] per-shard results (CUDA tensors) -> merged [nq, k] via the CUDA merge kernel."""
    import torch

    G, nq, k = D_parts.shape
    D_parts = D_parts.contiguous()
    I_parts = I_parts.contiguous()
    D = torch.empty((nq, k), dtype=torch.float32, device=D_parts.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=D_parts.device)
    stream = int(torch.cuda.current_stream(D_parts.device).cuda_stream) or 1  # 0x1 = cudaStreamLegacy
    C.check(C.load().b2f_merge_topk(int(metric), nq, k, G, D_parts.data_ptr(), I_parts.data_ptr(), D.data_ptr(),
                                    I.data_ptr(), D_parts.device.index or 0, ctypes.c_void_p(stream)))
    return D, I


# a rank's packed range hits [D | pad | I] of one all-gather stay below this; a query with more hits gets a gather
# of its own
RANGE_PART_BYTES = 256 << 20


def _range_layout(nhits: int) -> Tuple[int, int]:
    """Packed [D fp32 | pad | I int64] of nhits hits: (byte offset of I, part bytes), both multiples of 16."""
    off_i = (nhits * 4 + 15) // 16 * 16
    return off_i, (off_i + nhits * 8 + 15) // 16 * 16


def merge_range_strided(lims_parts, recv, part_bytes: int, off_i: int, D, I):
    """b2f_merge_range_strided over an all-gathered buffer: lims_parts [G, nq + 1] int64 (any base), recv [G * part_bytes]
    uint8 holding G packed parts [D | pad | I at off_i]; writes the label-ordered union into D / I [total] (CUDA
    tensors on one device, enqueued on the current torch stream)."""
    import torch

    G, nq = int(lims_parts.shape[0]), int(lims_parts.shape[1]) - 1
    lims_parts = lims_parts.contiguous()
    stream = int(torch.cuda.current_stream(recv.device).cuda_stream) or 1  # 0x1 = cudaStreamLegacy
    C.check(C.load().b2f_merge_range_strided(nq, G, lims_parts.data_ptr(), recv.data_ptr(), recv.data_ptr() + off_i,
                                             part_bytes, D.data_ptr(), I.data_ptr(), recv.device.index or 0,
                                             ctypes.c_void_p(stream)))


def merge_range(parts):
    """parts: G per-shard range results (lims [nq + 1], D [.], I [.]) as CUDA tensors on one device, labels disjoint
    across parts -> one (lims, D, I) with each query's hits in ascending label order, via the CUDA merge kernel."""
    import torch

    dev = parts[0][1].device
    lims_parts = torch.stack([p[0].to(device=dev, dtype=torch.int64) for p in parts])
    lims = lims_parts.sum(0) - lims_parts[:, :1].sum()
    nhits = [int(p[1].numel()) for p in parts]
    total = sum(nhits)
    D = torch.empty(total, dtype=torch.float32, device=dev)
    I = torch.empty(total, dtype=torch.int64, device=dev)
    if total == 0:
        return lims, D, I
    off_i, part = _range_layout(max(nhits))
    recv = torch.zeros(len(parts) * part, dtype=torch.uint8, device=dev)
    for g, (_, Dp, Ip) in enumerate(parts):
        recv[g * part: g * part + 4 * nhits[g]].view(torch.float32).copy_(Dp)
        recv[g * part + off_i: g * part + off_i + 8 * nhits[g]].view(torch.int64).copy_(Ip)
    merge_range_strided(lims_parts, recv, part, off_i, D, I)
    return lims, D, I


class ShardedIndexFlat:
    """IndexFlat surface over a torch.distributed process group, one shard per rank.

    `local_index` / `merge_fn` / `range_merge_fn` exist so the host logic (partitioning, label mapping, the
    collectives) can be exercised on CPU with the gloo backend in tests; the defaults are the CUDA index and the
    CUDA merge kernels.  range_merge_fn has merge_range_strided's signature.
    """

    def __init__(self, d: int, metric: int = METRIC_L2, *, storage: Optional[int] = None,
                 device: Optional[int] = None, group=None, local_index=None,
                 merge_fn: Optional[Callable] = None, range_merge_fn: Optional[Callable] = None):
        import torch.distributed as dist

        self._dist = dist
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.d = d
        self.metric_type = metric
        self.local = local_index if local_index is not None else IndexFlat(d, metric, storage=storage, device=device)
        self._merge = merge_fn if merge_fn is not None else merge_topk
        self._range_merge = range_merge_fn if range_merge_fn is not None else merge_range_strided
        self.segments = SegmentMap()
        self.ntotal = 0
        self.is_trained = True

    def __del__(self):
        ex = getattr(self, "_ex", None)
        if ex is not None:
            try:
                C.load().b2f_exchange_destroy(ex)
            except Exception:  # interpreter shutdown
                pass
            self._ex = None

    # -- ingest -----------------------------------------------------------------------------------
    def add(self, x):
        """x: the same [n, d] array on every rank; each rank keeps its contiguous slice."""
        n = int(x.shape[0])
        start, stop = partition_rows(n, self.world)[self.rank]
        if stop > start:
            self.local.add(x[start:stop])
        self.segments.append(self.ntotal + start, stop - start)
        self.ntotal += n

    def add_local(self, x_local, global_start: int):
        """This rank's rows only (already partitioned by the caller); labels start at global_start."""
        self.local.add(x_local)
        self.segments.append(int(global_start), int(x_local.shape[0]))

    def add_synthetic(self, seed: int, nrows: int, normalize: bool = False):
        """Every rank generates its slice of the synthetic matrix on its own device."""
        start, stop = partition_rows(nrows, self.world)[self.rank]
        if stop > start:
            self.local.add_synthetic(seed, self.ntotal + start, stop - start, normalize)
        self.segments.append(self.ntotal + start, stop - start)
        self.ntotal += nrows

    def set_total(self, ntotal: int):
        self.ntotal = int(ntotal)

    # -- search -----------------------------------------------------------------------------------
    def search_local(self, x, k: int):
        off = self.segments.single_offset()
        if hasattr(self.local, "set_search_params"):
            # always set: an offset left behind by an earlier single-segment search must not leak into the
            # multi-segment branch, whose labels are remapped below
            self.local.set_search_params(id_offset=off if off is not None else 0)
        if off is not None and hasattr(self.local, "set_search_params"):
            return self.local.search(x, k)
        D, I = self.local.search(x, k)
        if isinstance(I, np.ndarray):
            return D, self.segments.to_global_numpy(I)
        return D, self.segments.to_global_torch(I)

    def _peer_exchange(self, need_bytes: int):
        """The NVLink peer-memory exchange (csrc/exchange.cu), created on first use and re-created when a search needs
        bigger slots.  Collective: every rank takes the same decisions (same need_bytes on every rank).  Returns None
        when B200FLAT_EXCHANGE=nccl or the IPC set-up fails on any rank (then NCCL carries the exchange)."""
        import os

        if os.environ.get("B200FLAT_EXCHANGE", "peer").lower() == "nccl" or getattr(self, "_ex_failed", False):
            return None
        ex = getattr(self, "_ex", None)
        lib = C.load()
        if ex is not None and lib.b2f_exchange_slot_bytes(ex) >= need_bytes:
            return ex
        import torch

        torch.cuda.synchronize()
        if ex is not None:
            self._dist.barrier(group=self.group)   # nobody may still be reading our old buffers
            lib.b2f_exchange_destroy(ex)
            self._ex = None
        slot = max(1 << 20, 2 * need_bytes)
        h = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(64)
        rc = lib.b2f_exchange_create(self.local.device, self.rank, self.world, slot, ctypes.byref(h), handle)
        handles = [None] * self.world
        self._dist.all_gather_object(handles, bytes(handle.raw) if rc == 0 else None, group=self.group)
        ok = rc == 0 and all(b is not None for b in handles)
        if ok:
            ok = lib.b2f_exchange_connect(h, b"".join(handles)) == 0
        oks = [None] * self.world
        self._dist.all_gather_object(oks, bool(ok), group=self.group)
        if not all(oks):
            if rc == 0:
                lib.b2f_exchange_destroy(h)
            self._ex_failed = True
            return None
        self._ex = h
        return h

    def _search_packed(self, x, k: int, out=None):
        """CUDA path of search(): every rank writes its (D, I) into ONE message buffer (12 * nq * k bytes), one kernel
        pushes it to the peers over NVLink and merges the world parts (or: one NCCL all-gather + the merge kernel).
        out = (D [nq, k] float32, I [nq, k] int64) CUDA tensors to write into (else allocated here)."""
        import torch

        nq = int(x.shape[0])
        if out is not None:
            Dm, Im = out
            if not (Dm.is_cuda and Im.is_cuda and Dm.dtype == torch.float32 and Im.dtype == torch.int64
                    and Dm.is_contiguous() and Im.is_contiguous() and tuple(Dm.shape) == (nq, k) == tuple(Im.shape)):
                raise AssertionError("out must be contiguous CUDA tensors (D [nq, k] float32, I [nq, k] int64)")
        else:
            Dm = torch.empty((nq, k), dtype=torch.float32, device=x.device)
            Im = torch.empty((nq, k), dtype=torch.int64, device=x.device)
        if nq == 0:
            return Dm, Im
        if x.device.index != self.local.device:
            raise AssertionError("queries are on another GPU than this rank's shard")
        off_i = (nq * k * 4 + 15) // 16 * 16
        part = (off_i + nq * k * 8 + 15) // 16 * 16
        stream = int(torch.cuda.current_stream(x.device).cuda_stream) or 1  # 0x1 = cudaStreamLegacy
        off = self.segments.single_offset()
        ex = self._peer_exchange(part)
        if ex is not None and off is not None:
            # the whole sharded step behind one C call: local search into the exchange's message buffer, then
            # push over NVLink peer memory + flag + merge in one kernel -- no allocation, no second library call
            x = x.to(torch.float32).contiguous()
            p = C.SearchParams.from_buffer_copy(self.local._params)
            p.id_offset = off
            C.check(C.load().b2f_exchange_search(ex, self.local._h, nq, x.data_ptr(), k, Dm.data_ptr(), Im.data_ptr(),
                                                 ctypes.c_void_p(stream), ctypes.byref(p)))
            return Dm, Im
        send = torch.empty(part, dtype=torch.uint8, device=x.device)
        D = send[: nq * k * 4].view(torch.float32).view(nq, k)
        I = send[off_i: off_i + nq * k * 8].view(torch.int64).view(nq, k)
        self.local.set_search_params(id_offset=off if off is not None else 0)
        if off is not None:
            self.local.search_tensors_into(x, k, D, I)
        else:
            Dl, Il = self.local.search(x, k)
            D.copy_(Dl)
            I.copy_(self.segments.to_global_torch(Il))
        if ex is not None:
            # the one exchange step of the path, fused with the merge: push over NVLink peer memory, flag, merge
            C.check(C.load().b2f_exchange_merge(ex, send.data_ptr(), part, int(self.metric_type), nq, k, off_i,
                                                Dm.data_ptr(), Im.data_ptr(), ctypes.c_void_p(stream)))
            return Dm, Im
        recv = torch.empty(self.world * part, dtype=torch.uint8, device=x.device)
        self._dist.all_gather_into_tensor(recv, send, group=self.group)   # NCCL form of the same exchange
        C.check(C.load().b2f_merge_topk_strided(int(self.metric_type), nq, k, self.world, recv.data_ptr(),
                                                recv.data_ptr() + off_i, part, Dm.data_ptr(), Im.data_ptr(),
                                                x.device.index or 0, ctypes.c_void_p(stream)))
        return Dm, Im

    def search_host(self, x_host, k: int, D_out=None, I_out=None):
        """Host-resident replicated queries (the same pinned [nq, d] float32 tensor on every rank) -> merged (D, I)
        in host tensors.  Every rank uploads only ITS 1/G slice of the batch over PCIe and the slices are
        all-gathered over NVLink (8 ranks pulling the whole batch through the host at once is what limited the
        end-to-end rate at N = 8); then the usual sharded search; results come back with one D2H copy each."""
        import torch

        nq, d = int(x_host.shape[0]), int(x_host.shape[1])
        dev = torch.device("cuda", self.local.device)
        x = torch.empty((nq, d), dtype=torch.float32, device=dev)
        if self.world > 1 and nq % self.world == 0 and nq >= 8 * self.world:
            per = nq // self.world
            mine = x[self.rank * per:(self.rank + 1) * per]
            mine.copy_(x_host[self.rank * per:(self.rank + 1) * per], non_blocking=True)
            self._dist.all_gather_into_tensor(x, mine, group=self.group)
        else:
            x.copy_(x_host, non_blocking=True)
        D, I = self.search(x, k)
        if D_out is None or I_out is None:
            D_out = torch.empty((nq, k), dtype=torch.float32).pin_memory()
            I_out = torch.empty((nq, k), dtype=torch.int64).pin_memory()
        D_out.copy_(D, non_blocking=True)
        I_out.copy_(I, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return D_out, I_out

    def search(self, x, k: int, out=None):
        """Replicated queries -> identical merged (D, I) on every rank.  out: optional caller-owned CUDA result
        tensors (CUDA path only), so that a serving loop allocates nothing per search."""
        if (self.world > 1 and self._merge is merge_topk and hasattr(x, "is_cuda") and x.is_cuda
                and hasattr(self.local, "search_tensors_into")):
            return self._search_packed(x, k, out)
        D, I = self.search_local(x, k)
        if self.world == 1:
            return D, I
        import torch

        was_numpy = isinstance(D, np.ndarray)
        if was_numpy:
            D, I = torch.from_numpy(D), torch.from_numpy(I)
        nq, kk = D.shape
        # concatenated-along-dim-0 form ([G*nq, k]) is accepted by both NCCL and gloo
        Dg = torch.empty((self.world * nq, kk), dtype=D.dtype, device=D.device)
        Ig = torch.empty((self.world * nq, kk), dtype=I.dtype, device=I.device)
        # the one exchange step of the path: 12 * nq * k bytes per rank
        self._dist.all_gather_into_tensor(Dg, D.contiguous(), group=self.group)
        self._dist.all_gather_into_tensor(Ig, I.contiguous(), group=self.group)
        Dm, Im = self._merge(self.metric_type, Dg.view(self.world, nq, kk), Ig.view(self.world, nq, kk))
        if was_numpy and not isinstance(Dm, np.ndarray):
            Dm, Im = Dm.cpu().numpy(), Im.cpu().numpy()
        return Dm, Im

    def _all_gather(self, t):
        """[world, *t.shape] all-gather of t (the same shape on every rank), returned on t's device.  An NCCL group
        gathers device tensors; a gloo group gathers host copies (the CPU tier, or several ranks sharing one GPU)."""
        import torch

        host = not (t.is_cuda and "nccl" in str(self._dist.get_backend(self.group)))
        src = (t.cpu() if host else t).contiguous().view(-1)
        out = torch.empty(self.world * src.numel(), dtype=t.dtype, device=src.device)
        self._dist.all_gather_into_tensor(out, src, group=self.group)
        out = out.view((self.world,) + tuple(t.shape))
        return out.to(t.device) if host else out

    @staticmethod
    def _range_chunks(lims_host: np.ndarray) -> List[Tuple[int, int]]:
        """Query ranges [q0, q1) over which no rank's packed hits ([world, nq + 1] lims) exceed RANGE_PART_BYTES; a
        query with more hits than that on some rank is a range of its own."""
        budget = max((RANGE_PART_BYTES - 32) // 12, 0)   # _range_layout(budget)[1] <= RANGE_PART_BYTES
        nq = lims_host.shape[1] - 1
        chunks, q0 = [], 0
        while q0 < nq:
            q1 = min(int(np.searchsorted(lims, lims[q0] + budget, side="right")) - 1 for lims in lims_host)
            q1 = min(max(q1, q0 + 1), nq)
            chunks.append((q0, q1))
            q0 = q1
        return chunks

    def range_search(self, x, radius: float, *, params: Optional[C.SearchParams] = None):
        """index.range_search(x, radius) over the whole sharded index: replicated queries -> the same faiss
        RangeSearchResult (lims, D, I) on every rank, each query's hits in ascending label order, as IndexFlat returns
        it (numpy in: lims uint64, D float32, I int64 numpy arrays; CUDA tensor in: CUDA tensors).

        Each rank range-searches its shard; one all-gather of every rank's lims settles all sizes; the hits then move
        in all-gathers of at most RANGE_PART_BYTES per rank, each followed by the CUDA merge (b2f_merge_range_strided)
        into its slice of the result.  last_range_info: the local search's five numbers, `chunks` (hit all-gathers) and
        `gathered_bytes` (bytes this rank sent: its lims and its packed hits)."""
        import torch

        # checked on every rank before the first collective, so that a bad call leaves no rank waiting for another
        radius = float(radius)
        if radius != radius:
            raise C.B200FlatError(C.EINVAL, "range_search: radius is NaN")
        shape = tuple(x.shape)
        _assert(len(shape) == 2 and int(shape[1]) == self.d, f"dimension mismatch: got {shape}, index has d={self.d}")
        dev_in = _is_torch(x) and x.is_cuda
        nq = int(shape[0])

        off = self.segments.single_offset()
        if hasattr(self.local, "set_search_params"):
            self.local.set_search_params(id_offset=off if off is not None else 0)
        if params is not None:
            params = C.SearchParams.from_buffer_copy(params)
            params.id_offset = off if off is not None else 0
            lims, D, I = self.local.range_search(x, radius, params=params)
        else:
            lims, D, I = self.local.range_search(x, radius)
        info = dict(getattr(self.local, "last_range_info", {}))
        if isinstance(D, np.ndarray):
            lims, D, I = (torch.from_numpy(np.asarray(lims).astype(np.int64)), torch.from_numpy(D), torch.from_numpy(I))
        if off is None:
            I = self.segments.to_global_torch(I)
            if not self.segments.monotone():
                # a segment added below an earlier one: order each query's hits by label again
                qid = torch.repeat_interleave(torch.arange(nq, device=I.device), lims.diff(), output_size=I.numel())
                order = torch.argsort(I, stable=True)
                order = order[torch.argsort(qid[order], stable=True)]
                D, I = D[order], I[order]

        chunks, sent = 0, 0
        if self.world > 1:
            # the hits stay on the shard's GPU (a host-side stand-in for the local index keeps them on the host)
            work = torch.device("cuda", self.local.device) if isinstance(self.local, IndexFlat) else torch.device("cpu")
            lims, D, I = lims.to(work), D.to(work), I.to(work)
            lims_all = self._all_gather(lims)      # [world, nq + 1]: every rank's local lims (base 0)
            lims_host = lims_all.cpu().numpy()
            sent = 8 * (nq + 1)
            glims = lims_host.sum(0)
            Dm = torch.empty(int(glims[-1]), dtype=torch.float32, device=work)
            Im = torch.empty(int(glims[-1]), dtype=torch.int64, device=work)
            a_own = lims_host[self.rank]
            for q0, q1 in self._range_chunks(lims_host):
                nmax = int((lims_host[:, q1] - lims_host[:, q0]).max())
                if nmax == 0:   # decided from the gathered lims, so every rank skips the same gathers
                    continue
                off_i, part = _range_layout(nmax)
                a, b = int(a_own[q0]), int(a_own[q1])
                send = torch.empty(part, dtype=torch.uint8, device=work)
                send[: 4 * (b - a)].view(torch.float32).copy_(D[a:b])
                send[off_i: off_i + 8 * (b - a)].view(torch.int64).copy_(I[a:b])
                recv = self._all_gather(send).view(-1)
                g0, g1 = int(glims[q0]), int(glims[q1])
                self._range_merge(lims_all[:, q0:q1 + 1], recv, part, off_i, Dm[g0:g1], Im[g0:g1])
                chunks += 1
                sent += part
            lims, D, I = torch.from_numpy(glims), Dm, Im
        self.last_range_info = dict(info, chunks=chunks, gathered_bytes=sent)
        if dev_in:
            return lims.to(x.device), D.to(x.device), I.to(x.device)
        return lims.cpu().numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()

    def remove_ids(self, x) -> int:
        """index.remove_ids(sel) over the whole sharded index: x (IDSelectorRange, IDSelectorBatch or 1-D integer array)
        names global labels, the same on every rank.  Each rank removes the rows it holds and renumbers its segments;
        the labels of the concatenated database shift down as on one index.  No communication.  Returns the number of
        labels removed (the same on every rank)."""
        if isinstance(x, IDSelectorRange):
            labels = np.arange(max(x.imin, 0), min(x.imax, self.ntotal), dtype=np.int64)
        else:
            labels = x.ids if isinstance(x, IDSelectorBatch) else _id_array(x)
            labels = np.unique(labels[(labels >= 0) & (labels < self.ntotal)])
        local = self.segments.remove(labels)
        if len(local):
            self.local.remove_ids(local)
        self.ntotal -= int(len(labels))
        return int(len(labels))

    def reset(self):
        self.local.reset()
        if hasattr(self.local, "set_search_params"):
            self.local.set_search_params(id_offset=0)
        self.segments = SegmentMap()
        self.ntotal = 0
