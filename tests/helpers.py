"""Shared test helpers: oracle-backed stand-ins used ONLY to exercise host logic on CPU."""
import numpy as np

import oracle as orc


class OracleIndex:
    """Minimal IndexFlat look-alike over the CPU oracle (tests of host-side logic only)."""

    def __init__(self, d, metric=orc.METRIC_L2, **_):
        self.d = d
        self.metric_type = metric
        self.x = np.zeros((0, d), np.float32)
        self.is_trained = True
        self._offset = 0

    @property
    def ntotal(self):
        return self.x.shape[0]

    def add(self, x):
        x = np.ascontiguousarray(x, np.float32)
        if x.shape[1] != self.d:
            raise AssertionError("dimension mismatch")
        self.x = np.concatenate([self.x, x], 0)

    def set_search_params(self, id_offset=None, **_):
        if id_offset is not None:
            self._offset = int(id_offset)
        return self

    def search(self, q, k):
        if k <= 0:
            raise AssertionError("k must be > 0")
        D, I = orc.c_search(self.x, np.ascontiguousarray(q, np.float32), k, self.metric_type)
        I = np.where(I >= 0, I + self._offset, I)
        return D, I

    def reset(self):
        self.x = np.zeros((0, self.d), np.float32)
        # (the id offset is NOT cleared here: the sharded wrapper must reset it itself)


def np_merge(metric, Dg, Ig):
    """numpy restatement of the top-k merge kernel (b2f_merge_topk_strided) for [G, nq, k] inputs (torch CPU tensors or
    arrays)."""
    Dg = np.asarray(Dg)
    Ig = np.asarray(Ig)
    G, nq, k = Dg.shape
    keys = (Dg if metric == orc.METRIC_L2 else -Dg).transpose(1, 0, 2).reshape(nq, G * k).astype(np.float64)
    ids = Ig.transpose(1, 0, 2).reshape(nq, G * k)
    keys = np.where(ids < 0, np.inf, keys)
    tie = np.where(ids < 0, np.iinfo(np.int64).max, ids)
    order = np.lexsort((tie, keys), axis=1)[:, :k]
    I = np.take_along_axis(ids, order, 1)
    Dflat = Dg.transpose(1, 0, 2).reshape(nq, G * k)
    D = np.take_along_axis(Dflat, order, 1).astype(np.float32)
    fmax = np.finfo(np.float32).max
    D = np.where(I < 0, fmax if metric == orc.METRIC_L2 else -fmax, D).astype(np.float32)
    return D, I


def np_topk_merge_fn(metric, recv, part_bytes, off_i, D, I):
    """ShardedIndexFlat(merge_fn=...) stand-in for the CUDA merge: splits the all-gathered host buffer (uint8 [G *
    part_bytes], part g = [D fp32 | pad | I int64 at off_i], [nq, k] each) and merges with np_merge into D / I."""
    nq, k = D.shape
    buf = recv.numpy().reshape(-1, part_bytes)
    Dg = buf[:, : 4 * nq * k].copy().view(np.float32).reshape(-1, nq, k)
    Ig = buf[:, off_i: off_i + 8 * nq * k].copy().view(np.int64).reshape(-1, nq, k)
    D.numpy()[:], I.numpy()[:] = np_merge(metric, Dg, Ig)
