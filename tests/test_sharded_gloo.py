"""CPU tier: the N>1 path without the peer exchange (partition -> per-rank search into one packed message -> one
all-gather -> merge) on the gloo backend with world_size 2 and 3, using oracle-backed local shards and the numpy
restatement of the merge kernel.  Results must equal a single-index search of the concatenated database."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle as orc
from tests.helpers import OracleIndex, np_topk_merge_fn


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, metric, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from rag_faiss_embedding_b200.sharded import ShardedIndexFlat

        d, k = 32, 7
        xb1 = orc.np_synth_rows(11, 0, 501, d)
        xb2 = orc.np_synth_rows(11, 501, 77, d)
        xq = orc.np_synth_rows(12, 0, 9, d)

        ix = ShardedIndexFlat(d, metric, local_index=OracleIndex(d, metric), merge_fn=np_topk_merge_fn)
        ix.add(xb1)
        D0, I0 = ix.search(xq, k)   # single segment: the shard offset is applied by the local index ...
        ix.add(xb2)   # second add: labels continue after the first, shard holds two segments
        assert ix.ntotal == 578
        D, I = ix.search(xq, k)     # ... and must not leak into the multi-segment remap (add, search, add, search)
        Dk, Ik = ix.search(xq, 600)  # k > rows per shard and > ntotal: padding must survive the merge
        ix.reset()
        ix.add(xb2)
        Dr, Ir = ix.search(xq, k)   # after reset(): labels start at 0 again
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), D=D, I=I, Dk=Dk, Ik=Ik, D0=D0, I0=I0, Dr=Dr, Ir=Ir,
                 nlocal=ix.local.ntotal)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("metric", [orc.METRIC_L2, orc.METRIC_INNER_PRODUCT])
def test_sharded_equals_single(tmp_path, world, metric):
    port = _free_port()
    mp.spawn(_worker, args=(world, port, metric, str(tmp_path)), nprocs=world, join=True)
    d, k = 32, 7
    xb = orc.np_synth_rows(11, 0, 578, d)
    xq = orc.np_synth_rows(12, 0, 9, d)
    D_ref, I_ref = orc.c_search(xb, xq, k, metric)
    Dk_ref, Ik_ref = orc.c_search(xb, xq, 600, metric)
    D0_ref, I0_ref = orc.c_search(xb[:501], xq, k, metric)
    Dr_ref, Ir_ref = orc.c_search(xb[501:], xq, k, metric)
    total = 0
    for r in range(world):
        z = np.load(os.path.join(tmp_path, f"r{r}.npz"))
        assert np.array_equal(z["I"], I_ref), f"rank {r}"
        assert np.allclose(z["D"], D_ref, rtol=1e-6)
        assert np.array_equal(z["Ik"], Ik_ref)
        assert np.array_equal(z["Dk"], Dk_ref)
        assert np.array_equal(z["I0"], I0_ref) and np.allclose(z["D0"], D0_ref, rtol=1e-6)
        assert np.array_equal(z["Ir"], Ir_ref) and np.allclose(z["Dr"], Dr_ref, rtol=1e-6)
        total += int(z["nlocal"])
    assert total == 77
