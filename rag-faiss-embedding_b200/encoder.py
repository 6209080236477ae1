"""Tensor handoff from the sentence encoder to the index (SURVEY 8a9 / 8f rank 2).

The reference slices the CLS token, copies it to the host, turns it into a Python list of rows and
back into a numpy array for every batch of 32 texts (vectorization.py:38-47,
rag_datastore_manager.py:123-132).  Here the encoder's `last_hidden_state` stays on the device:
one fused kernel pools (CLS = reference semantics, or masked mean), optionally L2-normalises, and
writes the rows, their bf16 scan copy and norms straight into index storage.
"""
from __future__ import annotations

import ctypes

from . import _capi as C
from .index import _torch_stream


def pool_normalize(hidden, attention_mask=None, pool: str = "cls", normalize: bool = False):
    """hidden [B, T, d] CUDA fp32 -> [B, d] CUDA fp32 through the CUDA kernel (no torch math)."""
    import torch

    if not (hidden.is_cuda and hidden.dim() == 3):
        raise AssertionError("pool_normalize expects a CUDA tensor [B, T, d]")
    hidden = hidden.to(torch.float32).contiguous()
    B, T, d = hidden.shape
    out = torch.empty((B, d), dtype=torch.float32, device=hidden.device)
    mptr = None
    if attention_mask is not None:
        attention_mask = attention_mask.to(device=hidden.device, dtype=torch.int64).contiguous()
        mptr = attention_mask.data_ptr()
    C.check(C.load().b2f_pool_normalize(hidden.data_ptr(), mptr, B, T, d,
                                        C.POOL_MEAN if pool == "mean" else C.POOL_CLS, int(bool(normalize)),
                                        out.data_ptr(), hidden.device.index or 0, ctypes.c_void_p(_torch_stream(hidden))))
    return out


def synth_rows(seed: int, row0: int, nrows: int, d: int, normalize: bool = False, device: int = 0):
    """Rows of the counter-based synthetic matrix as a CUDA tensor (bit-identical to the oracle's)."""
    import torch

    out = torch.empty((nrows, d), dtype=torch.float32, device=f"cuda:{device}")
    C.check(C.load().b2f_synth_rows(int(seed), int(row0), int(nrows), int(d), int(bool(normalize)), out.data_ptr(),
                                    device, ctypes.c_void_p(_torch_stream(out))))
    return out
