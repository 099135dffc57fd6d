"""1:N identification against the prototype queue (csrc/identify_sm100.cu) and the closed-set accuracy helper.

The gallery is ``queue[0][s]`` of every resident LRU slot ``s < cur_idx``; the result for each query row is the k prototypes of
highest cosine, score descending, ties by smaller global slot.  Rows with fewer than k resident identities are padded with
slot -1, label INT64_MIN and score -inf.
"""
from __future__ import annotations

import ctypes as C
from collections import namedtuple

import torch

from . import _capi
from ._capi import check
from .tail import l2_normalize

Identification = namedtuple('Identification', 'scores labels slots')
Identification.__doc__ = 'Result of identify(): scores fp32 [N, k], labels int64 [N, k], slots int32 [N, k] (global), device tensors.'

LABEL_NONE = -(1 << 63)          # label of a padding entry (INT64_MIN, never a key)


def check_k(k):
    k = int(k)
    if not 1 <= k <= _capi.TOPK_MAX:
        raise _capi.FFCError(f'identify: k={k} outside [1, {_capi.TOPK_MAX}]')
    return k


def normalized_queries(x, D, dev):
    """fp32 / fp16 / bf16 rows on any device -> L2-normalised contiguous fp32 rows on `dev` (the tail kernel)."""
    x = torch.as_tensor(x)
    if x.dim() != 2 or x.shape[1] != D:
        raise ValueError(f'identify expects [N, {D}] embeddings, got {tuple(x.shape)}')
    x = x.to(device=dev, dtype=torch.float32).contiguous()
    return l2_normalize(x) if x.shape[0] else x


def empty(n, k, dev):
    return Identification(torch.full((n, k), float('-inf'), dtype=torch.float32, device=dev),
                          torch.full((n, k), LABEL_NONE, dtype=torch.int64, device=dev),
                          torch.full((n, k), -1, dtype=torch.int32, device=dev))


def search(lib, head, lru_handle, xn, k, queue, queue_bf16):
    """ffc_identify over unit rows `xn` [N, D] on the current stream, FFC_IDENTIFY_MAX_ROWS rows per call."""
    n, dev = xn.shape[0], xn.device
    out = empty(n, k, dev)
    s = torch.cuda.current_stream(dev).cuda_stream
    need = C.c_int64()
    ws = None
    for a in range(0, n, _capi.IDENTIFY_MAX_ROWS):
        m = min(_capi.IDENTIFY_MAX_ROWS, n - a)
        check(lib.ffc_identify_workspace_bytes(head, m, k, C.byref(need)))
        if ws is None or ws.numel() < need.value:
            ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
        check(lib.ffc_identify(head, lru_handle, xn.data_ptr() + a * xn.shape[1] * 4, m, k, queue.data_ptr(),
                               None if queue_bf16 is None else queue_bf16.data_ptr(), ws.data_ptr(), ws.numel(),
                               out.scores.data_ptr() + a * k * 4, out.labels.data_ptr() + a * k * 8, out.slots.data_ptr() + a * k * 4, s))
    return out


def merge(scores, labels, slots, k):
    """Per row, the k best of the candidates [N, C] by (score desc, slot asc); padding (slot -1) sorts last."""
    key_slot = torch.where(slots < 0, torch.full_like(slots, torch.iinfo(torch.int32).max), slots).long()
    order = torch.argsort(key_slot, dim=1, stable=True)                      # slot ascending ...
    s1 = torch.gather(scores, 1, order)
    order2 = torch.argsort(s1, dim=1, descending=True, stable=True)         # ... then score descending, stable
    idx = torch.gather(order, 1, order2)[:, :k]
    return Identification(torch.gather(scores, 1, idx), torch.gather(labels, 1, idx), torch.gather(slots, 1, idx))


def cmc(labels_topk, true_labels, ranks=(1, 5, 10)):
    """Closed-set cumulative match characteristic: {r: fraction of rows whose true label is among their first r results}.
    A row whose true identity is not resident in the gallery counts as a miss (it cannot be found).  ``labels_topk`` [N, k] is
    ``identify(...).labels``; ranks above k use all k results."""
    lab = torch.as_tensor(labels_topk)
    true = torch.as_tensor(true_labels).to(device=lab.device, dtype=lab.dtype).reshape(-1, 1)
    if lab.dim() != 2 or true.shape[0] != lab.shape[0]:
        raise ValueError(f'cmc: labels_topk [N, k] and true_labels [N] expected, got {tuple(lab.shape)} and {tuple(true.shape)}')
    hit = lab == true
    n = max(lab.shape[0], 1)
    return {int(r): float(hit[:, :int(r)].any(dim=1).sum()) / n for r in ranks}
