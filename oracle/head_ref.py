"""CPU restatement of the reference FFC head (one head pass and FFC.forward).

TEST INFRASTRUCTURE ONLY: only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s CPU-baseline / ``--impl reference`` legs may import this module;
the product path (``ffc_b200``) never does.

It restates /root/reference/ffc.py for the head (the backbones are replaced by
"embeddings in"), materialising the B x Q logit matrices exactly like the
reference does (that is what makes it the oracle and the CPU baseline):

  * bookkeeping loop            ffc.py:162-177 (commit) / ffc.py:214-235 (rollback)
  * enqueue scatter             ffc.py:179-182 / ffc.py:237-241 (last duplicate wins, CPU index_put)
  * probe labels                ffc.py:189-194 / ffc.py:242-246
  * logits 1, blend, logits 2   ffc.py:195-201 / ffc.py:248-253
  * add_margin (AM / Arc / SV + hard negatives)   ffc.py:60-138
  * rollback restore            ffc.py:255-259
  * forward = rollback pass (probe=x, gallery=y) + commit pass (probe=y, gallery=x)   ffc.py:264-267
  * hard_neg = min(max(int(Q*0.0002), 3), 10), mask_svfc = 1.2    ffc.py:47-48

Parity of this restatement is pinned against the reference itself run in the
build container (tests/golden/make_golden.py -> tests/golden/*.npz, and live in
tests/test_oracle_vs_reference.py when /root/reference is present).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from .lru_ref import LRU


def hard_neg_k(queue_size: int) -> int:
    """ffc.py:48"""
    return min(max(int(queue_size * 0.0002), 3), 10)


def init_queue(queue_size: int, feat_dim: int, seed: int = 0, dtype=torch.float32) -> torch.Tensor:
    """ffc.py:29-30: normalize(rand(2, Q, D)) (all-positive unit rows)."""
    gen = torch.Generator().manual_seed(seed)
    q = torch.rand(2, queue_size, feat_dim, generator=gen, dtype=torch.float32)
    return F.normalize(q, dim=2).to(dtype)


def add_margin(cos_theta, label, loss_type, margin, scale, k, mask_svfc=1.2):
    """ffc.py:60-138.  cos_theta [B,Q], label [B] in {-1} u [0,Q).  Returns a 0-dim tensor
    (or python 0 when both row sets are empty, like the reference)."""
    out_rows = torch.nonzero(label == -1).flatten()
    pos_rows = torch.nonzero(label != -1).flatten()
    cls_loss = 0
    neg_loss = 0
    if pos_rows.numel() > 0:
        z = cos_theta[pos_rows]
        if loss_type != 'AM':
            z = z.float() if z.dtype in (torch.float16, torch.bfloat16) else z
        tgt = label[pos_rows]
        ar = torch.arange(z.shape[0], device=z.device)
        gt = z[ar, tgt].view(-1, 1)
        if loss_type == 'AM':
            new_t = gt - margin
        elif loss_type == 'Arc':
            sin_t = torch.sqrt(1.0 - gt * gt)
            new_t = gt * math.cos(margin) - sin_t * math.sin(margin)
        else:  # 'SV'
            hard = z > (gt - margin)
            new_t = torch.where(gt > margin, gt - margin, gt)
            z = torch.where(hard, mask_svfc * z + mask_svfc - 1.0, z)
        z = z.scatter(1, tgt.view(-1, 1), new_t)
        cls_loss = F.cross_entropy(z * scale, tgt)
    if out_rows.numel() > 0:
        c = cos_theta[out_rows]
        top_idx = torch.argsort(c, dim=1, descending=True)[:, :k]
        neg_loss = torch.clamp(torch.gather(c, 1, top_idx), min=0).mean()
    return cls_loss + neg_loss


class HeadOracle:
    """State + one head pass, embeddings in.  ``queue`` is [2,Q,D]."""

    def __init__(self, feat_dim, queue_size, scale=32.0, loss_type='AM', margin=0.4,
                 queue=None, dtype=torch.float32, seed=0):
        assert loss_type in ('AM', 'Arc', 'SV')
        self.D, self.Q = feat_dim, queue_size
        self.scale, self.margin, self.loss_type = scale, margin, loss_type
        self.dtype = dtype
        self.queue = (init_queue(queue_size, feat_dim, seed, dtype) if queue is None
                      else queue.detach().clone().to(dtype))
        self.lru = LRU(queue_size)
        self.qpos = [0] * queue_size                        # ffc.py:41-43 queue_position_dict
        self.k = hard_neg_k(queue_size)
        self.trace = []                                     # per pass: dict(rows, cols, labels, ones)

    # -- ffc.py:162-177 / 214-235 -------------------------------------------------
    def bookkeeping(self, gallery_label, commit):
        rows, cols, ones, saved = [], [], [], {}
        seen_ones = set()
        for gl in gallery_label:
            known = gl in self.lru
            slot = self.lru.get(gl) if commit else self.lru.try_get(gl)
            if not commit and slot not in saved:
                saved[slot] = self.qpos[slot]
            if known:
                rows.append(self.qpos[slot])
                if slot not in seen_ones:
                    seen_ones.add(slot)
                    ones.append(slot)
                self.qpos[slot] ^= 1
            else:
                rows.append(0)
                self.qpos[slot] = 1
            cols.append(slot)
        return rows, cols, ones, saved

    def head_pass(self, p, g, probe_label, gallery_label, commit):
        """p [B,D] (may require grad), g [B,D]; labels: python int lists. Returns loss."""
        gl = [int(v) for v in gallery_label]
        pl = [int(v) for v in probe_label]
        rows, cols, ones, saved = self.bookkeeping(gl, commit)
        r = torch.tensor(rows, dtype=torch.long)
        c = torch.tensor(cols, dtype=torch.long)
        g = g.detach().to(self.dtype)
        if not commit:
            old = self.queue[r, c].clone()
        # ffc.py:182/241 ``queue[r, c] = g``: with a repeated (row, col) pair the reference's result is
        # "last occurrence wins" when index_put runs serially (CPU, one thread; probed) and undefined
        # otherwise.  The oracle pins the serial behaviour explicitly: keep the last writer only.
        last = {}
        for i, rc in enumerate(zip(rows, cols)):
            last[rc] = i
        keep = torch.tensor(sorted(last.values()), dtype=torch.long)
        self.queue[r[keep], c[keep]] = g[keep]
        labels = [self.lru.view(v) for v in pl]             # after this pass's inserts
        label = torch.tensor(labels, dtype=torch.long, device=self.queue.device)
        w0 = self.queue[0].clone()
        w2 = w0.clone()
        if ones:
            oi = torch.tensor(ones, dtype=torch.long)
            w2[oi] = self.queue[1][oi]                      # ffc.py:197-200: mask ? queue[1] : queue[0]
        p = p.to(self.dtype)
        cos1 = p @ w0.t()
        cos2 = p @ w2.t()
        loss = (add_margin(cos1, label, self.loss_type, self.margin, self.scale, self.k)
                + add_margin(cos2, label, self.loss_type, self.margin, self.scale, self.k))
        if not commit:                                      # ffc.py:255-259
            self.queue[r, c] = old
            for s, v in saved.items():
                self.qpos[s] = v
            self.lru.rollback_steps(len(gl))
        self.trace.append(dict(rows=rows, cols=cols, labels=labels, ones=sorted(ones)))
        return loss

    def forward(self, x, y, x_label, y_label):
        """ffc.py:264-267 with identity backbones (x, y are unit-norm embeddings)."""
        loss2 = self.head_pass(x, y, x_label, y_label, commit=False)
        loss1 = self.head_pass(y, x, y_label, x_label, commit=True)
        return loss1 + loss2


def dqueue_ref(p, queue, label, ones, loss_type, margin, scale, k):
    """dLoss/dQueue of ONE head pass by autograd, had the reference's `queue` required grad (it is a no-grad buffer, ffc.py:29; the
    optional mode of north_star): `queue` [2,Q,D] is the queue as the pass sweeps it (after its enqueue), `label` the probe labels
    (ffc.py:189-194), `ones` the slots whose second row the blended weight reads (ffc.py:197-200).  Returns (loss, dqueue [2,Q,D])."""
    w = queue.detach().clone().requires_grad_(True)
    w0 = w[0]
    if len(ones):
        m = torch.zeros(w.shape[1], 1, dtype=w.dtype)
        m[torch.as_tensor(ones, dtype=torch.long)] = 1.0
        w2 = m * w[1] + (1.0 - m) * w[0]                  # ffc.py:200
    else:
        w2 = w0
    p = p.detach().to(w.dtype)
    lab = torch.as_tensor(label, dtype=torch.long)
    loss = add_margin(p @ w0.t(), lab, loss_type, margin, scale, k) + add_margin(p @ w2.t(), lab, loss_type, margin, scale, k)
    (g,) = torch.autograd.grad(loss, w)
    return loss.detach(), g
