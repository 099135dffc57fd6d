"""fp64 restatement of the tcgen05 sweep's per-row statistics on the operands the sweep multiplies.

TEST INFRASTRUCTURE ONLY (like the rest of ``oracle/``): only ``tests/`` import it.

The bf16 head rounds the probe rows to bf16 (round to nearest even, ``head_prep_fused_kernel`` writing ``p16``) and multiplies them with
the bf16 queue mirror.  Every product of two bf16 numbers is exact in fp64, so the cosines below are the sweep's cosines up to the fp32
accumulation of the tensor cores alone, and the statistics differ from the kernel's only by fp32 accumulation order, ``ex2.approx`` and
the bf16 rounding of p~ before GEMM-2 -- each of which can be bounded per row (tests/test_gpu_sweep_rows.py).  The head's own parity
tests compare against the fp32 queue instead, which leaves a 1e-2 operand-rounding gap in which a kernel can be wrong for a few rows.

Layout follows include/ffc_b200.h (n rows, k = topk, D = feat_dim):
  tgt  [4][n]      target cosine under queue[0], under W2, owner flag, 0
  lsum [4][n]      sum of exp(s z(cos) - M) over: main columns under loss 1 (slot 0), main columns under loss 2 (slot 1, SV only),
                   the `ones` rows of queue[0] (slot 2) and of queue[1] (slot 3); main = every column except `ones` and the row's
                   target, side sets exclude the target's position
  osum [4][n][D]   sum of w exp(...) W_j over the same sets (w = 1.2 on SV-hard columns); rows of hard-negative-only rows are zero
Top-k lists are judged, not compared: see ``judge_topk``.
"""
from __future__ import annotations

import math

import numpy as np
import torch

SV_T = 1.2                      # ffc.py:47 mask_svfc
KEY_TRUNC = 2.0 ** -18          # a top-k key keeps the cosine with its low 5 mantissa bits replaced by the column: relative loss < 2^-18


def fixed_max(loss_type: str, scale: float) -> float:
    """csrc/head.cu fixed_max_of, in the fp32 arithmetic it is computed in."""
    f = np.float32
    s = f(scale)
    zmax = s * (f(2.0) * f(SV_T) - f(1.0)) if loss_type == 'SV' else s
    return float(f(0.5) * (zmax - s + f(20.0)))


def bf16_operands(p_f32: torch.Tensor, mirror: torch.Tensor):
    """The sweep's operands in fp64: P rounded to bf16 (RNE, as the prep kernel does), W0 / W1 = the mirror's two tables."""
    P = p_f32.to(torch.bfloat16).double()
    return P, mirror[0].double(), mirror[1].double()


def sv_thresholds(tgt: torch.Tensor, margin: float) -> torch.Tensor:
    """[2][n] SV hard thresholds as the prep kernel forms them from its fp32 target cosines (c - margin in fp32; +inf without target)."""
    n = tgt.shape[1]
    thr = (tgt[:2].float() - torch.tensor(margin, dtype=torch.float32)).double()
    return torch.where(tgt[2:3].expand(2, n) > 0, thr, torch.full_like(thr, math.inf))


class SweepRef:
    """Per-row sweep statistics in fp64.  ``label``: local slots or -1, ``ones``: the pass's `ones` slots in list order.
    ``thr`` ([2][n], SV only): the hard thresholds; pass the kernel's (``sv_thresholds`` of its checked tgt) so that both sides classify
    columns against the same number.  Everything runs on the device of the inputs, chunked over columns."""

    def __init__(self, p_f32, mirror, label, ones, loss_type, scale, margin, k, thr=None, col_chunk=1 << 14):
        self.P, self.W0, self.W1 = bf16_operands(p_f32, mirror)
        dev = self.P.device
        self.n, self.D = self.P.shape
        self.Q = self.W0.shape[0]
        self.label = torch.as_tensor(label, dtype=torch.long, device=dev)
        self.ones = torch.as_tensor(list(ones), dtype=torch.long, device=dev)
        self.loss_type, self.scale, self.margin, self.k = loss_type, float(scale), float(margin), int(k)
        self.M = fixed_max(loss_type, scale)
        self.col_chunk = col_chunk
        self.is_out = self.label < 0
        in_ones = torch.zeros(self.Q, dtype=torch.bool, device=dev)
        in_ones[self.ones] = True
        self.in_ones = in_ones
        pos_of = torch.full((self.Q,), -1, dtype=torch.long, device=dev)
        pos_of[self.ones] = torch.arange(len(self.ones), device=dev)
        t = self.label.clamp(min=0)
        self.tpos = torch.where(self.is_out, torch.full_like(t, -1), pos_of[t])
        self.thr = thr.to(dev).double() if thr is not None else torch.full((2, self.n), math.inf, dtype=torch.float64, device=dev)
        self._stats = None

    # -- target cosines -----------------------------------------------------------------------------------------------------------
    def tgt(self) -> torch.Tensor:
        t = self.label.clamp(min=0)
        c0 = (self.P * self.W0[t]).sum(1)
        w2 = torch.where((self.tpos >= 0).unsqueeze(1), self.W1[t], self.W0[t])
        c1 = (self.P * w2).sum(1)
        own = (~self.is_out).double()
        return torch.stack([c0 * own, c1 * own, own, torch.zeros_like(own)])

    # -- softmax statistics -------------------------------------------------------------------------------------------------------
    def _z(self, c, thr):
        if self.loss_type != 'SV':
            return c, torch.ones_like(c)
        hard = c > thr.unsqueeze(1)
        return torch.where(hard, SV_T * c + (SV_T - 1.0), c), torch.where(hard, torch.full_like(c, SV_T), torch.ones_like(c))

    def _accumulate(self, W, cols, excl_col, thr, delta=None):
        """lsum / osum over the columns `cols` of W (rows of W), excluding per row the column excl_col[i] (-1: none).  With `delta`:
        instead sum_j w p~_j |W_j| and the SV ambiguity sum_j |p~_j(hard) - p~_j(not hard)| over columns within delta of the threshold
        (the terms of the kernel's error bounds)."""
        pr = torch.nonzero(~self.is_out).flatten()     # hard-negative-only rows have no softmax term
        P, thr, excl_col = self.P[pr], thr[pr], excl_col[pr]
        L = torch.zeros(len(pr), dtype=torch.float64, device=self.P.device)
        O = torch.zeros(len(pr), self.D, dtype=torch.float64, device=self.P.device)
        for c0 in range(0, len(cols), self.col_chunk):
            cc = cols[c0:c0 + self.col_chunk]
            Wc = W[cc]
            c = P @ Wc.t()
            z, w = self._z(c, thr)
            e = torch.exp(self.scale * z - self.M)
            keep = cc.unsqueeze(0) != excl_col.unsqueeze(1)
            e = torch.where(keep, e, torch.zeros_like(e))
            if delta is None:
                L += e.sum(1)
                O += (e * w) @ Wc
            else:
                O += (e * w) @ Wc.abs()
                if self.loss_type == 'SV':
                    near = keep & ((c - thr.unsqueeze(1)).abs() <= delta)
                    both = (torch.exp(self.scale * (SV_T * c + (SV_T - 1.0)) - self.M) - torch.exp(self.scale * c - self.M)).abs()
                    L += torch.where(near, both, torch.zeros_like(both)).sum(1)
        Lf = torch.zeros(self.n, dtype=torch.float64, device=self.P.device)
        Of = torch.zeros(self.n, self.D, dtype=torch.float64, device=self.P.device)
        Lf[pr], Of[pr] = L, O
        return Lf, Of

    def abs_osum_and_ambiguous(self, delta):
        """(amb [4][n], absO [4][n][D]) for the statistics' slots: see ``_accumulate``."""
        dev = self.P.device
        main = torch.nonzero(~self.in_ones).flatten()
        t_main = torch.where(self.is_out, torch.full_like(self.label, -1), self.label)
        amb = torch.zeros(4, self.n, dtype=torch.float64, device=dev)
        absO = torch.zeros(4, self.n, self.D, dtype=torch.float64, device=dev)
        amb[0], absO[0] = self._accumulate(self.W0, main, t_main, self.thr[0], delta)
        if self.loss_type == 'SV':
            amb[1], absO[1] = self._accumulate(self.W0, main, t_main, self.thr[1], delta)
        if len(self.ones):
            pos = torch.arange(len(self.ones), device=dev)
            amb[2], absO[2] = self._accumulate(self.W0[self.ones], pos, self.tpos, self.thr[0], delta)
            amb[3], absO[3] = self._accumulate(self.W1[self.ones], pos, self.tpos, self.thr[1], delta)
        return amb, absO

    def stats(self):
        """(lsum [4][n], osum [4][n][D]); zero in the rows of hard-negative-only rows (the kernel's lsum there is unspecified)."""
        if self._stats is not None:
            return self._stats
        dev = self.P.device
        main = torch.nonzero(~self.in_ones).flatten()
        t_main = torch.where(self.is_out, torch.full_like(self.label, -1), self.label)
        lsum = torch.zeros(4, self.n, dtype=torch.float64, device=dev)
        osum = torch.zeros(4, self.n, self.D, dtype=torch.float64, device=dev)
        lsum[0], osum[0] = self._accumulate(self.W0, main, t_main, self.thr[0])
        if self.loss_type == 'SV':
            lsum[1], osum[1] = self._accumulate(self.W0, main, t_main, self.thr[1])
        if len(self.ones):
            # side sets: positions 0..n_ones-1 of the gathered rows; the excluded position is the target's place in `ones`
            pos = torch.arange(len(self.ones), device=dev)
            lsum[2], osum[2] = self._accumulate(self.W0[self.ones], pos, self.tpos, self.thr[0])
            lsum[3], osum[3] = self._accumulate(self.W1[self.ones], pos, self.tpos, self.thr[1])
        self._stats = (lsum, osum)
        return self._stats

    # -- hard-negative cosines ----------------------------------------------------------------------------------------------------
    def set_cosines(self, rows, which: int) -> torch.Tensor:
        """[len(rows), Q] fp64 cosines of the given rows over the slots of top-k set `which` (0 main under queue[0], 1 `ones` under
        queue[0], 2 `ones` under queue[1]); slots outside the set are -inf."""
        rows = torch.as_tensor(rows, dtype=torch.long, device=self.P.device)
        W = self.W1 if which == 2 else self.W0
        c = self.P[rows] @ W.t()
        elig = ~self.in_ones if which == 0 else self.in_ones
        return torch.where(elig.unsqueeze(0), c, torch.full_like(c, -math.inf))

    def loss_cosines(self, rows, l: int) -> torch.Tensor:
        """[len(rows), Q] cosines of loss l's logits (l = 0: queue[0]; l = 1: W2 = queue[1] on `ones`, queue[0] elsewhere)."""
        rows = torch.as_tensor(rows, dtype=torch.long, device=self.P.device)
        c0 = self.P[rows] @ self.W0.t()
        if l == 0 or not len(self.ones):
            return c0
        return torch.where(self.in_ones.unsqueeze(0), self.P[rows] @ self.W1.t(), c0)

    # -- finalize (row_coef_math) in fp64 -----------------------------------------------------------------------------------------
    def margin_fn(self, ct):
        """(f(ct), f'(ct)) of the loss, with the bf16 path's clamp of ct to +-(1 - 1e-6), rounded to fp32 as the one-GPU finalize
        forms it (0.99999899: 1 - ct is 1.3 % larger than with the exact bound, and Arc's f' near the clamp follows 1 / sqrt(1 - ct))."""
        b = float(np.float32(1.0 - 1e-6))
        ct = ct.clamp(-b, b)
        if self.loss_type == 'AM':
            return ct - self.margin, torch.ones_like(ct)
        if self.loss_type == 'Arc':
            sn = torch.sqrt((1.0 - ct) * (1.0 + ct))
            cm, sm = math.cos(self.margin), math.sin(self.margin)
            return ct * cm - sn * sm, cm + ct * sm / sn
        return torch.where(ct > self.margin, ct - self.margin, ct), torch.ones_like(ct)

    def positive_rows(self, lsum, tgt):
        """Per positive row and loss: (row loss [n], cO [2][n], cT [2][n], L [2][n]) from statistics laid out as the kernel's."""
        n_pos = int((~self.is_out).sum())
        loss = torch.zeros(self.n, dtype=torch.float64, device=self.P.device)
        cO = torch.zeros(2, self.n, dtype=torch.float64, device=self.P.device)
        cT = torch.zeros_like(cO)
        Ls = torch.zeros_like(cO)
        s, M = self.scale, self.M
        for l in range(2):
            ft, dft = self.margin_fn(tgt[l].double())
            zt = s * ft
            et = torch.exp(zt - M)
            cs = l if self.loss_type == 'SV' else 0
            L = lsum[cs].double() + lsum[2 + l].double() + et
            loss += (torch.log(L) + M - zt) / max(n_pos, 1)
            cO[l] = s / L / max(n_pos, 1)
            cT[l] = s * (et / L - 1.0) * dft / max(n_pos, 1)
            Ls[l] = L
        pos = ~self.is_out
        return loss * pos, cO * pos, cT * pos, Ls

    def dp_positive(self, lsum, osum, tgt):
        """dLoss/dp of the positive rows (outlier rows zero) from statistics in the kernel's layout."""
        _, cO, cT, _ = self.positive_rows(lsum, tgt)
        t = self.label.clamp(min=0)
        w1 = torch.where((self.tpos >= 0).unsqueeze(1), self.W1[t], self.W0[t])
        oc1 = osum[1] if self.loss_type == 'SV' else osum[0]
        dp = cO[0].unsqueeze(1) * (osum[0].double() + osum[2].double()) + cO[1].unsqueeze(1) * (oc1.double() + osum[3].double())
        dp += cT[0].unsqueeze(1) * self.W0[t] + cT[1].unsqueeze(1) * w1
        return dp * (~self.is_out).unsqueeze(1)

    def exact_lists(self):
        """topv / topi [3][n][k] as an exact kernel would report them: per outlier row and set the k largest POSITIVE fp64 cosines
        (ties by smaller slot), -inf / -1 padded; positive rows empty."""
        tv = torch.full((3, self.n, self.k), -math.inf, dtype=torch.float64)
        ti = torch.full((3, self.n, self.k), -1, dtype=torch.long)
        rows = torch.nonzero(self.is_out).flatten()
        for which in range(3):
            for r0 in range(0, len(rows), 1024):
                rr = rows[r0:r0 + 1024]
                c = self.set_cosines(rr, which)
                kk = min(self.k, c.shape[1])
                v, s = torch.topk(c, kk, dim=1, sorted=True)       # (values unique in the tests that rely on the order)
                keep = v > 0
                tv[which, rr.cpu(), :kk] = torch.where(keep, v, torch.full_like(v, -math.inf)).cpu()
                ti[which, rr.cpu(), :kk] = torch.where(keep, s, torch.full_like(s, -1)).cpu()
        return tv, ti

    def outlier_loss_from(self, merged):
        """Hard-negative term from finalize's selection (``merged_hard_negatives``): sum of max(v, 0) over n_out k."""
        n_out = int(self.is_out.sum())
        return sum(max(v, 0.0) for per_loss in merged.values() for sel in per_loss for v, _, _ in sel) / (max(n_out, 1) * self.k)

    def merged_hard_negatives(self, topv, topi):
        """finalize's merge for every outlier row and loss: main list first, then the loss's side list, the k largest values (ties:
        the earlier entry wins).  topv / topi [3][n][k] as the kernel reports them (global = local slots here).  Returns a list over
        rows of [(value, slot, table)] per loss, table 1 = queue[1]."""
        tv, ti = topv.double().cpu(), topi.long().cpu()
        out = {}
        for i in torch.nonzero(self.is_out).flatten().tolist():
            per_loss = []
            for l in range(2):
                cand = [(float(tv[0, i, q]), int(ti[0, i, q]), 0) for q in range(self.k) if int(ti[0, i, q]) >= 0]
                cand += [(float(tv[1 + l, i, q]), int(ti[1 + l, i, q]), l) for q in range(self.k) if int(ti[1 + l, i, q]) >= 0]
                order = sorted(range(len(cand)), key=lambda e: -cand[e][0])       # stable: main before side on equal values
                per_loss.append([cand[e] for e in order[:self.k]])
            out[i] = per_loss
        return out

    def dp_outlier(self, merged):
        """dLoss/dp of the hard-negative-only rows from the slots finalize selects (``merged_hard_negatives`` of the kernel's lists):
        the sum of the selected bf16 prototype rows with a non-negative value, over n_out k."""
        n_out = int(self.is_out.sum())
        dp = torch.zeros(self.n, self.D, dtype=torch.float64, device=self.P.device)
        w = 1.0 / (max(n_out, 1) * self.k)
        for i, per_loss in merged.items():
            for sel in per_loss:
                for v, slot, table in sel:
                    if v >= 0.0:
                        dp[i] += w * (self.W1[slot] if table == 1 else self.W0[slot])
        return dp

    def outlier_loss(self):
        """Hard-negative term of both losses from the exact cosines: mean over outlier rows and k of max(top-k cos, 0)."""
        rows = torch.nonzero(self.is_out).flatten()
        n_out = len(rows)
        if n_out == 0:
            return 0.0
        tot = 0.0
        for r0 in range(0, n_out, 1024):
            rr = rows[r0:r0 + 1024]
            for l in range(2):
                c = self.loss_cosines(rr, l)
                tot += float(torch.topk(c, self.k, dim=1).values.clamp(min=0).sum())
        return tot / (n_out * self.k)

    def loss(self, lsum=None, tgt=None):
        """The pass's loss (both add_margin terms) from the statistics (default: this reference's own)."""
        if lsum is None:
            lsum = self.stats()[0]
        if tgt is None:
            tgt = self.tgt()
        return float(self.positive_rows(lsum, tgt)[0].sum()) + self.outlier_loss()


def judge_topk(tv, ti, cos, k, delta):
    """Judge one row's reported top-k list of one set against the fp64 cosines of that set.

    tv / ti: the k reported values and slots; cos: [Q] fp64 cosines, -inf on slots outside the set; delta: bound on |fp32 MMA
    cosine - fp64 cosine|.  The kernel lists positive cosines only (keys start at 0; an exact +0.0 may appear), truncated to a key with
    the low 5 mantissa bits cleared: 0 <= cos_f32 - tv < 2^-18 cos_f32.  Returns the list of violations (empty: accepted).
      - entries are a prefix of valid, distinct slots of the set, then (-inf, -1) padding; values non-increasing;
      - each value is its slot's cosine within delta + the truncation;
      - the count lies between min(k, #cos > delta) and min(k, #cos >= -delta);
      - with c_k the k-th eligible cosine (0 when fewer), every slot with cos > c_k + 2 band is listed and every listed slot has
        cos >= c_k - 2 band (band = delta + truncation): the list is exact outside the tie band."""
    tv = [float(v) for v in tv]
    ti = [int(v) for v in ti]
    cos = cos.double().cpu()
    Q = cos.shape[0]
    bad = []
    nv = 0
    while nv < len(ti) and ti[nv] != -1:
        nv += 1
    for q in range(nv, len(ti)):
        if ti[q] != -1 or tv[q] != -math.inf:
            bad.append(f'entry {q}: ({tv[q]}, {ti[q]}) after the padding started')
    slots = ti[:nv]
    for q, s in enumerate(slots):
        if not (0 <= s < Q):
            bad.append(f'entry {q}: slot {s} is not a column')
        elif cos[s] == -math.inf:
            bad.append(f'entry {q}: slot {s} is not in the set')
    if len(set(slots)) != len(slots):
        bad.append(f'duplicate slots {slots}')
    if bad:
        return bad
    for q in range(1, nv):
        if not tv[q] <= tv[q - 1]:
            bad.append(f'values not descending at {q}: {tv[q - 1]} then {tv[q]}')
    band = delta + KEY_TRUNC
    for q, s in enumerate(slots):
        c = float(cos[s])
        if not (tv[q] >= 0.0 and tv[q] - delta <= c <= tv[q] + band):
            bad.append(f'entry {q}: value {tv[q]!r} for slot {s} whose cosine is {c!r}')
    finite = cos[cos > -math.inf]
    lo = min(k, int((finite > delta).sum()))
    hi = min(k, int((finite >= -delta).sum()))
    if not lo <= nv <= hi:
        bad.append(f'{nv} entries, expected {lo}..{hi}')
    ck = max(float(torch.topk(finite, k).values[-1]) if finite.numel() >= k else 0.0, 0.0)
    must = torch.nonzero(cos > ck + 2 * band).flatten().tolist()
    missing = sorted(set(must) - set(slots))
    if missing:
        bad.append(f'slots {missing} (cos > c_k + 2 band = {ck + 2 * band}) not listed')
    for q, s in enumerate(slots):
        if float(cos[s]) < ck - 2 * band:
            bad.append(f'entry {q}: slot {s} cos {float(cos[s])} below c_k - 2 band = {ck - 2 * band}')
    return bad
