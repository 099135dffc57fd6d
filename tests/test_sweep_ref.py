"""CPU pins of oracle/sweep_ref.py, the fp64 restatement of the sweep's per-row statistics that tests/test_gpu_sweep_rows.py judges the
tcgen05 kernels against: on bf16-exact operands the loss rebuilt from its statistics (finalize's formulas) must be HeadOracle's add_margin
loss to 1e-12, and the top-k judge must accept exact lists and swaps inside its tie band and reject everything a wrong kernel produces."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle.head_ref import add_margin, hard_neg_k
from oracle.sweep_ref import KEY_TRUNC, SweepRef, judge_topk


def _bf16_exact_case(seed, n, Q, D, ones, n_out, tgt_in_ones):
    gen = torch.Generator().manual_seed(seed)
    # bf16-representable operands: the reference's fp64 cosines are then the oracle's
    q = F.normalize(torch.rand(2, Q, D, generator=gen), dim=2).to(torch.bfloat16).float()
    p = F.normalize(torch.randn(n, D, generator=gen)).to(torch.bfloat16).float()
    label = torch.randint(0, Q, (n,), generator=gen)
    label[torch.randperm(n, generator=gen)[:n_out]] = -1
    if tgt_in_ones and ones:
        pos = torch.nonzero(label >= 0).flatten()[:3]
        label[pos] = torch.tensor(ones[:len(pos)])
    return p, q, label


@pytest.mark.parametrize('loss_type,margin', [('AM', 0.35), ('Arc', 0.5), ('SV', 0.35), ('SV', 0.9)])
@pytest.mark.parametrize('with_ones,n_out,tgt_in_ones', [(False, 0, False), (True, 0, True), (True, 5, True), (False, 7, False), (True, 20, False)])
def test_loss_from_statistics_is_add_margin(loss_type, margin, with_ones, n_out, tgt_in_ones):
    n, Q, D, scale = 20, 300, 32, 32.0
    k = hard_neg_k(Q)
    ones = [0, 31, 32, 127, 128, Q - 1] if with_ones else []
    p, q, label = _bf16_exact_case(7, n, Q, D, ones, n_out, tgt_in_ones)
    mirror = q.to(torch.bfloat16)
    r = SweepRef(p, mirror, label, ones, loss_type, scale, margin, k)
    tgt = r.tgt()
    if loss_type == 'SV':       # thresholds from the (here exact) target cosines, as the kernel's prep forms them
        thr = torch.where(tgt[2:3].expand(2, n) > 0, tgt[:2] - margin, torch.full_like(tgt[:2], math.inf))
        r = SweepRef(p, mirror, label, ones, loss_type, scale, margin, k, thr=thr)
    P, W0 = p.double(), q[0].double()
    W2 = W0.clone()
    if ones:
        W2[ones] = q[1].double()[ones]
    want = float(add_margin(P @ W0.t(), label, loss_type, margin, scale, k) + add_margin(P @ W2.t(), label, loss_type, margin, scale, k))
    lsum, _ = r.stats()
    got = r.loss(lsum, tgt)
    assert abs(got - want) <= 1e-12 * abs(want), (got, want)
    # the hard-negative term through finalize's merge of per-set lists (main + side of each loss) equals the direct top-k
    if n_out:
        tv, ti = r.exact_lists()
        merged = r.merged_hard_negatives(tv, ti)
        assert abs(r.outlier_loss_from(merged) - r.outlier_loss()) <= 1e-14
        for i in merged:
            for which in range(3):
                assert judge_topk(tv[which, i], ti[which, i], r.set_cosines([i], which)[0], k, 1e-6) == []
    # dLoss/dp of the positive rows from the statistics against autograd through add_margin
    if n_out < n:
        Pg = P.clone().requires_grad_(True)
        pos = label >= 0
        lab_pos = torch.where(pos, label, torch.full_like(label, -1))
        L = add_margin(Pg @ W0.t(), lab_pos, loss_type, margin, scale, k) + add_margin(Pg @ W2.t(), lab_pos, loss_type, margin, scale, k)
        # add_margin normalises the outlier term by the outlier count; the positive rows' gradient is independent of it
        (g,) = torch.autograd.grad(L, Pg)
        lsum, osum = r.stats()
        dp = r.dp_positive(lsum, osum, tgt)
        assert torch.allclose(dp[pos], g[pos], rtol=0, atol=1e-12 * float(g[pos].abs().max()))


def _judge_row(seed=3, Q=200, k=5):
    gen = torch.Generator().manual_seed(seed)
    cos = torch.rand(Q, generator=gen, dtype=torch.float64) * 2 - 1
    cos[::7] = -math.inf                          # slots outside the set
    order = torch.argsort(torch.where(cos > -math.inf, cos, torch.full_like(cos, -2.0)), descending=True)
    tv = cos[order[:k]].clone()
    ti = order[:k].clone()
    return cos, tv, ti


def test_judge_accepts_exact_list_and_truncated_keys():
    cos, tv, ti = _judge_row()
    assert judge_topk(tv, ti, cos, 5, 1e-6) == []
    # the kernel's values are the keys: low 5 mantissa bits of the fp32 cosine cleared
    keys = (tv.float().view(torch.int32) & ~31).view(torch.float32).double()
    assert judge_topk(keys, ti, cos, 5, 1e-6) == []


def test_judge_accepts_swap_inside_band_only():
    cos, tv, ti = _judge_row()
    k, delta = 5, 1e-6
    nxt = int(torch.argsort(torch.where(cos > -math.inf, cos, torch.full_like(cos, -2.0)), descending=True)[k])
    # plant the (k+1)-th inside the band below the k-th: either may be listed
    cos[nxt] = float(cos[ti[k - 1]]) - delta
    tv2, ti2 = tv.clone(), ti.clone()
    tv2[k - 1], ti2[k - 1] = cos[nxt], nxt
    assert judge_topk(tv2, ti2, cos, k, delta) == []
    # outside the band: rejected
    cos[nxt] = float(cos[ti[k - 1]]) - 10 * (delta + KEY_TRUNC)
    tv2[k - 1] = cos[nxt]
    assert judge_topk(tv2, ti2, cos, k, delta) != []


def test_judge_rejects_wrong_lists():
    cos, tv, ti = _judge_row()
    k, d = 5, 1e-6
    excluded = int(torch.nonzero(cos == -math.inf).flatten()[0])
    cases = {
        'duplicate': (tv, torch.tensor([ti[0], ti[0], ti[2], ti[3], ti[4]])),
        'excluded slot': (tv, torch.tensor([excluded, ti[1], ti[2], ti[3], ti[4]])),
        'seed marker': (tv, torch.tensor([ti[0], ti[1], -2, ti[3], ti[4]])),
        'missing entry': (torch.cat([tv[:4], torch.tensor([-math.inf], dtype=torch.float64)]), torch.cat([ti[:4], torch.tensor([-1])])),
        'not descending': (tv[[1, 0, 2, 3, 4]], ti[[1, 0, 2, 3, 4]]),
        'wrong value': (torch.cat([tv[:1] + 1e-3, tv[1:]]), ti),
        'padding in the middle': (torch.tensor([tv[0], -math.inf, tv[2], tv[3], tv[4]], dtype=torch.float64), torch.tensor([ti[0], -1, ti[2], ti[3], ti[4]])),
    }
    for name, (v, i) in cases.items():
        assert judge_topk(v, i, cos, k, d) != [], name


def test_judge_counts_positive_cosines_only():
    cos = torch.tensor([0.5, 0.25, -0.1, -0.2, -math.inf, 0.0], dtype=torch.float64)
    tv = torch.tensor([0.5, 0.25, -math.inf, -math.inf], dtype=torch.float64)
    ti = torch.tensor([0, 1, -1, -1])
    assert judge_topk(tv, ti, cos, 4, 1e-6) == []
    # an exact zero may be listed
    assert judge_topk(torch.tensor([0.5, 0.25, 0.0, -math.inf], dtype=torch.float64), torch.tensor([0, 1, 5, -1]), cos, 4, 1e-6) == []
    # a negative cosine may not
    assert judge_topk(torch.tensor([0.5, 0.25, -0.1, -math.inf], dtype=torch.float64), torch.tensor([0, 1, 2, -1]), cos, 4, 1e-6) != []
    # a row whose cosines are all negative has an empty list
    neg = torch.tensor([-0.5, -0.25, -0.1], dtype=torch.float64)
    assert judge_topk(torch.full((3,), -math.inf, dtype=torch.float64), torch.full((3,), -1), neg, 3, 1e-6) == []
    assert judge_topk(torch.tensor([-0.1, -math.inf, -math.inf], dtype=torch.float64), torch.tensor([2, -1, -1]), neg, 3, 1e-6) != []
