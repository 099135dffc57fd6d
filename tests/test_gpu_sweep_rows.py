"""Row-by-row checks of the bf16 tcgen05 sweep (csrc/head_sm100.cu, csrc/head_sm100_1cta.cu) and the reduce / finalize kernels that
consume its partials, against oracle/sweep_ref.py: fp64 statistics computed on the operands the kernels multiply (bf16 probe rows, the
bf16 queue mirror), so that the only honest differences are fp32 accumulation, ex2.approx and the bf16 rounding of p~.

The head's parity suites compare the summed loss and the norm of the whole gradient against an fp32-queue oracle to 1e-2; inside that a
kernel can be wrong for a few rows (an exclusion missed or doubled, a ragged-tail mask off by one, a wrong hard negative, a leaked seed
entry, a side tile read wrong).  Here every row's target cosines, softmax denominators, O sums, top-k lists and gradient row is checked,
on crafted inputs where tiles, column chunks, `ones` exclusions and the top-k meet.  The sweep is driven through the C ABI
(ffc_head_sweep for the statistics, ffc_head_pass_single for loss and dLoss/dp) with hand-built labels, `ones` list and cmask.

Tolerances (per row; u = 2^-24, the fp32 unit roundoff):
  cosine     delta_D = D u * 1.02: fp32 accumulation of D exact bf16 x bf16 products whose absolute sum is at most |p| |w| <= (1 + 2^-8)^2
             (worst case; used by the top-k judge, whose values are also truncated keys: 0 <= cos - topv < 2^-18 cos)
  tgt        1 fp32 ulp: prep sums the products in fp64 and rounds once
  lsum       relative  s delta_rw + (s + M) log2(e) u ln 2 + 2^-21 + 4 sqrt(64 + n_cols / 128) u, delta_rw = 4 sqrt(D) u: the cosine's
             accumulation error (as a random walk of D roundings, 4 sigma), the fp32 rounding of ex2's argument, ex2.approx, and the
             fp32 summation depth of a row (64 columns per lane and tile, then tiles and chunks); SV adds the exp mass of the columns
             within delta_D of the threshold under both classifications
  osum       elementwise  2^-8 sum_j w p~_j |W_jd| (bf16 rounding of p~ before GEMM-2) + lsum_tol sum_j w p~_j |W_jd|
  dp         positive rows: propagated from the lsum and osum bounds through finalize's coefficients, plus 2^-16 for its fp32 scalar
             part; hard-negative-only rows: 1e-6 relative to the sum of |terms| (fp32 sums of k bf16 rows over the kernel's slots)
  loss       fp64 reconstruction from the reference statistics and exact top-k, relative 1e-4 (measured near 1e-6)
The launch variants (FFC_SWEEP_* switches, read once per process) re-run this file in subprocesses; within one kernel the variants must
agree bit for bit on tgt and the top-k values (GEMM-1 of a (row, column) is the same MMA sequence in every launch shape), and on the
slots except for which members of a value tied at a list's last place are kept (see test_launch_variants_agree)."""
import ctypes as C
import math
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.sweep_ref import SweepRef, judge_topk, sv_thresholds

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24
DUMP = os.environ.get('FFC_SWEEP_ROWS_DUMP')          # set by the variant runs: where each case leaves tgt / topv / topi
JUDGE_ROWS = 384                                      # hard-negative-only rows judged per case (all planted rows, then a spread)


def _unit(x):
    return F.normalize(x, dim=-1)


def _plant_near(q, slots, p, gen, spread):
    """queue rows at `slots` := unit(max(p + e_j noise, 0)) with graded e_j: cosines to p spaced around a chosen k-th.  Non-negative
    like every queue row, so that minus the queue's mean direction stays a probe with no positive cosine."""
    for j, s in enumerate(slots):
        q[s] = _unit((p + spread * (1.0 + 0.15 * j) * torch.randn(p.shape[0], generator=gen) / math.sqrt(p.shape[0])).clamp(min=0))


def _plant_dense(q, slots, p, gen, c0, step):
    """queue rows at `slots` with cosines c0, c0 + step, ... to p (before bf16 rounding), in column order: each later column beats the
    row's running k-th by a hair, so the p~-space candidate filter must not round its threshold up."""
    pu = _unit(p)
    for j, s in enumerate(slots):
        u = torch.randn(p.shape[0], generator=gen, dtype=torch.float64)
        u = _unit(u - (u @ pu.double()) * pu.double())
        cj = c0 + step * j
        q[s] = _unit((cj * pu.double() + math.sqrt(1.0 - cj * cj) * u).float())


def _plant_ladder(q, p, gen, first_slot, n_steps, gap):
    """A ladder of hard negatives for a top-1 row: bf16-exact queue rows whose cosines to bf16(p) rise by `gap` from one column to the
    next, in column order, each one beating the running top-1 by less than a bf16 step of p~ (2^-8 relative: 2^-8 / s in cosine).
    The p~-space candidate filter must round its threshold down, or it skips some of them -- and the last one is the row's answer."""
    pb = p.to(torch.bfloat16).double()
    base = _unit(p)
    cand = _unit(base.unsqueeze(0) + 0.2 * torch.randn(4000, p.shape[0], generator=gen) / math.sqrt(p.shape[0])).to(torch.bfloat16)
    cos = cand.double() @ pb
    order = torch.argsort(cos)
    picked, last = [], -2.0
    for j in order[len(order) // 2:].tolist():      # from the median up, where the candidates are dense
        if float(cos[j]) >= last + gap:
            picked.append(j)
            last = float(cos[j])
        if len(picked) == n_steps:
            break
    for t, j in enumerate(picked):
        q[first_slot + 37 * t] = cand[j].float()
    return [first_slot + 37 * t for t in range(len(picked))]


def _case(name):
    """(params, p [n, D] fp32, queue [2, Q, D] fp32, label [n], ones list, planted outlier rows)."""
    gen = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    c = dict(CASES[name])
    D, Q, n = c['D'], c['Q'], c['n']
    q = _unit(torch.rand(2, Q, D, generator=gen))                     # ffc.py:29-30: all-positive unit rows
    p = _unit(torch.randn(n, D, generator=gen))
    label = torch.randint(0, Q, (n,), generator=gen)
    edges = [s for s in (0, 31, 32, 127, 128, Q - 1) if s < Q]
    ones = []
    if c['n_ones']:
        rest = [s for s in torch.randperm(Q, generator=gen).tolist() if s not in edges]
        ones = ([e for e in edges if not (c.get('last_col_main') and e == Q - 1)] + rest)[:c['n_ones']]
        ones = ones[len(ones) // 2:] + ones[:len(ones) // 2]            # list order is not slot order
    planted = []
    out = c.get('outliers', [])
    for i in out:
        label[i] = -1
    if c.get('tail_outliers'):
        label[n - c['tail_outliers']:] = -1
    pos = [i for i in range(n) if label[i] >= 0]
    # targets at the tile / word edges, inside `ones` and outside, and several rows sharing one target
    tg = edges + [s + 1 for s in edges if s + 1 < Q and s + 1 not in ones]
    for i, s in zip(pos[:len(tg)], tg):
        label[i] = s
    for i in pos[len(tg):len(tg) + 4]:
        label[i] = tg[-1]
    if ones:
        for i, s in zip(pos[len(tg) + 4:len(tg) + 10], ones[-6:]):   # targets deep in the list: past the first side tile when n_ones > 128
            label[i] = s
    # probe rows near their target: large target cosines (Arc clamp when equal, SV's gt > margin branch)
    for i in pos[len(tg) + 10:len(tg) + 16]:
        p[i] = _unit(q[0, label[i]] + 0.3 * torch.randn(D, generator=gen) / math.sqrt(D))
    if (out or c.get('tail_outliers')) and not c.get('ladders'):
        outl = [i for i in range(n) if label[i] < 0]
        k = c['k']
        # planted hard negatives straddling the k-th across column chunks (slots spread over the whole queue)
        if len(outl) >= 1:
            r = outl[0]
            slots = [s for s in torch.linspace(1, Q - 2, 2 * k + 2).long().tolist() if s not in ones]
            _plant_near(q[0], slots, p[r], gen, 0.4)
            planted.append(r)
        # exact duplicate queue rows among the planted: their cosines tie exactly
        if len(outl) >= 2 and Q > 64:
            r = outl[1]
            main = [s for s in range(2, Q - 1) if s not in ones]
            a = main[len(main) // 3]
            _plant_near(q[0], [a], p[r], gen, 0.2)
            for b in main[len(main) // 3 + 1:len(main) // 3 + 1 + k]:
                q[:, b] = q[:, a]
            planted.append(r)
        # hard negatives that exist only under queue[1] of `ones` slots: loss 1 and loss 2 select different sets
        if len(outl) >= 3 and ones:
            r = outl[2]
            _plant_near(q[1], ones[-min(len(ones), k + 2):], p[r], gen, 0.3)
            planted.append(r)
        # a row whose cosines are all negative: empty lists, zero loss term, zero gradient row
        if len(outl) >= 4:
            r = outl[3]
            p[r] = -_unit(q.reshape(-1, D).mean(0))
            planted.append(r)
            c['neg_row'] = r
        # hard negatives denser than one bf16 step of p~ above the running k-th, met one after another (positive probe: its planted
        # rows stay on the positive side of the queue's mean, away from the all-negative row)
        if len(outl) >= 5 and Q > 4 * k + 8:
            r = outl[4]
            p[r] = _unit(torch.randn(D, generator=gen).abs())
            slots = [s for s in torch.linspace(3, Q - 3, 4 * k).long().tolist() if s not in ones]
            _plant_dense(q[0], slots, p[r], gen, 0.95, 2e-5)
            planted.append(r)
        # k + 1 hard negatives on `ones` slots of queue[0] above every main cosine, and k on other `ones` slots of queue[1] between the
        # main k-th and those: loss 1's list is main + side 0, loss 2's main + side 1, so side 0's k-th must not cut side 1's list
        if len(outl) >= 6 and len(ones) >= 2 * k + 1:
            r = outl[5]
            _plant_near(q[0], ones[:k + 1], p[r], gen, 0.2)
            _plant_near(q[1], ones[k + 1:2 * k + 1], p[r], gen, 1.0)
            planted.append(r)
        # the last column of a ragged queue as a live main column: a row's top hard negative, and the dominant term of a positive row
        if c.get('last_col_main') and len(outl) >= 7:
            r = outl[6]
            _plant_near(q[0], [Q - 1], p[r], gen, 0.1)
            planted.append(r)
            i = next(i for i in pos[len(tg) + 16:] if label[i] != Q - 1)
            p[i] = _unit(q[0, Q - 1] + 0.3 * torch.randn(D, generator=gen) / math.sqrt(D))
    q = _unit(q)
    if c.get('ladders'):       # after the normalisation: the rungs are bf16-exact rows whose cosines were chosen on those bits
        outl = [i for i in range(n) if label[i] < 0]
        for t, r in enumerate(outl):
            _plant_ladder(q[0], p[r], gen, 1 + 5 * t, 24, 1.5 * 2.0 ** -8 / c['scale'] / 4)
            planted.append(r)
    if c.get('clamp_row') and len(pos) > len(tg) + 16:
        i = pos[len(tg) + 16]
        p[i] = q[0, label[i]] * (1.0 + 2.0 ** -7)                     # cos_t > 1 after rounding: finalize's clamp to 1 - 1e-6
    return c, p, q, label.to(torch.int32), ones, planted


# name -> D, Q, rows, loss, scale, margin, k, n_ones (+ max_rows, outlier rows, ...)
CASES = {
    # ragged rows (129), `ones` on the word / tile edges and beyond one side tile, targets on the edges, scale 64
    'am_d128_edges': dict(D=128, Q=4097, n=129, loss='AM', scale=64.0, margin=0.35, k=5, n_ones=206, max_rows=256, outliers=[3, 40, 41, 77, 100], tail_outliers=1),
    # n_ones > roundup128(n_rows): side rows past the prep grid (rows 128..299)
    'am_d512_two_rows_300_ones': dict(D=512, Q=4097, n=2, loss='AM', scale=32.0, margin=0.35, k=4, n_ones=300, max_rows=384, outliers=[1]),
    'arc_d256_q65569': dict(D=256, Q=65536 + 33, n=127, loss='Arc', scale=64.0, margin=0.5, k=10, n_ones=300, max_rows=320,
                            outliers=[5, 6, 7, 8, 100], clamp_row=True),
    'sv_d128': dict(D=128, Q=4097, n=129, loss='SV', scale=64.0, margin=0.35, k=5, n_ones=150, max_rows=160, outliers=[2, 50, 51, 52, 100, 101]),
    # the pair kernel's ragged tail with a live last main column (Q = 39 x 128 + 8), SV's separate side launches on the pair kernel
    'sv_d512_ragged': dict(D=512, Q=5000, n=130, loss='SV', scale=32.0, margin=0.35, k=4, n_ones=40, outliers=[1, 2, 3, 4, 60, 61, 62],
                           last_col_main=True),
    'sv_d256_scale32': dict(D=256, Q=6000, n=200, loss='SV', scale=32.0, margin=0.2, k=3, n_ones=40, outliers=[0, 1, 2, 3, 199]),
    # below one column tile, no `ones` (NULL cmask: side items without columns), the largest AM / Arc scale
    'arc_d64_q97_scale77': dict(D=64, Q=97, n=127, loss='Arc', scale=77.0, margin=0.5, k=3, n_ones=0, outliers=[1, 2, 3, 4, 60], clamp_row=True),
    'am_d64_q97_one_row': dict(D=64, Q=97, n=1, loss='AM', scale=64.0, margin=0.35, k=3, n_ones=0),
    # top-1 rows climbing ladders of hard negatives closer than one bf16 step of p~: one such row per warp of a positive row tile
    'am_d64_top1_ladders': dict(D=64, Q=4097, n=512, loss='AM', scale=32.0, margin=0.35, k=1, n_ones=0, outliers=list(range(5, 512, 32)),
                                ladders=True),
    # many column chunks
    'am_d512_q262144': dict(D=512, Q=262144, n=1000, loss='AM', scale=32.0, margin=0.35, k=10, n_ones=64, outliers=list(range(0, 1000, 8))),
    # the 8-way shard shape: 8192 rows, 7/8 of them hard-negative-only (whole row tiles), several waves: row map and seeded lists
    'arc_d512_8way': dict(D=512, Q=131072, n=8192, loss='Arc', scale=32.0, margin=0.5, k=10, n_ones=1000, tail_outliers=7168, outliers=[5, 700]),
}


def _kernel_of(D):
    return 'pair' if D == 512 or os.environ.get('FFC_SWEEP_PAIR', '0') not in ('', '0') else 'one'


def _cmask(ones, Q, dev):
    words = np.zeros(((Q + 127) // 128) * 4 + 4, dtype=np.uint32)
    for s in ones:
        words[s >> 5] |= np.uint32(1 << (s & 31))
    return torch.from_numpy(words.view(np.int32)).to(dev)


def _run(c, p, q, label, ones):
    from ffc_b200 import _capi
    from ffc_b200._capi import HeadConfig, HeadPass, HeadStats, check
    lib = _capi.lib()
    dev = torch.device('cuda')
    D, Q, n, k = c['D'], c['Q'], c['n'], c['k']
    max_rows = c.get('max_rows', n)
    cfg = HeadConfig(max_rows, Q, Q, 0, D, _capi.LOSS_TYPES[c['loss']], c['scale'], c['margin'], k, 0)
    h = C.c_void_p()
    check(lib.ffc_head_create(C.byref(cfg), C.byref(h)))
    try:
        s = torch.cuda.current_stream().cuda_stream
        qd = q.to(dev).contiguous()
        mirror = torch.empty(2, Q, D, dtype=torch.bfloat16, device=dev)
        check(lib.ffc_cast_bf16(qd.data_ptr(), mirror.data_ptr(), 2 * Q * D, s))
        assert torch.equal(mirror, qd.to(torch.bfloat16))               # the reference's W is the mirror, bit for bit
        pd, lab = p.to(dev).contiguous(), label.to(dev)
        ones_d = torch.full((max_rows,), -1, dtype=torch.int32, device=dev)
        if ones:
            ones_d[:len(ones)] = torch.tensor(ones, dtype=torch.int32)
        n_ones = torch.tensor([len(ones)], dtype=torch.int32, device=dev)
        cm = _cmask(ones, Q, dev) if ones else None
        hp = HeadPass(pd.data_ptr(), qd.data_ptr(), mirror.data_ptr(), lab.data_ptr(), ones_d.data_ptr(), n_ones.data_ptr(),
                      cm.data_ptr() if cm is not None else None, n)
        st = dict(lsum=torch.zeros(4, n, device=dev), osum=torch.zeros(4, n, D, device=dev), tgt=torch.zeros(4, n, device=dev),
                  topv=torch.zeros(3, n, k, device=dev), topi=torch.zeros(3, n, k, dtype=torch.int32, device=dev))
        hs = HeadStats(*(st[nm].data_ptr() for nm in ('lsum', 'osum', 'tgt', 'topv', 'topi')))
        check(lib.ffc_head_sweep(h, C.byref(hp), C.byref(hs), s))
        scratch = dict(lsum=torch.zeros(4, n, device=dev), osum=torch.zeros(4, n, D, device=dev), tgt=torch.zeros(4, n, device=dev),
                       topv=torch.zeros(3, n, k, device=dev), topi=torch.zeros(3, n, k, dtype=torch.int32, device=dev))
        hs2 = HeadStats(*(scratch[nm].data_ptr() for nm in ('lsum', 'osum', 'tgt', 'topv', 'topi')))
        loss = torch.zeros((), device=dev)
        dp = torch.zeros(n, D, device=dev)
        check(lib.ffc_head_pass_single(h, C.byref(hp), C.byref(hs2), loss.data_ptr(), dp.data_ptr(), s))
        torch.cuda.synchronize()
        return {**{nm: t.cpu() for nm, t in st.items()}, 'loss': float(loss), 'dp': dp.double(), 'mirror': mirror, 'p': pd}
    finally:
        lib.ffc_head_destroy(h)


def _ulp(x):
    a = x.abs().float().clamp(min=2.0 ** -126)
    return (torch.nextafter(a, torch.tensor(math.inf)) - a).double()


@pytest.mark.parametrize('name', list(CASES))
def test_sweep_rows(name):
    c, p, q, label, ones, planted = _case(name)
    D, Q, n, k, s = c['D'], c['Q'], c['n'], c['k'], c['scale']
    got = _run(c, p, q, label, ones)
    dev = torch.device('cuda')
    is_out = label < 0
    pos = ~is_out
    report = {}

    # target cosines: fp64 sums of the bf16 products, rounded once to fp32 by the kernel
    ref0 = SweepRef(got['p'], got['mirror'], label.to(dev), ones, c['loss'], s, c['margin'], k)
    tgt_ref = ref0.tgt().cpu()
    err = (got['tgt'].double() - tgt_ref).abs()
    assert bool((err[:2] <= _ulp(tgt_ref[:2])).all()), ('tgt', float(err.max()))
    assert torch.equal(got['tgt'][2:], tgt_ref[2:].float())
    report['tgt_ulps'] = float((err[:2] / _ulp(tgt_ref[:2])).max())

    delta = D * U * 1.02
    thr = sv_thresholds(got['tgt'], c['margin']) if c['loss'] == 'SV' else None
    ref = SweepRef(got['p'], got['mirror'], label.to(dev), ones, c['loss'], s, c['margin'], k, thr=thr)
    lsum_r, osum_r = (t.cpu() for t in ref.stats())
    amb, absO = (t.cpu() for t in ref.abs_osum_and_ambiguous(delta))

    # softmax denominators of the positive rows (slot 1 only for SV; slots 2 / 3 zero without `ones`)
    M = ref.M
    depth = 64 + -(-Q // 128)
    rel = s * 4 * math.sqrt(D) * U + (s + M) * math.log2(math.e) * U * math.log(2) + 2.0 ** -21 + 4 * math.sqrt(depth) * U
    slots = [0, 1, 2, 3] if c['loss'] == 'SV' else [0, 2, 3]
    for sl in slots:
        e = (got['lsum'][sl].double() - lsum_r[sl]).abs()[pos]
        tol = rel * lsum_r[sl][pos] + amb[sl][pos] + 1e-30
        assert bool((e <= tol).all()), ('lsum', sl, int(torch.nonzero(pos)[int(torch.argmax(e / tol))]), float((e / tol).max()))
        report[f'lsum{sl}'] = float((e / tol).max()) if e.numel() else 0.0
        # The per-row tolerance against the effect of one column with p~ = 1e-3 L (L: the row's whole denominator), over the rows without
        # SV columns within delta_D of the threshold (there the tolerance holds both classifications of such a column).  The aim is 0.1;
        # the cosine term s 4 sqrt(D) u alone exceeds 1e-4 once s sqrt(D) > 417 -- every case at scale 64 / 77 from D = 64 up and at
        # scale 32 from D = 256 up -- and there the bound resolves a column of p~ >= 3e-4 L instead (ratio <= 0.3).
        sure = pos & (amb[sl] == 0)
        ratio = (rel * lsum_r[sl] / (1e-3 * (lsum_r[0] + lsum_r[2] + lsum_r[3])))[sure]
        rule = 0.1 if s * math.sqrt(D) <= 417 else 0.3
        report[f'lsum{sl}_tol_over_1e-3L'] = float(ratio.max()) if ratio.numel() else 0.0
        assert report[f'lsum{sl}_tol_over_1e-3L'] <= rule, ('lsum tolerance against one column', sl, report[f'lsum{sl}_tol_over_1e-3L'], rule)
    # O sums: positive rows within the p~ rounding bound, hard-negative-only rows exactly zero
    for sl in slots:
        e = (got['osum'][sl].double() - osum_r[sl]).abs()[pos]
        tol = (2.0 ** -8 + rel) * absO[sl][pos] + amb[sl][pos].unsqueeze(1) * 1.2 + 1e-30
        assert bool((e <= tol).all()), ('osum', sl, float((e / tol).max()))
        report[f'osum{sl}'] = float((e / tol).max()) if e.numel() else 0.0
        assert bool((got['osum'][sl][is_out] == 0).all())

    # top-k lists: positive rows empty, hard-negative-only rows judged per set
    assert bool((got['topi'][:, pos] == -1).all()) and bool((got['topv'][:, pos] == -math.inf).all())
    out_rows = torch.nonzero(is_out).flatten().tolist()
    judged = planted + [r for r in out_rows[::max(1, len(out_rows) // JUDGE_ROWS)] if r not in planted]
    for r0 in range(0, len(judged), 256):
        rows = judged[r0:r0 + 256]
        for which in range(3):
            cos = ref.set_cosines(rows, which).cpu()
            for j, i in enumerate(rows):
                bad = judge_topk(got['topv'][which, i], got['topi'][which, i], cos[j], k, delta)
                assert not bad, (name, 'row', i, 'set', which, bad[:4])
    assert bool((got['topi'][:, is_out] >= -1).all())        # no seed marker (-2) leaks into any reported list

    # dLoss/dp per row: positive rows from the statistics' bounds, hard-negative-only rows from the kernel's accepted slots
    tgt_k = got['tgt'].double().to(dev)
    dp_ref = ref.dp_positive(*(t.to(dev) for t in ref.stats()), tgt_k).cpu()
    _, cO, cT, L = (t.cpu() for t in ref.positive_rows(ref.stats()[0], tgt_k))
    Wt = ref.W0[label.clamp(min=0).long().to(dev)].cpu()
    tpos = ref.tpos.cpu()
    W1t = torch.where((tpos >= 0).unsqueeze(1), ref.W1[label.clamp(min=0).long().to(dev)].cpu(), Wt)
    o1, ab1 = (osum_r[1], absO[1]) if c['loss'] == 'SV' else (osum_r[0], absO[0])
    # finalize: dp = sum_l cO_l (O_common + O_side,l) + cT_l W_l[t], cO = s / (L n_pos), cT = s (e_t / L - 1) f'(c_t) / n_pos.  A relative
    # error r of L moves cO by r cO and cT by r (|cT| + cO L |f'|); its fp32 scalar part adds 2^-16
    dft = [ref.margin_fn(tgt_k[l]).__getitem__(1).abs().cpu() for l in range(2)]
    tol = torch.zeros(n, D, dtype=torch.float64)
    for l, (oc, osd, ac, asd, w) in enumerate(((osum_r[0], osum_r[2], absO[0], absO[2], Wt), (o1, osum_r[3], ab1, absO[3], W1t))):
        cl = 1 if (l == 1 and c['loss'] == 'SV') else 0
        amb_l = amb[cl] + amb[2 + l]
        rL = (rel + 2.0 ** -16 + amb_l / L[l]).unsqueeze(1)
        tol += cO[l].unsqueeze(1) * ((2.0 ** -8 + rel) * (ac + asd) + 1.2 * amb_l.unsqueeze(1))
        tol += rL * (cO[l].abs().unsqueeze(1) * (oc + osd).abs() + (cT[l].abs() + cO[l].abs() * L[l] * dft[l]).unsqueeze(1) * w.abs())
    e = (got['dp'].cpu() - dp_ref).abs()
    assert bool((e[pos] <= tol[pos] + 1e-30).all()), ('dp positive', float((e[pos] / (tol[pos] + 1e-30)).max()))
    report['dp_pos'] = float((e[pos] / (tol[pos] + 1e-30)).max()) if bool(pos.any()) else 0.0
    merged = ref.merged_hard_negatives(got['topv'], got['topi'])
    dpo = ref.dp_outlier(merged).cpu()
    n_out = int(is_out.sum())
    if n_out:
        # 2k fp32 terms of size <= 1 / (n_out k) summed in order, and the fp32 weight itself
        tol_o = (2 * k + 2) * U * 2 * k / (n_out * k) * 1.01
        eo = (got['dp'].cpu() - dpo).abs()[is_out]
        assert float(eo.max()) <= tol_o, ('dp outlier', float(eo.max()), tol_o)
        report['dp_out'] = float(eo.max()) / tol_o
    if 'neg_row' in c:            # the all-negative row: no list, no loss term, zero gradient
        r = c['neg_row']
        assert bool((got['topi'][:, r] == -1).all()) and bool((got['dp'][r] == 0).all())

    # the pass's loss against the fp64 reconstruction (reference statistics, exact top-k)
    want = ref.loss(lsum_r.to(dev), tgt_ref.to(dev))
    report['loss_rel'] = abs(got['loss'] - want) / abs(want)
    assert report['loss_rel'] <= 1e-4, (got['loss'], want)
    print(f'\n{name} [{_kernel_of(D)}] ' + ' '.join(f'{kk}={v:.3g}' for kk, v in report.items()))
    if DUMP:
        torch.save({nm: got[nm] for nm in ('tgt', 'topv', 'topi')}, os.path.join(DUMP, f'{name}.pt'))


VARIANTS = {
    'default': {},
    'one_pair': dict(FFC_SWEEP_PAIRS='1'),
    'two_pairs_three_chunks_rowmap': dict(FFC_SWEEP_PAIRS='2', FFC_SWEEP_CHUNKS='3', FFC_SWEEP_ROWMAP='1'),
    'rowmap': dict(FFC_SWEEP_ROWMAP='1'),
    'no_seed': dict(FFC_SWEEP_NO_SEED='1'),
    'pair_kernel': dict(FFC_SWEEP_PAIR='1'),
}


def _variant_run(tag, env, out_dir):
    d = os.path.join(out_dir, tag)
    os.makedirs(d, exist_ok=True)
    r = subprocess.run([sys.executable, '-m', 'pytest', '-q', '-x', '-s', '-p', 'no:cacheprovider', os.path.join('tests', 'test_gpu_sweep_rows.py'),
                        '-k', 'test_sweep_rows'], cwd=ROOT, env=dict(os.environ, FFC_SWEEP_ROWS_DUMP=d, **env), capture_output=True, text=True,
                       timeout=1500)
    assert r.returncode == 0, (tag, (r.stdout + r.stderr)[-4000:])
    return d


def _same_kernel(name, env):
    D = CASES[name]['D']
    return D == 512 or 'FFC_SWEEP_PAIR' not in env


def test_launch_variants_agree():
    """Every launch variant is judged against the reference (the subprocess runs test_sweep_rows), and within one kernel the variants
    agree bit for bit on tgt, on the top-k values and on the slots above a list's last value."""
    with tempfile.TemporaryDirectory() as tmp:
        base = _variant_run('default', {}, tmp)
        for tag, env in VARIANTS.items():
            if tag == 'default':
                continue
            d = _variant_run(tag, env, tmp)
            for name in CASES:
                if not _same_kernel(name, env):
                    continue
                a, b = torch.load(os.path.join(base, f'{name}.pt')), torch.load(os.path.join(d, f'{name}.pt'))
                assert torch.equal(a['tgt'], b['tgt']), (tag, name)
                for which in range(3):
                    for i in range(a['topv'].shape[1]):
                        la = list(zip(a['topv'][which, i].tolist(), a['topi'][which, i].tolist()))
                        lb = list(zip(b['topv'][which, i].tolist(), b['topi'][which, i].tolist()))
                        # Which members of a value tied at a list's last place are kept is not fixed: a key orders equal truncated
                        # cosines by column, but the lists carry the truncated value only, and the merges of warpgroup and chunk lists
                        # compare values -- the first-merged member stays, and which warpgroup took which tile depends on the launch
                        # shape (seen with exact duplicate queue rows at the 8-way shape).
                        cut = la[-1][0]
                        assert sorted(v for v, _ in la) == sorted(v for v, _ in lb), (tag, name, which, i, 'topv')
                        assert sorted(x for x in la if x[0] > cut) == sorted(x for x in lb if x[0] > cut), (tag, name, which, i)
