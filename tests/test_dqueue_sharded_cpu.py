"""Queue gradient of the sharded head (ShardedFFCHead(queue_grad=True)) under gloo on the CPU.

The per-shard compute is the fp64 stand-in of tests/cpu_shard_backend.py, extended here by a `dqueue` in closed form from the
shard's reduced statistics (what csrc/head.cu's dQueue kernels compute from finalize's coefficients).  The expectation: rank r's
`dqueue_pass` equals rows [off_r, off_r + Q_r) of oracle.head_ref.dqueue_ref on the global queue as the pass swept it, the gathered
probe rows, global target slots and the union of the ranks' `ones` slots.  Rollback and commit passes, evictions, outlier rows;
AM / Arc / SV; 2 and 3 (uneven) ranks; the per-pass statistics flow and the per-pass record flow."""
import math
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from oracle.head_ref import dqueue_ref, hard_neg_k


def swept_queue(queue_after, tr, g, commit):
    """The global queue as a pass swept it: after a commit pass the oracle's queue is it; a rollback pass has restored its rows
    since, so its (last-writer) enqueue is applied again."""
    if commit:
        return queue_after.clone()
    q = queue_after.clone()
    last = {}
    for i, rc in enumerate(zip(tr['rows'], tr['cols'])):
        last[rc] = i
    for (r, c), i in last.items():
        q[r, c] = g[i].to(q.dtype)
    return q


def shard_dqueue_ref(p_all, g_all, oracle, commit, loss_type, margin, off, ql, scale=32.0):
    tr = oracle.trace[-1]
    q = swept_queue(oracle.queue, tr, g_all, commit)
    _, dq = dqueue_ref(p_all.double(), q.double(), tr['labels'], tr['ones'], loss_type, margin, scale, oracle.k)
    return dq[:, off:off + ql]


class DqueueMixin:
    """`dqueue` of the stand-in: dLoss/dQueue of the shard in closed form, fp64, from the statistics finalize was given (the
    all-reduced denominators and target cosines, the gathered top-k candidates) -- the coefficients csrc/head.cu exports."""

    def enable_dqueue(self):
        self.dq_enabled = True

    def finalize(self, p_all, label, st, n_ranks):
        self._dq_stats = (st, n_ranks)
        return super().finalize(p_all, label, st, n_ranks)

    def dqueue(self, p_all, label, out):
        st, n_ranks = self._dq_stats
        p = p_all.double()
        n, k, s, M, m, T = p.shape[0], self.k, self.scale, self._fixed_max(), self.margin, self.SV_T
        sv = self.loss_type == 'SV'
        tcol, tpos = self._row_info(label)
        is_out = label < 0
        n_pos, n_out = int((~is_out).sum()), int(is_out.sum())
        red = st['red']
        W0, W1 = self.queue[0], self.queue[1]
        in_c = torch.zeros(self.Ql, dtype=torch.bool)
        in_c[torch.tensor(self.ones, dtype=torch.long)] = True
        cos0 = p @ W0.t()
        cosl = (cos0, torch.where(in_c, p @ W1.t(), cos0))            # loss 2 reads queue[1] on `ones`
        c0 = torch.zeros(n, self.Ql, dtype=torch.float64)               # coefficient of p_i in dqueue[0][j] / dqueue[1][j]
        c1 = torch.zeros(n, self.Ql, dtype=torch.float64)
        for i in range(n):
            if is_out[i]:
                continue
            for l in range(2):
                ct = float(red[4 + l, i])
                cs = l if sv else 0
                if self.loss_type == 'AM':
                    ft, dft = ct - m, 1.0
                elif sv:
                    ft, dft = (ct - m if ct > m else ct), 1.0
                else:
                    sn = math.sqrt(1.0 - ct * ct)
                    ft, dft = ct * math.cos(m) - sn * math.sin(m), math.cos(m) + ct * math.sin(m) / sn
                et = math.exp(s * ft - M)
                L = float(red[cs, i] + red[2 + l, i]) + et
                c = cosl[l][i]
                if sv:
                    thr = ct - m if float(red[6, i]) > 0 else math.inf
                    hard = c > thr
                    z, h = torch.where(hard, T * c + T - 1.0, c), torch.where(hard, torch.full_like(c, T), torch.ones_like(c))
                else:
                    z, h = c, torch.ones_like(c)
                gcoef = (s / (n_pos * L)) * torch.exp(s * z - M) * h
                if tcol[i] >= 0:
                    gcoef[tcol[i]] = s * (et / L - 1.0) * dft / n_pos
                if l == 0:
                    c0[i] += gcoef
                else:
                    c0[i] += torch.where(in_c, 0.0, gcoef)
                    c1[i] += torch.where(in_c, gcoef, 0.0)
        dq = torch.stack([c0.t() @ p, c1.t() @ p])
        if n_out:
            wneg = 1.0 / (n_out * k)
            for i in range(n):
                if not is_out[i]:
                    continue
                for l in range(2):
                    cand = []
                    for r in range(n_ranks):
                        for src, setid in ((0, 0), (1, 1 + l)):
                            for q in range(k):
                                v, gi = float(st['topv'][r, setid, i, q]), int(st['topi'][r, setid, i, q])
                                if gi >= 0:
                                    cand.append((v, gi, src))
                    cand.sort(key=lambda t: -t[0])
                    for v, gi, src in cand[:k]:
                        loc = gi - self.off
                        if v >= 0 and 0 <= loc < self.Ql:
                            dq[l if src else 0, loc] += wneg * p[i]
        out.copy_(dq)


def _worker(rank, world, port, loss_type, record_flow, ret):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from cpu_shard_backend import CpuShardBackend, CpuShardBackendM
        from test_dist_cpu import ShardedOracle
        from ffc_b200.dist import ShardedFFCHead
        base = CpuShardBackendM if record_flow else CpuShardBackend
        Backend = type('DqBackend', (DqueueMixin, base), {})
        torch.manual_seed(0)
        D, Q, B, n_ids, steps = 16, {2: 64, 3: 67}[world], 12, 90, 4
        margin = 0.5 if loss_type == 'Arc' else 0.4
        q0 = F.normalize(torch.rand(2, Q, D, dtype=torch.float64), dim=2)
        head = ShardedFFCHead(D, Q, 32.0, loss_type, margin, max_batch=B, queue_grad=True,
                              backend_factory=lambda ql, off, n: Backend(D, ql, Q, off, n, 32.0, loss_type, margin, hard_neg_k(Q),
                                                                         queue=q0[:, off:off + ql]))
        assert head.merged is False and head.dqueue.shape == (2, head.Ql, D)
        oracle = ShardedOracle(world, D, Q, 32.0, loss_type, margin, queue=q0, dtype=torch.float64)
        gen = torch.Generator().manual_seed(5)
        cen = F.normalize(torch.randn(n_ids, D, generator=gen, dtype=torch.float64))
        acc = torch.zeros(2, head.Ql, D, dtype=torch.float64)
        n_out_seen = 0
        for step in range(steps):
            xl = torch.randint(0, n_ids, (world * B,), generator=gen)
            yl = torch.cat([xl[:world * B // 2], torch.randint(0, n_ids, (world * B - world * B // 2,), generator=gen)])
            x = F.normalize(cen[xl] + 0.4 * torch.randn(world * B, D, generator=gen, dtype=torch.float64))
            y = F.normalize(cen[yl] + 0.4 * torch.randn(world * B, D, generator=gen, dtype=torch.float64))
            sl = slice(rank * B, (rank + 1) * B)
            if step % 2 == 0:
                # one pass at a time: the rollback pass's gradient is of the queue it swept, not of the restored one
                for commit, (p, g, pl, gl) in ((False, (x, y, xl, yl)), (True, (y, x, yl, xl))):
                    head.head_pass(p[sl], g[sl], pl[sl], gl[sl], commit)
                    oracle.head_pass(p, g, pl.tolist(), gl.tolist(), commit)
                    ref = shard_dqueue_ref(p, g, oracle, commit, loss_type, margin, head.off, head.Ql)
                    n_out_seen += sum(v < 0 for v in oracle.trace[-1]['labels'])
                    err = float((head.dqueue_pass - ref).abs().max())
                    assert err <= 1e-9 * float(ref.abs().max()), (step, commit, err)
                    acc += ref
            else:
                # both passes of a step through forward_pair: dqueue_pass is the commit pass's, dqueue has both
                head.forward_pair(x[sl], y[sl], xl[sl], yl[sl])
                oracle.head_pass(x, y, xl.tolist(), yl.tolist(), False)
                acc += shard_dqueue_ref(x, y, oracle, False, loss_type, margin, head.off, head.Ql)
                oracle.head_pass(y, x, yl.tolist(), xl.tolist(), True)
                ref = shard_dqueue_ref(y, x, oracle, True, loss_type, margin, head.off, head.Ql)
                acc += ref
                assert float((head.dqueue_pass - ref).abs().max()) <= 1e-9 * float(ref.abs().max()), step
            assert head._last['label'].tolist() == oracle.trace[-1]['labels']
        assert float((head.dqueue - acc).abs().max()) <= 1e-9 * float(acc.abs().max())
        assert n_out_seen > 0                      # outlier rows (hard negatives) were part of it
        head.zero_dqueue()
        assert float(head.dqueue.abs().max()) == 0.0
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


def _run(world, loss_type, record_flow):
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, loss_type, record_flow, ret), nprocs=world, join=True)
    assert dict(ret) == {r: 'ok' for r in range(world)}


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('loss_type', ['AM', 'Arc', 'SV'])
def test_sharded_dqueue_matches_global_reference_gloo(world, loss_type):
    _run(world, loss_type, record_flow=False)


@pytest.mark.parametrize('loss_type', ['AM', 'Arc'])
def test_sharded_dqueue_record_flow_gloo(loss_type):
    """a backend that speaks the merged-step protocol (bf16 AM / Arc on the GPU) runs the per-pass record flow with queue_grad"""
    _run(2, loss_type, record_flow=True)


def test_sharded_default_keeps_merged_flow_gloo():
    """without queue_grad nothing changes: the merged flow is selected and no gradient buffers exist"""
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from cpu_shard_backend import CpuShardBackendM
    from ffc_b200.dist import ShardedFFCHead
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=0, world_size=1)
    try:
        D, Q = 16, 64
        head = ShardedFFCHead(D, Q, 32.0, 'AM', 0.4, max_batch=8,
                              backend_factory=lambda ql, off, n: CpuShardBackendM(D, ql, Q, off, n, 32.0, 'AM', 0.4, hard_neg_k(Q)))
        assert head.merged is True and head.queue_grad is False
        assert head.dqueue is None and head.dqueue_pass is None
        head.zero_dqueue()
    finally:
        dist.destroy_process_group()
