"""world_size-2 gloo test (CPU) of the sharded head's collective choreography (ffc_b200/dist.py).

The per-shard compute is the torch stand-in of tests/cpu_shard_backend.py; the expectation is the dense oracle run
on the concatenated global batch with the sharded bookkeeping (one reference LRU(Q/R) per rank, keys routed by
id mod R, global slot = rank*Q/R + local slot)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from oracle.head_ref import hard_neg_k
from oracle.shard_ref import ShardedOracle


def _worker(rank, world, port, loss_type, ret):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from cpu_shard_backend import CpuShardBackend
        from ffc_b200.dist import ShardedFFCHead
        torch.manual_seed(0)
        D, Q, B, n_ids, steps = 16, {2: 64, 3: 67, 4: 70}[world], 12, 90, 4          # 67 / 3 and 70 / 4: uneven shards (the first Q % R one slot longer)
        margin = 0.5 if loss_type == 'Arc' else 0.4
        q0 = F.normalize(torch.rand(2, Q, D, dtype=torch.float64), dim=2)
        head = ShardedFFCHead(D, Q, 32.0, loss_type, margin, max_batch=B,
                              backend_factory=lambda ql, off, n: CpuShardBackend(D, ql, Q, off, n, 32.0, loss_type, margin, hard_neg_k(Q),
                                                                                 queue=q0[:, off:off + ql]))
        oracle = ShardedOracle(world, D, Q, 32.0, loss_type, margin, queue=q0, dtype=torch.float64)
        gen = torch.Generator().manual_seed(5)
        cen = F.normalize(torch.randn(n_ids, D, generator=gen, dtype=torch.float64))
        for s in range(steps):
            # the same global batch on every rank; each rank feeds its own slice
            xl = torch.randint(0, n_ids, (world * B,), generator=gen)
            yl = torch.cat([xl[:world * B // 2], torch.randint(0, n_ids, (world * B - world * B // 2,), generator=gen)])
            x = F.normalize(cen[xl] + 0.4 * torch.randn(world * B, D, generator=gen, dtype=torch.float64))
            y = F.normalize(cen[yl] + 0.4 * torch.randn(world * B, D, generator=gen, dtype=torch.float64))
            sl = slice(rank * B, (rank + 1) * B)
            xs = x[sl].clone().requires_grad_(True)
            ys = y[sl].clone().requires_grad_(True)
            loss = head.forward(xs, ys, xl[sl], yl[sl])
            loss.backward()
            xo = x.clone().requires_grad_(True)
            yo = y.clone().requires_grad_(True)
            ref = oracle.forward(xo, yo, xl.tolist(), yl.tolist())
            ref.backward()
            assert abs(float(loss) - float(ref)) <= 1e-9 * abs(float(ref)), (s, float(loss), float(ref))
            assert torch.allclose(xs.grad, xo.grad[sl], rtol=1e-8, atol=1e-12), s
            assert torch.allclose(ys.grad, yo.grad[sl], rtol=1e-8, atol=1e-12), s
            # per-shard LRU == reference LRU(Q/R) fed the keys it owns
            assert head.backend.lru.state_dict() == oracle.lrus[rank].state_dict()
            # labels agree with the oracle's global slots
            assert head._last['label'].tolist() == oracle.trace[-1]['labels']
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


def _worker_prefetch(rank, world, port, ret, all_hits=False):
    """prefetch(labels) + forward_pair(x, y) == forward_pair(x, y, labels), step for step (loss, gradients, LRU, queue), including a
    prefetch that is discarded because other labels arrive"""
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from cpu_shard_backend import CpuShardBackend
        from ffc_b200.dist import ShardedFFCHead
        D, Q, B, n_ids, steps = 16, 64, 12, (62 if all_hits else 90), 5
        q0 = F.normalize(torch.rand(2, Q, D, dtype=torch.float64), dim=2)
        mk = lambda: ShardedFFCHead(D, Q, 32.0, 'Arc', 0.5, max_batch=B,
                                    backend_factory=lambda ql, off, n: CpuShardBackend(D, ql, Q, off, n, 32.0, 'Arc', 0.5, hard_neg_k(Q),
                                                                                       queue=q0[:, off:off + ql]))
        plain, pre = mk(), mk()
        if all_hits:        # bench.py's regime: every identity resident (identities <= queue), every gallery key a hit, `ones` = all of them
            plain.prefill_identity(Q), pre.prefill_identity(Q)
        gen = torch.Generator().manual_seed(6)
        cen = F.normalize(torch.randn(n_ids, D, generator=gen, dtype=torch.float64))
        batches = []
        for s in range(steps):
            xl = torch.randint(0, n_ids, (B,), generator=gen)
            yl = torch.cat([xl[:B // 2], torch.randint(0, n_ids, (B - B // 2,), generator=gen)])
            g2 = torch.Generator().manual_seed(100 * s + rank)
            x = F.normalize(cen[xl] + 0.4 * torch.randn(B, D, generator=g2, dtype=torch.float64))
            y = F.normalize(cen[yl] + 0.4 * torch.randn(B, D, generator=g2, dtype=torch.float64))
            batches.append((x, y, xl + rank, yl + rank))       # different labels per rank (< 64 in the all-hit variant)
        pre.prefetch(batches[0][2], batches[0][3])
        for s, (x, y, xl, yl) in enumerate(batches):
            a = plain.forward_pair(x, y, xl, yl)
            if s == 2:      # stale prefetch: labels of another batch were handed over, then this batch arrives with its own
                pre.prefetch(batches[4][2], batches[4][3])
                b = pre.forward_pair(x, y, xl, yl)
            elif s == 3:    # prefetched labels, passed again as the same objects
                b = pre.forward_pair(x, y, xl, yl)
            else:
                b = pre.forward_pair(x, y)
            if s + 1 < steps and s + 1 != 2:
                pre.prefetch(batches[s + 1][2], batches[s + 1][3])
            for u, v in zip(a, b):
                assert torch.equal(u, v), s
            assert plain.backend.lru.state_dict() == pre.backend.lru.state_dict()
            assert plain.backend.qpos == pre.backend.qpos and torch.equal(plain.backend.queue, pre.backend.queue)
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


def _worker_resume(rank, world, port, ret):
    """ShardedFFCHead.checkpoint() / load_checkpoint(): a head resumed from the per-rank snapshot continues exactly like the original
    (through torch.save / torch.load, i.e. the file a trainer would write)"""
    import io
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from cpu_shard_backend import CpuShardBackend
        from ffc_b200.dist import ShardedFFCHead
        D, Q, B, n_ids = 16, 64, 12, 90
        q0 = F.normalize(torch.rand(2, Q, D, dtype=torch.float64, generator=torch.Generator().manual_seed(3)), dim=2)
        mk = lambda q: ShardedFFCHead(D, Q, 32.0, 'AM', 0.4, max_batch=B,
                                      backend_factory=lambda ql, off, n: CpuShardBackend(D, ql, Q, off, n, 32.0, 'AM', 0.4, hard_neg_k(Q),
                                                                                         queue=q[:, off:off + ql]))
        gen = torch.Generator().manual_seed(11 + rank)
        cen = F.normalize(torch.randn(n_ids, D, generator=torch.Generator().manual_seed(12), dtype=torch.float64))

        def batch():
            xl = torch.randint(0, n_ids, (B,), generator=gen)
            yl = torch.cat([xl[:B // 2], torch.randint(0, n_ids, (B - B // 2,), generator=gen)])
            return (F.normalize(cen[xl] + 0.4 * torch.randn(B, D, generator=gen, dtype=torch.float64)),
                    F.normalize(cen[yl] + 0.4 * torch.randn(B, D, generator=gen, dtype=torch.float64)), xl, yl)
        a = mk(q0)
        for _ in range(3):
            a.forward_pair(*batch())
        a.prefetch(*batch()[2:])                     # a pending prefetch must not leak into the snapshot
        buf = io.BytesIO()
        torch.save(a.checkpoint(), buf)
        buf.seek(0)
        ck = torch.load(buf, weights_only=False)
        assert set(ck) == {'lru', 'fc', 'qp', 'shard'} and ck['shard'] == (rank, world, Q) and tuple(ck['fc'].shape) == (2, Q // world, D)
        assert all(0 <= s < Q // world for _, s in ck['lru']) and all(k % world == rank for k, _ in ck['lru'])
        b = mk(torch.zeros_like(q0))                 # wrong queue, empty LRU: everything must come from the snapshot
        b.load_checkpoint(ck)
        for _ in range(2):
            bt = batch()
            ra, rb = a.forward_pair(*bt), b.forward_pair(*bt)
            for u, v in zip(ra, rb):
                assert torch.equal(u, v)
            assert a.backend.lru.state_dict() == b.backend.lru.state_dict() and a.backend.qpos == b.backend.qpos
            assert torch.equal(a.backend.queue, b.backend.queue)
        wrong = dict(ck, shard=((rank + 1) % world, world, Q))
        try:
            b.load_checkpoint(wrong)
            raise RuntimeError('a snapshot of another shard was accepted')
        except AssertionError:
            pass
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


def test_sharded_head_checkpoint_resume_world2_gloo():
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker_resume, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: 'ok', 1: 'ok'}


@pytest.mark.parametrize('all_hits', [False, True])
def test_sharded_head_label_prefetch_world2_gloo(all_hits):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker_prefetch, args=(2, port, ret, all_hits), nprocs=2, join=True)
    assert dict(ret) == {0: 'ok', 1: 'ok'}


def _worker_merged(rank, world, port, loss_type, ret):
    """The product's merged step (ShardedFFCHead._forward_pair_merged: one statistics exchange per step, the rollback pass's finalize
    through the overlay) with the stand-in backend: results must equal the dense oracle, and must NOT without the overlay."""
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from cpu_shard_backend import CpuShardBackendM
        from ffc_b200.dist import ShardedFFCHead
        torch.manual_seed(0)
        # few identities, small queue: in-batch duplicates, evictions, targets and hard negatives inside the rows both passes overwrite
        D, Q, B, n_ids, steps = 16, 32, 12, 40, 6
        margin = 0.5 if loss_type == 'Arc' else 0.4
        q0 = F.normalize(torch.rand(2, Q, D, dtype=torch.float64), dim=2)
        mk = lambda ov: ShardedFFCHead(D, Q, 32.0, loss_type, margin, max_batch=B,
                                       backend_factory=lambda ql, off, n: CpuShardBackendM(D, ql, Q, off, n, 32.0, loss_type, margin, hard_neg_k(Q),
                                                                                           queue=q0[:, off:off + ql], use_overlay=ov))
        head, naive = mk(True), mk(False)
        assert head.merged and naive.merged
        oracle = ShardedOracle(world, D, Q, 32.0, loss_type, margin, queue=q0, dtype=torch.float64)
        gen = torch.Generator().manual_seed(9)
        cen = F.normalize(torch.randn(n_ids, D, generator=gen, dtype=torch.float64))
        naive_wrong = 0
        for s in range(steps):
            xl = torch.randint(0, n_ids, (world * B,), generator=gen)
            yl = torch.cat([xl[:world * B // 2], torch.randint(0, n_ids, (world * B - world * B // 2,), generator=gen)])
            x = F.normalize(cen[xl] + 0.4 * torch.randn(world * B, D, generator=gen, dtype=torch.float64))
            y = F.normalize(cen[yl] + 0.4 * torch.randn(world * B, D, generator=gen, dtype=torch.float64))
            sl = slice(rank * B, (rank + 1) * B)
            if s % 2:        # labels handed over one step ahead: the rollback bookkeeping lands in the OTHER rollback set (0 / 2 alternate)
                head.prefetch(xl[sl], yl[sl])
                loss, dx, dy = head.forward_pair(x[sl], y[sl])
            else:
                loss, dx, dy = head.forward_pair(x[sl], y[sl], xl[sl], yl[sl])
            _, dx_n, dy_n = naive.forward_pair(x[sl], y[sl], xl[sl], yl[sl])
            xo, yo = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
            ref = oracle.forward(xo, yo, xl.tolist(), yl.tolist())
            ref.backward()
            assert abs(float(loss) - float(ref)) <= 1e-9 * abs(float(ref)), (s, float(loss), float(ref))
            assert torch.allclose(dx, xo.grad[sl], rtol=1e-8, atol=1e-12), s
            assert torch.allclose(dy, yo.grad[sl], rtol=1e-8, atol=1e-12), s
            assert head.backend.lru.state_dict() == oracle.lrus[rank].state_dict()
            assert torch.allclose(head.backend.queue, oracle.queue[:, head.off:head.off + head.Ql].double(), atol=0, rtol=0)
            naive_wrong += int(not torch.allclose(dx_n, xo.grad[sl], rtol=1e-8, atol=1e-12))
        t = torch.tensor([naive_wrong, head.backend.overlay_reads, head.prefetch_hits])
        dist.all_reduce(t)
        assert int(t[0]) > 0 and int(t[1]) > 0 and int(t[2]) == world * (steps // 2), t.tolist()       # the overlay was needed, and it was read
        assert head.barrier_timeouts() == 0            # (no in-kernel barriers on the CPU stand-in: the counter exists and reads 0)
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,loss_type', [(2, 'Arc'), (2, 'AM'), (3, 'Arc')])
def test_merged_step_one_exchange_gloo(world, loss_type):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker_merged, args=(world, port, loss_type, ret), nprocs=world, join=True)
    assert dict(ret) == {r: 'ok' for r in range(world)}


def _run(world, loss_type):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, loss_type, ret), nprocs=world, join=True)
    assert dict(ret) == {r: 'ok' for r in range(world)}


@pytest.mark.parametrize('loss_type', ['AM', 'Arc', 'SV'])
def test_sharded_head_world2_gloo(loss_type):
    _run(2, loss_type)


@pytest.mark.parametrize('world,loss_type', [(3, 'Arc'), (4, 'SV')])
def test_sharded_head_more_ranks_gloo(world, loss_type):
    """3 ranks (queue 67) and 4 ranks (queue 70) -- queue sizes the rank count does not divide: candidate sets of several ranks merged per
    outlier row, target cosines owned by any of them"""
    _run(world, loss_type)
