"""NCCL worker for tests/test_gpu_dist.py: R ranks, one GPU each, sharded head vs the sharded oracle."""
import os
import sys

import torch
import torch.distributed as dist
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'very-large-scale-face-recognition_b200'), os.path.join(ROOT, 'tests')]


def main():
    from ffc_b200.dist import ShardedFFCHead
    from oracle.shard_ref import ShardedOracle
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    routes = set()
    if os.environ.get('DIST_DBG_POISON'):      # debug aid: NaN bit patterns in the caching allocator's free blocks (reads of unwritten memory show up)
        junk = [torch.full((sz,), float('nan'), device=dev) for sz in (1 << 24, 1 << 20, 1 << 16, 1 << 12, 256, 16) for _ in range(6)]
        torch.cuda.synchronize()
        del junk
    if os.environ.get('DIST_DBG_PAD'):
        keep = torch.empty(int(os.environ['DIST_DBG_PAD']), device=dev)
    for precision, tol, D, Q, B, n_ids, loss_type, margin in (('bf16', 1e-2, 128, 1024, 96, 1500, 'Arc', 0.5),
                                                               ('fp32', 1e-5, 64, 512, 40, 700, 'AM', 0.4),
                                                               ('bf16', 1e-2, 512, 4096, 128, 4096, 'AM', 0.4),
                                                               ('bf16', 1e-2, 128, 7409, 64, 9000, 'Arc', 0.5),      # ffc.py:11's default queue_size: uneven shards
                                                               ('bf16', 1e-2, 128, 1024, 96, 1500, 'SV', 0.4),
                                                               ('fp32', 1e-5, 64, 512, 40, 700, 'SV', 0.4)):
        torch.manual_seed(0)
        q0 = F.normalize(torch.rand(2, Q, D), dim=2)
        head = ShardedFFCHead(D, Q, 32.0, loss_type, margin, precision=precision, max_batch=B, device=dev)
        head.backend.set_queue(q0[:, head.off:head.off + head.Ql])
        oracle = ShardedOracle(world, D, Q, 32.0, loss_type, margin, queue=q0, dtype=torch.float64)
        gen = torch.Generator().manual_seed(5)
        cen = F.normalize(torch.randn(n_ids, D, generator=gen))
        for s in range(6):
            n = world * B
            xl = torch.randint(0, n_ids, (n,), generator=gen)
            yl = torch.cat([xl[:n // 2], torch.randint(0, n_ids, (n - n // 2,), generator=gen)])
            x = F.normalize(cen[xl] + 0.7 * torch.randn(n, D, generator=gen))
            y = F.normalize(cen[yl] + 0.7 * torch.randn(n, D, generator=gen))
            sl = slice(rank * B, (rank + 1) * B)
            xs = x[sl].to(dev).requires_grad_(True)
            ys = y[sl].to(dev).requires_grad_(True)
            if s == 2:      # the two-pass entry used by bench.py, fed through the staging views: the backbone tail (csrc/tail.cu,
                # l2_normalize with out=) writes the unit-norm rows straight into the packed all-gather input -- no [B, D] copy
                from ffc_b200 import l2_normalize
                sx, sy = head.staging()
                px = l2_normalize(xs.detach() * 3.0, out=sx)          # any positive row scale: the tail normalises
                py = l2_normalize(ys.detach() * 0.5, out=sy)
                assert px.data_ptr() == sx.data_ptr() and py.data_ptr() == sy.data_ptr()
                loss, gx, gy = head.forward_pair(px, py, xl[sl], yl[sl])
                xs.grad, ys.grad = gx, gy
            elif s == 3:    # labels handed over early (CPU tensors): the rollback bookkeeping runs on the bookkeeping stream
                head.prefetch(xl[sl], yl[sl])
                assert head._pre is not None and head.prefetch_hits == 0
                loss, gx, gy = head.forward_pair(xs.detach(), ys.detach())
                assert head.prefetch_hits == 1
                xs.grad, ys.grad = gx, gy
            elif s == 4:    # a stale prefetch (other labels) is discarded without a trace, then the same objects are accepted
                mine = (xl[sl], yl[sl])
                head.prefetch(yl[sl].clone(), xl[sl].clone())
                head.prefetch(*mine)
                loss, gx, gy = head.forward_pair(xs.detach(), ys.detach(), *mine)
                assert head._pre is None and head.prefetch_hits == 2
                xs.grad, ys.grad = gx, gy
            elif s == 5:    # stale prefetch followed by the autograd entry
                head.prefetch(yl[sl].clone(), xl[sl].clone())
                loss = head.forward(xs, ys, xl[sl], yl[sl])
                loss.backward()
                assert head._pre is None and head.prefetch_hits == 2
            else:
                loss = head.forward(xs, ys, xl[sl], yl[sl])
                loss.backward()
            xo, yo = x.double().requires_grad_(True), y.double().requires_grad_(True)
            q_pre = oracle.queue.clone()                    # the queue before this step (the rollback pass sweeps it + its own enqueue)
            ref = oracle.forward(xo, yo, xl.tolist(), yl.tolist())
            ref.backward()
            assert head._last['label'].tolist() == oracle.trace[-1]['labels'], (precision, s, 'labels')
            assert head.backend.lru.state_dict() == oracle.lrus[rank].state_dict(), (precision, s, 'lru')
            # queue positions (ffc.py:41-43) of the shard, and the queue rows themselves (enqueue is a pure copy)
            assert head.backend.qpos.cpu().tolist() == oracle.qpos[head.off:head.off + head.Ql], (precision, s, 'qpos')
            qerr = float((head.backend.queue.cpu().double() - oracle.queue[:, head.off:head.off + head.Ql]).abs().max())
            assert qerr < 1e-6, (precision, s, 'queue', qerr)
            assert abs(float(loss) - float(ref)) <= tol * abs(float(ref)), (precision, s, float(loss), float(ref))
            for name, got, want, pemb, tr in (('dx', xs.grad, xo.grad[sl], x, oracle.trace[-2]), ('dy', ys.grad, yo.grad[sl], y, oracle.trace[-1])):
                got = got.double().cpu()
                row_err = (got - want).norm(dim=1) / (want.norm(dim=1) + 1e-30)
                skip = torch.zeros(B, dtype=torch.bool)
                if precision == 'bf16':
                    # An outlier row's gradient is the mean of its top-k prototype rows (ffc.py:88-90): when the k-th and (k+1)-th
                    # largest cosines are closer than the bf16 operand rounding, either selection is a correct bf16 result but the
                    # row's gradient differs by a whole prototype.  Such rows are left out of the gradient comparison (the loss,
                    # which moves by ~1e-4 only, is still compared).
                    lab = torch.tensor(tr['labels'][rank * B:(rank + 1) * B])
                    for b in torch.nonzero(row_err > 10 * tol).flatten().tolist():
                        assert int(lab[b]) < 0, (precision, s, name, 'positive row off', b, float(row_err[b]))
                        if name == 'dx':            # the queue as it was during the rollback sweep: the pre-step queue + that pass's enqueue
                            Wq = q_pre.clone()
                            for i, (r_, c_) in enumerate(zip(tr['rows'], tr['cols'])):
                                Wq[r_, c_] = y.double()[i]
                        else:                       # the commit pass sweeps the queue it leaves behind
                            Wq = oracle.queue.clone()
                        # a near-tie at the top-k boundary under either loss's weights (loss 2 reads queue[1] on the `ones` slots)
                        W2 = Wq[0].clone()
                        W2[tr['ones']] = Wq[1][tr['ones']]
                        gaps = []
                        for Wl in (Wq[0], W2):
                            top = torch.topk(pemb.double()[rank * B + b] @ Wl.t(), oracle.k + 1).values
                            gaps.append(float(top[-2] - top[-1]))
                        if not min(gaps) < 3e-3:
                            diff = got[b] - want[b]
                            enq = set(zip(tr['rows'], tr['cols']))
                            other = oracle.trace[-1] if name == 'dx' else oracle.trace[-2]
                            enq2 = set(zip(other['rows'], other['cols']))
                            for r_ in (0, 1):
                                proj = Wq[r_] @ diff / (Wq[r_].norm(dim=1) ** 2)
                                t4 = torch.topk(proj.abs(), 3)
                                print(f'[rank {rank}] {name} row {b} queue[{r_}] components: ' + ', '.join(
                                    f'slot {int(j)} ({"this-pass-enq " if (r_, int(j)) in enq else ""}{"other-pass-enq " if (r_, int(j)) in enq2 else ""}{"ones" if int(j) in tr["ones"] else ""}) {float(proj[j]):+.2e}'
                                    for j in t4.indices), flush=True)
                            t0_ = torch.topk(pemb.double()[rank * B + b] @ Wq[0].t(), oracle.k + 1)
                            print(f'[rank {rank}]   top cosines under queue[0] (sweep-time): ' + ', '.join(f'{int(j)}:{float(v):.4f}' for v, j in zip(t0_.values, t0_.indices)) + f'; shard offsets {oracle.offs}', flush=True)
                        assert min(gaps) < 3e-3, (precision, D, Q, loss_type, s, name, 'outlier row off without a near-tie', b, gaps, 'rows off', int((row_err > 10 * tol).sum()))
                        skip[b] = True
                err = float((got[~skip] - want[~skip]).norm() / want[~skip].norm())
                assert err <= tol and int(skip.sum()) <= max(3, B // 16), (precision, s, name, err, int(skip.sum()))
        if precision == 'bf16' and loss_type != 'SV':
            assert os.environ.get('FFC_DIST_NO_MERGE') or (head.merged and head._route is not None)   # one exchange per step, reduce-scatter folded into finalize
            routes.add(head._route['kind'] if head._route else 'per-pass')
            if any(isinstance(r, dict) and 'peer' in r for r in head._stats.values()):
                routes.add('records by peer stores')
        assert head.barrier_timeouts() == 0, 'an in-kernel cross-rank barrier timed out'
        del head
    sharded_checkpoint_resume(rank, world, dev)
    long_run_odd_queue(rank, world, dev)
    dist.barrier()
    if rank == 0:
        print('DIST_GPU_OK', world, 'routes', sorted(routes))
    dist.destroy_process_group()


def sharded_checkpoint_resume(rank, world, dev):
    """ShardedFFCHead.checkpoint() / load_checkpoint() over NCCL: a head resumed from the per-rank snapshot continues bit-identically."""
    import io
    from ffc_b200.dist import ShardedFFCHead
    D, Q, B, N = 128, 4096, 64, 6000
    gen = torch.Generator().manual_seed(40 + rank)

    def batch():
        xl = torch.randint(0, N, (B,), generator=gen)
        yl = torch.cat([xl[:B // 2], torch.randint(0, N, (B - B // 2,), generator=gen)])
        return F.normalize(torch.randn(B, D, generator=gen)).to(dev), F.normalize(torch.randn(B, D, generator=gen)).to(dev), xl, yl
    torch.manual_seed(1)
    a = ShardedFFCHead(D, Q, 32.0, 'Arc', 0.5, max_batch=B, device=dev)
    for _ in range(4):
        a.forward_pair(*batch())
    buf = io.BytesIO()
    torch.save(a.checkpoint(), buf)
    buf.seek(0)
    b = ShardedFFCHead(D, Q, 32.0, 'Arc', 0.5, max_batch=B, device=dev)
    b.load_checkpoint(torch.load(buf, weights_only=False))
    for _ in range(3):
        bt = batch()
        for u, v in zip(a.forward_pair(*bt), b.forward_pair(*bt)):
            assert torch.equal(u, v)
        assert a.backend.lru.state_dict() == b.backend.lru.state_dict() and torch.equal(a.backend.queue, b.backend.queue)


def long_run_odd_queue(rank, world, dev):
    """A queue size that is not a power of two and R*B >= 4096 keys per pass (several chunks of the LRU's resolve CTA in one call, ring
    space reserved per pass): 40 steps with evictions; every rank's LRU stays equal to the oracle's LRU(Q/R) fed the keys it owns."""
    from ffc_b200.dist import ShardedFFCHead
    from oracle.lru_ref import LRU as RefLRU
    D, B = 64, 4096 // world
    Q = 1000 * world
    N = 5 * Q
    torch.manual_seed(2)
    head = ShardedFFCHead(D, Q, 32.0, 'AM', 0.4, max_batch=B, device=dev)
    ref = RefLRU(Q // world)
    gen = torch.Generator().manual_seed(9)
    for s in range(40):
        n = world * B
        xl = torch.randint(0, N, (n,), generator=gen)
        yl = torch.randint(0, N, (n,), generator=gen)
        x = F.normalize(torch.randn(n, D, generator=gen))
        y = F.normalize(torch.randn(n, D, generator=gen))
        sl = slice(rank * B, (rank + 1) * B)
        loss, _, _ = head.forward_pair(x[sl].to(dev), y[sl].to(dev), xl[sl], yl[sl])
        for k in xl.tolist():                       # the commit pass's gallery keys, global batch order; the rollback pass undoes itself
            if k % world == rank:
                ref.get(k)
        if s % 8 == 7:
            assert head.backend.lru.state_dict() == ref.state_dict(), ('odd queue', s)
            assert bool(torch.isfinite(loss))


if __name__ == '__main__':
    main()
