"""Queue gradient (queue_grad=True) for every head configuration: the check mode (fp32, fp64-accumulated SIMT kernels) for AM / Arc /
SV, the SV mode of the bf16 swapped tcgen05 sweep, and column shards -- emulated on one GPU with one CudaShardBackend per rank, and
over NCCL when two GPUs are present.  The reference is autograd on a queue that requires grad (oracle/head_ref.py dqueue_ref, fp64);
on a shard, rows [off, off + q_local) of it on the global queue."""
import os
import socket
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle.head_ref import HeadOracle, dqueue_ref, hard_neg_k

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_dqueue_sharded_cpu import swept_queue  # noqa: E402

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-30))


def _center(i, D, seed):
    return torch.randn(D, generator=torch.Generator().manual_seed(seed * 1000003 + int(i)))


def _clustered(ids, D, seed, noise, gen):
    c = torch.stack([_center(i, D, seed) for i in ids.tolist()])
    return F.normalize(F.normalize(c) + noise * torch.randn(len(ids), D, generator=gen) / D ** 0.5)


def _regions(got, ref, special, tol, what):
    Q = got.shape[1]
    plain = torch.ones(Q, dtype=torch.bool)
    plain[special] = False
    assert _rel(got[0][plain], ref[0][plain]) <= tol, ('bulk rows', what, _rel(got[0][plain], ref[0][plain]))
    assert _rel(got[0][special], ref[0][special]) <= tol, ('target / ones rows', what, _rel(got[0][special], ref[0][special]))
    assert _rel(got[1], ref[1]) <= tol, ('queue[1]', what, _rel(got[1], ref[1]))


def _bf16_values(t):
    """SV's loss jumps at the hard-example threshold (1.2 z + 0.2 multiplies a term by ~e^8 there): rounding an operand to bf16 that moves a
    cosine across it changes that term by thousands of times, which no tolerance absorbs.  The bf16 tests therefore feed embeddings and
    prototypes that are bf16 values already, so that the fp64 reference sees the operands the tensor cores see."""
    return t.to(torch.bfloat16).float()


def _run_head(D, Q, B, n_ids, loss_type, margin, precision, steps, seed=4):
    """Rollback and commit passes through FFCHead(queue_grad=True); yields (dqueue_pass, reference, special slots, outlier count)."""
    q_ = _bf16_values if precision == 'bf16' else (lambda t: t)
    import ffc_b200
    dev = torch.device('cuda')
    torch.manual_seed(0)
    h = ffc_b200.FFCHead(D, Q, 32.0, loss_type, margin, precision=precision, max_batch=B, device=dev, queue_grad=True)
    with torch.no_grad():      # zero-mean prototypes: SV's hard-example branch fires for a few columns per row, not for all
        h.queue.copy_(q_(F.normalize(torch.randn(2, Q, D, generator=torch.Generator().manual_seed(seed + 1)), dim=2)))
    h._ensure()
    o = HeadOracle(D, Q, 32.0, loss_type, margin, queue=h.queue.cpu(), dtype=torch.float64)
    gen = torch.Generator().manual_seed(seed)
    for step in range(steps):
        xl = torch.randint(0, n_ids, (B,), generator=gen)
        yl = torch.cat([xl[:B // 2], torch.randint(0, n_ids, (B - B // 2,), generator=gen)])
        x = q_(_clustered(xl, D, 5, 0.7, gen))
        y = q_(_clustered(yl, D, 5, 0.7, gen))
        for commit, (p, g, pl, gl) in ((False, (x, y, xl, yl)), (True, (y, x, yl, xl))):
            h.head(p.to(dev), g.to(dev), pl, gl, commit=commit)
            o.head_pass(p.double(), g.double(), pl.tolist(), gl.tolist(), commit=commit)
            tr = o.trace[-1]
            q = swept_queue(o.queue, tr, g.double(), commit)
            _, ref = dqueue_ref(p.double(), q, tr['labels'], tr['ones'], loss_type, margin, 32.0, o.k)
            special = sorted(set(tr['ones']) | {l for l in tr['labels'] if l >= 0})
            yield h, h.dqueue_pass.double().cpu(), ref, special, sum(l < 0 for l in tr['labels']), (commit, step)


@pytest.mark.parametrize('D', [64, 132, 512])
@pytest.mark.parametrize('loss_type,margin', [('AM', 0.4), ('Arc', 0.5), ('SV', 0.4)])
def test_check_mode_dqueue(D, loss_type, margin):
    """fp32 head: 1e-5 per region against fp64 autograd on the same fp32 inputs, rollback and commit passes (the rollback pass's
    gradient is of the queue it swept: one taken after the restore fails), identities > queue (evictions, outlier rows)"""
    Q, B = 1000, 96
    acc = None
    for h, got, ref, special, n_out, what in _run_head(D, Q, B, 1300, loss_type, margin, 'fp32', 3):
        assert torch.isfinite(got).all()
        _regions(got, ref, special, 1e-5, (what, n_out))
        acc = ref.clone() if acc is None else acc + ref
    assert _rel(h.dqueue.double().cpu(), acc) <= 1e-5


@pytest.mark.parametrize('loss_type,margin', [('AM', 0.4), ('SV', 0.4)])
def test_check_mode_dqueue_is_bit_identical(loss_type, margin):
    runs = [[got for _, got, *_ in _run_head(132, 1000, 96, 1300, loss_type, margin, 'fp32', 2)] for _ in range(2)]
    assert all(torch.equal(a, b) for a, b in zip(*runs))


@pytest.mark.parametrize('D', [128, 256, 512])
def test_bf16_sv_dqueue(D):
    """the SV mode of the swapped sweep: per region 1e-2 without outlier rows, 5e-2 in aggregate with them (a near-tie at a row's
    top-k boundary moves a whole prototype row between two slots); rollback and commit passes"""
    Q, B = {128: 2000, 256: 2000, 512: 4096}[D], {128: 96, 256: 128, 512: 256}[D]
    seen_out = seen_clean = 0
    # few identities (all resident after the first commit pass: no outlier rows from then on), then more identities than slots
    for n_ids, kind, steps in ((B // 3, 'clean', 4), (Q * 5 // 4, 'outliers', 2)):
        for h, got, ref, special, n_out, what in _run_head(D, Q, B, n_ids, 'SV', 0.4, 'bf16', steps):
            assert torch.isfinite(got).all()
            if n_out == 0:
                _regions(got, ref, special, 1e-2, what)
                seen_clean += 1
            else:
                seen_out += 1
            assert _rel(got, ref) <= (1e-2 if n_out == 0 else 5e-2), (what, kind, _rel(got, ref), n_out)
    assert seen_clean and seen_out


def _sv_pass_on_both_precisions(D, Q, B):
    """commit passes of a bf16 and an fp32 SV head on identical inputs (bf16 values, see _bf16_values)"""
    import ffc_b200
    dev = torch.device('cuda')
    gen = torch.Generator().manual_seed(9)
    q0 = _bf16_values(F.normalize(torch.randn(2, Q, D, generator=gen), dim=2))
    xl = torch.randint(0, Q * 7 // 10, (B,), generator=gen)
    yl = torch.cat([xl[:B // 2], torch.randint(0, Q * 7 // 10, (B - B // 2,), generator=gen)])
    x, y = _bf16_values(_clustered(xl, D, 5, 0.7, gen)), _bf16_values(_clustered(yl, D, 5, 0.7, gen))
    out = {}
    for prec in ('bf16', 'fp32'):
        torch.manual_seed(0)
        h = ffc_b200.FFCHead(D, Q, 32.0, 'SV', 0.4, precision=prec, max_batch=B, device=dev, queue_grad=True)
        with torch.no_grad():
            h.queue.copy_(q0)
        h._ensure()
        for _ in range(2):          # a second pass: the first one's gallery rows are resident (targets, `ones`)
            h.head(y.to(dev), x.to(dev), yl, xl, commit=True)
        out[prec] = h.dqueue_pass.double().cpu()
    return out


@pytest.mark.parametrize('D', [128, 512])
def test_bf16_sv_dqueue_against_check_mode(D):
    out = _sv_pass_on_both_precisions(D, 2000, 128)
    assert _rel(out['bf16'], out['fp32']) <= 1e-2, _rel(out['bf16'], out['fp32'])


def _set_ones(cmask, ones_list, n_ones, local):
    cmask.zero_()
    for j, s in enumerate(local):
        cmask[s >> 5] |= (1 << (s & 31)) if (s & 31) < 31 else -(1 << 31)
        ones_list[j] = s
    n_ones.fill_(len(local))


@pytest.mark.parametrize('precision,loss_type,margin', [('bf16', 'AM', 0.4), ('bf16', 'Arc', 0.5), ('bf16', 'SV', 0.4), ('fp32', 'AM', 0.4),
                                                        ('fp32', 'Arc', 0.5), ('fp32', 'SV', 0.4)])
@pytest.mark.parametrize('R', [2, 4])
def test_emulated_shards_dqueue(R, precision, loss_type, margin):
    """R CudaShardBackends on one GPU (uneven shards), the collectives of ffc_b200/dist.py done by hand: every shard's dqueue equals
    its slice of the gradient of the global queue"""
    from ffc_b200.dist import CudaShardBackend
    D, Q, n = 128, 4099, 200
    base, rem = divmod(Q, R)
    Qls = [base + (1 if r < rem else 0) for r in range(R)]
    offs = [r * base + min(r, rem) for r in range(R)]
    gen = torch.Generator().manual_seed(13)
    dev = torch.device('cuda')
    queue = F.normalize(torch.randn(2, Q, D, generator=gen), dim=2)
    if precision == 'bf16':
        queue = _bf16_values(queue)
    label = torch.randint(0, Q, (n,), generator=gen)
    label[torch.rand(n, generator=gen) < 0.2] = -1
    ones_global = torch.randperm(Q, generator=gen)[:40].sort().values
    label[:10] = ones_global[:10]
    known = label >= 0
    p = torch.randn(n, D, generator=gen)
    p[known] = queue[0][label[known]] + 0.12 * p[known]
    p = F.normalize(p)
    if precision == 'bf16':
        p = _bf16_values(p)
    _, ref = dqueue_ref(p.double(), queue.double(), label.tolist(), ones_global.tolist(), loss_type, margin, 32.0, hard_neg_k(Q))
    p_d, label_d = p.to(dev), label.to(torch.int32).to(dev)
    torch.manual_seed(0)
    shards = [CudaShardBackend(D, Qls[r], Q, offs[r], n, 32.0, loss_type, margin, hard_neg_k(Q), precision, dev) for r in range(R)]
    for r, be in enumerate(shards):
        be.enable_dqueue()
        be.set_queue(queue[:, offs[r]:offs[r] + Qls[r]])
        be.use_set(0)
        _set_ones(be.cmask, be.ones_list, be.n_ones, [int(g) - offs[r] for g in ones_global.tolist() if offs[r] <= int(g) < offs[r] + Qls[r]])
    if shards[0].record_path:
        # bf16 AM / Arc: the record flow (one record per rank, all-gathered, finalize from the records)
        recs = [be.new_records(n, R) for be in shards]
        for be, rec in zip(shards, recs):
            be.sweep_record(p_d, label_d, rec)
        for rec in recs:
            rec['all'].copy_(torch.stack([rr['own'] for rr in recs]))
        for be, rec in zip(shards, recs):
            be.finalize_gathered(p_d, label_d, rec, R)
    else:
        stats = [be.new_stats(n, R) for be in shards]
        for r, be in enumerate(shards):
            be.prep(p_d, label_d, stats[r], r)
        tgt = sum(st['red'][4:] for st in stats)
        for r, be in enumerate(shards):
            stats[r]['red'][4:].copy_(tgt)
            be.sweep_prepared(p_d, label_d, stats[r], r)
        lsum = sum(st['red'][:4] for st in stats)
        topv = torch.stack([stats[r]['topv'][r] for r in range(R)])
        topi = torch.stack([stats[r]['topi'][r] for r in range(R)])
        for r, be in enumerate(shards):
            stats[r]['red'][:4].copy_(lsum)
            stats[r]['topv'].copy_(topv)
            stats[r]['topi'].copy_(topi)
            be.finalize(p_d, label_d, stats[r], R)
    got = []
    for r, be in enumerate(shards):
        out = torch.empty(2, Qls[r], D, device=dev)
        be.dqueue(p_d, label_d, out)
        got.append(out.double().cpu())
    got = torch.cat(got, dim=1)
    # (outlier rows take part: a bf16 near-tie at a top-k boundary moves a whole row, hence the aggregate bound there)
    special = sorted(set(ones_global.tolist()) | {int(l) for l in label.tolist() if l >= 0})
    if precision == 'fp32':
        _regions(got, ref, special, 1e-5, R)
    else:
        assert _rel(got, ref) <= 5e-2, _rel(got, ref)


def test_sharded_head_default_keeps_merged_flow():
    """without queue_grad the sharded head still takes the merged step and allocates no gradient buffers; with it, the per-pass flow"""
    import torch.distributed as dist
    from ffc_b200.dist import ShardedFFCHead
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=0, world_size=1)
    try:
        off = ShardedFFCHead(128, 4096, 32.0, 'AM', 0.4, precision='bf16', max_batch=64, device='cuda')
        assert off.merged is True and off.dqueue is None and off.dqueue_pass is None
        on = ShardedFFCHead(128, 4096, 32.0, 'AM', 0.4, precision='bf16', max_batch=64, device='cuda', queue_grad=True)
        assert on.merged is False and on.dqueue.shape == (2, 4096, 128) and on.dqueue.is_cuda
    finally:
        dist.destroy_process_group()


def _nccl_worker(rank, world, port, loss_type, margin, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world)
    try:
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from test_dist_cpu import ShardedOracle
        from ffc_b200.dist import ShardedFFCHead
        dev = torch.device('cuda', rank)
        D, Q, B, n_ids = 128, 4099, 64, 3000
        torch.manual_seed(0)
        head = ShardedFFCHead(D, Q, 32.0, loss_type, margin, precision='bf16', max_batch=B, device=dev, queue_grad=True)
        q0 = F.normalize(torch.randn(2, Q, D, generator=torch.Generator().manual_seed(3)), dim=2)
        head.backend.set_queue(q0[:, head.off:head.off + head.Ql])
        oracle = ShardedOracle(world, D, Q, 32.0, loss_type, margin, queue=q0, dtype=torch.float64)
        gen = torch.Generator().manual_seed(5)
        for step in range(3):
            xl = torch.randint(0, n_ids, (world * B,), generator=gen)
            yl = torch.cat([xl[:world * B // 2], torch.randint(0, n_ids, (world * B - world * B // 2,), generator=gen)])
            x, y = _clustered(xl, D, 5, 0.7, gen), _clustered(yl, D, 5, 0.7, gen)
            sl = slice(rank * B, (rank + 1) * B)
            for commit, (p, g, pl, gl) in ((False, (x, y, xl, yl)), (True, (y, x, yl, xl))):
                head.head_pass(p[sl].to(dev), g[sl].to(dev), pl[sl], gl[sl], commit)
                oracle.head_pass(p.double(), g.double(), pl.tolist(), gl.tolist(), commit)
                tr = oracle.trace[-1]
                q = swept_queue(oracle.queue, tr, g.double(), commit)
                _, ref = dqueue_ref(p.double(), q, tr['labels'], tr['ones'], loss_type, margin, 32.0, oracle.k)
                ref = ref[:, head.off:head.off + head.Ql]
                n_out = sum(l < 0 for l in tr['labels'])
                got = head.dqueue_pass.double().cpu()
                assert _rel(got, ref) <= (1e-2 if n_out == 0 else 5e-2), (rank, step, commit, _rel(got, ref))
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason='needs two GPUs')
@pytest.mark.parametrize('loss_type,margin', [('Arc', 0.5), ('SV', 0.4)])
def test_nccl_sharded_dqueue_two_gpus(loss_type, margin):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, port, loss_type, margin, ret), nprocs=2, join=True)
    assert dict(ret) == {0: 'ok', 1: 'ok'}


@pytest.mark.parametrize('loss_type,precision', [('SV', 'bf16'), ('AM', 'fp32'), ('SV', 'fp32')])
def test_dqueue_c_abi_checks(loss_type, precision):
    """ffc_head_set_dqueue accepts every loss type and precision; ffc_head_dqueue rejects a bad pass description, the operand its
    precision needs missing, and a handle without the mode -- before any launch"""
    import ctypes as C
    import ffc_b200
    from ffc_b200 import _capi
    lib = _capi.lib()
    dev = torch.device('cuda')
    h = ffc_b200.FFCHead(64, 256, 32.0, loss_type, 0.4, precision=precision, max_batch=32, device=dev)
    h._ensure()
    out = torch.empty(2, 256, 64, device=dev)
    p = torch.zeros(32, 64, device=dev)
    good = dict(p_f32=p.data_ptr(), queue_f32=h.queue.data_ptr(), queue_bf16=h.queue_bf16.data_ptr(), label=h.label.data_ptr(),
                ones_list=h.ones_list.data_ptr(), n_ones=h.n_ones.data_ptr(), cmask=h.cmask.data_ptr(), n_rows=32)
    launches = lib.ffc_launch_count()
    assert lib.ffc_head_dqueue(h._h, C.byref(_capi.HeadPass(**good)), out.data_ptr(), None) != 0 and b'enable the mode' in lib.ffc_last_error()
    _capi.check(lib.ffc_head_set_dqueue(h._h, 1))
    missing = ['n_rows', 'ones_list', 'n_ones'] + (['queue_bf16'] if precision == 'bf16' else ['p_f32', 'queue_f32'])
    for field in missing:
        assert lib.ffc_head_dqueue(h._h, C.byref(_capi.HeadPass(**dict(good, **{field: 0}))), out.data_ptr(), None) != 0, field
    assert lib.ffc_head_dqueue(h._h, C.byref(_capi.HeadPass(**dict(good, n_rows=33))), out.data_ptr(), None) != 0
    assert lib.ffc_launch_count() == launches
    _capi.check(lib.ffc_head_set_dqueue(h._h, 0))
