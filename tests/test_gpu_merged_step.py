"""The sharded head's merged step (ShardedFFCHead._forward_pair_merged) on ONE GPU.

The merged step is the bf16 AM / Arc step of the multi-GPU head: one statistics exchange per step, the rollback pass finalized
after its queue rows have been restored and re-enqueued (it reads them through the overlay map), dLoss/dp routed to the owner
ranks' staging buffers by the finalize kernel itself and summed there.  Every kernel of that path runs on one device when the
ranks' buffers all live on it, and the in-kernel barriers return at once when their flag words already hold the epoch -- so
each kernel is checked here bit for bit against a plain torch restatement, and the whole step, driven for R emulated ranks in
lock step, against the per-pass record flow (bit for bit) and the fp64 sharded oracle.

No barrier kernel is ever launched before the flag words it waits on hold its epoch (the 5 s timeout path is not exercised).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SENT = 12345.0              # sentinel of words a kernel must not write
TAG = 0x40000000            # overlay table-1 marks (csrc/queue_scatter.cu)


def _lib():
    from ffc_b200 import _capi
    return _capi.lib()


def _check(rc):
    from ffc_b200._capi import check
    check(rc)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptrs(ts, off_words=0):
    return torch.tensor([t.data_ptr() + 4 * off_words for t in ts], dtype=torch.int64, device='cuda')


# ---- packed position lists and their plain restatements ------------------------------------------------------------------------

def _packed_list(gen, n, live, Ql):
    """A rank's packed (rows, cols) list of n positions: `live` positions first, then padding (cols = -1, stale rows), and a source
    permutation of the n gathered rows.  Columns come from a narrow range (duplicates everywhere); three more duplicate pairs are
    planted more than 128 positions (one scan chunk) apart, the last one ending at the last live position."""
    rows = torch.randint(0, 2, (n,), generator=gen, dtype=torch.int32)
    cols = torch.randint(0, min(Ql, max(8, live // 2)), (n,), generator=gen, dtype=torch.int32)
    cols[live:] = -1
    for j1, j2 in ((3, 3 + 129), (10, 10 + 300), (live // 3, live - 1)):
        if j1 < j2 < live:
            rows[j2], cols[j2] = rows[j1], cols[j1]
    src = torch.randperm(n, generator=gen).to(torch.int32)
    return rows, cols, src


def _winners(rows, cols):
    """Positions that write, in position order: the last occurrence of every (row, col) pair of the live prefix (serial index_put)."""
    live = int((cols < 0).nonzero()[0]) if bool((cols < 0).any()) else cols.numel()
    last = {}
    for i, rc in enumerate(zip(rows[:live].tolist(), cols[:live].tolist())):
        last[rc] = i
    return torch.tensor(sorted(last.values()), dtype=torch.long)


def _ref_scatter(q, mp, rows, cols, g, src, table, undo_shape):
    """fp32 queue, overlay map and undo buffer after one enqueue of the packed list (ffc_queue_scatter_overlay restated)."""
    q, mp = q.clone(), mp.clone()
    w = _winners(rows, cols)
    r, c = rows[w].long(), cols[w].long()
    undo = torch.full(undo_shape, SENT)
    undo[w] = q[r, c]
    q[r, c] = g[src[w].long()]
    if table == 0:
        mp[r, c] = src[w]
    elif table == 1:
        free = mp[r, c] < 0
        mp[r[free], c[free]] = (TAG | w[free]).to(torch.int32)
    return q, mp, undo


@pytest.mark.parametrize('D,Ql,n,live0,live1', [(64, 300, 1000, 300, 263), (128, 1001, 2048, 389, 352), (512, 8192, 8192, 1101, 1064)])
def test_scatter_overlay_clear_and_restore(D, Ql, n, live0, live1):
    """ffc_queue_scatter_overlay tables 0 and 1 (table 1 on top of table 0), ffc_overlay_clear, ffc_queue_restore_packed."""
    lib, s = _lib(), _stream()
    gen = torch.Generator().manual_seed(D + n)
    q0 = torch.randn(2, Ql, D, generator=gen)
    g = torch.randn(n, D, generator=gen)
    la, lb = _packed_list(gen, n, live0, Ql), _packed_list(gen, n, live1, Ql)
    cu = lambda t: t.cuda().contiguous()
    qf, qh, gd = cu(q0), cu(q0.to(torch.bfloat16)), cu(g)
    mp = torch.full((2, Ql), -1, dtype=torch.int32, device='cuda')
    ua, ub = torch.full((n, D), SENT, device='cuda'), torch.full((n, D), SENT, device='cuda')
    (ra, ca, sa), (rb, cb, sb) = [tuple(cu(t) for t in l) for l in (la, lb)]

    def scatter(rows, cols, src, undo, table):
        _check(lib.ffc_queue_scatter_overlay(qf.data_ptr(), qh.data_ptr(), rows.data_ptr(), cols.data_ptr(), gd.data_ptr(), src.data_ptr(), n, Ql, D,
                                             undo.data_ptr(), mp.data_ptr(), table, s))

    # table 0 (a rollback pass's enqueue), then table 1 (the commit pass's enqueue) on top of it
    q_ref, mp_ref = q0, torch.full((2, Ql), -1, dtype=torch.int32)
    for (rows, cols, src), (rd, cd, sd), undo, table in ((la, (ra, ca, sa), ua, 0), (lb, (rb, cb, sb), ub, 1)):
        scatter(rd, cd, sd, undo, table)
        q_ref, mp_ref, u_ref = _ref_scatter(q_ref, mp_ref, rows, cols, g, src, table, (n, D))
        assert torch.equal(qf.cpu(), q_ref), table
        assert torch.equal(qh.cpu(), q_ref.to(torch.bfloat16)), table
        assert torch.equal(undo.cpu(), u_ref), table
        assert torch.equal(mp.cpu(), mp_ref), table
    # both kinds of table-1 position occurred: entries a table-0 mark held, and fresh table-1 marks
    wb = _winners(*lb[:2])
    held = mp_ref[lb[0][wb].long(), lb[1][wb].long()]
    assert bool((held & TAG == 0).any()) and bool((held & TAG != 0).any())

    # overlay_clear: exactly the live entries of the list return to -1
    for (rows, cols, _), (rd, cd, _) in ((la, (ra, ca, sa)), (lb, (rb, cb, sb))):
        _check(lib.ffc_overlay_clear(mp.data_ptr(), rd.data_ptr(), cd.data_ptr(), n, Ql, s))
        live = cols >= 0
        mp_ref[rows[live].long(), cols[live].long()] = -1
        assert torch.equal(mp.cpu(), mp_ref)
    assert bool((mp_ref == -1).all())

    # restore_packed after an undo-saving scatter of the same packed list: the queue is the original one, bit for bit
    qf.copy_(q0)
    qh.copy_(q0.to(torch.bfloat16))
    scatter(ra, ca, sa, ua, 0)
    assert not torch.equal(qf.cpu(), q0)
    _check(lib.ffc_queue_restore_packed(qf.data_ptr(), qh.data_ptr(), ra.data_ptr(), ca.data_ptr(), ua.data_ptr(), n, Ql, D, s))
    assert torch.equal(qf.cpu(), q0)
    assert torch.equal(qh, qf.to(torch.bfloat16))


# ---- slab sums and barriers ----------------------------------------------------------------------------------------------------

def _slab_case(n_slabs, n, seed):
    gen = torch.Generator().manual_seed(seed)
    stride = n + 36
    # magnitudes spread over six decades: a different summation order rounds differently
    slabs = (torch.randn(n_slabs * stride, generator=gen) * torch.exp(6 * torch.rand(n_slabs * stride, generator=gen))).cuda()
    ref = slabs[:n].clone()
    for r in range(1, n_slabs):
        ref += slabs[r * stride:r * stride + n]
    buf = torch.full((n + 16,), SENT, device='cuda')        # 8 sentinel words on either side of the output
    return slabs, stride, ref, buf


def _check_out(buf, ref, n):
    assert torch.equal(buf[8:8 + n], ref)
    assert bool((buf[:8] == SENT).all()) and bool((buf[8 + n:] == SENT).all())


@pytest.mark.parametrize('n_slabs', [1, 2, 3, 8])
def test_sum_slabs(n_slabs):
    lib, s = _lib(), _stream()
    for n in (4, 1000, 2 * 1024 * 512):
        slabs, stride, ref, buf = _slab_case(n_slabs, n, n_slabs * 7 + n)
        _check(lib.ffc_sum_slabs(slabs.data_ptr(), n_slabs, stride, n, buf.data_ptr() + 32, s))
        _check_out(buf, ref, n)


@pytest.mark.parametrize('R', [1, 2, 3, 8])
def test_sum_slabs_barrier_preseeded(R):
    """ffc_sum_slabs_barrier for every rank of R, the flag words it waits on already at the epoch (one of them ahead: the words only
    grow): the sums are the plain ones, no timeout, and every peer's word [my_rank] now holds the epoch."""
    lib, s = _lib(), _stream()
    epoch = 5
    for n in (4, 1000, 2 * 1024 * 512):
        for me in range(R):
            slabs, stride, ref, buf = _slab_case(R, n, 31 * R + me + n)
            flags = torch.full((R, R), epoch - 1, dtype=torch.int32, device='cuda')
            flags[me] = epoch
            if R > 1:
                flags[me, (me + 1) % R] = epoch + 3
            err = torch.zeros(1, dtype=torch.int32, device='cuda')
            _check(lib.ffc_sum_slabs_barrier(slabs.data_ptr(), R, stride, n, buf.data_ptr() + 32, _ptrs(list(flags)).data_ptr(), me, R, epoch,
                                             err.data_ptr(), s))
            _check_out(buf, ref, n)
            assert int(err) == 0
            assert bool((flags[:, me] == epoch).all())


# ---- emulated ranks ------------------------------------------------------------------------------------------------------------

def _shards(Q, R):
    """ShardedFFCHead's slot ranges: contiguous, the first Q % R ranks one slot longer."""
    base, rem = divmod(Q, R)
    return [base + (1 if r < rem else 0) for r in range(R)], [r * base + min(r, rem) for r in range(R)]


def _backend(D, Q, R, r, B, loss_type, q0):
    """Rank r's shard of R (B rows per rank), loaded with its slice of q0."""
    from ffc_b200.dist import CudaShardBackend
    from ffc_b200.ffc import hard_neg_k
    Qls, offs = _shards(Q, R)
    be = CudaShardBackend(D, Qls[r], Q, offs[r], R * B, 32.0, loss_type, 0.5 if loss_type == 'Arc' else 0.4, hard_neg_k(Q), 'bf16',
                          torch.device('cuda'))
    be.set_queue(q0[:, offs[r]:offs[r] + Qls[r]])
    return be


def _backends(D, Q, R, B, loss_type, q0):
    return [_backend(D, Q, R, r, B, loss_type, q0) for r in range(R)]


def _peer_records(be, n, R):
    """ShardedFFCHead._peer_records with every rank's buffer on this device: [R ranks][2 passes][16-byte aligned record] + R flag words."""
    w = be.new_records(n, 1, passes=1)['words']
    ws = (w + 3) // 4 * 4
    bufs = [torch.zeros(R * 2 * ws + 64, device='cuda') for _ in range(R)]
    recs = []
    for r in range(R):
        recs.append(dict(own=torch.zeros(2, ws, device='cuda'), all=bufs[r][:R * 2 * ws].view(R, 2, ws), words=ws, passes=2, buf=bufs[r],
                         peer=dict(ptrs=_ptrs(bufs), flags=_ptrs(bufs, R * 2 * ws), err=torch.zeros(1, dtype=torch.int32, device='cuda'), epoch=0)))
    return recs


def _peer_barrier_all(bes, recs):
    """One ffc_peer_barrier per rank, every flag word published beforehand."""
    R = len(bes)
    epoch = recs[0]['peer']['epoch'] + 1
    for rc in recs:
        rc['peer']['epoch'] = epoch
        n0 = R * 2 * rc['words']
        rc['buf'][n0:n0 + R].view(torch.int32).fill_(epoch)
    for r, (be, rc) in enumerate(zip(bes, recs)):
        be.peer_barrier(rc['peer']['flags'], r, R, epoch, rc['peer']['err'])
    for rc in recs:
        n0 = R * 2 * rc['words']
        assert int(rc['peer']['err']) == 0 and bool((rc['buf'][n0:n0 + R].view(torch.int32) == epoch).all())


def _pass_inputs(gen, n, D, Q, frac_out=0.33):
    p = F.normalize(torch.randn(n, D, generator=gen)).cuda()
    label = torch.randint(0, Q, (n,), generator=gen, dtype=torch.int32)
    label[torch.rand(n, generator=gen) < frac_out] = -1
    return p, label.cuda()


def _set_ones(be, gen, n_ones):
    """A pass's `ones` set on the backend's current bookkeeping set: n_ones random local slots (list + bitmask)."""
    local = torch.randperm(be.Ql, generator=gen)[:n_ones].sort().values
    words = np.zeros(be.cmask.numel(), dtype=np.uint32)
    np.bitwise_or.at(words, local.numpy() >> 5, np.left_shift(np.uint32(1), (local.numpy() & 31).astype(np.uint32)))
    be.cmask.copy_(torch.from_numpy(words.view(np.int32)))
    be.ones_list[:n_ones] = local.to(torch.int32).cuda()
    be.n_ones.fill_(n_ones)
    return local


@pytest.mark.parametrize('D,Q,R,B', [(128, 2048, 2, 96), (512, 8192, 8, 128)])
def test_push_record_and_peer_barrier(D, Q, R, B):
    """ffc_head_push_record into R sentinel-filled buffers of the _peer_records layout: the per-row scalar words land at every
    destination, the top-k words only for hard-negative-only rows (label -1), every other word keeps its sentinel."""
    gen = torch.Generator().manual_seed(D + R)
    q0 = F.normalize(torch.rand(2, Q, D, generator=gen), dim=2)
    be = _backend(D, Q, R, 1, B, 'Arc', q0)
    n = R * B
    recs = _peer_records(be, n, R)
    w, ws = be.new_records(n, 1)['words'], recs[0]['words']
    k = be.k
    for rc in recs:
        rc['buf'][:R * 2 * ws].fill_(SENT)
    be.use_set(0)
    _set_ones(be, gen, 40)
    for which in (0, 1):
        p, label = _pass_inputs(gen, n, D, Q)
        be.sweep_record(p, label, recs[1], which)
        be.push_record(p, recs[1], which, 1)
        src = recs[1]['own'][which, :w].clone()
        out = (label < 0).cpu()
        want = torch.full((ws,), SENT)
        want[:8 * n] = src[:8 * n].cpu()
        top = src[8 * n:].cpu().view(6, n, k)
        want[8 * n:w].view(6, n, k)[:, out] = top[:, out]
        for dst in recs:
            got = dst['all'][1, which].cpu()
            assert torch.equal(got.view(torch.int32), want.view(torch.int32)), which
    for dst in recs:        # the other source ranks' slots were not touched
        assert bool((dst['all'][[r for r in range(R) if r != 1]] == SENT).all())
    _peer_barrier_all([be] * R, recs)


@pytest.mark.parametrize('D,Q,R,B', [(128, 3001, 3, 96), (512, 8192, 4, 128)])
def test_finalize_routed_rows(D, Q, R, B):
    """ffc_head_finalize_gathered_ex with dp_peer routing against the same finalize into dp_out: row i lands in buffer i / B at the
    slot offset + (i % B) * D, bit-equal to its dp_out row; every other word of the stage buffers keeps its sentinel; equal loss."""
    gen = torch.Generator().manual_seed(D + Q)
    q0 = F.normalize(torch.rand(2, Q, D, generator=gen), dim=2)
    be = _backend(D, Q, R, R - 1, B, 'Arc', q0)
    n = R * B
    be.use_set(0)
    local = _set_ones(be, gen, 48)
    p, label = _pass_inputs(gen, n, D, Q)
    label[:16] = (local[:16] + be.off).to(torch.int32).cuda()            # targets inside `ones`
    label[16:48] = torch.randint(be.off, be.off + be.Ql, (32,), generator=gen, dtype=torch.int32).cuda()
    rec = be.new_records(n, 1)
    be.sweep_record(p, label, rec)
    rec['all'].copy_(rec['own'])
    loss_a, dp_a = be.finalize_gathered(p, label, rec, 1)
    slab = 2 * B * D
    stage = [torch.full((R * slab + 64,), SENT, device='cuda') for _ in range(R)]
    off = (R - 1) * slab + B * D + 4           # a source rank's commit-pass slot, plus four words
    be.sweep_record(p, label, rec)
    loss_b, dp_b = be.finalize_gathered(p, label, rec, 1, route=(_ptrs(stage), B, off))
    assert dp_b is None
    assert torch.equal(loss_a, loss_b)
    for q in range(R):
        got = stage[q].cpu()
        assert torch.equal(got[off:off + B * D].view(B, D), dp_a[q * B:(q + 1) * B].cpu()), q
        rest = torch.cat([got[:off], got[off + B * D:]])
        assert bool((rest == SENT).all()), q


@pytest.mark.parametrize('D,Q,R,B', [(128, 256, 2, 96), (512, 512, 2, 128)])
def test_finalize_reads_rewritten_rows_through_overlay(D, Q, R, B):
    """The overlay read of ffc_head_finalize_gathered_ex (w_row / w_load4).  Every queue row of the shard is rewritten after the sweep,
    and the map sends each (row, slot) entry to its sweep-time fp32 row: even entries through table 0 (overlay_g), odd ones through
    table 1 (the undo rows).  Loss and dLoss/dp must then equal, bit for bit, those of the finalize that read the bf16 mirror before
    the rewrite.  The rows are plain fp32, so this holds only if finalize rounds them to nearest-even, as the mirror was."""
    gen = torch.Generator().manual_seed(D + Q + 1)
    q0 = F.normalize(torch.rand(2, Q, D, generator=gen), dim=2)
    be = _backend(D, Q, R, 1, B, 'Arc', q0)
    n, Ql = R * B, be.Ql
    be.use_set(0)
    local = _set_ones(be, gen, 24)
    p, label = _pass_inputs(gen, n, D, Q)
    label[:8] = (local[:8] + be.off).to(torch.int32).cuda()            # targets inside `ones`: their loss-2 row is queue[1]
    label[8:40] = torch.randint(be.off, be.off + Ql, (32,), generator=gen, dtype=torch.int32).cuda()
    rec = be.new_records(n, 1)
    be.sweep_record(p, label, rec)
    rec['all'].copy_(rec['own'])
    loss_a, dp_a = be.finalize_gathered(p, label, rec, 1)
    be.sweep_record(p, label, rec)                                       # the same sweep again, then every row changes under it
    swept = be.queue.view(2 * Ql, D).clone()
    assert not torch.equal(swept, swept.to(torch.bfloat16).float())      # the rounding is observable
    be.set_queue(F.normalize(torch.rand(2, Ql, D, generator=gen), dim=2))
    even, odd = torch.arange(0, 2 * Ql, 2), torch.arange(1, 2 * Ql, 2)
    g_idx = torch.randperm(2 * Ql + 17, generator=gen)[:even.numel()]
    u_idx = torch.randperm(n, generator=gen)[:odd.numel()]
    ovl_g = torch.full((2 * Ql + 17, D), SENT, device='cuda')
    ovl_g[g_idx.cuda()] = swept[even.cuda()]
    be.undo_rows_cm.fill_(SENT)
    be.undo_rows_cm[u_idx.cuda()] = swept[odd.cuda()]
    mp = torch.empty(2 * Ql, dtype=torch.int32)
    mp[even], mp[odd] = g_idx.to(torch.int32), (TAG | u_idx).to(torch.int32)
    be.ovl_map.copy_(mp)
    loss_b, dp_b = be.finalize_gathered(p, label, rec, 1, overlay_g=ovl_g)
    assert torch.equal(loss_b, loss_a)
    assert torch.equal(dp_b, dp_a), _rel(dp_b, dp_a)


# ---- the merged step, emulated ------------------------------------------------------------------------------------------------

class _Ranks:
    """R CudaShardBackend instances on one device, driven in lock step.  Collectives are plain tensor operations: the label all-reduce
    MAX is torch.stack(...).amax(0), the record all-gather a stack of the ranks' rec['own'], the reduce-scatter a sum over the ranks
    in rank order (per-pass flow) or the symmetric-memory layout -- one [R][2][B][D] stage buffer per owner, finalize's routed stores,
    ffc_sum_slabs per owner (merged step)."""

    def __init__(self, D, Q, R, B, loss_type, q0, prefill, exchange='gather', overlay=True):
        self.D, self.Q, self.R, self.B = D, Q, R, B
        self.bes = _backends(D, Q, R, B, loss_type, q0)
        for be, (keys, slots) in zip(self.bes, prefill):
            be.lru.restore_arrays(keys, slots)
        self.exchange, self.overlay = exchange, overlay
        self.rb_set = 0
        self.recs = self.recs1 = None
        self.slab = 2 * B * D
        self.stage = [torch.empty(R * self.slab, device='cuda') for _ in range(R)]
        self.ptrs = _ptrs(self.stage)

    def bookkeep(self, pl_all, gl_all, commit, set_idx):
        """ShardedFFCHead._bookkeep on every rank, then the label all-reduce MAX."""
        orders, labels = [], []
        for r, be in enumerate(self.bes):
            be.use_set(set_idx)
            keys_c, order, n_mine = be.route(gl_all, self.R, r)
            be.assign(keys_c, n_mine, journal=not commit)
            loc = be.view(pl_all)
            labels.append(torch.where(loc >= 0, loc + be.off, loc).to(torch.int32))
            if not commit:
                be.undo_bookkeeping()
            orders.append(order)
        return dict(order=orders, label=torch.stack(labels).amax(0), set=set_idx)

    def merged_step(self, x_all, y_all, xl_all, yl_all):
        """ShardedFFCHead.forward_pair without a bookkeeping stream, merged (no prefetch; the rollback set alternates 2, 0, 2, ...):
            bookkeep_rb (set 2 / 0) -> [scatter y, overlay table 0, undo -> sweep_record x (pass 0) -> (peer: push_record 0) -> restore
            -> end_pass] -> bookkeep_cm (set 1) -> [scatter x, overlay table 1, undo_cm -> sweep_record y (pass 1) -> end_pass] ->
            record exchange (all-gather, or push_record 1 + ONE peer_barrier) -> [finalize_gathered 0 (set rb, overlay_g = y, route
            slot r * slab) -> finalize_gathered 1 (set 1, route slot r * slab + B * D) -> overlay_clear(rb) -> overlay_clear(1)] ->
            sum_slabs per owner.
        A reordering of _forward_pair_merged needs the same change here."""
        R, B, D = self.R, self.B, self.D
        n = x_all.shape[0]
        if self.recs is None:
            self.recs = _peer_records(self.bes[0], n, R) if self.exchange == 'peer' else [be.new_records(n, R, passes=2) for be in self.bes]
        recs = self.recs
        self.rb_set = rb_set = 2 - self.rb_set
        ctx_rb = self.bookkeep(xl_all, yl_all, False, rb_set)
        for r, be in enumerate(self.bes):
            be.use_set(rb_set)
            be.scatter(y_all, ctx_rb['order'][r], save_undo=True, overlay_table=0)
            be.sweep_record(x_all, ctx_rb['label'], recs[r], 0)
            if self.exchange == 'peer':
                be.push_record(x_all, recs[r], 0, r)
            be.restore_queue()
            be.end_pass()
        ctx_cm = self.bookkeep(yl_all, xl_all, True, 1)
        for r, be in enumerate(self.bes):
            be.use_set(1)
            be.scatter(x_all, ctx_cm['order'][r], save_undo=True, overlay_table=1)
            be.sweep_record(y_all, ctx_cm['label'], recs[r], 1)
            be.end_pass()
        if self.exchange == 'peer':
            for r, be in enumerate(self.bes):
                be.push_record(y_all, recs[r], 1, r)
            _peer_barrier_all(self.bes, recs)
        else:
            gathered = torch.stack([rc['own'] for rc in recs])
            for rc in recs:
                rc['all'].copy_(gathered)
        for st in self.stage:
            st.fill_(float('nan'))
        losses = []
        for r, be in enumerate(self.bes):
            be.use_set(rb_set)
            l2, _ = be.finalize_gathered(x_all, ctx_rb['label'], recs[r], R, 0, overlay_g=y_all if self.overlay else None,
                                         route=(self.ptrs, B, r * self.slab))
            be.use_set(1)
            l1, _ = be.finalize_gathered(y_all, ctx_cm['label'], recs[r], R, 1, route=(self.ptrs, B, r * self.slab + B * D))
            be.overlay_clear(rb_set)
            be.overlay_clear(1)
            losses.append((l2, l1))
        outs = []
        for be, st in zip(self.bes, self.stage):
            out = torch.empty(2, B, D, device='cuda')
            be.sum_slabs(st, R, self.slab, self.slab, out)
            outs.append(out)
        return losses, [o[0] for o in outs], [o[1] for o in outs]

    def per_pass_step(self, x_all, y_all, xl_all, yl_all):
        """ShardedFFCHead.forward_pair through the per-pass record flow (_finish with backend.record_path):
            bookkeep_rb (set 0) -> scatter y (undo) -> sweep_record x -> all-gather -> finalize_gathered -> reduce-scatter -> restore ->
            end_pass; bookkeep_cm (set 1) -> scatter x -> sweep_record y -> all-gather -> finalize_gathered -> reduce-scatter -> end_pass."""
        R, B = self.R, self.B
        n = x_all.shape[0]
        if self.recs1 is None:
            self.recs1 = [be.new_records(n, R) for be in self.bes]
        losses, grads = [[None, None] for _ in range(R)], []
        for which, (p_all, g_all, pl, gl, commit) in enumerate(((x_all, y_all, xl_all, yl_all, False), (y_all, x_all, yl_all, xl_all, True))):
            ctx = self.bookkeep(pl, gl, commit, 1 if commit else 0)
            for r, be in enumerate(self.bes):
                be.use_set(ctx['set'])
                be.scatter(g_all, ctx['order'][r], save_undo=not commit)
                be.sweep_record(p_all, ctx['label'], self.recs1[r])
            gathered = torch.stack([rc['own'] for rc in self.recs1])
            dps = []
            for r, be in enumerate(self.bes):
                self.recs1[r]['all'].copy_(gathered)
                loss, dp = be.finalize_gathered(p_all, ctx['label'], self.recs1[r], R)
                losses[r][which] = loss
                dps.append(dp)
            own = []
            for q in range(R):          # reduce-scatter: the owner's rows summed over the ranks in rank order, fp32
                acc = dps[0][q * B:(q + 1) * B].clone()
                for r in range(1, R):
                    acc += dps[r][q * B:(q + 1) * B]
                own.append(acc)
            grads.append(own)
            for be in self.bes:
                if not commit:
                    be.restore_queue()
                be.end_pass()
        return [tuple(l) for l in losses], grads[0], grads[1]


def _prefill(Q, R, B):
    """Nearly full shards: identity key r + R j in local slot j of rank r (most- to least-recent), a few slots still free."""
    Qls, _ = _shards(Q, R)
    out = []
    for r, ql in enumerate(Qls):
        n0 = ql - min(ql // 8, 16)
        keys = torch.arange(r, r + R * n0, R, dtype=torch.int64)
        out.append((keys, torch.arange(n0, dtype=torch.int32)))
    return out


def _step_batch(gen, n, D, Q):
    """Global batch of one step: 2/3 of the rows share their identity between x and y (drawn with replacement from 2 Q identities,
    with planted repeats: duplicates within the batch; often resident, so targets inside `ones`), the rest are identities from a
    pool of 100 Q (rarely resident: about a third of the probe rows are hard-negative-only).  Plain fp32 rows, NOT bf16-representable:
    the rows the rollback finalize reads through the overlay carry bits below bf16 precision, so only a finalize that rounds them to
    nearest-even, as the mirror was, stays bit-identical to the per-pass flow."""
    m = 2 * n // 3
    shared = torch.randint(0, 2 * Q, (m,), generator=gen)
    shared[1::7] = shared[0::7][:shared[1::7].numel()]
    xl = torch.cat([shared, torch.randint(2 * Q, 100 * Q, (n - m,), generator=gen)])
    yl = torch.cat([shared, torch.randint(2 * Q, 100 * Q, (n - m,), generator=gen)])
    perm = torch.randperm(n, generator=gen)
    xl, yl = xl[perm], yl[perm]
    x = F.normalize(torch.randn(n, D, generator=gen))
    y = F.normalize(x + 0.7 * F.normalize(torch.randn(n, D, generator=gen)))
    return x.cuda(), y.cuda(), xl.cuda(), yl.cuda()


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


@pytest.mark.parametrize('D,Q,R,B,loss_type,peer', [
    (512, 4096, 2, 128, 'Arc', False),
    (512, 4096, 2, 128, 'Arc', True),
    (128, 3001, 3, 96, 'AM', False),
    (64, 1000, 4, 64, 'Arc', False),
    (512, 65536, 8, 256, 'Arc', False),
    (512, 65536, 8, 256, 'Arc', True),
])
def test_merged_step_on_one_gpu(D, Q, R, B, loss_type, peer):
    """Six merged steps of R emulated ranks against the per-pass record flow on twin backends (bit-identical loss, dL/dx, dL/dy,
    queue, mirror, queue positions, LRU), the fp64 sharded oracle (bookkeeping and queue exact, loss / gradients 1e-2), and a third
    set finalizing the rollback pass WITHOUT the overlay, which must go wrong in at least one step (the overlay was needed).  peer:
    records exchanged by ffc_head_push_record + ffc_peer_barrier (FFC_DIST_PEER_RECORDS=1), bit-identical to the all-gather."""
    from oracle.shard_ref import ShardedOracle
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(D * R + Q)
    q0 = F.normalize(torch.rand(2, Q, D, generator=gen), dim=2)
    margin = 0.5 if loss_type == 'Arc' else 0.4
    pre = _prefill(Q, R, B)
    merged = _Ranks(D, Q, R, B, loss_type, q0, pre)
    per_pass = _Ranks(D, Q, R, B, loss_type, q0, pre)
    naive = _Ranks(D, Q, R, B, loss_type, q0, pre, overlay=False)
    peered = _Ranks(D, Q, R, B, loss_type, q0, pre, exchange='peer') if peer else None
    oracle = ShardedOracle(R, D, Q, 32.0, loss_type, margin, queue=q0.cuda(), dtype=torch.float64)
    for r, (keys, slots) in enumerate(pre):
        oracle.lrus[r].restore(list(zip(keys.tolist(), slots.tolist())))
    Qls, offs = _shards(Q, R)
    naive_wrong, n_out, n_ones_t = 0, 0, 0
    for step in range(6):
        x, y, xl, yl = _step_batch(gen, R * B, D, Q)
        assert not torch.equal(y, y.to(torch.bfloat16).float()), 'overlay rows must not be bf16-exact'
        lm, dxm, dym = merged.merged_step(x, y, xl, yl)
        lp, dxp, dyp = per_pass.per_pass_step(x, y, xl, yl)
        _, dxn, _ = naive.merged_step(x, y, xl, yl)
        for r in range(R):
            assert torch.equal(lm[r][0], lm[0][0]) and torch.equal(lm[r][1], lm[0][1]), (step, r, 'loss differs between ranks')
            assert torch.equal(lm[r][0], lp[r][0]) and torch.equal(lm[r][1], lp[r][1]), (step, r, 'loss')
            assert torch.equal(dxm[r], dxp[r]), (step, r, 'dx', _rel(dxm[r], dxp[r]))
            assert torch.equal(dym[r], dyp[r]), (step, r, 'dy', _rel(dym[r], dyp[r]))
            a, b = merged.bes[r], per_pass.bes[r]
            assert torch.equal(a.queue, b.queue) and torch.equal(a.queue_bf16, b.queue_bf16) and torch.equal(a.qpos, b.qpos), (step, r)
            assert torch.equal(a.queue_bf16, a.queue.to(torch.bfloat16)) and torch.equal(b.queue_bf16, b.queue.to(torch.bfloat16)), (step, r)
            assert bool((a.ovl_map == -1).all()) and bool((naive.bes[r].ovl_map == -1).all()), (step, r, 'overlay left set')
            assert a.lru.state_dict() == b.lru.state_dict(), (step, r)
        if peered is not None:
            lq, dxq, dyq = peered.merged_step(x, y, xl, yl)
            for r in range(R):
                assert torch.equal(lq[r][0], lm[r][0]) and torch.equal(lq[r][1], lm[r][1]), (step, r, 'peer loss')
                assert torch.equal(dxq[r], dxm[r]) and torch.equal(dyq[r], dym[r]), (step, r, 'peer grads')
                assert bool((peered.bes[r].ovl_map == -1).all())
        naive_wrong += int(any(not torch.equal(dxn[r], dxm[r]) for r in range(R)))
        # the fp64 oracle on the same global batch
        xo, yo = x.double().requires_grad_(True), y.double().requires_grad_(True)
        ref = oracle.forward(xo, yo, xl.tolist(), yl.tolist())
        ref.backward()
        n_out += sum(1 for v in oracle.trace[-2]['labels'] if v < 0)
        n_ones_t += sum(1 for i, v in enumerate(oracle.trace[-2]['labels']) if v >= 0 and v in set(oracle.trace[-2]['ones']))
        for r in range(R):
            be = merged.bes[r]
            assert be.lru.state_dict() == oracle.lrus[r].state_dict(), (step, r, 'lru')
            assert be.qpos.cpu().tolist() == oracle.qpos[offs[r]:offs[r] + Qls[r]], (step, r, 'qpos')
            assert torch.equal(be.queue.double(), oracle.queue[:, offs[r]:offs[r] + Qls[r]]), (step, r, 'queue')
        loss = float(lm[0][0] + lm[0][1])
        ref = float(ref.detach())
        assert abs(loss - ref) <= 1e-2 * abs(ref), (step, loss, ref)
        assert _rel(torch.cat(dxm), xo.grad) <= 1e-2, (step, 'dx', _rel(torch.cat(dxm), xo.grad))
        assert _rel(torch.cat(dym), yo.grad) <= 1e-2, (step, 'dy', _rel(torch.cat(dym), yo.grad))
    # the regime the step was meant to reach: hard-negative-only rows, targets inside `ones`, evictions, and the overlay was needed
    assert n_out > 0 and n_ones_t > 0
    for r, (keys, _) in enumerate(pre):
        resident = {k for k, _ in oracle.lrus[r].state_dict()}
        assert len(resident) == Qls[r] and not set(keys.tolist()) <= resident, (r, 'no evictions')
    print(f'merged step D={D} Q={Q} R={R} B={B} {loss_type} peer={peer}: no-overlay finalize differed in {naive_wrong} of 6 steps')
    assert naive_wrong > 0
