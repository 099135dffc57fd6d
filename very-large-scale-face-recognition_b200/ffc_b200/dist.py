"""Column-sharded FFC head over the GPUs of one node (partial-FC style; nothing like it exists in the reference,
which is single-process -- SURVEY.md section 8(e)).

Partition: rank r of R owns a contiguous range of about Q/R queue slots (the first Q mod R ranks one more) -- fp32 rows, bf16 mirror, queue positions -- and the
LRU of the identities with ``id mod R == r`` (an exact, balanced "identity hash" for dense class indices).  A rank's
LRU is bit-exact with the reference ``LRU(Q/R)`` fed the keys it owns in global batch order (rank-major, then row).

One head pass (embeddings in) per rank:
  all-gather p, g, probe/gallery labels            (NCCL over NVLink)
  own gallery keys  -> device LRU assign + enqueue scatter into the local shard      (ffc.py:162-182 / 214-241)
  probe labels      -> local view, global slot = r*Q/R + local, all-reduce MAX       (ffc.py:189-194)
  sweep of the local shard for ALL R*B rows        (same tcgen05 kernel as on one GPU)
  [SV only: the target cosines are all-reduced BEFORE the sweep -- its hard-example threshold is gt - margin, ffc.py:121-122]
  all-reduce SUM of the per-row softmax denominators / target cosines, all-gather of the top-k candidates
  finalize -> loss (identical on every rank) and this rank's partial dLoss/dp for all rows
  reduce-scatter SUM -> dLoss/dp of the rank's own B rows
No collective touches the B x Q logits (they never exist); the exchanged bytes are O(R*B*D).

The per-rank compute sits behind a small backend interface so that the collective choreography can be exercised on
CPU (gloo, world_size 2) by the tests with a torch stand-in; the product backend is :class:`CudaShardBackend`.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.distributed as dist

from . import _capi
from ._capi import HeadConfig, HeadPass, HeadStats, check
from . import identify as _ident
from .ffc import hard_neg_k
from .lru import LRU


class CudaShardBackend:
    """One rank's shard on the device, through the C ABI (no fallback)."""

    def __init__(self, feat_dim, q_local, q_total, col_offset, max_rows, scale, loss_type, margin, topk, precision, device):
        if not torch.cuda.is_available():
            raise _capi.FFCError('the sharded FFC head needs CUDA devices (no CPU fallback)')
        self.lib = _capi.lib()
        self.dev = torch.device(device)
        self.D, self.Ql, self.Q, self.off, self.R_rows, self.k = feat_dim, q_local, q_total, col_offset, max_rows, topk
        dev, D, Ql, n = self.dev, feat_dim, q_local, max_rows
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            self.lru = LRU(Ql, device=dev)
            q = torch.rand(2, Ql, D, device=dev)
            q /= q.norm(dim=2, keepdim=True).clamp_min(1e-12)
            self.queue = q
            self.queue_bf16 = torch.empty(2, Ql, D, dtype=torch.bfloat16, device=dev)
            self.qpos = torch.zeros(Ql, dtype=torch.uint8, device=dev)
            # per-pass bookkeeping state, three sets: 1 = commit pass; 0 and 2 = the rollback passes of alternating steps (the next
            # step's rollback bookkeeping -- label prefetch -- is computed while the current step still needs its own)
            self._sets = [dict(cmask=torch.zeros((Ql + 31) // 32 + 8, **i32), rows=torch.zeros(n, **i32), cols=torch.full((n,), -1, **i32),
                               ones_list=torch.empty(n, **i32), n_ones=torch.zeros(1, **i32), n=0) for _ in range(3)]
            self.use_set(0)
            self.undo_rows = torch.empty(n, D, **f32)
            cfg = HeadConfig(n, Ql, q_total, col_offset, D, _capi.LOSS_TYPES[loss_type], scale, margin, topk, _capi.PRECISIONS[precision])
            h = C.c_void_p()
            check(self.lib.ffc_head_create(C.byref(cfg), C.byref(h)))
            self._h, self._cfg = h, cfg
            self.record_path = precision == 'bf16' and loss_type in ('AM', 'Arc')
            # merged step (one statistics exchange per FFC.forward): both passes' sweep results are outstanding at once, so the commit
            # pass gets its own head workspace; the rollback pass's finalize reads rewritten queue rows through the overlay map
            self.merged = self.record_path
            self._h2 = None
            if self.merged:
                h2 = C.c_void_p()
                check(self.lib.ffc_head_create(C.byref(cfg), C.byref(h2)))
                self._h2 = h2
                self.undo_rows_cm = torch.empty(n, D, **f32)
                self.ovl_map = torch.full((2 * Ql,), -1, **i32)
        self.sync_mirror()

    def __del__(self):
        for name in ('_h', '_h2'):
            h = self.__dict__.pop(name, None)
            if h:
                try:
                    self.lib.ffc_head_destroy(h)
                except Exception:
                    pass

    def _s(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def use_set(self, i):
        st = self._sets[i]
        self._set = st
        self.cmask, self.rows, self.cols, self.ones_list, self.n_ones = st['cmask'], st['rows'], st['cols'], st['ones_list'], st['n_ones']

    def sync_mirror(self):
        check(self.lib.ffc_cast_bf16(self.queue.data_ptr(), self.queue_bf16.data_ptr(), self.queue.numel(), self._s()))

    def set_queue(self, q):
        self.queue.copy_(q.to(self.dev))
        self.sync_mirror()

    def new_stats(self, n, n_ranks):
        dev, D, k = self.dev, self.D, self.k
        red = torch.zeros(8, n, dtype=torch.float32, device=dev)          # rows 0-3 lsum, 4-7 tgt: one all-reduce
        return dict(red=red, osum=torch.empty(4, n, D, dtype=torch.float32, device=dev),
                    topv=torch.empty(n_ranks, 3, n, k, dtype=torch.float32, device=dev),
                    topi=torch.empty(n_ranks, 3, n, k, dtype=torch.int32, device=dev))

    def identify_local(self, x, k):
        """Top-k of the rows `x` [n, D] (L2-normalised here) over this shard's resident slots: global slots, labels from this
        rank's LRU (FFCHead.identify's semantics)."""
        xn = _ident.normalized_queries(x, self.D, self.dev)
        return _ident.search(self.lib, self._h, self.lru._h, xn, k, self.queue, self.queue_bf16 if self._cfg.precision == _capi.PRECISIONS['bf16'] else None)

    # -- pass steps -------------------------------------------------------------------------------
    def assign(self, keys_compact, n_dev, journal):
        n = keys_compact.numel()
        self.n_ones.zero_()
        self.cols[:n].fill_(-1)
        self.lru.assign(keys_compact, journal=journal, qpos=self.qpos, rows=self.rows, cols=self.cols, ones_list=self.ones_list,
                        n_ones=self.n_ones, cmask=self.cmask, n_dev=n_dev)
        self._set['n'] = n

    def route(self, keys_all, n_ranks, rank):
        """Stable partition of the gathered gallery keys: this rank's keys first (global batch order).  One launch."""
        n = keys_all.numel()
        keys_c = torch.empty_like(keys_all)
        order = torch.empty(n, dtype=torch.int32, device=self.dev)
        n_mine = torch.empty(1, dtype=torch.int32, device=self.dev)
        check(self.lib.ffc_route_keys(keys_all.data_ptr(), n, n_ranks, rank, keys_c.data_ptr(), order.data_ptr(), n_mine.data_ptr(), self._s()))
        return keys_c, order, n_mine

    def scatter(self, g_all, order, save_undo, overlay_table=None):
        """Enqueue this rank's gallery rows straight out of the all-gathered embeddings (row j of the bookkeeping <- g_all[order[j]]).
        overlay_table (merged step): 0 = a rollback pass's enqueue, 1 = the commit pass's enqueue that follows it in the same step --
        every winning write is recorded in the overlay map (see ffc_queue_scatter_overlay); the commit pass then saves the rows it
        replaces in its own undo buffer."""
        assert g_all.dtype == torch.float32 and g_all.is_contiguous() and order.dtype == torch.int32
        undo = (self.undo_rows_cm if overlay_table == 1 else self.undo_rows) if save_undo else None
        check(self.lib.ffc_queue_scatter_overlay(self.queue.data_ptr(), self.queue_bf16.data_ptr(), self.rows.data_ptr(), self.cols.data_ptr(),
                                                 g_all.data_ptr(), order.data_ptr(), self._set['n'], self.Ql, self.D,
                                                 None if undo is None else undo.data_ptr(),
                                                 None if overlay_table is None else self.ovl_map.data_ptr(), overlay_table or 0, self._s()))

    def overlay_clear(self, set_idx):
        st = self._sets[set_idx]
        check(self.lib.ffc_overlay_clear(self.ovl_map.data_ptr(), st['rows'].data_ptr(), st['cols'].data_ptr(), st['n'], self.Ql, self._s()))

    def undo_bookkeeping(self):
        """lru.py:252-255 + ffc.py:256-257: the LRU / queue positions of a rollback pass can be restored as soon as the probe
        labels have been read (the sweep only needs labels, `ones` and the queue rows)."""
        self.lru.undo(-1, self.qpos)

    def restore_queue(self):
        check(self.lib.ffc_queue_restore_packed(self.queue.data_ptr(), self.queue_bf16.data_ptr(), self.rows.data_ptr(), self.cols.data_ptr(),
                                         self.undo_rows.data_ptr(), self._set['n'], self.Ql, self.D, self._s()))

    def view(self, keys):
        return self.lru.view_batch(keys)

    def _structs(self, p_all, label, st, slot):
        n = p_all.shape[0]
        hp = HeadPass(p_all.data_ptr(), self.queue.data_ptr(), self.queue_bf16.data_ptr(), label.data_ptr(), self.ones_list.data_ptr(),
                      self.n_ones.data_ptr(), self.cmask.data_ptr(), n)
        red = st['red']
        hs = HeadStats(red.data_ptr(), st['osum'].data_ptr(), red.data_ptr() + 4 * n * 4, st['topv'][slot].data_ptr(), st['topi'][slot].data_ptr())
        return hp, hs

    # -- record path (one all-gather per pass instead of all-reduce + all-gather; see include/ffc_b200.h) --------------------
    def new_records(self, n, n_ranks, passes=1):
        """Record buffers: `own` [passes, words] written by sweep_record, `all` [n_ranks, passes, words] filled by ONE all-gather."""
        w = C.c_int64()
        check(self.lib.ffc_head_record_words(C.byref(self._cfg), n, C.byref(w)))
        return dict(own=torch.empty(passes, w.value, dtype=torch.float32, device=self.dev),
                    all=torch.empty(n_ranks, passes, w.value, dtype=torch.float32, device=self.dev), words=w.value, passes=passes)

    def _pass_struct(self, p_all, label):
        return HeadPass(p_all.data_ptr(), self.queue.data_ptr(), self.queue_bf16.data_ptr(), label.data_ptr(), self.ones_list.data_ptr(),
                        self.n_ones.data_ptr(), self.cmask.data_ptr(), p_all.shape[0])

    def sweep_record(self, p_all, label, rec, which=0):
        """prep + sweep + scalar reduction of one pass into rec['own'][which]; pass `which` (0 rollback / 1 commit of a merged step) uses
        its own head workspace, so both passes' partial results can be outstanding until the step's single exchange"""
        hp = self._pass_struct(p_all, label)
        check(self.lib.ffc_head_sweep_record(self._h2 if which else self._h, C.byref(hp), rec['own'][which].data_ptr(), self._s()))

    def finalize_gathered(self, p_all, label, rec, n_ranks, which=0, overlay_g=None, route=None):
        """finalize of pass `which` from the gathered records.  overlay_g: the gathered gallery embeddings of this (rollback) pass -- its
        queue rows have been restored / re-enqueued since the sweep and are read through the overlay map.  route = (peer pointer table,
        rows per rank, slot offset): dLoss/dp rows go straight to their owner rank's staging buffer (no dp tensor is returned)."""
        hp = self._pass_struct(p_all, label)
        loss = torch.empty((), dtype=torch.float32, device=self.dev)
        dp = None if route is not None else torch.empty(p_all.shape[0], self.D, dtype=torch.float32, device=self.dev)
        opts = _capi.FinalizeOpts()
        if overlay_g is not None:
            assert overlay_g.dtype == torch.float32 and overlay_g.is_contiguous()
            opts.overlay_map, opts.overlay_g, opts.overlay_undo = self.ovl_map.data_ptr(), overlay_g.data_ptr(), self.undo_rows_cm.data_ptr()
        if route is not None:
            opts.dp_peer, opts.dp_rows_per_rank, opts.dp_slot_offset = route[0].data_ptr(), int(route[1]), int(route[2])
        w, passes = rec['words'], rec['passes']
        check(self.lib.ffc_head_finalize_gathered_ex(self._h2 if which else self._h, C.byref(hp), rec['all'].data_ptr() + 4 * w * which, n_ranks,
                                                     w * passes, C.byref(opts), loss.data_ptr(), None if dp is None else dp.data_ptr(), self._s()))
        return loss, dp

    def push_record(self, p_all, rec, which, rank):
        """Record exchange by peer stores: this rank's record of pass `which` into every rank's gathered buffer (top-k slots only for
        hard-negative-only rows); ffc_head_push_record."""
        pr = rec['peer']
        check(self.lib.ffc_head_push_record(self._h2 if which else self._h, p_all.shape[0], rec['own'][which].data_ptr(), pr['ptrs'].data_ptr(),
                                            (rank * rec['passes'] + which) * rec['words'], pr['ptrs'].numel(), self._s()))

    def peer_barrier(self, flags, rank, ranks, epoch, err):
        check(self.lib.ffc_peer_barrier(flags.data_ptr(), rank, ranks, epoch & 0x7fffffff, err.data_ptr(), self._s()))

    def sum_slabs(self, slabs, n_slabs, stride, n, out, barrier=None):
        """out = sum of the slabs in order; barrier = (flag pointer table, rank, ranks, epoch, error flag): first meet the peers whose
        finalize kernels wrote the slabs (one launch)"""
        if barrier is None:
            check(self.lib.ffc_sum_slabs(slabs.data_ptr(), n_slabs, stride, n, out.data_ptr(), self._s()))
        else:
            fp, rank, ranks, epoch, err = barrier
            check(self.lib.ffc_sum_slabs_barrier(slabs.data_ptr(), n_slabs, stride, n, out.data_ptr(), fp.data_ptr(), rank, ranks, epoch & 0x7fffffff,
                                                 err.data_ptr(), self._s()))

    def sweep(self, p_all, label, st, rank_slot):
        hp, hs = self._structs(p_all, label, st, rank_slot)
        check(self.lib.ffc_head_sweep(self._h, C.byref(hp), C.byref(hs), self._s()))

    def prep(self, p_all, label, st, rank_slot):
        """first half of :meth:`sweep`: target cosines / owner flags into st['red'][4:8] (SV: summed over the ranks before the sweep)"""
        hp, hs = self._structs(p_all, label, st, rank_slot)
        check(self.lib.ffc_head_prep(self._h, C.byref(hp), C.byref(hs), self._s()))

    def sweep_prepared(self, p_all, label, st, rank_slot):
        hp, hs = self._structs(p_all, label, st, rank_slot)
        check(self.lib.ffc_head_sweep_prepared(self._h, C.byref(hp), C.byref(hs), self._s()))

    def finalize(self, p_all, label, st, n_ranks):
        hp, hs = self._structs(p_all, label, st, 0)
        dp = torch.empty(p_all.shape[0], self.D, dtype=torch.float32, device=self.dev)
        loss = torch.empty((), dtype=torch.float32, device=self.dev)
        check(self.lib.ffc_head_finalize(self._h, C.byref(hp), C.byref(hs), n_ranks, loss.data_ptr(), dp.data_ptr(), self._s()))
        return loss, dp

    def end_pass(self):
        self.cmask.zero_()

    # -- checkpoint of the shard (host-sync) ------------------------------------------------------
    def export_state(self):
        return dict(lru=self.lru.state_dict(), queue=self.queue.detach().cpu(), qpos=self.qpos.cpu().tolist())

    def import_state(self, st):
        assert tuple(st['queue'].shape) == tuple(self.queue.shape), (tuple(st['queue'].shape), tuple(self.queue.shape))
        self.lru.clear()
        self.lru.restore([(int(k), int(v)) for k, v in st['lru']])
        self.queue.copy_(st['queue'].to(self.dev))
        self.sync_mirror()
        self.qpos.copy_(torch.tensor([int(v) for v in st['qpos']], dtype=torch.uint8).to(self.dev))

    def set_timing(self, enable):
        check(self.lib.ffc_head_set_timing(self._h, 1 if enable else 0))

    def get_timing(self):
        ms, n = C.c_double(), C.c_int64()
        check(self.lib.ffc_head_get_timing(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value


class _ShardedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, head, g, probe_label, gallery_label, commit):
        loss, dp = head.head_pass(p.detach(), g, probe_label, gallery_label, commit)
        ctx.save_for_backward(dp)
        ctx.p_dtype = p.dtype
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (dp,) = ctx.saved_tensors
        return (dp * grad_out).to(ctx.p_dtype), None, None, None, None, None


class ShardedFFCHead:
    """R-way column-sharded head.  ``backend_factory(q_local, col_offset, max_rows) -> backend`` is for the CPU tests."""

    def __init__(self, feat_dim, queue_size, scale=32.0, loss_type='AM', margin=0.4, precision='bf16', max_batch=1024, device=None,
                 group=None, backend_factory=None):
        assert dist.is_initialized(), 'torch.distributed must be initialised (one process per GPU)'
        assert loss_type in ('AM', 'Arc', 'SV')
        self.loss_type = loss_type
        self.group = group
        self.R = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        assert queue_size >= self.R, 'fewer queue slots than ranks'
        # contiguous slot ranges, the first queue_size % R ranks one slot longer: any queue size shards (the reference's default is 7409, ffc.py:11)
        base, rem = divmod(queue_size, self.R)
        self.D, self.Q, self.Ql = feat_dim, queue_size, base + (1 if self.rank < rem else 0)
        self.B = max_batch
        self.k = hard_neg_k(queue_size)
        self.off = self.rank * base + min(self.rank, rem)
        n = self.R * self.B
        if backend_factory is None:
            self.backend = CudaShardBackend(feat_dim, self.Ql, queue_size, self.off, n, scale, loss_type, margin, self.k, precision, device)
            self.dev = torch.device(device)
        else:
            self.backend = backend_factory(self.Ql, self.off, n)
            self.dev = torch.device('cpu')
        self._nccl = dist.get_backend(group) == 'nccl'
        self._stats = {}
        self._timing = [] if (os.environ.get('FFC_DIST_TIMING') and self._nccl) else None
        # bookkeeping stream, high priority: its short kernels get the SMs a sweep CTA frees before the sweep's own pending CTAs do
        self._side = (torch.cuda.Stream(device=self.dev, priority=_capi.side_stream_priority())
                      if (self._nccl and not os.environ.get('FFC_DIST_NO_OVERLAP')) else None)
        self._pre = None            # labels + rollback-pass bookkeeping of the next forward_pair (see prefetch)
        self.prefetch_hits = 0      # forward_pair calls that consumed prefetched bookkeeping
        # prefetch's collectives get their own communicator: torch's NCCL backend runs all collectives of one process group on one
        # internal stream in issue order, so on the main group they would queue behind the current step's record all-gather /
        # reduce-scatter, i.e. behind the very sweeps they are meant to run under
        self._side_group = None
        if self._side is not None:
            ranks = dist.get_process_group_ranks(group) if group is not None else None
            self._side_group = dist.new_group(ranks=ranks, backend='nccl')      # its communicator is built on first use (first prefetch)
        self._rb_done = None        # event: the last pass that used bookkeeping set 0 has finished with it
        self._lru_main_ev = None    # event: the last bookkeeping enqueued on the caller's stream (the LRU state prefetch builds on)
        # merged step (bf16 AM / Arc): ONE statistics exchange per forward_pair instead of one per pass, the rollback pass's finalize
        # reading through the overlay; rollback bookkeeping alternates between sets 0 and 2 so that the next step's (prefetch) never
        # touches the set the current step still needs
        self.merged = bool(getattr(self.backend, 'merged', False)) and not os.environ.get('FFC_DIST_NO_MERGE')
        self._rb_set = 0
        self._set_free = {}         # bookkeeping set -> event: the step that used it last has finished with it
        self._route = None
        if self.merged and self._nccl:
            self._init_route(os.environ.get('FFC_DIST_NO_SYMM') is None)

    def _init_route(self, try_symm):
        """Staging for the reduce-scatter folded into finalize.  Preferred: a symmetric-memory buffer [R sources][2 passes][B][D] per
        rank (torch.distributed._symmetric_memory: peer-mapped over NVLink, torch only provides the mapping and the barrier) -- every
        rank's finalize kernels store the dLoss/dp rows of rank r's samples straight into r's buffer, one barrier, and r adds the R
        slabs in rank order (ffc_sum_slabs: deterministic).  Fallback (no peer mapping): the same stores into a local
        [R][2][B][D] buffer followed by ONE NCCL reduce-scatter per step."""
        R, B, D, dev = self.R, self.B, self.D, self.dev
        slab = 2 * B * D
        self._route = dict(kind='nccl', slab=slab)
        if try_symm:
            try:
                import torch.distributed._symmetric_memory as symm_mem
                stage = symm_mem.empty(R * slab + 64, dtype=torch.float32, device=dev)          # + the barrier's flag words (int32[R])
                hdl = symm_mem.rendezvous(stage, self.group if self.group is not None else dist.group.WORLD)
                ptrs = [int(p) for p in hdl.buffer_ptrs]
                assert len(ptrs) == R and ptrs[self.rank] == stage.data_ptr() and R <= 64
                stage.zero_()
                ok = torch.ones(1, device=dev)
                self._route.update(kind='symm', stage=stage, hdl=hdl, ptrs=torch.tensor(ptrs, dtype=torch.int64, device=dev),
                                   flags=torch.tensor([p + 4 * R * slab for p in ptrs], dtype=torch.int64, device=dev),
                                   err=torch.zeros(1, dtype=torch.int32, device=dev), epoch=0)
            except Exception as e:      # noqa: BLE001 -- any failure of the optional peer mapping selects the NCCL route
                ok = torch.zeros(1, device=dev)
                self._route['symm_error'] = repr(e)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)     # all ranks take the same route
            if float(ok) == 0.0:
                self._route = dict(kind='nccl', slab=slab, symm_error=self._route.get('symm_error'))
        if self._route['kind'] == 'nccl':
            stage = torch.empty(R * slab, dtype=torch.float32, device=dev)
            self._route.update(stage=stage, ptrs=torch.tensor([stage.data_ptr() + 4 * r * slab for r in range(R)], dtype=torch.int64, device=dev))

    def _peer_records(self, n):
        """Gathered-record buffers of the merged step in symmetric memory: [R ranks][2 passes][words] + the barrier's flag words, peer-mapped
        like the gradient staging.  The ranks then exchange their records by peer stores (ffc_head_push_record: the scalars of every row,
        the top-k slots only of hard-negative-only rows -- 12 % of the bytes an all-gather moves when there are none) and ONE
        ffc_peer_barrier.  None when the peer route is not available or not asked for (NCCL all-gather then)."""
        be, R, dev = self.backend, self.R, self.dev
        # Opt-in (FFC_DIST_PEER_RECORDS=1): NCCL parity tests green at 2 and 8 GPUs with it on, the exchange itself 0.14 -> 0.08 ms per step at
        # 8 GPUs, but the one 8-GPU run measured with it showed the step's [x | y] all-gather at 0.50 ms against 0.13 in every run before, with
        # no GPU budget left to tell a slow box from a side effect (profiles/r2_dist_8gpu.md) -- the all-gather stays the default.
        if self._route is None or self._route.get('kind') != 'symm' or not os.environ.get('FFC_DIST_PEER_RECORDS'):
            return None
        import torch.distributed._symmetric_memory as symm_mem
        w = be.new_records(n, 1, passes=1)['words']
        ws = (w + 3) // 4 * 4                                    # 16-byte aligned records
        buf = symm_mem.empty(R * 2 * ws + 64, dtype=torch.float32, device=dev)
        hdl = symm_mem.rendezvous(buf, self.group if self.group is not None else dist.group.WORLD)
        ptrs = [int(p) for p in hdl.buffer_ptrs]
        assert len(ptrs) == R and ptrs[self.rank] == buf.data_ptr()
        buf.zero_()
        dist.barrier(group=self.group)                           # every rank's flag words are zero before anyone signals
        return dict(own=torch.zeros(2, ws, dtype=torch.float32, device=dev), all=buf[:R * 2 * ws].view(R, 2, ws), words=ws, passes=2, buf=buf, hdl=hdl,
                    peer=dict(ptrs=torch.tensor(ptrs, dtype=torch.int64, device=dev),
                              flags=torch.tensor([p + 4 * R * 2 * ws for p in ptrs], dtype=torch.int64, device=dev),
                              err=torch.zeros(1, dtype=torch.int32, device=dev), epoch=0))

    # -- helpers ----------------------------------------------------------------------------------
    def shard_of(self, keys):
        """Owner rank of each identity: floor-mod (exact and balanced for dense class indices)."""
        return torch.remainder(keys, self.R)

    def _all_gather(self, t, group=None):
        out = torch.empty((self.R * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t.contiguous(), group=group if group is not None else self.group)
        return out

    def _reduce_scatter(self, t):
        B = t.shape[0] // self.R
        if self._nccl:
            out = torch.empty((B,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
            dist.reduce_scatter_tensor(out, t, group=self.group)
            return out
        dist.all_reduce(t, group=self.group)                       # gloo (CPU tests): no reduce_scatter
        return t[self.rank * B:(self.rank + 1) * B].clone()

    def prefill_identity(self, n_ids):
        """Steady state for benchmarks: identities 0..n_ids-1 resident, id i in local slot i // R of rank i % R."""
        keys = torch.arange(self.rank, n_ids, self.R, dtype=torch.int64)[:self.Ql]
        self.backend.lru.restore_arrays(keys, torch.arange(keys.numel(), dtype=torch.int32))

    # -- one pass ---------------------------------------------------------------------------------
    def _mark(self, name):
        # optional per-phase device timing (FFC_DIST_TIMING=1): CUDA events on the current stream, read by phase_times()
        if self._timing is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self._timing.append((name, ev))

    def phase_times(self):
        """{phase: total ms} accumulated since construction (synchronises); needs FFC_DIST_TIMING=1."""
        out = {}
        if self._timing:
            torch.cuda.synchronize()
            for (n0, e0), (n1, e1) in zip(self._timing[:-1], self._timing[1:]):
                if n1 != 'start':
                    out[n1] = out.get(n1, 0.0) + e0.elapsed_time(e1)
        return out

    def gather(self, emb, label):
        """All-gather one side of the batch (embeddings [B,D] + labels [B]) -> ([R*B,D], int64 [R*B])."""
        be, dev = self.backend, self.dev
        assert emb.shape[0] == self.B, f'every rank must feed max_batch={self.B} rows (got {emb.shape[0]})'
        fdt = getattr(be, 'dtype', torch.float32)
        e_all = self._all_gather(emb.detach().to(device=dev, dtype=fdt))
        l_all = self._all_gather(torch.as_tensor(label).to(device=dev, dtype=torch.int64))
        return e_all, l_all

    def staging(self):
        """The rank's slice of the packed all-gather input, as two fp32 [B, D] views (x, y).  Hand them to the backbone tail
        (``FFCTail(...)(feat, out=view)`` / ``l2_normalize(feat, out=view)``, csrc/tail.cu) and pass the results to
        :meth:`forward_pair`: the unit-norm rows are then written ONCE, where the exchange reads them (SURVEY 8(f) rank 3's
        "all-gather staging"); any other tensors are copied in.  The views stay valid for the life of the head; a step's rows must
        be written after the previous forward_pair call has returned."""
        if getattr(self, '_own', None) is None:
            ne = self.B * self.D
            self._own = torch.empty(2 * ne + 4 * self.B, dtype=torch.float32, device=self.dev)      # [x | y | x_label, y_label (int64)]
        ne = self.B * self.D
        return self._own[:ne].view(self.B, self.D), self._own[ne:2 * ne].view(self.B, self.D)

    def gather_pair(self, x, y, x_label=None, y_label=None):
        """Both sides of the batch in ONE all-gather (NCCL): each rank contributes [x | y | x_label | y_label] as one packed
        buffer of 4-byte words.  Returns (x_all, xl_all, y_all, yl_all) in global batch order (rank-major); without labels
        (they were exchanged by :meth:`prefetch`) the buffer is [x | y] and the label entries are None."""
        with_labels = x_label is not None
        if not self._nccl:
            if with_labels:
                return self.gather(x, x_label) + self.gather(y, y_label)
            fdt = getattr(self.backend, 'dtype', torch.float32)
            return (self._all_gather(x.detach().to(device=self.dev, dtype=fdt)), None, self._all_gather(y.detach().to(device=self.dev, dtype=fdt)), None)
        dev, B, D, R = self.dev, self.B, self.D, self.R
        assert x.shape == (B, D) and y.shape == (B, D), f'every rank must feed max_batch={B} rows of {D} features'
        ne = B * D
        sx, sy = self.staging()
        own = self._own if with_labels else self._own[:2 * ne]
        # rows the backbone tail already wrote into the staging views (FFCTail / l2_normalize `out=`) are not copied again
        if not (x.data_ptr() == sx.data_ptr() and x.is_contiguous() and x.dtype == torch.float32):
            sx.copy_(x.detach())
        if not (y.data_ptr() == sy.data_ptr() and y.is_contiguous() and y.dtype == torch.float32):
            sy.copy_(y.detach())
        if with_labels:
            lab = own[2 * ne:].view(torch.int64)
            lab[:B].copy_(torch.as_tensor(x_label).reshape(B), non_blocking=True)
            lab[B:].copy_(torch.as_tensor(y_label).reshape(B), non_blocking=True)
        buf = torch.empty(R, own.numel(), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(buf, own, group=self.group)
        x_all, y_all = buf[:, :ne].reshape(R * B, D), buf[:, ne:2 * ne].reshape(R * B, D)
        if not with_labels:
            return x_all, None, y_all, None
        labs = buf[:, 2 * ne:].view(torch.int64)                      # [R, 2B]
        return x_all, labs[:, :B].reshape(R * B), y_all, labs[:, B:].reshape(R * B)

    # -- label prefetch (SURVEY 8(f) rank 4: the labels of a step are known long before its embeddings) --------------------------
    def prefetch(self, x_label, y_label):
        """Hand over the labels of the NEXT :meth:`forward_pair` now.  They are all-gathered and the rollback pass's bookkeeping
        (route, LRU try_get + undo, probe labels: ffc.py:214-235, 242-246, 256-259) is enqueued on the bookkeeping stream, where
        it runs underneath the sweeps already queued on the caller's stream (it only needs the LRU state the previous commit
        pass left, and bookkeeping set 0, which the previous rollback pass has released).  The next forward_pair must be given
        these same label objects (or none); any other call discards the prefetched work, which leaves no trace (a rollback
        pass's bookkeeping undoes itself).  Pass CPU tensors (the reference's contract, main.py:59-60): CUDA labels make the
        bookkeeping stream wait for the caller's stream, i.e. no overlap."""
        self._discard_prefetch()
        if self._side is None:
            xl_all, yl_all = self._gather_labels(x_label, y_label)
            ctx = self._bookkeep(xl_all, yl_all, False, self._next_rb_set())
            self._pre = dict(xl=xl_all, yl=yl_all, ctx=ctx, ev=None, src=(x_label, y_label))
            return
        main = torch.cuda.current_stream(self.dev)
        on_dev = any(torch.is_tensor(t) and t.is_cuda for t in (x_label, y_label))
        with torch.cuda.stream(self._side):
            if on_dev:
                ev_in = torch.cuda.Event()
                ev_in.record(main)
                self._side.wait_event(ev_in)
            rb_set = self._next_rb_set()
            for e in (self._set_free.get(rb_set) if self.merged else self._rb_done, self._lru_main_ev):
                if e is not None:
                    self._side.wait_event(e)
            timing, self._timing = self._timing, None
            xl_all, yl_all = self._gather_labels(x_label, y_label, self._side_group)
            ctx = self._bookkeep(xl_all, yl_all, False, rb_set, group=self._side_group)
            self._timing = timing
            ev = torch.cuda.Event()
            ev.record(self._side)
        self._pre = dict(xl=xl_all, yl=yl_all, ctx=ctx, ev=ev, src=(x_label, y_label))

    prefetch_labels = prefetch          # the name ffc_b200/train.py looks for (same hook on the one-GPU head)

    def _gather_labels(self, x_label, y_label, group=None):
        B, R = self.B, self.R
        own = torch.empty(2 * B, dtype=torch.int64, device=self.dev)
        own[:B].copy_(torch.as_tensor(x_label).reshape(B), non_blocking=True)
        own[B:].copy_(torch.as_tensor(y_label).reshape(B), non_blocking=True)
        labs = self._all_gather(own, group).view(R, 2 * B)
        return labs[:, :B].reshape(R * B), labs[:, B:].reshape(R * B)

    def _next_rb_set(self):
        """bookkeeping set of the NEXT rollback pass: merged steps alternate between 0 and 2, the per-pass flow always uses 0"""
        return (2 - self._rb_set) if self.merged else 0

    def _discard_prefetch(self):
        pre, self._pre = self._pre, None
        if pre is None:
            return
        # the LRU / queue positions were restored by the bookkeeping itself; only the set's `ones` mask has to be cleared
        be = self.backend
        set_idx = pre['ctx']['set']
        if self._side is not None:
            with torch.cuda.stream(self._side):
                if hasattr(be, 'use_set'):
                    be.use_set(set_idx)
                be.end_pass()
                ev = torch.cuda.Event()
                ev.record(self._side)
            torch.cuda.current_stream(self.dev).wait_event(ev)
        else:
            if hasattr(be, 'use_set'):
                be.use_set(set_idx)
            be.end_pass()

    def _take_prefetch(self, x_label, y_label):
        pre = self._pre
        if pre is None:
            return None
        if (x_label is None and y_label is None) or (x_label is pre['src'][0] and y_label is pre['src'][1]):
            self._pre = None
            self.prefetch_hits += 1
            return pre
        self._discard_prefetch()
        return None

    def head_pass(self, p, g, probe_label, gallery_label, commit):
        self._discard_prefetch()
        self._mark('start')
        p_all, pl_all = self.gather(p, probe_label)
        g_all, gl_all = self.gather(g, gallery_label)
        self._mark('all_gather')
        return self.head_pass_gathered(p_all, g_all, pl_all, gl_all, commit)

    def forward_pair(self, x, y, x_label=None, y_label=None):
        """ffc.py:264-267 on embeddings without autograd glue: both passes share ONE all-gather of (x, x_label) and
        (y, y_label), since the commit pass only swaps the roles.  Returns (loss, dLoss/dx, dLoss/dy) for the rank's rows.
        After :meth:`prefetch` the labels (and the rollback pass's bookkeeping) are already there: only [x | y] is gathered."""
        self._mark('start')
        pre = self._take_prefetch(x_label, y_label)
        if pre is None:
            assert x_label is not None and y_label is not None, 'labels are required unless they were handed to prefetch()'
            x_all, xl_all, y_all, yl_all = self.gather_pair(x, y, x_label, y_label)
            self._mark('all_gather')
            ctx_rb = self._bookkeep(xl_all, yl_all, False, self._next_rb_set())
        else:
            x_all, _, y_all, _ = self.gather_pair(x, y)
            self._mark('all_gather')
            xl_all, yl_all, ctx_rb = pre['xl'], pre['yl'], pre['ctx']
            if pre['ev'] is not None:
                main = torch.cuda.current_stream(self.dev)
                main.wait_event(pre['ev'])
                for t in list(ctx_rb.values()) + [xl_all, yl_all]:
                    if torch.is_tensor(t):
                        t.record_stream(main)
        if self.merged:
            return self._forward_pair_merged(x_all, y_all, xl_all, yl_all, ctx_rb)
        if self._nccl and self._side is not None:
            # the commit pass's bookkeeping (LRU assign, probe labels) only needs the LRU state, which the rollback pass has
            # already restored: run it on a side stream underneath the rollback pass's sweep
            main = torch.cuda.current_stream(self.dev)
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(self._side):
                self._side.wait_event(ev)
                timing, self._timing = self._timing, None
                ctx_cm = self._bookkeep(yl_all, xl_all, True, 1)
                self._timing = timing
                ev_cm = torch.cuda.Event()
                ev_cm.record(self._side)
            for t in ctx_cm.values():
                if torch.is_tensor(t):
                    t.record_stream(main)
            l2, dx = self._finish(x_all, y_all, ctx_rb, False)
            main.wait_event(ev_cm)
        else:
            l2, dx = self._finish(x_all, y_all, ctx_rb, False)
            ctx_cm = self._bookkeep(yl_all, xl_all, True, 1)
        self._mark('start')
        l1, dy = self._finish(y_all, x_all, ctx_cm, True)
        return l1 + l2, dx, dy

    def _forward_pair_merged(self, x_all, y_all, xl_all, yl_all, ctx_rb):
        """One step with ONE statistics exchange (bf16 AM / Arc):
            enqueue_rb -> sweep_rb -> restore -> enqueue_cm -> sweep_cm -> all-gather of both passes' records -> finalize_rb (through the
            overlay: its queue rows have been restored / re-enqueued since its sweep) -> finalize_cm -> dLoss/dp of both passes to their
            owner ranks.
        Three rendezvous per step ([x | y] all-gather, records, gradient rows) instead of five, the rank skew of two sweeps absorbed once;
        the reduce-scatter is folded into finalize (peer stores + one barrier + a local fixed-order sum) when the ranks' staging buffers
        are peer-mapped, and is one NCCL reduce-scatter per step otherwise."""
        be, R, B, D = self.backend, self.R, self.B, self.D
        n = x_all.shape[0]
        rec = self._stats.get(('rec2', n))
        if rec is None:
            rec = self._peer_records(n) if self._nccl else None
            if rec is None:
                rec = be.new_records(n, R, passes=2)
            self._stats[('rec2', n)] = rec
        rb_set = ctx_rb['set']
        self._rb_set = rb_set
        main = torch.cuda.current_stream(self.dev) if self._nccl else None
        # commit pass's bookkeeping: on the side stream underneath the rollback sweep (it only needs the LRU, which the rollback
        # bookkeeping has already restored)
        if self._side is not None:
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(self._side):
                self._side.wait_event(ev)
                if self._set_free.get(1) is not None:
                    self._side.wait_event(self._set_free[1])
                timing, self._timing = self._timing, None
                ctx_cm = self._bookkeep(yl_all, xl_all, True, 1)
                self._timing = timing
                ev_cm = torch.cuda.Event()
                ev_cm.record(self._side)
            for t in ctx_cm.values():
                if torch.is_tensor(t):
                    t.record_stream(main)
        else:
            ctx_cm = None
        # rollback pass: enqueue (+ overlay marks), sweep, restore
        be.use_set(rb_set)
        be.scatter(y_all, ctx_rb['order'], save_undo=True, overlay_table=0)
        self._mark('scatter')
        be.sweep_record(x_all, ctx_rb['label'], rec, 0)
        if 'peer' in rec:
            be.push_record(x_all, rec, 0, self.rank)
        self._mark('sweep')
        be.restore_queue()
        be.end_pass()
        self._mark('restore')
        # commit pass: enqueue (+ overlay marks, previous rows saved), sweep
        if ctx_cm is None:
            ctx_cm = self._bookkeep(yl_all, xl_all, True, 1)
        else:
            main.wait_event(ev_cm)
        be.use_set(1)
        be.scatter(x_all, ctx_cm['order'], save_undo=True, overlay_table=1)
        self._mark('scatter')
        be.sweep_record(y_all, ctx_cm['label'], rec, 1)
        be.end_pass()
        self._mark('sweep')
        # the step's single statistics exchange: by peer stores + one barrier, or one NCCL all-gather
        if 'peer' in rec:
            be.push_record(y_all, rec, 1, self.rank)
            pr = rec['peer']
            pr['epoch'] += 1
            be.peer_barrier(pr['flags'], self.rank, R, pr['epoch'], pr['err'])
        else:
            dist.all_gather_into_tensor(rec['all'].view(-1, rec['words']), rec['own'], group=self.group)
        self._mark('stat_exchange')
        route = self._route
        if route is not None:
            slab = route['slab']
            base = self.rank * slab if route['kind'] == 'symm' else 0
            r_rb, r_cm = (route['ptrs'], B, base), (route['ptrs'], B, base + B * D)
        else:
            r_rb = r_cm = None
        be.use_set(rb_set)
        l2, dx_part = be.finalize_gathered(x_all, ctx_rb['label'], rec, R, 0, overlay_g=y_all, route=r_rb)
        be.use_set(1)
        l1, dy_part = be.finalize_gathered(y_all, ctx_cm['label'], rec, R, 1, route=r_cm)
        be.overlay_clear(rb_set)
        be.overlay_clear(1)
        self._mark('finalize')
        if route is None:                              # CPU stand-in (gloo): plain sum of both passes' partial gradients
            both = torch.stack([dx_part, dy_part])
            dist.all_reduce(both, group=self.group)
            sl = slice(self.rank * B, (self.rank + 1) * B)
            dx, dy = both[0, sl].clone(), both[1, sl].clone()
        else:
            out = torch.empty(2, B, D, dtype=torch.float32, device=self.dev)
            if route['kind'] == 'symm':
                # one launch: meet the peers (their finalize stores have landed in this rank's staging buffer), then add the R slabs
                route['epoch'] += 1
                be.sum_slabs(route['stage'], R, route['slab'], route['slab'], out,
                             barrier=(route['flags'], self.rank, R, route['epoch'], route['err']))
            else:
                dist.reduce_scatter_tensor(out.view(-1), route['stage'], group=self.group)
            dx, dy = out[0], out[1]
        self._mark('reduce_scatter')
        if self._side is not None:
            for st_idx in (rb_set, 1):
                self._set_free[st_idx] = torch.cuda.Event()
                self._set_free[st_idx].record()
        self._last = dict(label=ctx_cm['label'], n_mine=ctx_cm['n_mine'])
        return l1 + l2, dx, dy

    def _bookkeep(self, pl_all, gl_all, commit, set_idx, group=None):
        """Route this rank's gallery keys, run the LRU (+ immediate undo on a rollback pass) and resolve the probe labels.
        Touches only LRU state and bookkeeping set `set_idx`; never the queue rows."""
        be = self.backend
        if hasattr(be, 'use_set'):
            be.use_set(set_idx)
        if hasattr(be, 'route'):
            keys_c, order, n_mine = be.route(gl_all, self.R, self.rank)
        else:
            mine = self.shard_of(gl_all) == self.rank
            order = torch.argsort((~mine).to(torch.int8), stable=True)
            n_mine = mine.sum().to(torch.int32).reshape(1)
            keys_c = gl_all[order].contiguous()
        self._mark('route')
        be.assign(keys_c, n_mine, journal=not commit)
        self._mark('lru_assign')
        # probe labels: only the owner's LRU can know the key; everyone else answers -1
        loc = be.view(pl_all)
        label = torch.where(loc >= 0, loc + self.off, loc).to(torch.int32)
        if not commit:
            be.undo_bookkeeping()
        dist.all_reduce(label, op=dist.ReduceOp.MAX, group=group if group is not None else self.group)
        self._mark('labels')
        if self._side is not None and torch.cuda.current_stream(self.dev) != self._side:
            self._lru_main_ev = torch.cuda.Event()
            self._lru_main_ev.record()
        return dict(order=order, label=label, n_mine=n_mine, set=set_idx)

    def _finish(self, p_all, g_all, ctx, commit):
        be, R = self.backend, self.R
        n = p_all.shape[0]
        if hasattr(be, 'use_set'):
            be.use_set(ctx['set'])
        be.scatter(g_all, ctx['order'], save_undo=not commit)
        self._mark('scatter')
        label = ctx['label']
        if getattr(be, 'record_path', False):
            # one record per rank and pass, one all-gather, finalize straight from the sweep partials
            rec = self._stats.get(('rec', n))
            if rec is None:
                rec = self._stats[('rec', n)] = be.new_records(n, R)
            be.sweep_record(p_all, label, rec)
            self._mark('sweep')
            dist.all_gather_into_tensor(rec['all'].view(-1, rec['words']), rec['own'], group=self.group)
            self._mark('stat_exchange')
            loss, dp_part = be.finalize_gathered(p_all, label, rec, R)
            self._mark('finalize')
            return self._finish_tail(be, dp_part, loss, label, ctx, commit)
        st = self._stats.get(n)
        if st is None:
            st = self._stats[n] = be.new_stats(n, R)
        if self.loss_type == 'SV':
            # ffc.py:121-122: the hard-example threshold of a row is its target cosine - margin, known only to the rank that owns the
            # target column: sum the target cosines over the ranks first (owner's value + zeros), then sweep
            be.prep(p_all, label, st, self.rank)
            dist.all_reduce(st['red'][4:], group=self.group)
            be.sweep_prepared(p_all, label, st, self.rank)
            self._mark('sweep')
            dist.all_reduce(st['red'][:4], group=self.group)
        else:
            be.sweep(p_all, label, st, self.rank)
            self._mark('sweep')
            dist.all_reduce(st['red'], group=self.group)
        if R > 1 and st['topv'].dtype != torch.float32:     # CPU stand-in backend (fp64 values): two plain gathers
            tv, ti = st['topv'][self.rank].clone(), st['topi'][self.rank].clone()
            dist.all_gather_into_tensor(st['topv'].view(R * 3, n, -1), tv, group=self.group)
            dist.all_gather_into_tensor(st['topi'].view(R * 3, n, -1), ti, group=self.group)
        elif R > 1:
            # one all-gather for values and indices: both are 4-byte words
            k = st['topv'].shape[-1]
            mine_pack = torch.cat([st['topv'][self.rank].view(torch.int32), st['topi'][self.rank]], dim=0)    # [6, n, k]
            pack = torch.empty(R * 6, n, k, dtype=torch.int32, device=mine_pack.device)
            dist.all_gather_into_tensor(pack, mine_pack, group=self.group)
            pack = pack.view(R, 2, 3, n, k)
            st['topv'].copy_(pack[:, 0].view(torch.float32))
            st['topi'].copy_(pack[:, 1])
        self._mark('stat_exchange')
        loss, dp_part = be.finalize(p_all, label, st, R)
        self._mark('finalize')
        return self._finish_tail(be, dp_part, loss, label, ctx, commit)

    def _finish_tail(self, be, dp_part, loss, label, ctx, commit):
        dp = self._reduce_scatter(dp_part)
        self._mark('reduce_scatter')
        if not commit:
            be.restore_queue()
        be.end_pass()
        if self._side is not None and ctx['set'] == 0:
            self._rb_done = torch.cuda.Event()
            self._rb_done.record()
        if self._side is not None and self.merged:      # a single pass between merged steps: its set is busy until here
            self._set_free[ctx['set']] = torch.cuda.Event()
            self._set_free[ctx['set']].record()
        self._mark('restore')
        self._last = dict(label=label, n_mine=ctx['n_mine'])
        return loss, dp

    # -- checkpoint / resume: one dict per rank, the reference's wire format (main.py:84-85) for the rank's shard -----------------
    def checkpoint(self):
        """``{'lru': [(key, local slot)] most -> least recently used (lru.py:102-108), 'fc': the rank's [2, Q/R, D] queue rows on the
        CPU, 'qp': {local slot: 0 / 1} (ffc.py:41-43), 'shard': (rank, ranks, queue_size)}`` -- what main.py:85 saves, per shard: the
        recency order of a sharded LRU exists per shard only (each is the reference LRU(Q/R) of the identities it owns).  Save one
        file per rank; resume with the same number of ranks."""
        self._discard_prefetch()
        if self._side is not None:
            self._side.synchronize()
        st = self.backend.export_state()
        return {'lru': st['lru'], 'fc': st['queue'], 'qp': dict(enumerate(st['qpos'])), 'shard': (self.rank, self.R, self.Q)}

    def load_checkpoint(self, ckpt):
        assert tuple(ckpt['shard']) == (self.rank, self.R, self.Q), f"checkpoint of shard {tuple(ckpt['shard'])}, this is {(self.rank, self.R, self.Q)}"
        self._discard_prefetch()
        if self._side is not None:
            self._side.synchronize()
        self.backend.import_state(dict(lru=ckpt['lru'], queue=ckpt['fc'], qpos=[ckpt['qp'][i] for i in range(self.Ql)]))
        if self._side is not None:      # the bookkeeping stream must see the imported state
            torch.cuda.current_stream(self.dev).synchronize()

    def head_pass_gathered(self, p_all, g_all, pl_all, gl_all, commit):
        ctx = self._bookkeep(pl_all, gl_all, commit, 0)
        return self._finish(p_all, g_all, ctx, commit)

    def head(self, p, g, probe_label, gallery_label, commit=True):
        return _ShardedFn.apply(p, self, g, probe_label, gallery_label, commit)

    def forward(self, x, y, x_label, y_label):
        """ffc.py:264-267 with embeddings in (rollback pass, then commit pass)."""
        return self.head(x, y.detach(), x_label, y_label, commit=False) + self.head(y, x.detach(), y_label, x_label, commit=True)

    def identify(self, x, k=1):
        """1:N identification across the shards (collective: every rank calls it with its own rows, any number of them).  The
        queries are all-gathered, every rank searches its shard (its LRU's resident slots) with :meth:`FFCHead.identify`'s
        semantics, one all-gather exchanges the packed candidates, and each rank merges its own rows by (score desc, slot asc):
        the result equals a one-GPU search over the union of the shards.  Returns ``Identification`` [N, k] for this rank's rows."""
        k = _ident.check_k(k)
        be, R, dev = self.backend, self.R, self.dev
        with torch.no_grad():
            if self._side is not None:
                torch.cuda.current_stream(dev).wait_stream(self._side)    # bookkeeping already enqueued (a prefetch undoes itself)
            x = torch.as_tensor(x)
            n = x.shape[0] if x.dim() >= 1 else 0
            counts = self._all_gather(torch.tensor([n], dtype=torch.int64, device=dev)).tolist()
            n_max = max(counts)
            if n_max == 0:
                return _ident.empty(0, k, dev)
            if n and (x.dim() != 2 or x.shape[1] != self.D):
                raise ValueError(f'identify expects [N, {self.D}] embeddings, got {tuple(x.shape)}')
            pad = torch.zeros(n_max, self.D, dtype=getattr(be, 'dtype', torch.float32), device=dev)
            pad[:n] = x.to(device=dev, dtype=pad.dtype)
            x_all = self._all_gather(pad)                                    # [R * n_max, D] raw rows (zero rows pad)
            loc = be.identify_local(x_all, k)
            # one all-gather of (score, label, slot) packed as 3 x 8-byte words per entry
            pack = torch.stack([loc.scores.double().view(torch.int64), loc.labels, loc.slots.long()], dim=-1)     # [R * n_max, k, 3]
            allp = self._all_gather(pack).view(R, R, n_max, k, 3)[:, self.rank, :n]     # [source rank, own rows, k, 3]
            cand = allp.permute(1, 0, 2, 3).reshape(n, R * k, 3)
            out = _ident.merge(cand[..., 0].contiguous().view(torch.float64).float(), cand[..., 1], cand[..., 2].to(torch.int32), k)
            if self._side is not None:
                self._lru_main_ev = torch.cuda.Event()
                self._lru_main_ev.record()                                   # a later prefetch must not rewrite the LRU under the search
        return out

    def barrier_timeouts(self):
        """Number of in-kernel cross-rank barriers (gradient slabs, record exchange) that gave up waiting for a peer (5 s) since
        construction; anything but 0 means wrong results.  Synchronises."""
        n = 0
        if self._route is not None and 'err' in self._route:
            n += int(self._route['err'].item())
        for rec in self._stats.values():
            if isinstance(rec, dict) and 'peer' in rec:
                n += int(rec['peer']['err'].item())
        return n

    def set_timing(self, enable):
        self.backend.set_timing(enable)

    def get_timing(self):
        return self.backend.get_timing()
