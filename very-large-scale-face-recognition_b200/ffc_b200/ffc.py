"""Drop-in for the reference ``ffc.FFC`` (ffc.py:10-267) with the head on hand-written sm_100a kernels.

``FFC(net_type, feat_dim, queue_size, scale, loss_type, margin, momentum, ...)`` and
``FFC.forward(x, y, x_label, y_label) -> loss`` keep the reference's contract (main.py:64-65,116-117); the
attributes callers read (``probe_net``, ``gallery_net``, ``queue``, ``lru``, ``queue_position_dict``, ``mask``)
are there.  The head-level entry named by the build spec is :meth:`FFCHead.head`:
``head(p, g, probe_label, gallery_label, commit) -> loss`` differentiable w.r.t. ``p``.

Everything below the Python surface goes through the C ABI in include/ffc_b200.h; there is no PyTorch or CPU
fallback for the head (a missing library or device raises).
"""
from __future__ import annotations

import ctypes as C

import torch
from torch.nn import Module

from . import _capi
from . import identify as _ident
from ._capi import HeadConfig, HeadPass, HeadStats, check
from .lru import LRU
from .tail import l2_normalize


def hard_neg_k(queue_size: int) -> int:
    """ffc.py:48"""
    return min(max(int(queue_size * 0.0002), 3), 10)


class NormalizeNet(Module):
    """Head-only stand-in backbone (``net_type='identity'``): L2-normalise the input embeddings, which is what
    every reference backbone ends with (mobilefacenet_def.py:114, resnet_arcface.py:151, resnet_std.py:202)."""

    def __init__(self, feat_dim=None, **_):
        super().__init__()
        self.dummy = torch.nn.Parameter(torch.zeros(1))

    def forward(self, x):
        return l2_normalize(x + 0.0 * self.dummy)       # csrc/tail.cu: the head normalises the embeddings it is fed


def _default_create_net(net_type, **kwargs):
    if net_type in ('identity', 'none', None):
        return NormalizeNet(**kwargs)
    try:  # inside the reference tree this resolves to model/__init__.py:create_net
        from model import create_net as ref_create_net
        if net_type == 'ir100':   # C4's backbone: defined in the reference (resnet_arcface.py:177) but not registered in its create_net
            from model.resnet_arcface import iresnet100
            return iresnet100(**kwargs)
    except ImportError as e:
        raise ValueError(f"net_type {net_type!r}: backbones are outside this package; run inside the reference tree "
                         "(its model/ package on sys.path), pass nn.Module instances via probe_net=/gallery_net=, "
                         "or use net_type='identity' for head-only use") from e
    return ref_create_net(net_type, **kwargs)


create_net = _default_create_net


class _HeadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, head, g, probe_label, gallery_label, commit):
        loss, dp = head._pass(p.detach(), g, probe_label, gallery_label, commit)
        ctx.save_for_backward(dp)
        ctx.p_dtype = p.dtype
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (dp,) = ctx.saved_tensors
        return (dp * grad_out).to(ctx.p_dtype), None, None, None, None, None


class _HeadPairFn(torch.autograd.Function):
    """Both passes of ffc.py:264-267 in one call, so that the commit pass's bookkeeping can run under the rollback sweep."""

    @staticmethod
    def forward(ctx, p_rb, p_cm, head, g_rb, g_cm, x_label, y_label):
        loss, d_rb, d_cm = head.forward_pair(p_rb.detach(), g_rb, p_cm.detach(), g_cm, x_label, y_label)
        ctx.save_for_backward(d_rb, d_cm)
        ctx.dtypes = (p_rb.dtype, p_cm.dtype)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        d_rb, d_cm = ctx.saved_tensors
        return (d_rb * grad_out).to(ctx.dtypes[0]), (d_cm * grad_out).to(ctx.dtypes[1]), None, None, None, None, None


class FFCHead(Module):
    """State and kernels of the FFC head: prototype queue [2,Q,D] (+ bf16 mirror), device LRU, queue positions."""

    def __init__(self, feat_dim, queue_size, scale=32.0, loss_type='AM', margin=0.4, precision='bf16', max_batch=1024, device=None, queue_grad=False):
        super().__init__()
        assert loss_type in ('AM', 'Arc', 'SV')
        assert precision in _capi.PRECISIONS
        self.feat_dim, self.queue_size = int(feat_dim), int(queue_size)
        self.scale, self.margin, self.loss_type = float(scale), float(margin), loss_type
        self.precision = precision
        self.hard_neg = hard_neg_k(self.queue_size)
        self.max_batch = int(max_batch)
        # Optional, off by default (the reference's queue is a no-grad buffer, ffc.py:29): also compute dLoss/dQueue.  After every head
        # pass `dqueue_pass` [2, Q, D] holds d(loss of that pass)/d(queue as the pass swept it) for an upstream gradient of 1, and
        # `dqueue` accumulates it over passes until zero_dqueue() -- a caller that trains the prototypes applies it after
        # loss.backward(), multiplied by whatever factor scales the loss (a GradScaler's).  Every loss type, both precisions (the
        # check mode's gradient is fp64-accumulated and bit-identical from run to run); ShardedFFCHead has the same option per shard.
        self.queue_grad = bool(queue_grad)
        self.dqueue = self.dqueue_pass = None
        q = torch.rand(2, self.queue_size, self.feat_dim, device=device)                                     # ffc.py:29-30
        q /= q.norm(dim=2, keepdim=True).clamp_min(1e-12)
        self.register_buffer('queue', q)
        self.register_buffer('mask', torch.zeros(self.queue_size, 1, device=device))                        # ffc.py:45
        self._dev = None
        self._lru = None
        self._compact = {}
        self._pending_lru = None
        self._pending_qpos = None
        self._mirror_version, self._mirror_ptr = -1, 0
        self._pre = None                # rollback-pass bookkeeping of the next forward_pair (prefetch_labels)
        self.prefetch_hits = 0          # forward_pair calls that consumed prefetched bookkeeping

    # -- lazy device state ------------------------------------------------------------------------
    def _ensure(self):
        q = self.queue
        if not q.is_cuda:
            raise _capi.FFCError('the FFC head runs on a CUDA device only: move the module with .cuda() (no CPU fallback)')
        if self._dev == q.device and self._lru is not None:
            # a torch-level write to `queue` since the mirror was made (module.load_state_dict(), queue.copy_(), ...) bumps the buffer's
            # version counter; the kernels' own writes go through raw pointers and keep fp32 rows and mirror in step
            if q._version != self._mirror_version or q.data_ptr() != self._mirror_ptr:
                self.sync_mirror()
            return
        dev = q.device
        if self._lru is not None:
            # the module was moved to another device after use: carry the LRU (order and slots) and the queue positions over, and
            # release the old device's head
            self._side.synchronize()
            self._pending_lru = self._lru.state_dict()
            self._pending_qpos = self.qpos.cpu()
            self._lib.ffc_head_destroy(self.__dict__.pop('_h'))
            self._lru, self._pre = None, None
        self._lib = _capi.lib()
        Q, D, R = self.queue_size, self.feat_dim, self.max_batch
        with torch.cuda.device(dev):
            self._lru = LRU(Q, device=dev)
            self.qpos = torch.zeros(Q, dtype=torch.uint8, device=dev)
            self.queue_bf16 = torch.empty(2, Q, D, dtype=torch.bfloat16, device=dev)
            self._alloc_batch(R)
            # LRU bookkeeping runs on its own stream, ahead of the sweeps of the main stream (see forward_pair)
            # (high priority: its short kernels take the SMs a sweep CTA frees before the sweep's next CTAs do, instead of queueing
            # behind the whole sweep grid)
            self._side = torch.cuda.Stream(device=dev, priority=_capi.side_stream_priority())
            self._lru_sync_main = True
            cfg = HeadConfig(R, Q, Q, 0, D, _capi.LOSS_TYPES[self.loss_type], self.scale, self.margin, self.hard_neg,
                             _capi.PRECISIONS[self.precision])
            h = C.c_void_p()
            check(self._lib.ffc_head_create(C.byref(cfg), C.byref(h)))
            self._h, self._cfg = h, cfg
            if self.queue_grad:
                check(self._lib.ffc_head_set_dqueue(h, 1))
                self.dqueue = torch.zeros(2, Q, D, dtype=torch.float32, device=dev)
                self.dqueue_pass = torch.empty(2, Q, D, dtype=torch.float32, device=dev)
        self._dev = dev
        self.sync_mirror()
        if self._pending_lru is not None:
            self._lru.restore(self._pending_lru)
            self._pending_lru = None
        if self._pending_qpos is not None:
            self.qpos.copy_(self._pending_qpos.to(dev))
            self._pending_qpos = None

    def _alloc_batch(self, R):
        dev, D, k = self.queue.device, self.feat_dim, self.hard_neg
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        Q = self.queue_size
        # per-pass bookkeeping state, two sets (rollback pass / commit pass): the bookkeeping of a pass may be computed while
        # the previous pass is still sweeping
        self._sets = [dict(rows=torch.empty(R, **i32), cols=torch.empty(R, **i32), label=torch.empty(R, **i32), ones_list=torch.empty(R, **i32),
                           n_ones=torch.zeros(1, **i32), cmask=torch.zeros((Q + 31) // 32 + 1, **i32), free=None) for _ in range(2)]
        self._use_set(0)
        self.undo_rows = torch.empty(R, D, **f32)
        self.stats = dict(lsum=torch.empty(4, R, **f32), osum=torch.empty(4, R, D, **f32), tgt=torch.empty(4, R, **f32),
                          topv=torch.empty(3, R, k, **f32), topi=torch.empty(3, R, k, **i32))

    def _use_set(self, i):
        st = self._sets[i]
        self.rows, self.cols, self.label, self.ones_list, self.n_ones, self.cmask = (st[k] for k in ('rows', 'cols', 'label', 'ones_list', 'n_ones', 'cmask'))
        return st

    def __del__(self):
        h = self.__dict__.pop('_h', None)
        if h:
            try:
                self._lib.ffc_head_destroy(h)
            except Exception:
                pass

    @property
    def lru(self):
        """The device LRU (reference attribute ``ffc_net.lru``, main.py:85); created on first use."""
        self._ensure()
        self._side.synchronize()          # bookkeeping enqueued by earlier passes
        self._lru_sync_main = True        # whatever the caller does with it happens on the caller's stream
        return self._lru

    def zero_dqueue(self):
        """Reset the accumulated queue gradient (queue_grad=True)."""
        if self.dqueue is not None:
            self.dqueue.zero_()

    def set_timing(self, enable):
        """Bracket every main-sweep launch with CUDA events (roofline evidence for bench.py)."""
        self._ensure()
        check(self._lib.ffc_head_set_timing(self._h, 1 if enable else 0))

    def get_timing(self):
        ms, n = C.c_double(), C.c_int64()
        check(self._lib.ffc_head_get_timing(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def sync_mirror(self):
        """Refresh the bf16 mirror from the fp32 queue (after construction / checkpoint load)."""
        q = self.queue
        assert q.is_contiguous() and q.dtype == torch.float32
        check(self._lib.ffc_cast_bf16(q.data_ptr(), self.queue_bf16.data_ptr(), q.numel(), torch.cuda.current_stream(q.device).cuda_stream))
        self._mirror_version, self._mirror_ptr = q._version, q.data_ptr()

    # -- reference attribute: ffc.py:41-43 ------------------------------------------------------------
    @property
    def queue_position_dict(self):
        if self._lru is None:
            src = self._pending_qpos if self._pending_qpos is not None else torch.zeros(self.queue_size, dtype=torch.uint8)
        else:
            self._side.synchronize()
            src = self.qpos
        return dict(enumerate(src.cpu().tolist()))

    @queue_position_dict.setter
    def queue_position_dict(self, d):
        t = torch.tensor([int(d[i]) for i in range(self.queue_size)], dtype=torch.uint8)
        if self._lru is None:
            self._pending_qpos = t
        else:
            self._side.synchronize()
            self._lru_sync_main = True
            self.qpos.copy_(t.to(self.qpos.device))

    def _labels_dev(self, lab, n):
        t = torch.as_tensor(lab)
        assert t.numel() == n, (t.numel(), n)
        return t.to(device=self._dev, dtype=torch.int64, non_blocking=True).contiguous()

    # -- one head pass ------------------------------------------------------------------------------
    def _bookkeep(self, set_idx, gallery_label, probe_label, B, commit, main, labels_on_main):
        """LRU side of a pass on the bookkeeping stream: ffc.py:162-177 / 214-235 (get / try_get, rows, cols, `ones`), the probe
        labels (ffc.py:189-194 / 242-246) and, on a rollback pass, the LRU / queue-position undo (ffc.py:256-259) -- the sweep
        only needs the labels, `ones` and the queue rows, never the LRU.  Returns the event the main stream has to wait for."""
        side, st = self._side, self._sets[set_idx]
        if labels_on_main or self._lru_sync_main:
            ev_in = torch.cuda.Event()
            ev_in.record(main)
            side.wait_event(ev_in)
            self._lru_sync_main = False
        if st['free'] is not None:
            side.wait_event(st['free'])           # the pass that used this set last has finished with it
        with torch.cuda.stream(side):
            kg = self._labels_dev(gallery_label, B)
            kp = self._labels_dev(probe_label, B)
            st['n_ones'].zero_()
            self._lru.assign(kg, journal=not commit, qpos=self.qpos, rows=st['rows'], cols=st['cols'], ones_list=st['ones_list'],
                             n_ones=st['n_ones'], cmask=st['cmask'])
            self._lru.view_batch(kp, st['label'])
            if not commit:
                self._lru.undo(B, self.qpos)
            done = torch.cuda.Event()
            done.record(side)
        return done

    def _finish(self, set_idx, p, g, B, commit, main):
        """Queue and sweep side of a pass on the caller's stream."""
        lib, dev = self._lib, self._dev
        Q, D = self.queue_size, self.feat_dim
        st = self._use_set(set_idx)
        p32 = p.to(device=dev, dtype=torch.float32).contiguous()
        g32 = g.detach().to(device=dev, dtype=torch.float32).contiguous()
        s = main.cuda_stream
        # ffc.py:179-182 / 237-241: enqueue (fp32 queue + bf16 mirror), old rows saved on a rollback pass
        check(lib.ffc_queue_scatter(self.queue.data_ptr(), self.queue_bf16.data_ptr(), self.rows.data_ptr(), self.cols.data_ptr(),
                                    g32.data_ptr(), B, Q, D, None if commit else self.undo_rows.data_ptr(), s))
        hp = HeadPass(p32.data_ptr(), self.queue.data_ptr(), self.queue_bf16.data_ptr(), self.label.data_ptr(),
                      self.ones_list.data_ptr(), self.n_ones.data_ptr(), self.cmask.data_ptr(), B)
        hs = HeadStats(*(self._stat_ptr(name, B) for name in ('lsum', 'osum', 'tgt', 'topv', 'topi')))
        dp = torch.empty(B, D, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        # ffc.py:195-202 / 248-254 + backward
        check(lib.ffc_head_pass_single(self._h, C.byref(hp), C.byref(hs), loss.data_ptr(), dp.data_ptr(), s))
        if self.queue_grad:      # while the queue still is what the pass swept (a rollback pass restores its rows next)
            check(lib.ffc_head_dqueue(self._h, C.byref(hp), self.dqueue_pass.data_ptr(), s))
            self.dqueue.add_(self.dqueue_pass)
        if not commit:   # ffc.py:255: the queue rows come back; the LRU was undone by the bookkeeping stream
            check(lib.ffc_queue_restore(self.queue.data_ptr(), self.queue_bf16.data_ptr(), self.rows.data_ptr(), self.cols.data_ptr(),
                                        self.undo_rows.data_ptr(), B, Q, D, s))
        self.cmask.zero_()
        st['free'] = torch.cuda.Event()
        st['free'].record(main)
        self._last = dict(rows=self.rows[:B], cols=self.cols[:B], label=self.label[:B], ones=self.ones_list, n_ones=self.n_ones)
        return loss, dp

    def _check_batch(self, p, g):
        B, D = p.shape[0], self.feat_dim
        assert p.shape == (B, D) and g.shape == (B, D), (p.shape, g.shape)
        assert 1 <= B <= self.max_batch, f'batch {B} > max_batch {self.max_batch}'
        assert self.queue.is_contiguous()
        return B

    @staticmethod
    def _on_device(lab):
        return torch.is_tensor(lab) and lab.is_cuda

    def _pass(self, p, g, probe_label, gallery_label, commit):
        self._ensure()
        self._drop_prefetch()
        B = self._check_batch(p, g)
        with torch.cuda.device(self._dev):
            main = torch.cuda.current_stream(self._dev)
            done = self._bookkeep(0 if not commit else 1, gallery_label, probe_label, B, commit, main,
                                  self._on_device(probe_label) or self._on_device(gallery_label))
            main.wait_event(done)
            return self._finish(0 if not commit else 1, p, g, B, commit, main)

    def prefetch_labels(self, x_label, y_label):
        """Hand over the labels of the NEXT :meth:`forward` / :meth:`forward_pair` now (SURVEY 8(f) rank 4: they are CPU tensors the
        loader has long before the images have gone through the backbones, main.py:59-60).  The rollback pass's LRU bookkeeping
        (ffc.py:214-235, 242-246, 256-259) is enqueued on the bookkeeping stream at once, behind the previous step's commit bookkeeping
        and the release of bookkeeping set 0 -- i.e. it runs under the previous step's sweeps and the backbones' kernels.  The next call
        must pass these same label objects; anything else discards the prefetched work (a rollback pass's bookkeeping undoes itself on
        the LRU; only set 0's `ones` mask is cleared)."""
        self._ensure()
        self._drop_prefetch()
        B = int(torch.as_tensor(x_label).numel())
        assert 1 <= B <= self.max_batch and int(torch.as_tensor(y_label).numel()) == B
        with torch.cuda.device(self._dev):
            main = torch.cuda.current_stream(self._dev)
            done = self._bookkeep(0, y_label, x_label, B, False, main, self._on_device(x_label) or self._on_device(y_label))
        self._pre = (x_label, y_label, B, done)

    def _drop_prefetch(self):
        pre, self._pre = self._pre, None
        if pre is not None:
            with torch.cuda.stream(self._side):
                self._sets[0]['cmask'].zero_()

    def _take_prefetch(self, x_label, y_label, B):
        pre = self._pre
        if pre is None:
            return None
        if pre[0] is x_label and pre[1] is y_label and pre[2] == B:
            self._pre = None
            self.prefetch_hits += 1
            return pre[3]
        self._drop_prefetch()
        return None

    def forward_pair(self, p_rb, g_rb, p_cm, g_cm, x_label, y_label):
        """ffc.py:264-267 with embeddings in and no autograd glue: the rollback pass (probe p_rb with labels x_label, gallery g_rb
        with labels y_label) then the commit pass (probe p_cm / y_label, gallery g_cm / x_label).  Both passes' LRU bookkeeping is
        enqueued first on the bookkeeping stream -- a rollback pass leaves the LRU as it found it, so the commit pass's
        bookkeeping does not depend on the rollback sweep and runs underneath it (on the SMs the sweep leaves free); with host
        labels (the reference's contract, main.py:59-60) it even runs under the previous step's sweep.
        Returns (loss1 + loss2, dLoss/dp_rb, dLoss/dp_cm)."""
        self._ensure()
        B = self._check_batch(p_rb, g_rb)
        assert self._check_batch(p_cm, g_cm) == B
        with torch.cuda.device(self._dev):
            main = torch.cuda.current_stream(self._dev)
            on_main = self._on_device(x_label) or self._on_device(y_label)
            done_rb = self._take_prefetch(x_label, y_label, B)
            if done_rb is None:
                done_rb = self._bookkeep(0, y_label, x_label, B, False, main, on_main)
            done_cm = self._bookkeep(1, x_label, y_label, B, True, main, False)
            main.wait_event(done_rb)
            l2, d_rb = self._finish(0, p_rb, g_rb, B, False, main)
            main.wait_event(done_cm)
            l1, d_cm = self._finish(1, p_cm, g_cm, B, True, main)
        return l1 + l2, d_rb, d_cm

    def forward(self, x, y, x_label, y_label):
        """``FFC.forward`` (ffc.py:264-267) with embeddings in: ``x`` / ``y`` are the two views' embeddings [B, D]; gradients flow
        to both (each is the probe of one pass and the no-grad gallery of the other)."""
        return _HeadPairFn.apply(x, y, self, y.detach(), x.detach(), x_label, y_label)

    def _stat_ptr(self, name, B):
        # the stats arrays are laid out [slots][n_rows][...] for the n_rows of THIS pass: use compact per-pass views
        t = self.stats[name]
        if B == t.shape[1]:
            return t.data_ptr()
        c = self._compact.get((name, B))
        if c is None:
            c = torch.empty((t.shape[0], B) + tuple(t.shape[2:]), dtype=t.dtype, device=t.device)
            self._compact[(name, B)] = c
        return c.data_ptr()

    def head(self, p, g, probe_label, gallery_label, commit=True):
        """One head pass: ``forward_impl`` (commit=True, ffc.py:153-204) or ``forward_impl_rollback`` (commit=False,
        ffc.py:208-260) with embeddings in.  Returns the loss; gradients flow to ``p`` only."""
        return _HeadFn.apply(p, self, g, probe_label, gallery_label, commit)

    @torch.no_grad()
    def identify(self, x, k=1):
        """1:N identification of embeddings ``x`` [N, D] (fp32 / fp16 / bf16, any device; raw features or unit rows: they are
        L2-normalised here) against the resident prototypes ``queue[0][s]``, ``s < lru.cur_idx``.  Returns
        ``Identification(scores, labels, slots)``, device tensors [N, k]: cosine (fp32), the identity's label, its slot; ordered by
        score descending, ties by smaller slot; fewer than k resident -> slot -1, label INT64_MIN, score -inf.  ``precision='fp32'``
        heads select by the fp32 score (the check mode), bf16 heads by the tcgen05 bf16 cosine and rescore the k winners in fp32.
        Leaves queue, mirror, LRU (contents and recency), queue positions and a pending :meth:`prefetch_labels` untouched."""
        k = _ident.check_k(k)
        self._ensure()
        with torch.cuda.device(self._dev):
            main = torch.cuda.current_stream(self._dev)
            ev = torch.cuda.Event()
            ev.record(self._side)              # the bookkeeping enqueued so far (a prefetch's rollback has undone itself by then)
            main.wait_event(ev)
            xn = _ident.normalized_queries(x, self.feat_dim, self._dev)
            if xn.shape[0] == 0:
                return _ident.empty(0, k, self._dev)
            out = _ident.search(self._lib, self._h, self._lru._h, xn, k, self.queue, self.queue_bf16 if self.precision == 'bf16' else None)
            self._lru_sync_main = True         # the next bookkeeping must not rewrite the LRU while the search reads it
        return out

    def last_bookkeeping(self):
        """(rows, cols, labels, ones) of the most recent pass as Python lists (debug / parity tests; synchronises)."""
        l = self._last
        n1 = int(l['n_ones'].item())
        return (l['rows'].tolist(), l['cols'].tolist(), l['label'].tolist(), sorted(l['ones'][:n1].tolist()))


class FFC(FFCHead):
    """ffc.py:10-267.  Buffers ``queue`` / ``mask`` live on this module, as in the reference state_dict."""

    def __init__(self, net_type, feat_dim, queue_size=7409, scale=32.0, loss_type='AM', margin=0.4, momentum=0.99,
                 neg_margin=0.25, pretrained_model_path=None, num_class=None, *, precision='bf16', max_batch=1024,
                 probe_net=None, gallery_net=None, device=None, queue_grad=False):
        FFCHead.__init__(self, feat_dim, queue_size, scale, loss_type, margin, precision=precision, max_batch=max_batch, device=device,
                         queue_grad=queue_grad)
        self.probe_net = probe_net if probe_net is not None else create_net(net_type, feat_dim=feat_dim, fp16=True)
        self.gallery_net = gallery_net if gallery_net is not None else create_net(net_type, feat_dim=feat_dim, fp16=True)
        self.neg_margin = neg_margin          # stored, unused (as in the reference, ffc.py:44)
        self.m = momentum
        self.mask_svfc = 1.2
        for param_p, param_g in zip(self.probe_net.parameters(), self.gallery_net.parameters()):   # ffc.py:53-55
            param_g.data.copy_(param_p.data)
            param_g.requires_grad = False

    def _apply(self, fn, *args, **kwargs):
        self._ema_probe = None            # .to() / .cuda() / .float() move the parameters: rebuild the EMA chunk table
        return super()._apply(fn, *args, **kwargs)

    @torch.no_grad()
    def _momentum_update_gallery(self):
        """ffc.py:139-145 ``param_g = param_g * m + param_p * (1 - m)`` for every parameter, as ONE launch over all
        tensors (`ffc_ema_update`; the reference launches three eager kernels per tensor).  Bit-identical to the reference
        expression (same fp32 roundings, no FMA)."""
        pg = [q for q in self.gallery_net.parameters()]
        pp = [q for q in self.probe_net.parameters()]
        if not pg:
            return
        # the chunk table is keyed on the parameter storage; a full key costs ~0.1 ms of Python for a 240-tensor backbone, so it is
        # rebuilt only when the module was moved / cast (`_apply`) or the end points of the parameter lists changed storage
        probe = (len(pg), pg[0].data_ptr(), pp[0].data_ptr(), pg[-1].data_ptr(), pp[-1].data_ptr())
        if getattr(self, '_ema_probe', None) != probe:
            self._ema_probe = probe
            import numpy as np
            lib = _capi.lib()
            step = lib.ffc_ema_chunk_elems()
            rows = []
            for g, p in zip(pg, pp):
                if not (g.is_cuda and p.is_cuda and g.dtype == torch.float32 and p.dtype == torch.float32 and g.is_contiguous() and p.is_contiguous()
                        and g.numel() == p.numel()):
                    raise _capi.FFCError('gallery EMA: parameters must be contiguous fp32 CUDA tensors of equal size (no CPU fallback)')
                for a in range(0, g.numel(), step):
                    rows.append((g.data_ptr() + 4 * a, p.data_ptr() + 4 * a, min(step, g.numel() - a)))
            tab = np.zeros(len(rows), dtype=np.dtype([('g', np.uint64), ('p', np.uint64), ('n', np.int32), ('pad', np.int32)]))
            for i, (a, b, n) in enumerate(rows):
                tab[i] = (a, b, n, 0)
            self._ema_table = torch.from_numpy(tab.view(np.uint8).copy()).to(pg[0].device)
            self._ema_chunks = len(rows)
        m32 = float(torch.tensor(self.m, dtype=torch.float32))
        om32 = float(torch.tensor(1. - self.m, dtype=torch.float32))       # ffc.py:145: the Python double (1. - m), rounded to fp32 by the multiply
        check(_capi.lib().ffc_ema_update(self._ema_table.data_ptr(), self._ema_chunks, m32, om32,
                                         torch.cuda.current_stream(pg[0].device).cuda_stream))

    # -- checkpoint wire format of the reference (main.py:84-85) + the resume path it lacks (SURVEY 8(f) rank 2) ----------------
    def checkpoint(self):
        """The dict ``main.py:85`` saves: ``{'state_dict': probe_net.state_dict(), 'lru': lru.state_dict(), 'fc': queue.cpu(),
        'qp': queue_position_dict}``.  ``lru`` is the reference's recency-ordered ``[(key, slot)]`` list (lru.py:102-108)."""
        return {'state_dict': self.probe_net.state_dict(), 'lru': self.lru.state_dict(), 'fc': self.queue.detach().cpu(),
                'qp': self.queue_position_dict}

    def load_checkpoint(self, ckpt):
        """Resume from :meth:`checkpoint` (or a snapshot written by the reference's ``main.py``): probe weights, queue (+ bf16
        mirror), LRU (order and slots) and queue positions.  The gallery network restarts as a copy of the probe network, as
        in ``ffc.py:53-55`` (the reference does not save it)."""
        self.probe_net.load_state_dict(ckpt['state_dict'])
        with torch.no_grad():
            for param_p, param_g in zip(self.probe_net.parameters(), self.gallery_net.parameters()):
                param_g.data.copy_(param_p.data)
            self.queue.copy_(ckpt['fc'].to(self.queue.device))
        self._ensure()
        self.sync_mirror()
        lru = self.lru
        lru.clear()
        lru.restore([(int(k), int(v)) for k, v in ckpt['lru']])
        self.queue_position_dict = ckpt['qp']

    def forward_impl(self, p_data, g_data, probe_label, gallery_label):            # ffc.py:153-204
        p = self.probe_net(p_data)
        with torch.no_grad():
            g = self.gallery_net(g_data)
        return self.head(p, g, probe_label, gallery_label, commit=True)

    def forward_impl_rollback(self, p_data, g_data, probe_label, gallery_label):   # ffc.py:208-260
        p = self.probe_net(p_data)
        with torch.no_grad():
            self._momentum_update_gallery()
            g = self.gallery_net(g_data)
        return self.head(p, g, probe_label, gallery_label, commit=False)

    def forward(self, x, y, x_label, y_label):                                     # ffc.py:264-267
        """loss2 = forward_impl_rollback(x, y, ...), loss1 = forward_impl(y, x, ...), returned as loss1 + loss2.  The four backbone
        calls are issued in the reference's order (probe(x), EMA, gallery(y), probe(y), gallery(x)); the two head passes then
        run as one pair so that their bookkeeping overlaps the sweeps."""
        p_rb = self.probe_net(x)
        with torch.no_grad():
            self._momentum_update_gallery()
            g_rb = self.gallery_net(y)
        p_cm = self.probe_net(y)
        with torch.no_grad():
            g_cm = self.gallery_net(x)
        return _HeadPairFn.apply(p_rb, p_cm, self, g_rb, g_cm, x_label, y_label)
