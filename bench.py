#!/usr/bin/env python
"""Benchmark of the FFC head hot path (BASELINE.json metric: head fwd+bwd samples/s, % of bf16 tensor peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c4] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one reference ``FFC.forward`` over one synthetic batch, embeddings in: a rollback head pass
(probe=x, gallery=y) plus a commit head pass (probe=y, gallery=x) -- ffc.py:264-267 -- i.e. 2*B probe rows
("samples") per GPU, each through LRU bookkeeping, enqueue scatter, the fused margin-softmax sweep (loss and
dEmb, both add_margin terms) and, on the rollback pass, the restore.  Workloads (SURVEY.md section 8):
  c3 (default)  B=1024 rows/GPU, 1,048,576 identities, queue 1,048,576 (column-sharded over N GPUs), D=512, Arc
  c2            B=512, 100k identities, queue 65,536, D=512, Arc (single GPU)
  c4            B=512 rows/GPU, 10,000,000 identities, queue 1,048,576 (LRU-managed: evictions, unknown labels), D=512, Arc
`value` is device-timed with the inputs resident in HBM; `e2e` is the same metric through the public
``FFCHead.head`` API from pinned host buffers (H2D of embeddings+labels and a D2H read of the loss inside the
timed region).  `--impl reference` times the reference's own head (unmodified ffc.py / lru.py, staged under oracle/_ref by
oracle/make_ref.py; the oracle port only if neither /root/reference nor the staging exists) on all host cores, on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'very-large-scale-face-recognition_b200'))

WORKLOADS = {
    'c3': dict(name='C3: FFC head only, 512-d embeddings, batch 1024/GPU, 1M identities, queue 1M', B=1024, N=1 << 20, Q=1 << 20, D=512,
               loss_type='Arc', margin=0.5, scale=32.0),
    'c2': dict(name='C2: FFC head, batch 512, 100k identities, queue 64k, D=512', B=512, N=100000, Q=65536, D=512,
               loss_type='Arc', margin=0.5, scale=32.0),
    # head of C4 (the backbone is outside the path): ten identities per queue slot, so instance rows mostly miss (LRU eviction path)
    # and most probe labels of the instance half are unknown (hard-negative rows).  Not the default; not measured in round 1.
    'c4': dict(name='C4 head: batch 512/GPU, 10M identities, LRU-managed queue 1M, D=512', B=512, N=10_000_000, Q=1 << 20, D=512,
               loss_type='Arc', margin=0.5, scale=32.0),
}
CPU_SAMPLE = dict(B=1024, Q=32768)   # bounded CPU sample: rows per pass (the workload's own, up to 1024) and queue slice; scaled linearly in Q


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(burst=d['bf16_tflops'], sustained=d.get('bf16_tflops_sustained', d['bf16_tflops']), hbm=d['hbm_gbs'], src='measured')
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src='fallback')


def sweep_traffic(w, world):
    """DRAM bytes of one main-sweep launch from the committed ncu --set full capture (C3 at one GPU only)."""
    if world == 1 and w is WORKLOADS['c3']:
        for name in ('r2_sweep_traffic.json', 'r1_sweep_traffic.json'):       # the newest capture of this kernel
            p = os.path.join(ROOT, 'profiles', name)
            if os.path.isfile(p):
                return json.load(open(p))['dram_bytes_per_launch']
    return None


def config_of(w, world):
    """The `config` object of the JSON line: the same for our arm and the reference arm."""
    return dict(workload=w['name'], rows_per_pass_per_gpu=w['B'], passes_per_step=2, identities=w['N'], queue=w['Q'], feat_dim=w['D'],
                loss=w['loss_type'], margin=w['margin'], scale=w['scale'], sharding=('none' if world == 1 else f'queue columns /{world}'),
                l2_policy='working set (bf16 queue %.0f MB per rank) exceeds the 126 MB L2' % (w['Q'] // world * w['D'] * 2 / 1e6),
                labels='pinned host int64 tensors (the reference passes CPU LongTensors, main.py:59-60); embeddings resident in HBM')


def make_batches(w, n_batches, seed, rank=0, world=1):
    """SURVEY.md 8(d): id half = chunks of a seeded permutation (same ids in x and y), instance halves iid uniform."""
    import torch
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(seed + 7919 * rank)
    B, N, D = w['B'], w['N'], w['D']
    h = B // 2
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(seed))
    out = []
    for s in range(n_batches):
        base = ((s * world + rank) * h) % max(1, N - h)
        ids = perm[base:base + h]
        xl = torch.cat([ids, torch.randint(0, N, (B - h,), generator=g)])
        yl = torch.cat([ids, torch.randint(0, N, (B - h,), generator=g)])
        x = F.normalize(torch.randn(B, D, generator=g))
        y = F.normalize(torch.randn(B, D, generator=g))
        out.append((x, y, xl, yl))
    return out


# --------------------------------------------------------------------------------------------------
# CPU baseline: the reference's own head (ffc.py / lru.py, unmodified, through oracle/ref_shim.py: /root/reference in the build
# container, the byte-for-byte staging oracle/_ref on the GPU box) on the host cores; the oracle port only where neither exists.
# Bounded sample: the workload's full rows per pass against a SLICE of the queue; per-sample cost is linear in the queue size
# (blend, both GEMMs, softmax; the argsort is Q log Q), so samples/s at the full queue = sample figure * Qs / Q -- an extrapolation
# that favours the CPU, and is labelled as such in the reference arm's `config`.
# --------------------------------------------------------------------------------------------------
def host_threads():
    """All the host threads the CPU arm can use (torchrun exports OMP_NUM_THREADS=1 to its workers: override it)."""
    import torch
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def sample_of(w):
    Bs, Qs = min(CPU_SAMPLE['B'], w['B']), min(CPU_SAMPLE['Q'], w['Q'])
    return dict(w, B=Bs, N=max(Qs, int(w['N'] * Qs / w['Q'])), Q=Qs)


def cpu_head_runner(ws):
    """-> (kind, step(x, y, xl, yl)) for one FFC.forward + backward on the CPU at shape `ws`, LRU pre-filled (steady state)."""
    import torch
    from oracle import ref_shim
    if ref_shim.available():
        m = ref_shim.make_ffc(ws['D'], ws['Q'], ws['scale'], ws['loss_type'], ws['margin'])
        m.lru.restore([(i, i) for i in range(ws['Q'])])

        def step(x, y, xl, yl):
            return ref_shim.forward_backward(m, x, y, xl, yl)[0]
        return 'reference', step
    from oracle.head_ref import HeadOracle
    o = HeadOracle(ws['D'], ws['Q'], ws['scale'], ws['loss_type'], ws['margin'], dtype=torch.float32)
    o.lru.restore([(i, i) for i in range(ws['Q'])])

    def step(x, y, xl, yl):
        x = x.clone().requires_grad_(True)
        y = y.clone().requires_grad_(True)
        loss = o.forward(x, y, xl.tolist(), yl.tolist())
        loss.backward()
        return float(loss)
    return 'port', step


def time_cpu(ws, steps, warmup, seed=1234):
    """Mean seconds per step over `steps` timed steps."""
    kind, step = cpu_head_runner(ws)
    batches = make_batches(ws, min(4, steps + warmup), seed=seed)
    times = []
    for s in range(warmup + steps):
        b = batches[s % len(batches)]
        t0 = time.perf_counter()
        step(*b)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    return kind, sum(times) / len(times)


def cpu_reference(w, steps, warmup):
    import torch
    cores = host_threads()
    ws = sample_of(w)
    kind, t = time_cpu(ws, steps, warmup)
    Bs, Qs = ws['B'], ws['Q']
    raw = 2 * Bs / t                               # samples/s at the sample's queue size
    scaled = raw * Qs / w['Q']                     # per-sample cost is linear in Q
    what = ('the unmodified reference head (ffc.py FFC.forward + backward, lru.py; fp32 CPU, normalise-only backbones)' if kind == 'reference'
            else 'oracle port (torch fp32, materialised B x Q logits, argsort top-k, autograd backward)')
    sample = (f'{what} on B={Bs} rows/pass, queue {Qs}, D={w["D"]}: {t * 1e3:.0f} ms/step = {raw:.0f} samples/s'
              + (f', scaled by {Qs}/{w["Q"]} to the full queue (extrapolated)' if Qs != w['Q'] else ' (full configuration, not extrapolated)'))
    cb = dict(value=scaled, unit='samples/s', cores=cores, kind=kind, sample=sample, sample_rows_per_pass=Bs, sample_queue=Qs,
              extrapolated=bool(Qs != w['Q'] or Bs != w['B']), torch=torch.__version__)
    return cb, t


def cpu_extras():
    """BASELINE.json configs[0] (C1: the reference's own CPU-runnable case, head shape batch 64 / 10k identities / queue 4096, D = 128 and
    512) timed IN FULL on the host cores, and the Python LRU's get() rate (SURVEY.md 8(d)): the LRU baseline."""
    out = {}
    for D in (128, 512):
        ws = dict(name='C1', B=64, N=10000, Q=4096, D=D, loss_type='Arc', margin=0.5, scale=32.0)
        kind, t = time_cpu(ws, 10, 2, seed=77)
        out[f'c1_head_d{D}'] = dict(samples_per_s=2 * 64 / t, ms_per_step=t * 1e3, kind=kind, extrapolated=False,
                                    shape='B=64 rows/pass, 10k identities, queue 4096, Arc, fp32')
    from oracle import ref_shim
    if ref_shim.available():
        lru_cls, lk = ref_shim.load()[1].LRU, 'reference'
    else:
        from oracle.lru_ref import LRU as lru_cls
        lk = 'port'
    import random
    rng = random.Random(0)
    lru = lru_cls(65536)
    keys = [rng.randrange(1 << 20) for _ in range(400000)]
    for k in keys[:100000]:
        lru.get(k)
    t0 = time.perf_counter()
    for k in keys[100000:]:
        lru.get(k)
    dt = time.perf_counter() - t0
    out['lru_get'] = dict(keys_per_s=300000 / dt, kind=lk, cores=1, shape='capacity 65536, uniform keys over 2^20 (94 % misses -> evictions)')
    return out


def run_reference(args, w):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cb, t = cpu_reference(w, args.steps, args.warmup)
    cfg = dict(config_of(w, max(1, args.gpus)),
               reference_sample=dict(rows_per_pass=cb['sample_rows_per_pass'], queue=cb['sample_queue'], extrapolated=cb['extrapolated'],
                                     rule='samples/s measured on the sample, multiplied by sample queue / full queue (cost per sample is linear in the queue size)'))
    line = dict(metric='ffc_head_fwd_bwd_samples_per_s', value=cb['value'], unit='samples/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=t * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic', impl='reference',
                config=cfg, cpu_baseline=cb,
                e2e=dict(value=cb['value'], unit='samples/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------------------------------
class Clocks:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '20'],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            pass

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(', ') for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx, pw = [], set(), None, []
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                pw.append(float(r[3]))
                for n, v in zip(names, r[4:8]):
                    if v.strip().lower().startswith('active'):
                        reasons.add(n)
            except Exception:
                continue
        if sm:
            sm.sort()
            out = dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm), power_w_max=max(pw) if pw else None)
        return out


# --------------------------------------------------------------------------------------------------
# the HBM-bound kernels of the path, each timed alone (CUDA events on the launch stream, 50 launches after 5 warm-ups): achieved GB/s =
# ALGORITHMIC bytes (SURVEY.md 8(d)) / time, against the measured copy bandwidth.  They are latency-bound by construction (a few KB to a
# few MB per launch); the figure that matters is microseconds per batch and keys/s.
# --------------------------------------------------------------------------------------------------
def kernel_micro(head, w, dev, world):
    import torch
    import ctypes as C
    from ffc_b200 import _capi
    lib, pk = _capi.lib(), peaks()
    B, Q, D, N = w['B'], w['Q'], w['D'], w['N']
    g = torch.Generator().manual_seed(99)
    s = torch.cuda.current_stream(dev).cuda_stream

    def timed(fn, n=50, warm=5):
        for _ in range(warm):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n * 1e3            # microseconds per launch group

    out = {}
    lru, qpos = head._lru, head.qpos
    keys = [torch.randint(0, N, (B,), generator=g).to(dev) for _ in range(8)]
    cols, rows = torch.empty(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev)
    ones, n_ones = torch.empty(B, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)
    cmask = torch.zeros((Q + 31) // 32 + 1, dtype=torch.int32, device=dev)
    it = [0]

    def lru_rollback():       # try_get x B + undo: the LRU side of a rollback pass, state unchanged afterwards
        k = keys[it[0] % 8]
        it[0] += 1
        n_ones.zero_()
        lru.assign(k, journal=True, qpos=qpos, rows=rows, cols=cols, ones_list=ones, n_ones=n_ones, cmask=cmask)
        lru.undo(B, qpos)
    us = timed(lru_rollback)
    by = 41.0 * B * 2                                    # ~41 B / key algorithmic (key, table entry, recency, outputs), assign + undo
    out['lru_try_get_plus_undo'] = dict(us_per_batch=us, keys_per_s=B / (us * 1e-6), achieved_gbs=by / (us * 1e-6) / 1e9, peak_gbs=pk['hbm'],
                                        frac=by / (us * 1e-6) / 1e9 / pk['hbm'], algorithmic_bytes=by, keys=B)
    lab = torch.empty(B, dtype=torch.int32, device=dev)
    us = timed(lambda: lru.view_batch(keys[0], lab))
    by = 28.0 * B
    out['lru_view'] = dict(us_per_batch=us, keys_per_s=B / (us * 1e-6), achieved_gbs=by / (us * 1e-6) / 1e9, peak_gbs=pk['hbm'],
                           frac=by / (us * 1e-6) / 1e9 / pk['hbm'], algorithmic_bytes=by, keys=B)
    cmask.zero_()
    # enqueue scatter + restore (the rollback pass's pair): B rows of D floats into random distinct slots
    r = torch.zeros(B, dtype=torch.int32, device=dev)
    c = torch.randperm(Q, generator=g)[:B].to(torch.int32).to(dev)
    gl = torch.nn.functional.normalize(torch.randn(B, D, generator=g)).to(dev)
    undo = torch.empty(B, D, device=dev)

    def scatter_restore():
        _capi.check(lib.ffc_queue_scatter(head.queue.data_ptr(), head.queue_bf16.data_ptr(), r.data_ptr(), c.data_ptr(), gl.data_ptr(), B, Q, D, undo.data_ptr(), s))
        _capi.check(lib.ffc_queue_restore(head.queue.data_ptr(), head.queue_bf16.data_ptr(), r.data_ptr(), c.data_ptr(), undo.data_ptr(), B, Q, D, s))
    us = timed(scatter_restore)
    by = float(B * D * (4 + 4 + 2 + 8) + B * D * (4 + 4 + 2))       # scatter with undo (read g, old row; write row, undo, mirror) + restore
    out['queue_scatter_plus_restore'] = dict(us_per_batch=us, rows_per_s=B / (us * 1e-6), achieved_gbs=by / (us * 1e-6) / 1e9, peak_gbs=pk['hbm'],
                                             frac=by / (us * 1e-6) / 1e9 / pk['hbm'], algorithmic_bytes=by, rows=B)
    return out


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def l2_to_sm_note(rows, q_local, D, sweep_ms):
    """What bounds the D = 512 sweep (DESIGN.md 4.3, profiles/r2_sweep_ncu_summary.md): every 128-column tile of W (128 x D bf16) is streamed
    from L2 into BOTH CTAs of its pair, once per 128-row tile of probe rows.  The byte count is the kernel's tiling, the rate follows from
    the measured launch time; ncu's l1tex__m_xbar2l1tex_read_bytes of the C3 launch is 19.38 GB: the 17.18 GB counted here + 2.15 GB of
    p~ tiles handed from the S-CTA to the O-CTA over DSMEM (32 KB per tile, delivered through the same crossbar) + P tiles and side sweeps."""
    if D != 512 or sweep_ms <= 0:
        return None
    row_tiles, col_tiles = (rows + 127) // 128, (q_local + 127) // 128
    w_bytes = 2.0 * row_tiles * col_tiles * 128 * D * 2
    return dict(what='L2 -> SM delivery of the queue tiles (both CTAs of a pair stream every tile), not the tensor pipe',
                w_tile_bytes_per_launch=w_bytes, delivered_tb_per_s=w_bytes / (sweep_ms * 1e-3) / 1e12,
                evidence='profiles/r2_sweep_ncu_summary.md, profiles/r2_persistent_sweep.md')


def softmax_rows(head, rows):
    """Rows of the last pass that have a softmax term (label known), rounded up to whole 128-row tiles: the rows GEMM-2 runs for."""
    lab = None
    if getattr(head, '_last', None) is not None:                      # ShardedFFCHead: the commit pass's all-reduced labels
        lab = head._last['label']
    elif getattr(head, '_sets', None) is not None:                    # FFCHead: bookkeeping set 1 = the commit pass
        lab = head._sets[1]['label']
    if lab is None:
        return rows
    n_soft = int((lab[:rows] >= 0).sum().item())
    return min(rows, (n_soft + 127) // 128 * 128)


def dump_outputs(out_dir, out, rank, world):
    """Write what the last timed step returned -- the loss and dLoss/dx, dLoss/dy ([B, D]) -- as float32 out_dir/<name>.npy (a rank
    suffix when sharded), so that two builds of the project can be compared output for output.  At most 4 MB per rank (B = 1024,
    D = 512)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    suffix = '' if world == 1 else f'_rank{rank}'
    for name, t in zip(('loss', 'dx', 'dy'), out):
        np.save(os.path.join(out_dir, f'{name}{suffix}.npy'), t.detach().float().cpu().numpy())


def run_ours(args, w):
    import torch
    import torch.distributed as dist
    import ffc_b200
    from ffc_b200 import _capi

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _capi.lib()
    B, N, Q, D = w['B'], w['N'], w['Q'], w['D']
    # the initial queue (each rank's shard of it) is drawn from torch's global generators, which torch seeds differently in every
    # process: seed them, so that every run with the same arguments (and every build of the project) starts from the same queue
    torch.manual_seed(1234 + rank)

    if world == 1:
        head = ffc_b200.FFCHead(D, Q, w['scale'], w['loss_type'], w['margin'], precision='bf16', max_batch=B, device=dev)
        head._ensure()
        # steady state: LRU full (SURVEY 8(d)): ids 0..Q-1 resident, slot i <- id i, recency = id order
        head.lru.restore_arrays(torch.arange(Q, dtype=torch.int64), torch.arange(Q, dtype=torch.int32))

        def step(x, y, xl, yl):          # rollback pass (probe x, gallery y) + commit pass (probe y, gallery x): (loss, dLoss/dx, dLoss/dy)
            return head.forward_pair(x, y, y, x, xl, yl)

        def step_api(x, y, xl, yl):      # public API (FFC.forward with embeddings in), gradients requested
            return head(x.requires_grad_(True), y.requires_grad_(True), xl, yl)
        prefetch = None                  # one GPU: host labels already run ahead on the bookkeeping stream
    else:
        from ffc_b200.dist import ShardedFFCHead
        head = ShardedFFCHead(D, Q, w['scale'], w['loss_type'], w['margin'], max_batch=B, device=dev)
        head.prefill_identity(N)

        def step(x, y, xl, yl):          # (loss, dLoss/dx, dLoss/dy) of this rank's rows
            return head.forward_pair(x, y, xl, yl)

        def step_api(x, y, xl, yl):
            return step(x, y, xl, yl)[0]
        # the sharded head takes the NEXT step's labels (CPU tensors, main.py:59-60) as soon as the loader has them:
        # their all-gather and the rollback pass's LRU bookkeeping then run under the current step's sweeps
        prefetch = None if os.environ.get('FFC_BENCH_NO_PREFETCH') else head.prefetch

    # one distinct batch per step: re-feeding an embedding that is already in the queue makes the target cosine
    # exactly 1, the reference's Arc NaN hazard (SURVEY.md 3.4)
    n_b = args.steps + args.warmup
    host = make_batches(w, n_b, seed=1234, rank=rank, world=world)
    # embeddings device-resident; labels stay on the host (pinned), as in the reference's loop (main.py:59-60: CPU LongTensors) -- at
    # every N, so that the per-N values are comparable: host labels let the LRU bookkeeping of a step run ahead on the bookkeeping
    # stream (one GPU) / be handed over by prefetch() (sharded head), under the previous step's sweeps
    devb = [(x.to(dev), y.to(dev), xl.pin_memory(), yl.pin_memory()) for x, y, xl, yl in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value) ----
    clocks = Clocks(local) if rank == 0 else None
    for s in range(args.warmup):
        step(*devb[s % n_b])
        if prefetch:
            prefetch(*devb[(s + 1) % n_b][2:])
    barrier()
    if getattr(head, '_timing', None):
        head._timing.clear()
    head.set_timing(True)
    l0 = lib.ffc_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        out = step(*devb[(args.warmup + s) % n_b])
        if prefetch and s + 1 < args.steps:
            prefetch(*devb[(args.warmup + s + 1) % n_b][2:])
    e1.record()
    barrier()
    launches = lib.ffc_launch_count() - l0
    ms = e0.elapsed_time(e1)
    sweep_ms, sweep_n = head.get_timing()
    head.set_timing(False)
    clk = clocks.stop() if clocks else None
    loss_val = float(out[0])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, rank, world)

    # ---- end to end through the public API from pinned host buffers (e2e) ----
    # fresh batches (other embeddings AND other identities' rows than the ones just enqueued: a re-fed embedding makes its target
    # cosine exactly 1 -- the Arc clamp regime -- and the loss would not be comparable with the device-timed phase)
    pinned = [tuple(t.pin_memory() for t in b) for b in make_batches(w, n_b, seed=4321, rank=rank, world=world)]
    phase_ms = head.phase_times() if getattr(head, '_timing', None) else None
    if phase_ms is not None:
        head._timing = None
    barrier()
    # The loop a trainer runs: the H2D copy of step k+1's embeddings goes up on a copy stream while step k computes, and the loss
    # of step k is read back (pinned buffer, async copy) once step k+1 has been enqueued.  Every step's inputs cross PCIe and
    # every step's loss is read on the host inside the timed region.
    main = torch.cuda.current_stream(dev)
    copy_stream = torch.cuda.Stream(device=dev)
    loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]

    def stage(s):
        x, y, xl, yl = pinned[(args.warmup + s) % n_b]
        with torch.cuda.stream(copy_stream):
            xd, yd = x.to(dev, non_blocking=True), y.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return xd, yd, xl, yl, ev

    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    nxt, pending, lv = stage(0), None, 0.0
    for s in range(args.steps):
        xd, yd, xl, yl, ev = nxt
        main.wait_event(ev)
        xd.record_stream(main)
        yd.record_stream(main)
        loss_e = step_api(xd, yd, xl, yl)
        buf = loss_host[s & 1]
        buf.copy_(loss_e.detach().reshape(1), non_blocking=True)
        ev_l = torch.cuda.Event()
        ev_l.record(main)
        if s + 1 < args.steps:
            nxt = stage(s + 1)
            if prefetch:
                prefetch(nxt[2], nxt[3])
        if pending is not None:
            pending[1].synchronize()
            lv = float(pending[0])                    # D2H read of the previous step's loss
        pending = (buf, ev_l)
    pending[1].synchronize()
    lv = float(pending[0])
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)

    t_all = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t_all[0]), float(t_all[1])
    samples = 2 * B * world * args.steps
    value = samples / (ms * 1e-3)
    pk = peaks()
    rows_per_sweep = B * world
    q_local = Q // world
    # Algorithmic FLOPs of one main sweep launch: 2*rows*Q*D for the cosines of every row + 2*rows'*Q*D for the gradient sum of the rows
    # that have a softmax term (a row whose label is unknown -- ffc.py:61, label -1 -- only takes part in the hard-negative top-k of its
    # cosines: no p~, no second GEMM; the kernel sweeps such rows last and skips GEMM-2 for row tiles made of them).  rows' is counted
    # in whole 128-row tiles from the labels of the last timed pass; C3 (every label known) has rows' = rows, i.e. 4*B*Q*D.
    soft_rows = softmax_rows(head, rows_per_sweep)
    flops = 2.0 * (rows_per_sweep + soft_rows) * q_local * D
    ach = flops * sweep_n / (sweep_ms * 1e-3) / 1e12 if sweep_ms > 0 else 0.0
    # the burst figure for a kernel timed in a short region, the sustained one when the timed region is long enough for the board to
    # settle at its power cap (MEASURED_PEAKS.json: best of 10 vs back to back for 4 s)
    long_run = ms >= 2000.0
    peak = pk['sustained'] if long_run else pk['burst']
    aux = kernel_micro(head, w, dev, world) if (world == 1 and not args.no_aux) else None
    if rank == 0:
        cb, _ = cpu_reference(w, 2, 1) if world == 1 and not args.no_cpu else (None, None)
        line = dict(metric='ffc_head_fwd_bwd_samples_per_s', value=value, unit='samples/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='bf16', data='synthetic',
                    config=config_of(w, world),
                    e2e=dict(value=samples / (ms_e2e * 1e-3), unit='samples/s', h2d_bytes_per_step=2 * B * D * 4 + 2 * B * 8, d2h_bytes_per_step=4,
                             ms_per_step=ms_e2e / args.steps, last_loss=lv,
                             pipeline='H2D of step k+1 on a copy stream under step k; loss of step k read on the host after step k+1 is enqueued'),
                    gpu_launches=int(launches),
                    roofline=dict(bound='tensor', achieved=ach, peak=peak, unit='TFLOP/s', frac=ach / peak, traffic=sweep_traffic(w, world),
                                  kernel='ffc_head_sweep_sm100_kernel (main sweep)', launches=int(sweep_n), avg_ms=sweep_ms / max(1, sweep_n),
                                  algorithmic_flops_per_launch=flops, rows_per_launch=rows_per_sweep, rows_with_softmax_term=soft_rows,
                                  peak_kind=('bf16_tflops_sustained' if long_run else 'bf16_tflops (burst)') + f' ({pk["src"]}; timed region {ms / 1e3:.2f} s)',
                                  frac_of_burst=ach / pk['burst'], frac_of_sustained=ach / pk['sustained'], sweep_share_of_step=sweep_ms / ms,
                                  limiter=l2_to_sm_note(rows_per_sweep, q_local, D, sweep_ms / max(1, sweep_n))),
                    clocks=clk, loss=loss_val)
        if cb is not None:
            line['cpu_baseline'] = cb
        if aux is not None:
            line['hbm_kernels'] = aux
        if world == 1 and not args.no_cpu:
            line['cpu_extras'] = cpu_extras()
        if world > 1 and os.environ.get('FFC_DIST_TIMING'):
            line['phase_ms_total'] = phase_ms
        if world > 1:
            line['barrier_timeouts'] = head.barrier_timeouts()      # in-kernel cross-rank barriers that gave up (must be 0)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='c3', choices=sorted(WORKLOADS))
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-aux', action='store_true', help='skip the per-kernel HBM micro timings')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the loss and embedding gradients of the last timed step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes what our kernels computed: --impl ours only')
    w = WORKLOADS[args.workload]
    if args.impl == 'reference':
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == '__main__':
    main()
