"""Cost of the queue gradient (queue_grad=True) at C3 (B = 1024 rows per pass, Q = 1 M prototypes, D = 512).

One JSON line per measurement:
  * step: ms per forward_pair (rollback + commit pass) with queue_grad off and on, AM and SV (CUDA events over --iters steps after
    warm-up, a distinct batch per step, the LRU full as in bench.py);
  * dqueue: ms per ffc_head_dqueue call (CUDA events), and the swapped tcgen05 sweep inside it on its own (torch.profiler, CUDA
    activity, in a separate run of --iters calls): achieved TFLOP/s = 4 n Q D / sweep time (the SV mode does the same GEMM FLOPs)
    and its fraction of bench.peaks()['burst'].
The card's name and power limit are read in the same run.  One GPU by default; under torchrun (WORLD_SIZE 2 or 8) the step lines
are for ShardedFFCHead, each rank timing its own shard (n = R B rows, Q / R slots).

    python tools/dqueue_bench.py [--iters 20] [--out dqueue_bench.jsonl]
    torchrun --nproc_per_node 8 tools/dqueue_bench.py
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'very-large-scale-face-recognition_b200')]

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import bench  # noqa: E402
import ffc_b200  # noqa: E402
from ffc_b200 import _capi  # noqa: E402

B, Q, D = 1024, 1 << 20, 512
MARGIN = dict(AM=0.4, SV=0.4)


def gpu_info(index):
    r = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else torch.cuda.get_device_name(index)


def batches(n, rows, n_ids, dev, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        xl = torch.randint(0, n_ids, (rows,), generator=g)
        yl = torch.cat([xl[:rows // 2], torch.randint(0, n_ids, (rows - rows // 2,), generator=g)])
        x = F.normalize(torch.randn(rows, D, generator=g)).to(dev)
        y = F.normalize(torch.randn(rows, D, generator=g)).to(dev)
        out.append((x, y, xl.pin_memory(), yl.pin_memory()))
    return out


def time_steps(step, data, warmup):
    for b in data[:warmup]:
        step(*b)
    torch.cuda.synchronize()
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for b in data[warmup:]:
        step(*b)
    e.record()
    torch.cuda.synchronize()
    return a.elapsed_time(e) / (len(data) - warmup)


def make_head(loss_type, queue_grad, world, dev):
    torch.manual_seed(1234)
    if world == 1:
        h = ffc_b200.FFCHead(D, Q, 32.0, loss_type, MARGIN[loss_type], precision='bf16', max_batch=B, device=dev, queue_grad=queue_grad)
        h._ensure()
        h.lru.restore_arrays(torch.arange(Q, dtype=torch.int64), torch.arange(Q, dtype=torch.int32))
        return h, lambda x, y, xl, yl: h.forward_pair(x, y, y, x, xl, yl)
    from ffc_b200.dist import ShardedFFCHead
    h = ShardedFFCHead(D, Q, 32.0, loss_type, MARGIN[loss_type], max_batch=B, device=dev, queue_grad=queue_grad)
    h.prefill_identity(Q)
    return h, lambda x, y, xl, yl: h.forward_pair(x, y, xl, yl)


def dqueue_call(h, dev):
    """ffc_head_dqueue again on the head's last (commit) pass: what every pass adds to a step with queue_grad"""
    last = h._last
    n = last['label'].numel()
    hp = _capi.HeadPass(h._p_last.data_ptr(), h.queue.data_ptr(), h.queue_bf16.data_ptr(), last['label'].data_ptr(), last['ones'].data_ptr(),
                        last['n_ones'].data_ptr(), h.cmask.data_ptr(), n)
    s = torch.cuda.current_stream(dev).cuda_stream
    return lambda: _capi.check(h._lib.ffc_head_dqueue(h._h, C.byref(hp), h.dqueue_pass.data_ptr(), s))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('dqueue_bench needs a CUDA device')
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank, local = int(os.environ.get('RANK', '0')), int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    info, burst = gpu_info(local), bench.peaks()['burst']
    lines = []

    def emit(d):
        d.update(gpu=info, world=world, rank=rank, B=B, Q=Q, D=D)
        lines.append(d)
        print(json.dumps(d), flush=True)

    data = batches(args.warmup + args.iters, B, Q, dev, 1234 + rank)      # ids of resident identities (bench.py: the LRU full)
    for loss_type in ('AM', 'SV'):
        for qg in (False, True):
            h, step = make_head(loss_type, qg, world, dev)
            ms = time_steps(step, data, args.warmup)
            emit(dict(kind='step', loss_type=loss_type, queue_grad=qg, ms=ms, merged=getattr(h, 'merged', None)))
            if qg and world == 1:
                # the probe rows of the head's last pass, for re-running its dqueue
                h._p_last = data[-1][1].float().contiguous()
                call = dqueue_call(h, dev)
                ms_dq = time_steps(lambda *a: call(), [()] * (args.warmup + args.iters), args.warmup)
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(args.iters):
                        call()
                    torch.cuda.synchronize()
                sweep_us = sum(getattr(e, 'device_time_total', 0) or e.cuda_time_total for e in prof.key_averages() if 'ffc_head_sweep_sm100_kernel' in e.key) / args.iters
                flops = 4.0 * B * Q * D
                tflops = flops / (sweep_us * 1e-6) / 1e12
                emit(dict(kind='dqueue', loss_type=loss_type, ms=ms_dq, sweep_ms=sweep_us / 1e3, sweep_tflops=tflops, frac_burst=tflops / burst,
                          burst_tflops=burst))
            del h
            torch.cuda.empty_cache()
    if args.out and rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            for d in lines:
                f.write(json.dumps(d) + '\n')
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
