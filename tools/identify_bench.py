"""Time FFCHead.identify (tcgen05 search + merge) against the torch baseline `topk(x @ queue_bf16[0, :cur].T)` on one GPU.

One JSON line per (workload, arm): ms per call (CUDA events over >= 20 calls after warm-up), TFLOP/s = 2 N cur_idx D / time,
its fraction of bench.peaks()['burst'], and the GPU name / power limit read in the same run.  The baseline materialises the
bf16 logits; where N x cur_idx of them would not fit in 8 GB it runs in chunks of 4 096 query rows (the line says so).
The gallery (1 M x 512 bf16 = 1 GB) exceeds the 126 MB L2, so every call streams it from HBM.

    python tools/identify_bench.py [--iters 20] [--out identify_bench.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'very-large-scale-face-recognition_b200')]

import torch  # noqa: E402

import bench  # noqa: E402
import ffc_b200  # noqa: E402

WORKLOADS = [(1024, 1 << 20, 512), (8192, 1 << 20, 512), (65536, 1 << 20, 512), (1024, 1 << 20, 128), (1024, 1 << 16, 512)]
K = 10
LOGIT_BUDGET = 8 << 30       # bytes of bf16 logits the baseline may materialise at once
CHUNK = 4096


def gpu_info():
    r = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else torch.cuda.get_device_name(0)


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('identify_bench needs a CUDA device')
    assert args.iters >= 20
    dev = torch.device('cuda', 0)
    info, burst = gpu_info(), bench.peaks()['burst']
    lines = []
    heads = {}
    for N, Q, D in WORKLOADS:
        if (Q, D) not in heads:
            heads.clear()
            torch.cuda.empty_cache()
            m = ffc_b200.FFCHead(D, Q, max_batch=64).to(dev)
            m.lru.restore_arrays(torch.arange(Q), torch.arange(Q, dtype=torch.int32))
            heads[(Q, D)] = m
        m = heads[(Q, D)]
        x = torch.randn(N, D, device=dev)
        flop = 2.0 * N * Q * D
        ours = timed(lambda: m.identify(x, k=K), args.iters)
        xb = torch.nn.functional.normalize(x).to(torch.bfloat16)
        W = m.queue_bf16[0, :Q]
        chunked = N * Q * 2 > LOGIT_BUDGET

        def base():
            for a in range(0, N, CHUNK if chunked else N):
                torch.topk(xb[a:a + (CHUNK if chunked else N)] @ W.t(), K, dim=1)
        ref = timed(base, args.iters)
        for arm, ms in (('identify', ours), ('torch_matmul_topk', ref)):
            tf = flop / ms / 1e9
            line = dict(arm=arm, N=N, cur_idx=Q, D=D, k=K, ms_per_call=round(ms, 4), tflops=round(tf, 1), frac_of_burst=round(tf / burst, 3),
                        burst_tflops=burst, gpu=info, iters=args.iters,
                        baseline_chunked_rows=(CHUNK if chunked else None) if arm != 'identify' else None)
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            for l in lines:
                f.write(json.dumps(l) + '\n')


if __name__ == '__main__':
    main()
