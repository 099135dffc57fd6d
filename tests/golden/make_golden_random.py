"""Record the expected values of the randomised cross-checks in tests/test_oracle_vs_reference.py, so that the same seeds and
configurations are checked on every machine (tests/golden/random_lru_streams.json.gz, tests/golden/random_head_configs.npz).

    python tests/golden/make_golden_random.py --source reference     # the unmodified reference tree (oracle/ref_shim.py)
    python tests/golden/make_golden_random.py --source oracle        # oracle/lru_ref.py + oracle/head_ref.py

Both files name their source.  The committed files were recorded with ``--source oracle``: the reference's source is not part of this
repository.  The oracle code these cases run (LRU, HeadOracle.forward) is unchanged since the live cross-checks of the same seeds against
the reference were added and passing, so the stored values are the ones those checks accepted.  Re-record with ``--source reference``
wherever the reference tree is available.

The op streams and configurations are drawn exactly as the live tests draw them (same seeds, same order of random calls).
"""
import argparse
import gzip
import json
import os
import random
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402
from oracle.head_ref import HeadOracle  # noqa: E402
from oracle.lru_ref import LRU  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
LRU_SEEDS = range(6)
HEAD_SEEDS, HEAD_LOSSES = range(4), ('AM', 'Arc', 'SV')


def lru_stream(seed, lru_cls):
    """test_lru_random_streams(seed): the op stream and what `lru_cls` returns along it"""
    rng = random.Random(seed)
    cap = rng.choice([1, 2, 3, 5, 8, 13, 32])
    universe = rng.choice([cap, cap + 1, 2 * cap + 3, 10 * cap])
    lru, ops, pending = lru_cls(cap), [], 0

    def state():
        sd = [list(kv) for kv in lru.state_dict()]
        it = [list(kv) for kv in lru]
        keys = sorted(lru.keys())
        return ['state', sd, lru.cur_idx, None if it == sd else it, None if keys == sorted(k for k, _ in sd) else keys]
    for step in range(1500):
        r, key = rng.random(), rng.randrange(universe)
        if r < 0.40 and pending == 0:
            ops.append(['get', key, lru.get(key)])
        elif r < 0.70:
            ops.append(['try_get', key, lru.try_get(key)])
            pending += 1
        elif r < 0.80 and pending:
            n = rng.randrange(1, pending + 1)
            lru.rollback_steps(n)
            pending -= n
            ops.append(['rollback_steps', n])
        elif r < 0.85 and pending:
            lru.rollback_one_step()
            pending -= 1
            ops.append(['rollback_one_step'])
        elif r < 0.92:
            ops.append(['view', key, lru.view(key), key in lru])
        elif r < 0.97:
            ops.append(state())
        elif pending == 0:
            kvs = lru.state_dict()
            lru = lru_cls(cap)
            lru.restore(kvs)
            ops.append(['restore', [list(kv) for kv in kvs]])
    ops.append(state())
    return dict(seed=seed, capacity=cap, ops=ops)


def head_config(seed, loss_type):
    """test_head_random_configs(seed, loss_type): D, Q, B, identity count and margin"""
    rng = random.Random(100 * seed + len(loss_type))
    D = rng.choice([4, 16, 32])
    Q = rng.choice([6, 17, 40])
    B = rng.choice([4, 6, 10])
    n_ids = rng.choice([Q // 2 + 2, Q + 3, 3 * Q])
    return D, Q, B, n_ids, (0.5 if loss_type == 'Arc' else 0.4)


def head_batches(seed, loss_type):
    """the 5 batches (x, y, x_label, y_label) of test_head_random_configs(seed, loss_type)"""
    D, Q, B, n_ids, _ = head_config(seed, loss_type)
    gen = torch.Generator().manual_seed(seed + 50)
    for s in range(5):
        ids = torch.randperm(n_ids, generator=gen)[:B // 2]
        xl = torch.cat([ids, torch.randint(0, n_ids, (B - B // 2,), generator=gen)])
        yl = torch.cat([ids, torch.randint(0, n_ids, (B - B // 2,), generator=gen)])
        x = F.normalize(torch.randn(B, D, generator=gen))
        y = F.normalize(torch.randn(B, D, generator=gen))
        yield x, y, xl, yl


def head_case(seed, loss_type, source, rec):
    """Per case `<loss>_<seed>_<name>`, stacked over the 5 steps: the batches' checksums (`inputs`: sums of x, y, x_label, y_label), loss,
    dx, dy, both passes' bookkeeping (`trace` [step, pass, rows/cols/labels/ones, B], `ones` padded with -1), LRU state (padded with -1)
    and cur_idx, queue positions; the queue before the first and after the last step."""
    D, Q, B, n_ids, margin = head_config(seed, loss_type)
    torch.manual_seed(seed)
    if source == 'reference':
        m = ref_shim.make_ffc(D, Q, 32.0, loss_type, margin)
        queue = lambda: m.queue                                                    # noqa: E731
    else:
        q = torch.rand(2, Q, D)                                                    # ffc.py:29-30
        q /= q.norm(dim=2, keepdim=True)
        o = HeadOracle(D, Q, 32.0, loss_type, margin, queue=q, dtype=torch.float32)
        queue = lambda: o.queue                                                    # noqa: E731
    p = f'{loss_type}_{seed}_'
    rec[p + 'queue0'] = queue().detach().float().numpy().copy()
    out = dict(inputs=[], loss=[], dx=[], dy=[], trace=[], lru=[], cur_idx=[], qpos=[])
    for x, y, xl, yl in head_batches(seed, loss_type):
        if source == 'reference':
            loss, dx, dy, trace = ref_shim.forward_backward(m, x, y, xl.tolist(), yl.tolist())
            lru, qpos = m.lru, [m.queue_position_dict[i] for i in range(Q)]
        else:
            xo, yo = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
            lo = o.forward(xo, yo, xl.tolist(), yl.tolist())
            if torch.is_tensor(lo) and lo.requires_grad:
                lo.backward()
            loss = float(lo)
            dx, dy = (torch.zeros(B, D) if t.grad is None else t.grad for t in (xo, yo))
            trace, lru, qpos = o.trace[-2:], o.lru, o.qpos
        out['inputs'].append([float(x.double().sum()), float(y.double().sum()), int(xl.sum()), int(yl.sum())])
        out['loss'].append(loss)
        out['dx'].append(dx.numpy())
        out['dy'].append(dy.numpy())
        out['trace'].append([[tr[k] + [-1] * (B - len(tr[k])) for k in ('rows', 'cols', 'labels', 'ones')] for tr in trace])
        out['lru'].append([list(kv) for kv in lru.state_dict()] + [[-1, -1]] * (Q - len(lru.state_dict())))
        out['cur_idx'].append(lru.cur_idx)
        out['qpos'].append(list(qpos))
    for k, v in out.items():
        rec[p + k] = np.array(v, dtype=np.float32 if k in ('dx', 'dy') else np.float64 if k in ('inputs', 'loss') else np.int64)
    rec[p + 'queue_final'] = queue().detach().float().numpy().copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--source', choices=['reference', 'oracle'], required=True)
    args = ap.parse_args()
    if args.source == 'reference':
        assert ref_shim.available(), 'reference tree not present (set FFC_REFERENCE_ROOT)'
        lru_cls = ref_shim.load()[1].LRU
    else:
        lru_cls = LRU
    torch.set_num_threads(1)          # serial index_put: "last duplicate wins" (make_golden.py)
    streams = [lru_stream(seed, lru_cls) for seed in LRU_SEEDS]
    with gzip.GzipFile(os.path.join(OUT, 'random_lru_streams.json.gz'), 'wb', mtime=0) as f:          # mtime 0: same bytes on every run
        f.write(json.dumps(dict(source=args.source, streams=streams), separators=(',', ':')).encode())
    rec = dict(source=np.array(args.source))
    for seed in HEAD_SEEDS:
        for loss_type in HEAD_LOSSES:
            head_case(seed, loss_type, args.source, rec)
    np.savez_compressed(os.path.join(OUT, 'random_head_configs.npz'), **rec)


if __name__ == '__main__':
    main()
