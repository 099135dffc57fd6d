"""Randomised cross-checks of the oracle.

  * oracle/lru_ref.py  vs  reference lru.py:   random op streams (get / try_get / rollback / view / contains / state_dict / restore)
  * oracle/head_ref.py vs  reference ffc.py:   random small FFC configurations, several FFC.forward + backward steps each -- integer
                                               bookkeeping bit-exact, loss / gradients / queue within fp32 tolerance
  * oracle/tail_ref.py vs  torch's BatchNorm1d + F.normalize (what resnet_arcface.py:151 calls), random shapes and modes

The LRU and head checks run live against the UNMODIFIED reference tree (see oracle/ref_shim.py) where it is present, and against the
values recorded for the same seeds and configurations (tests/golden/make_golden_random.py, which names the source it recorded from)
everywhere.  The tail check needs torch only.
"""
import gzip
import importlib.util
import json
import os
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_shim, tail_ref
from oracle.head_ref import HeadOracle
from oracle.lru_ref import LRU

needs_ref = pytest.mark.skipif(not ref_shim.available(), reason='reference tree not present: the recorded replays cover the same seeds')

_spec = importlib.util.spec_from_file_location('make_golden_random', os.path.join(os.path.dirname(__file__), 'golden', 'make_golden_random.py'))
recorded = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(recorded)


@needs_ref
@pytest.mark.parametrize('seed', range(6))
def test_lru_random_streams(seed):
    _, lru_mod = ref_shim.load()
    rng = random.Random(seed)
    cap = rng.choice([1, 2, 3, 5, 8, 13, 32])
    universe = rng.choice([cap, cap + 1, 2 * cap + 3, 10 * cap])
    ref, ora = lru_mod.LRU(cap), LRU(cap)
    pending = 0
    for step in range(1500):
        r, key = rng.random(), rng.randrange(universe)
        if r < 0.40 and pending == 0:
            assert ora.get(key) == ref.get(key)
        elif r < 0.70:
            assert ora.try_get(key) == ref.try_get(key)
            pending += 1
        elif r < 0.80 and pending:
            n = rng.randrange(1, pending + 1)
            ref.rollback_steps(n), ora.rollback_steps(n)
            pending -= n
        elif r < 0.85 and pending:
            ref.rollback_one_step(), ora.rollback_one_step()
            pending -= 1
        elif r < 0.92:
            assert ora.view(key) == ref.view(key) and (key in ora) == (key in ref)
        elif r < 0.97:
            assert ora.state_dict() == ref.state_dict() and ora.cur_idx == ref.cur_idx and sorted(ora.keys()) == sorted(ref.keys())
            assert list(ora) == list(ref)
        elif pending == 0:
            # restore round trip into fresh caches (lru.py:113-128)
            kvs = ref.state_dict()
            ref, ora = lru_mod.LRU(cap), LRU(cap)
            ref.restore(kvs), ora.restore(kvs)
    assert ora.state_dict() == ref.state_dict() and ora.cur_idx == ref.cur_idx


@needs_ref
@pytest.mark.parametrize('seed', range(4))
@pytest.mark.parametrize('loss_type', ['AM', 'Arc', 'SV'])
def test_head_random_configs(seed, loss_type):
    rng = random.Random(100 * seed + len(loss_type))
    D = rng.choice([4, 16, 32])
    Q = rng.choice([6, 17, 40])
    B = rng.choice([4, 6, 10])
    n_ids = rng.choice([Q // 2 + 2, Q + 3, 3 * Q])          # all-hit, mixed and eviction-heavy regimes
    margin = 0.5 if loss_type == 'Arc' else 0.4
    torch.manual_seed(seed)
    m = ref_shim.make_ffc(D, Q, 32.0, loss_type, margin)
    o = HeadOracle(D, Q, 32.0, loss_type, margin, queue=m.queue.detach().clone(), dtype=torch.float32)
    gen = torch.Generator().manual_seed(seed + 50)
    for step in range(5):
        ids = torch.randperm(n_ids, generator=gen)[:B // 2]
        xl = torch.cat([ids, torch.randint(0, n_ids, (B - B // 2,), generator=gen)])
        yl = torch.cat([ids, torch.randint(0, n_ids, (B - B // 2,), generator=gen)])
        x = F.normalize(torch.randn(B, D, generator=gen))
        y = F.normalize(torch.randn(B, D, generator=gen))
        loss_ref, dx_ref, dy_ref, trace = ref_shim.forward_backward(m, x, y, xl.tolist(), yl.tolist())
        xo, yo = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        loss = o.forward(xo, yo, xl.tolist(), yl.tolist())
        if torch.is_tensor(loss) and loss.requires_grad:
            loss.backward()
        for got, want in zip(o.trace[-2:], trace):
            for k in ('rows', 'cols', 'labels', 'ones'):
                assert got[k] == want[k], (step, k)
        assert o.lru.state_dict() == m.lru.state_dict() and o.lru.cur_idx == m.lru.cur_idx
        assert o.qpos == [m.queue_position_dict[i] for i in range(Q)]
        if np.isfinite(loss_ref):       # Arc: |cos_t| can reach 1 (sqrt(1 - 1) has an infinite slope, ffc.py:101): NaN on both sides
            assert abs(float(loss) - loss_ref) <= 2e-5 * abs(loss_ref) + 1e-6, (step, float(loss), loss_ref)
            for got, want in ((xo.grad, dx_ref), (yo.grad, dy_ref)):
                got = torch.zeros_like(want) if got is None else got
                assert (got - want).norm() <= 5e-5 * want.norm() + 1e-6, step
        else:
            assert not np.isfinite(float(loss))
        assert torch.allclose(o.queue.float(), m.queue.float(), atol=1e-6)


@pytest.mark.parametrize('seed', recorded.LRU_SEEDS)
def test_lru_random_streams_recorded(golden_dir, seed):
    """test_lru_random_streams against the stored stream of the same seed"""
    with gzip.open(os.path.join(golden_dir, 'random_lru_streams.json.gz'), 'rt') as f:
        stream = json.load(f)['streams'][seed]
    assert stream['seed'] == seed and len(stream['ops']) > 1000
    cap = stream['capacity']
    lru = LRU(cap)
    for op in stream['ops']:
        kind = op[0]
        if kind == 'get':
            assert lru.get(op[1]) == op[2]
        elif kind == 'try_get':
            assert lru.try_get(op[1]) == op[2]
        elif kind == 'rollback_steps':
            lru.rollback_steps(op[1])
        elif kind == 'rollback_one_step':
            lru.rollback_one_step()
        elif kind == 'view':
            assert lru.view(op[1]) == op[2] and (op[1] in lru) == op[3]
        elif kind == 'restore':             # restore round trip into a fresh cache (lru.py:113-128)
            assert [list(kv) for kv in lru.state_dict()] == op[1]
            lru = LRU(cap)
            lru.restore([tuple(kv) for kv in op[1]])
        else:
            _, sd, cur_idx, it, keys = op
            assert [list(kv) for kv in lru.state_dict()] == sd and lru.cur_idx == cur_idx
            assert [list(kv) for kv in lru] == (sd if it is None else it)
            assert sorted(lru.keys()) == (sorted(k for k, _ in sd) if keys is None else keys)


@pytest.mark.parametrize('seed', recorded.HEAD_SEEDS)
@pytest.mark.parametrize('loss_type', recorded.HEAD_LOSSES)
def test_head_random_configs_recorded(golden_dir, seed, loss_type):
    """test_head_random_configs against the stored values of the same configuration, with the same tolerances"""
    z = np.load(os.path.join(golden_dir, 'random_head_configs.npz'))
    rec = {k[len(f'{loss_type}_{seed}_'):]: z[k] for k in z.files if k.startswith(f'{loss_type}_{seed}_')}
    D, Q, B, n_ids, margin = recorded.head_config(seed, loss_type)
    o = HeadOracle(D, Q, 32.0, loss_type, margin, queue=torch.from_numpy(rec['queue0']), dtype=torch.float32)
    n_steps = 0
    for step, (x, y, xl, yl) in enumerate(recorded.head_batches(seed, loss_type)):
        inputs = rec['inputs'][step]
        assert abs(float(x.double().sum()) - inputs[0]) <= 1e-9 and abs(float(y.double().sum()) - inputs[1]) <= 1e-9, 'seeded batches changed'
        assert [int(xl.sum()), int(yl.sum())] == inputs[2:].astype(np.int64).tolist(), 'seeded labels changed'
        xo, yo = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
        loss = o.forward(xo, yo, xl.tolist(), yl.tolist())
        if torch.is_tensor(loss) and loss.requires_grad:
            loss.backward()
        for got, want in zip(o.trace[-2:], rec['trace'][step]):
            for k, w in zip(('rows', 'cols', 'labels', 'ones'), want.tolist()):
                assert got[k] == (w if k != 'ones' else [v for v in w if v >= 0]), (step, k)
        assert [list(kv) for kv in o.lru.state_dict()] == [kv for kv in rec['lru'][step].tolist() if kv != [-1, -1]], step
        assert o.lru.cur_idx == rec['cur_idx'][step] and o.qpos == rec['qpos'][step].tolist(), step
        loss_ref = float(rec['loss'][step])
        if np.isfinite(loss_ref):       # Arc: |cos_t| can reach 1 (ffc.py:101): NaN on both sides
            assert abs(float(loss) - loss_ref) <= 2e-5 * abs(loss_ref) + 1e-6, (step, float(loss), loss_ref)
            for got, want in ((xo.grad, rec['dx'][step]), (yo.grad, rec['dy'][step])):
                want = torch.from_numpy(want)
                got = torch.zeros_like(want) if got is None else got
                assert (got - want).norm() <= 5e-5 * want.norm() + 1e-6, step
        else:
            assert not np.isfinite(float(loss))
        n_steps += 1
    assert n_steps == 5
    assert torch.allclose(o.queue.float(), torch.from_numpy(rec['queue_final']), atol=1e-6)


@pytest.mark.parametrize('seed', range(5))
def test_tail_against_torch(seed):
    rng = np.random.default_rng(seed)
    B, D = int(rng.integers(2, 40)), int(rng.integers(1, 70))
    for training in (True, False):
        for affine in (True, False):
            bn = torch.nn.BatchNorm1d(D, eps=1e-05, affine=affine).double()
            with torch.no_grad():
                bn.running_mean.normal_(0, 0.3)
                bn.running_var.uniform_(0.5, 2.0)
                if affine:
                    bn.weight.uniform_(0.5, 1.5)
                    bn.bias.normal_(0, 0.3)
            bn.train(training)
            rm0, rv0 = bn.running_mean.numpy().copy(), bn.running_var.numpy().copy()
            x = torch.tensor(rng.normal(0.2, 1.5, size=(B, D)), requires_grad=True)
            dp = torch.tensor(rng.normal(size=(B, D)))
            p = F.normalize(bn(x))
            p.backward(dp)
            w = bn.weight.detach().numpy() if affine else None
            b = bn.bias.detach().numpy() if affine else None
            po, cache, rm, rv = tail_ref.tail_forward(x.detach().numpy(), w, b, rm0, rv0, training=training)
            dx, dw, db = tail_ref.tail_backward(dp.numpy(), cache)
            np.testing.assert_allclose(po, p.detach().numpy(), rtol=1e-10, atol=1e-12)
            np.testing.assert_allclose(dx, x.grad.numpy(), rtol=1e-8, atol=1e-11)
            np.testing.assert_allclose(rm, bn.running_mean.numpy(), rtol=1e-12, atol=1e-14)
            np.testing.assert_allclose(rv, bn.running_var.numpy(), rtol=1e-12, atol=1e-14)
            if affine:
                np.testing.assert_allclose(dw, bn.weight.grad.numpy(), rtol=1e-8, atol=1e-11)
                np.testing.assert_allclose(db, bn.bias.grad.numpy(), rtol=1e-8, atol=1e-11)
