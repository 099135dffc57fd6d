"""Host-side contract of bench.py (no GPU): synthetic batch composition (SURVEY.md 8(d)), the shared `config` object, and the JSON line
of the reference arm (`--impl reference`: the reference algorithm's CPU port on the host cores)."""
import importlib.util
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_make_batches_follow_the_reference_composition():
    b = _bench()
    w = dict(b.WORKLOADS['c3'], B=64, N=5000, D=16)
    for rank, world in ((0, 1), (1, 4)):
        batches = b.make_batches(w, 3, seed=1234, rank=rank, world=world)
        again = b.make_batches(w, 3, seed=1234, rank=rank, world=world)
        for (x, y, xl, yl), (x2, _, xl2, _) in zip(batches, again):
            assert torch.equal(x, x2) and torch.equal(xl, xl2)                          # seeded
            assert x.shape == y.shape == (64, 16) and xl.dtype == torch.int64 and not xl.is_cuda
            assert torch.allclose(x.norm(dim=1), torch.ones(64), atol=1e-5)             # unit-norm embeddings (ffc.py:157)
            assert torch.equal(xl[:32], yl[:32]) and len(set(xl[:32].tolist())) == 32   # id half: same ids in x and y, distinct (main.py:58-60)
            assert int(xl.max()) < 5000 and int(xl.min()) >= 0
    a = b.make_batches(w, 1, seed=1234, rank=0, world=2)[0]
    c = b.make_batches(w, 1, seed=1234, rank=1, world=2)[0]
    assert not set(a[2][:32].tolist()) & set(c[2][:32].tolist())                        # ranks draw different chunks of the permutation


def test_config_object_is_shared_by_both_arms():
    b = _bench()
    c1, c8 = b.config_of(b.WORKLOADS['c3'], 1), b.config_of(b.WORKLOADS['c3'], 8)
    assert c1['workload'].startswith('C3') and c1['queue'] == 1 << 20 and c1['identities'] == 1 << 20 and c1['feat_dim'] == 512
    assert c1['rows_per_pass_per_gpu'] == 1024 and c1['passes_per_step'] == 2 and 'model' not in c1
    assert c1['sharding'] == 'none' and c8['sharding'] == 'queue columns /8' and 'L2' in c1['l2_policy']


def test_reference_arm_json_line():
    env = dict(os.environ, OMP_NUM_THREADS='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'c2', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['metric'] == 'ffc_head_fwd_bwd_samples_per_s' and line['unit'] == 'samples/s'
    assert line['higher_is_better'] is True and line['value'] > 0 and line['vs_baseline'] is None
    # the shared keys are our arm's config; the reference arm adds the shape it really ran and says that the figure is extrapolated
    ours = _bench().config_of(_bench().WORKLOADS['c2'], 1)
    assert {k: line['config'][k] for k in ours} == ours
    rs = line['config']['reference_sample']
    assert rs['rows_per_pass'] == 512 and rs['queue'] == 32768 and rs['extrapolated'] is True
    cb = line['cpu_baseline']
    from oracle import ref_shim
    assert cb['kind'] == ('reference' if ref_shim.available() else 'port') and cb['value'] == line['value'] and 'queue' in cb['sample']
    assert cb['cores'] >= min(4, os.cpu_count())          # all host threads, whatever OMP_NUM_THREADS says (torchrun exports 1)
    assert line['e2e'] == {'value': line['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    # a non-zero rank of a torchrun launch exits 0 without work
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=120, env=dict(env, RANK='1', WORLD_SIZE='2'))
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_dump_outputs_files(tmp_path):
    """--dump-outputs: one float32 .npy per returned array (loss, dLoss/dx, dLoss/dy), a rank suffix when sharded"""
    import numpy as np
    b = _bench()
    out = (torch.tensor(3.25), torch.randn(6, 4), torch.randn(6, 4, dtype=torch.float64))
    b.dump_outputs(str(tmp_path / 'one'), out, 0, 1)
    assert sorted(os.listdir(tmp_path / 'one')) == ['dx.npy', 'dy.npy', 'loss.npy']
    for name, t in zip(('loss', 'dx', 'dy'), out):
        a = np.load(tmp_path / 'one' / f'{name}.npy')
        assert a.dtype == np.float32 and a.shape == tuple(t.shape) and np.array_equal(a, t.float().numpy())
    b.dump_outputs(str(tmp_path / 'sharded'), out, 3, 4)
    assert sorted(os.listdir(tmp_path / 'sharded')) == ['dx_rank3.npy', 'dy_rank3.npy', 'loss_rank3.npy']


def test_steps_and_dump_arguments_are_checked():
    for extra in (['--steps', '0'], ['--warmup', '-1'], ['--impl', 'reference', '--dump-outputs', 'x']):
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and r.stdout == '', (extra, r.stderr)


def test_executed_flop_accounting_and_limiter_note():
    """roofline.achieved counts executed tensor FLOPs: every row's cosines, and the gradient sum only for the row tiles that hold a row with a
    softmax term (hard-negative-only rows are swept last and skip GEMM-2); the limiter note counts the W tiles both CTAs of a pair stream."""
    b = _bench()

    class OneGpu:          # FFCHead: bookkeeping set 1 = the commit pass
        def __init__(self, lab):
            self._sets = [dict(label=None), dict(label=lab)]

    class Sharded:         # ShardedFFCHead: the commit pass's all-reduced labels
        def __init__(self, lab):
            self._last = dict(label=lab)

    lab = torch.full((512,), -1, dtype=torch.int32)
    lab[:130] = 7                                     # 130 rows with a known label -> two row tiles run GEMM-2
    assert b.softmax_rows(OneGpu(lab), 512) == 256 and b.softmax_rows(Sharded(lab), 512) == 256
    assert b.softmax_rows(OneGpu(torch.zeros(1024, dtype=torch.int32)), 1024) == 1024       # C3: every label known -> 4*B*Q*D
    assert b.softmax_rows(OneGpu(torch.full((300,), -1, dtype=torch.int32)), 300) == 0
    assert b.softmax_rows(object(), 77) == 77         # unknown head type: assume every row
    note = b.l2_to_sm_note(1024, 1 << 20, 512, 1.443)
    assert note['w_tile_bytes_per_launch'] == 2 * 8 * 8192 * 128 * 512 * 2 and 11.5 < note['delivered_tb_per_s'] < 12.5
    assert b.l2_to_sm_note(1024, 1 << 20, 128, 0.45) is None          # the one-CTA kernel loads every tile once: no such note
