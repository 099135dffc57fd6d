"""bench.py on the device: --steps sets the number of timed steps, and --dump-outputs writes what the last timed step returned, from
inputs that are the same on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(out_dir, steps, warmup):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'c2', '--steps', str(steps), '--warmup', str(warmup),
                        '--no-cpu', '--no-aux', '--dump-outputs', str(out_dir)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line['steps'] == steps and line['roofline']['launches'] == 2 * steps          # one main sweep per pass, two passes per step
    return line, {n: np.load(out_dir / f'{n}.npy') for n in ('loss', 'dx', 'dy')}


def test_bench_dumps_the_last_timed_step(tmp_path):
    # --steps 3 --warmup 1 and --steps 2 --warmup 2 run the same four batches from the same seeded queue and end on the same step: the
    # dumps are equal bit for bit.  --steps 2 --warmup 1 ends one batch earlier (its last step is the third step of the first run).
    line, a = _run(tmp_path / 'a', 3, 1)
    _, b = _run(tmp_path / 'b', 2, 2)
    _, c = _run(tmp_path / 'c', 2, 1)
    assert a['loss'].dtype == a['dx'].dtype == a['dy'].dtype == np.float32
    assert a['loss'].shape == () and a['dx'].shape == a['dy'].shape == (512, 512)      # C2: B = 512, D = 512
    assert float(a['loss']) == line['loss'] and np.isfinite(a['dx']).all() and np.isfinite(a['dy']).all()
    for n in ('loss', 'dx', 'dy'):
        assert np.array_equal(a[n], b[n]), n
        assert not np.array_equal(a[n], c[n]), n
    assert not np.array_equal(a['dx'], a['dy'])
