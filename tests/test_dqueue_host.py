"""Queue-gradient mode on the host: argument checks of the C ABI before any device work, the missing-device error, and what the
compiler made of the SV mode of the swapped tcgen05 sweep."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'


def test_dqueue_argument_checks_run_on_the_host():
    from ffc_b200 import _capi
    lib = _capi.lib()
    launches = lib.ffc_launch_count()
    hp = _capi.HeadPass()
    assert lib.ffc_head_set_dqueue(None, 1) != 0 and b'NULL handle' in lib.ffc_last_error()
    assert lib.ffc_head_dqueue(None, C.byref(hp), 0x1000, None) != 0 and b'NULL argument' in lib.ffc_last_error()
    assert lib.ffc_head_dqueue(None, None, 0x1000, None) != 0 and b'NULL argument' in lib.ffc_last_error()
    assert lib.ffc_launch_count() == launches


@pytest.mark.parametrize('loss_type,precision', [('SV', 'bf16'), ('AM', 'fp32'), ('SV', 'fp32')])
def test_queue_grad_without_cuda_raises(loss_type, precision):
    import ffc_b200
    m = ffc_b200.FFCHead(16, 32, loss_type=loss_type, precision=precision, queue_grad=True)
    assert m.queue_grad and m.dqueue is None
    with pytest.raises(ffc_b200.FFCError):
        m.head(torch.randn(4, 16), torch.randn(4, 16), [0, 1, 2, 3], [0, 1, 2, 3])


def test_sv_swapped_sweep_sass_is_tcgen05():
    if not os.path.isfile(CUOBJDUMP):
        pytest.skip('cuobjdump not available')
    import importlib.util
    spec = importlib.util.spec_from_file_location('ffc_build', os.path.join(ROOT, 'very-large-scale-face-recognition_b200', 'build.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    lib = mod.build()
    r = subprocess.run([CUOBJDUMP, '-sass', lib], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    fns, name = {}, None
    for line in r.stdout.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            name = m.group(1)
            fns[name] = []
        elif name is not None:
            fns[name].append(line)
    # ffc_head_sweep_sm100_kernel<false, D, true>: the DQ_SV instantiations
    kern = {n: '\n'.join(v) for n, v in fns.items() if re.search(r'ffc_head_sweep_sm100_kernelILb0ELi\d+ELb1E', n)}
    assert len(kern) == 4                                   # D = 64 / 128 / 256 / 512
    for n, body in kern.items():
        for mnemonic in ('UTCHMMA', 'LDTM', 'UTMALDG'):
            assert mnemonic in body, (n, mnemonic)
        assert not re.search(r'\bHMMA\b', body), n
