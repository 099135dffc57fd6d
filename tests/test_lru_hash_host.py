"""Host checks of the key crafting that the device LRU's adversarial tests rely on (oracle/lru_keys.py): mix64 and its
inverse, keys for a chosen home window / local cell, and the table size, pinned to the CUDA sources."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import lru_keys as K

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'very-large-scale-face-recognition_b200', 'csrc')

EDGES = [0, 1, 2, (1 << 63) - 1, 1 << 63, (1 << 63) + 1, (1 << 63) + 2, (1 << 64) - 1, (1 << 64) - 2, 0x5555555555555555,
         0xaaaaaaaaaaaaaaaa, 1 << 33, (1 << 33) - 1]


def _inputs(n):
    rng = np.random.default_rng(1234)
    r = [int(v) for v in rng.integers(0, 1 << 63, size=n - len(EDGES), dtype=np.uint64)]
    return EDGES + [v | ((i & 1) << 63) for i, v in enumerate(r)]


def test_unmix_inverts_mix():
    for x in _inputs(10000):
        assert K.unmix64(K.mix64(x)) == x and K.mix64(K.unmix64(x)) == x
    assert K.mix64(0) == 0 and K.mix64(1) != 1


def test_numpy_mix_matches_scalar():
    xs = _inputs(10000)
    signed = np.array([K.to_signed(x) for x in xs], dtype=np.int64)
    assert [int(v) for v in K.mix64_np(signed)] == [K.mix64(x) for x in xs]


def test_table_size_formula_is_ffc_lru_create():
    """The one place the tests state T: ffc_lru_create's formula, read from the source, and its values at the capacities the
    adversarial tests use."""
    src = open(os.path.join(CSRC, 'lru.cu')).read()
    assert re.search(r'h->T = std::max<int64_t>\(next_pow2\(4 \* capacity\), \(int64_t\)1 << 18\);', src)
    assert re.search(r'LHSZ = 4096;', src)
    for cap, t in ((1, 1 << 18), (64, 1 << 18), (7409, 1 << 18), (65536, 1 << 18), (65537, 1 << 19), (1 << 17, 1 << 19),
                   (1 << 20, 1 << 22), (3 << 18, 1 << 22)):
        assert K.table_cells(cap) == t, cap
        assert K.table_windows(cap) == t // 32


@pytest.mark.parametrize('nwin', [8192, 16384, 131072])
def test_keys_in_window(nwin):
    rng = np.random.default_rng(nwin)
    for w in (0, 1, nwin // 3, nwin - 1):
        keys = K.keys_in_window(w, nwin, 300, rng)
        assert len(set(keys)) == 300
        assert all(K.KEY_TOMB < k < (1 << 63) for k in keys)
        assert all(K.mix64(k) & (nwin - 1) == w for k in keys)
        counts = K.home_window_counts(keys, nwin)
        assert counts[w] == 300 and counts.sum() == 300


def test_keys_in_local_cell():
    rng = np.random.default_rng(7)
    for c in (0, 17, K.LHSZ - 1):
        keys = K.keys_in_local_cell(c, 1024, rng)
        assert len(set(keys)) == 1024
        assert all(K.mix64(k) & (K.LHSZ - 1) == c for k in keys)


def _nvcc():
    env = os.environ.get('NVCC')
    if env and os.path.isfile(env):
        return env
    return shutil.which('nvcc') or next((p for p in ('/usr/local/cuda/bin/nvcc',) if os.path.isfile(p)), None)


PIN_SRC = r'''
#include <cstdio>
#include "ffc_common.cuh"
int main() {
  unsigned long long x;
  while (std::scanf("%llx", &x) == 1) std::printf("%016llx\n", (unsigned long long)ffc::mix64(x));
  return 0;
}
'''


def test_mix64_pinned_to_the_header(tmp_path):
    """The Python mix64 against ffc::mix64 of csrc/ffc_common.cuh, compiled into a host program: 10 000 values."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip('nvcc not found')
    src = tmp_path / 'pin.cu'
    src.write_text(PIN_SRC)
    exe = tmp_path / 'pin'
    subprocess.run([nvcc, '-std=c++17', '-I', CSRC, str(src), '-o', str(exe)], check=True, capture_output=True, text=True)
    xs = _inputs(10000)
    r = subprocess.run([str(exe)], input=''.join(f'{x:x}\n' for x in xs), check=True, capture_output=True, text=True)
    got = [int(v, 16) for v in r.stdout.split()]
    assert got == [K.mix64(x) for x in xs]
