"""1:N identification on the build host: the fp64 oracle against brute force, the C ABI's argument checks, the missing-device
error, the sharded search's collectives under gloo (world 2, torch stand-in shards), the cmc helper and the search kernel's SASS."""
import os
import re
import shutil
import socket
import subprocess

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import identify_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
NVCC = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'


def _brute(x, state, q0, k, off=0):
    """per row: sort every resident slot by (-cos, global slot) with Python's sort"""
    xn = x / np.linalg.norm(x, axis=1, keepdims=True)
    res = []
    for row in xn:
        c = sorted(((-float(row @ q0[s]), s + off, key) for key, s in state))
        c = c[:k] + [(np.inf, -1, identify_ref.LABEL_NONE)] * max(0, k - len(c))
        res.append(c)
    return res


@pytest.mark.parametrize('seed', range(4))
def test_oracle_matches_brute_force(seed):
    rng = np.random.default_rng(seed)
    Q, D, k = 50, 8, 6
    q0 = rng.standard_normal((Q, D))
    q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    q0[7] = q0[3]                                   # exact tie: slot 3 before slot 7
    n_res = int(rng.integers(1, Q))
    slots = rng.permutation(n_res)                  # resident set is [0, n_res), listed in recency order
    state = [(int(1000 + 17 * s), int(s)) for s in slots]
    x = rng.standard_normal((9, D))
    x[0] = q0[3]
    x[1] = -q0[3]
    sc, lab, slo, _, _ = identify_ref.identify(x, state, q0, k, col_offset=100)
    want = _brute(x, state, q0, k, off=100)
    for i in range(x.shape[0]):
        assert [s for _, s, _ in want[i]] == slo[i].tolist()
        assert [l for _, _, l in want[i]] == lab[i].tolist()
        np.testing.assert_allclose([-c for c, _, _ in want[i]], sc[i], rtol=0, atol=1e-12)
    if n_res > 7:
        assert slo[0, :2].tolist() == [103, 107]     # tie order


def test_oracle_all_negative_cosines():
    rng = np.random.default_rng(7)
    q0 = np.abs(rng.standard_normal((30, 8)))
    q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    x = -np.abs(rng.standard_normal((5, 8)))          # every cosine < 0
    state = [(int(s) * 3, int(s)) for s in range(30)]
    sc, lab, slo, cos, _ = identify_ref.identify(x, state, q0, 4)
    assert (cos < 0).all() and (sc < 0).all()
    want = _brute(x, state, q0, 4)
    assert slo.tolist() == [[s for _, s, _ in w] for w in want]


def test_oracle_padding_and_empty_gallery():
    q0 = np.eye(4)
    sc, lab, slo, _, _ = identify_ref.identify(np.ones((2, 4)), [(5, 0), (9, 1)], q0, 3)
    assert slo.tolist() == [[0, 1, -1]] * 2 and lab[:, 2].tolist() == [identify_ref.LABEL_NONE] * 2 and np.isneginf(sc[:, 2]).all()
    sc, lab, slo, _, _ = identify_ref.identify(np.ones((2, 4)), [], q0, 2)
    assert (slo == -1).all() and (lab == identify_ref.LABEL_NONE).all() and np.isneginf(sc).all()


def test_identify_argument_checks_run_on_the_host():
    """ffc_identify validates n, k and its handles before touching the device"""
    import ctypes as C
    from ffc_b200 import _capi
    lib = _capi.lib()
    launches = lib.ffc_launch_count()
    need = C.c_int64()
    args = lambda n, k, h=None, lru=None: (h, lru, 0x1000, n, k, 0x2000, 0x3000, 0x4000, 1 << 20, 0x5000, 0x6000, 0x7000, None)
    assert lib.ffc_identify(*args(4, 11)) != 0 and b'k=11' in lib.ffc_last_error()
    assert lib.ffc_identify(*args(4, 0)) != 0 and b'k=0' in lib.ffc_last_error()
    assert lib.ffc_identify(*args(0, 5)) != 0 and b'n=0' in lib.ffc_last_error()
    assert lib.ffc_identify(*args(65537, 5)) != 0 and b'n=65537' in lib.ffc_last_error()
    assert lib.ffc_identify(*args(4, 5)) != 0 and b'NULL head' in lib.ffc_last_error()
    assert lib.ffc_identify_workspace_bytes(None, 4, 12, C.byref(need)) != 0 and b'k=12' in lib.ffc_last_error()
    assert lib.ffc_identify_workspace_bytes(None, 4, 5, C.byref(need)) != 0 and b'NULL' in lib.ffc_last_error()
    assert lib.ffc_launch_count() == launches


def test_identify_without_cuda_raises():
    import ffc_b200
    m = ffc_b200.FFCHead(16, 32)
    with pytest.raises(ffc_b200.FFCError):
        m.identify(torch.randn(3, 16), k=2)
    with pytest.raises(ffc_b200.FFCError, match='k=11'):
        m.identify(torch.randn(3, 16), k=11)


def test_cmc_hand_made():
    from ffc_b200 import cmc
    labels = torch.tensor([[5, 7, 9], [1, 2, 3], [4, 4, 4], [8, 6, 0]])
    true = torch.tensor([5, 3, 7, 6])            # rank 1, rank 3, not found (not resident), rank 2
    assert cmc(labels, true, ranks=(1, 2, 3, 10)) == {1: 0.25, 2: 0.5, 3: 0.75, 10: 0.75}
    with pytest.raises(ValueError):
        cmc(labels, true[:3])


# -- sharded search under gloo ------------------------------------------------------------------------------------------------
def _identify_backend_cls():
    from cpu_shard_backend import CpuShardBackend
    from ffc_b200.identify import Identification, LABEL_NONE

    class IdentifyCpuShardBackend(CpuShardBackend):
        """stand-in shard with the search of CudaShardBackend.identify_local, in fp64 torch"""

        def identify_local(self, x, k):
            xn = torch.nn.functional.normalize(x.double(), dim=1)
            st = self.lru.state_dict()
            n = xn.shape[0]
            scores = torch.full((n, k), float('-inf'), dtype=torch.float32)
            labels = torch.full((n, k), LABEL_NONE, dtype=torch.int64)
            slots = torch.full((n, k), -1, dtype=torch.int32)
            if st:
                sl = torch.tensor([s for _, s in st])
                keys = torch.tensor([key for key, _ in st])
                cos = xn @ self.queue[0][sl].t()
                for i in range(n):
                    order = sorted(range(len(st)), key=lambda j: (-float(cos[i, j]), int(sl[j])))[:k]
                    m = len(order)
                    scores[i, :m] = cos[i, order].float()
                    labels[i, :m] = keys[order]
                    slots[i, :m] = (sl[order] + self.off).int()
            return Identification(scores, labels, slots)
    return IdentifyCpuShardBackend


def _worker_identify(rank, world, port, ret):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from ffc_b200.dist import ShardedFFCHead
        from ffc_b200.ffc import hard_neg_k
        Backend = _identify_backend_cls()
        D, Q, k = 16, 67, 5                                 # 34 + 33 slots: uneven shards
        q0 = torch.nn.functional.normalize(torch.randn(2, Q, D, dtype=torch.float64, generator=torch.Generator().manual_seed(3)), dim=2)
        head = ShardedFFCHead(D, Q, 32.0, 'AM', 0.4, max_batch=4,
                              backend_factory=lambda ql, off, n: Backend(D, ql, Q, off, n, 32.0, 'AM', 0.4, hard_neg_k(Q), queue=q0[:, off:off + ql]))
        # rank 0 holds 20 identities (even keys), rank 1 only 3 (odd keys): most identities are resident on one rank only
        n_res = 20 if rank == 0 else 3
        keys = torch.arange(rank, 2 * n_res, 2, dtype=torch.int64)
        head.backend.lru.restore_arrays(keys, torch.randperm(n_res, generator=torch.Generator().manual_seed(rank)).int())
        states = [None, None]
        dist.all_gather_object(states, (head.backend.lru.state_dict(), head.off))
        union = identify_ref.union_state(states)
        gen = torch.Generator().manual_seed(11)
        x_all = torch.randn(9, D, dtype=torch.float64, generator=gen)
        x_all[0] = q0[0, 2]                                  # planted: global slot 2 (rank 0)
        x_all[5] = q0[0, head.off + 1] if rank == 1 else q0[0, 35]   # rank 1's own rows: 5 on rank 0 (rows 0-4), 4 on rank 1
        x_all[6] = -x_all[6].abs()
        mine = slice(0, 5) if rank == 0 else slice(5, 9)
        res = head.identify(x_all[mine], k=k)
        sc, lab, slo, _, _ = identify_ref.identify(x_all[mine].numpy(), union, q0[0].numpy(), k)
        assert res.slots.tolist() == slo.tolist(), (rank, res.slots, slo)
        assert res.labels.tolist() == lab.tolist()
        np.testing.assert_allclose(res.scores.double().numpy(), sc, rtol=0, atol=1e-6)
        if rank == 0:
            assert int(res.slots[0, 0]) == 2
        empty = head.identify(x_all[:0], k=2)            # every rank may pass no rows at all
        assert empty.slots.shape == (0, 2)
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


def test_sharded_identify_world2_gloo():
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker_identify, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: 'ok', 1: 'ok'}


# -- what the compiler made of the search kernel ------------------------------------------------------------------------------
def test_identify_kernel_sass_is_tcgen05():
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
    kern = {n: '\n'.join(v) for n, v in fns.items() if 'ffc_identify_sm100_kernel' in n}
    assert len(kern) == 4                                   # D = 64 / 128 / 256 / 512
    for n, body in kern.items():
        for mnemonic in ('UTCHMMA', 'LDTM', 'UTMALDG'):
            assert mnemonic in body, (n, mnemonic)
        assert not re.search(r'\bHMMA\b', body), n


def test_identify_kernels_do_not_spill():
    if not os.path.isfile(NVCC):
        pytest.skip('nvcc not available')
    import importlib.util
    spec = importlib.util.spec_from_file_location('ffc_build', os.path.join(ROOT, 'very-large-scale-face-recognition_b200', 'build.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        r = subprocess.run([mod.NVCC] + mod.FLAGS + ['-Xptxas', '-v', '-c', os.path.join(mod.CSRC, 'identify_sm100.cu'), '-o', os.path.join(td, 'i.o')],
                           capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    spills = re.findall(r'(\d+) bytes spill stores, (\d+) bytes spill loads', r.stderr)
    assert len(spills) >= 6                               # 4 tensor-core instances + check-mode search + merge
    assert all(a == '0' and b == '0' for a, b in spills), spills
