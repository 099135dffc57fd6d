"""GPU parity: device LRU vs the oracle (oracle/lru_ref.py) and the reference traces.  Bit-exact."""
import json
import os
import random

import pytest
import torch

from oracle.lru_ref import LRU as RefLRU
from oracle.lru_ref import ref_batch as _ref_batch

pytestmark = pytest.mark.gpu


def _dev_lru(cap, **kw):
    import ffc_b200
    return ffc_b200.LRU(cap, **kw)


def test_reference_traces_scalar_api(golden_dir):
    with open(os.path.join(golden_dir, 'lru_traces.json')) as f:
        cases = json.load(f)
    n = 0
    for case in cases:
        lru = _dev_lru(case['capacity'])
        if 'restore' in case:
            lru.restore([tuple(kv) for kv in case['restore']])
            assert [lru.get(k) for k in case['gets']] == case['slots']
            assert [list(kv) for kv in lru.state_dict()] == case['final']
            assert sorted(lru.keys()) == sorted(k for k, _ in case['final'])
            continue
        ops = case['ops'] if case['capacity'] <= 16 else case['ops'][:400]
        for op in ops:
            kind, arg = op[0], op[1]
            if kind == 'get':
                assert lru.get(arg) == op[2], (case['capacity'], n)
            elif kind == 'try_get':
                assert lru.try_get(arg) == op[2], (case['capacity'], n)
            elif kind == 'rollback_steps':
                lru.rollback_steps(arg)
            elif kind == 'view':
                assert lru.view(arg) == op[2]
            elif kind == 'contains':
                assert (arg in lru) == op[2]
            else:
                assert [list(kv) for kv in lru.state_dict()] == op[2]
                assert lru.cur_idx == op[3]
            n += 1
    assert n > 1000


@pytest.mark.parametrize('cap,universe,batch', [(1, 5, 7), (2, 6, 16), (7, 12, 16), (64, 90, 48), (64, 4000, 64),
                                                 (1000, 1500, 256), (1000, 100000, 512), (5000, 5200, 1024), (300, 100000, 1024)])
def test_batched_assign_matches_oracle(cap, universe, batch):
    dev = torch.device('cuda')
    rng = random.Random(cap * 7919 + batch)
    lru = _dev_lru(cap)
    ref = RefLRU(cap)
    qpos = torch.zeros(cap, dtype=torch.uint8, device=dev)
    ref_qpos = [0] * cap
    cmask = torch.zeros(cap // 32 + 2, dtype=torch.int32, device=dev)
    for step in range(14):
        n = batch if step % 3 else rng.randrange(1, batch + 1)
        # mix of fresh ids, repeats inside the batch and old ids
        keys = [rng.randrange(universe) for _ in range(n)]
        if step % 4 == 1:
            keys = [keys[rng.randrange(max(1, n // 3))] for _ in range(n)]
        journal = step % 2 == 1
        kt = torch.tensor(keys, dtype=torch.int64, device=dev)
        rows = torch.empty(n, dtype=torch.int32, device=dev)
        cols = torch.empty(n, dtype=torch.int32, device=dev)
        hit = torch.empty(n, dtype=torch.uint8, device=dev)
        ones_list = torch.empty(n, dtype=torch.int32, device=dev)
        n_ones = torch.zeros(1, dtype=torch.int32, device=dev)
        before = ref.state_dict()
        q_before = list(ref_qpos)
        lru.assign(kt, journal=journal, qpos=qpos, rows=rows, cols=cols, hit=hit, ones_list=ones_list, n_ones=n_ones, cmask=cmask)
        r_rows, r_cols, r_hits, r_ones = _ref_batch(ref, ref_qpos, keys, journal)
        assert cols.tolist() == r_cols, (step, journal)
        assert rows.tolist() == r_rows
        assert hit.tolist() == r_hits
        no = int(n_ones.item())
        assert sorted(ones_list[:no].tolist()) == sorted(r_ones)
        bits = set()
        for w, v in enumerate(cmask.tolist()):
            v &= 0xffffffff
            while v:
                b = (v & -v).bit_length() - 1
                bits.add(w * 32 + b)
                v &= v - 1
        assert bits == r_ones
        cmask.zero_()
        # probe view after the batch
        probe = [rng.randrange(universe) for _ in range(37)] + keys[:5]
        pv = lru.view_batch(torch.tensor(probe, dtype=torch.int64, device=dev)).tolist()
        assert pv == [ref.view(k) for k in probe]
        assert lru.state_dict() == ref.state_dict()
        assert qpos.cpu().tolist() == ref_qpos
        if journal:
            if step % 4 == 3 and n > 2:      # partial rollback first (lru.py:252-255 semantics)
                part = rng.randrange(1, n)
                lru.undo(part, qpos)
                ref.rollback_steps(part)
                assert lru.state_dict() == ref.state_dict()
                lru.undo(n - part, qpos)
                ref.rollback_steps(n - part)
            else:
                lru.undo(n, qpos)
                ref.rollback_steps(n)
            ref_qpos[:] = q_before
            assert lru.state_dict() == before
            assert qpos.cpu().tolist() == q_before
            assert lru.cur_idx == ref.cur_idx
            assert lru.journal_len == 0


def test_long_run_compaction_and_rebuild():
    """Enough batches to force ring compaction and hash-table rebuilds (capacity 512 -> ring 16384)."""
    dev = torch.device('cuda')
    rng = random.Random(5)
    cap = 512
    lru, ref = _dev_lru(cap), RefLRU(cap)
    for step in range(80):
        universe = 600 if step % 2 else 100000
        keys = [rng.randrange(universe) for _ in range(1024)]
        cols = lru.assign(torch.tensor(keys, dtype=torch.int64, device=dev))
        assert cols.tolist() == [ref.get(k) for k in keys], step
    assert lru.state_dict() == ref.state_dict()


def test_export_import_round_trip():
    dev = torch.device('cuda')
    rng = random.Random(9)
    a, ref = _dev_lru(100), RefLRU(100)
    keys = [rng.randrange(400) for _ in range(700)]
    a.assign(torch.tensor(keys, dtype=torch.int64, device=dev))
    for k in keys:
        ref.get(k)
    sd = a.state_dict()
    assert sd == ref.state_dict()
    b = _dev_lru(100)
    b.restore(sd)
    ref2 = RefLRU(100)
    ref2.restore(sd)
    more = [rng.randrange(500) for _ in range(300)]
    assert b.assign(torch.tensor(more, dtype=torch.int64, device=dev)).tolist() == [ref2.get(k) for k in more]
    assert b.state_dict() == ref2.state_dict()
    b.clear()
    assert b.state_dict() == [] and b.cur_idx == 0
    assert b.get(77) == 0


@pytest.mark.parametrize('cap,pass_keys', [(7409, 8192), (1024, 4096), (100, 3000)])
def test_long_run_multi_chunk_passes(cap, pass_keys):
    """A sharded head's pattern (ffc_b200/dist.py): every pass brings R*B keys -- several 1024-key chunks of the resolve CTA -- as ONE
    ffc_lru_assign call, journaled passes are undone, commit passes stay; capacities that are not powers of two (the reference's
    default queue_size is 7409, ffc.py:11).  Ring space for the whole pass is reserved before its first chunk: 60 steps never hit
    'recency ring full', and the state matches the oracle after every pass."""
    dev = torch.device('cuda')
    rng = random.Random(cap + pass_keys)
    lru, ref = _dev_lru(cap), RefLRU(cap)
    qpos = torch.zeros(cap, dtype=torch.uint8, device=dev)
    ref_qpos = [0] * cap
    universe = 6 * cap
    for step in range(60):
        for journal in (True, False):
            keys = [rng.randrange(universe) for _ in range(pass_keys)]
            kt = torch.tensor(keys, dtype=torch.int64, device=dev)
            rows = torch.empty(pass_keys, dtype=torch.int32, device=dev)
            cols = torch.empty(pass_keys, dtype=torch.int32, device=dev)
            q_before = list(ref_qpos)
            lru.assign(kt, journal=journal, qpos=qpos, rows=rows, cols=cols)
            r_rows, r_cols, _, _ = _ref_batch(ref, ref_qpos, keys, journal)
            assert cols.tolist() == r_cols and rows.tolist() == r_rows, (step, journal)
            if journal:
                lru.undo(-1, qpos)
                ref.rollback_steps(pass_keys)
                ref_qpos[:] = q_before
                assert lru.journal_len == 0
        if step % 10 == 9:
            assert lru.state_dict() == ref.state_dict() and qpos.cpu().tolist() == ref_qpos
    assert lru.state_dict() == ref.state_dict() and lru.cur_idx == ref.cur_idx


def test_device_side_key_count_stops_the_chunk_walk():
    """n_dev (a rank's share of an all-gathered batch, known only on the device): keys [0, *n_dev) are processed -- across chunk
    boundaries -- and the outputs of the remaining positions stay untouched."""
    dev = torch.device('cuda')
    rng = random.Random(77)
    cap, n = 3000, 8192
    lru, ref = _dev_lru(cap), RefLRU(cap)
    for n_eff in (1100, 0, 1024, 2500, 8192, 1):
        keys = [rng.randrange(5 * cap) for _ in range(n)]
        kt = torch.tensor(keys, dtype=torch.int64, device=dev)
        cols = torch.full((n,), -7, dtype=torch.int32, device=dev)
        nd = torch.tensor([n_eff], dtype=torch.int32, device=dev)
        lru.assign(kt, cols=cols, n_dev=nd)
        got = cols.tolist()
        assert got[:n_eff] == [ref.get(k) for k in keys[:n_eff]] and all(v == -7 for v in got[n_eff:])
        assert lru.state_dict() == ref.state_dict()
