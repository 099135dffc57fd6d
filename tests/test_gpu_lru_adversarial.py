"""Device LRU against the oracle where random keys never reach: crafted hash collisions in the global table (chains over
many 32-cell windows, the wrap from the last window to window 0, tombstones inside chains, many warps inserting into one
full window, undo re-inserting evicted keys into chains, rebuild and compaction with chains live), crowded shared-memory
hashes of the resolve CTA, the boundaries of its closed-form path and chunk walk, extreme and reserved key values.

Keys are built by inverting mix64 (oracle/lru_keys.py).  Every call compares, bit for bit, cols / rows / hit / the `ones`
list and mask with the oracle (oracle/lru_ref.py), and then state_dict, cur_idx, the journal length, qpos and view_batch."""
import random

import numpy as np
import pytest
import torch

from oracle import lru_keys as K
from oracle.lru_ref import LRU as RefLRU
from oracle.lru_ref import ref_batch

pytestmark = pytest.mark.gpu

NB = 1024            # keys per chunk of the resolve CTA (FFC_LRU_MAX_BATCH)
MAX_KEYS = 65536     # keys per ffc_lru_assign call (FFC_LRU_MAX_KEYS)
INT64_MAX = (1 << 63) - 1


class Counters:
    """The host-side conservative counters of csrc/lru.cu (lru_maintain_for, ffc_lru_assign, ffc_lru_undo), to know when a pass
    compacted the ring or rebuilt the table: neither changes observable state, so the stream has to be steered onto them."""

    def __init__(self, cap):
        self.cap, self.T, self.RC = cap, K.table_cells(cap), K.table_cells(cap)
        self.ring = self.ht = self.jl = 0
        self.rebuilds = self.compactions = 0

    def maintain(self, reserve):
        if self.jl == 0 and self.ring + reserve + 2 * NB > self.RC:
            self.compactions += 1
            self.ring = self.cap
        if self.jl == 0 and self.ht + 2 * reserve + 2 * NB > self.T // 2:
            self.rebuilds += 1
            self.ht = self.cap

    def assign(self, n, journal):
        for a in range(0, n, MAX_KEYS):
            m = min(MAX_KEYS, n - a)
            self.maintain(m)
            self.ring += m
            self.ht += m
            self.jl += m if journal else 0

    def undo(self, steps):
        m = min(self.jl if steps < 0 else steps, self.jl)
        self.jl -= m
        self.ring -= m
        self.ht += m


def _eq(got, want, what):
    if got == want:
        return
    if len(got) != len(want):
        raise AssertionError(f'{what}: length {len(got)} != {len(want)}')
    i = next(i for i, (a, b) in enumerate(zip(got, want)) if a != b)
    raise AssertionError(f'{what}: first difference at {i}: device {got[i]!r}, oracle {want[i]!r}')


def _bits(mask):
    out = set()
    for w, v in enumerate(mask.tolist()):
        v &= 0xffffffff
        while v:
            b = (v & -v).bit_length() - 1
            out.add(w * 32 + b)
            v &= v - 1
    return out


class Twin:
    """A device LRU and the oracle fed the same stream."""

    def __init__(self, cap, journal_capacity=0):
        import ffc_b200
        self.cap = cap
        self.dev = torch.device('cuda')
        self.lru = ffc_b200.LRU(cap, journal_capacity=journal_capacity)
        self.ref = RefLRU(cap)
        self.qpos = torch.zeros(cap, dtype=torch.uint8, device=self.dev)
        self.ref_qpos = [0] * cap
        self.qlog = []                       # (slot, qpos before) per outstanding journaled access
        self.cmask = torch.zeros(cap // 32 + 1, dtype=torch.int32, device=self.dev)
        self.ctr = Counters(cap)

    def tensor(self, keys):
        return torch.tensor(list(keys), dtype=torch.int64, device=self.dev)

    def assign(self, keys, journal, probe=(), state=True):
        keys = list(keys)
        n = len(keys)
        dev = self.dev
        rows = torch.full((n,), -5, dtype=torch.int32, device=dev)
        cols = torch.full((n,), -5, dtype=torch.int32, device=dev)
        hit = torch.full((n,), 7, dtype=torch.uint8, device=dev)
        ones_list = torch.full((n,), -5, dtype=torch.int32, device=dev)
        n_ones = torch.zeros(1, dtype=torch.int32, device=dev)
        self.cmask.zero_()
        self.lru.assign(self.tensor(keys), journal=journal, qpos=self.qpos, rows=rows, cols=cols, hit=hit, ones_list=ones_list,
                        n_ones=n_ones, cmask=self.cmask)
        self.ctr.assign(n, journal)
        r_rows, r_cols, r_hits, r_ones = ref_batch(self.ref, self.ref_qpos, keys, journal, self.qlog if journal else None)
        _eq(cols.tolist(), r_cols, 'cols')
        _eq(rows.tolist(), r_rows, 'rows')
        _eq(hit.tolist(), r_hits, 'hit')
        ol = ones_list[:int(n_ones.item())].tolist()
        assert len(ol) == len(set(ol)) and set(ol) == r_ones, 'ones_list'
        assert _bits(self.cmask) == r_ones, 'cmask'
        if state:
            self.check(keys[:NB] + keys[-NB:] + list(probe))
        return r_cols

    def undo(self, steps, probe=()):
        self.lru.undo(steps, self.qpos)
        m = min(len(self.ref.op_stack) if steps < 0 else steps, len(self.ref.op_stack))
        self.ref.rollback_steps(m)
        for _ in range(m):
            s, q = self.qlog.pop()
            self.ref_qpos[s] = q
        self.ctr.undo(steps)
        self.check(probe)

    def maintain(self):
        from ffc_b200._capi import check
        check(self.lru._lib.ffc_lru_maintain(self.lru._h, self.lru._s()))
        self.ctr.maintain(0)
        self.check()

    def check(self, probe=()):
        assert self.lru.cur_idx == self.ref.cur_idx, 'cur_idx'
        assert self.lru.journal_len == len(self.ref.op_stack), 'journal length'
        _eq(self.lru.state_dict(), self.ref.state_dict(), 'state_dict')
        _eq(self.qpos.cpu().tolist(), self.ref_qpos, 'qpos')
        probe = list(probe)
        if probe:
            _eq(self.lru.view_batch(self.tensor(probe)).tolist(), [self.ref.view(k) for k in probe], 'view_batch')


# ------------------------------------------------------------------------------------------------------------------------
# global table: chains over many windows
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cap', [64, 1000, 7409, 1 << 17])
def test_window_chains(cap):
    """Home windows holding 33, 72 and 300 keys (chains of 2, 3 and > 8 windows), 300 keys homed in the last window (probing wraps
    to window 0) and a chunk of 1024 distinct keys of one window (32 warps CAS into the same full windows).  Journaled passes undone
    in full, in part and across chunks, two journaled passes outstanding at once, committed passes with evictions (tombstones inside
    chains, reused by later inserts), explicit maintenance, and 65 536-key passes until the table has been rebuilt and the ring
    compacted with the chains live; the same stream then goes on."""
    nwin = K.table_windows(cap)
    assert nwin == (8192 if cap <= 65536 else 4 * cap // 32)
    rng = np.random.default_rng(cap)
    prng = random.Random(cap)
    sizes = ((nwin // 7, 33), (nwin // 3, 72), (nwin // 2, 300), (nwin - 1, 300))
    crafted = [k for w, m in sizes for k in K.keys_in_window(w, nwin, m, rng)]
    flood = K.keys_in_window(nwin // 5, nwin, NB, rng)
    universe = 8 * cap + 4096
    t = Twin(cap, journal_capacity=1 << 17)

    def batch(n, share=0.5):
        return [prng.choice(crafted) if prng.random() < share else prng.randrange(universe) for _ in range(n)]

    order = list(crafted)
    prng.shuffle(order)
    t.assign(order, journal=True, probe=crafted)
    t.undo(-1, probe=crafted)
    t.assign(order, journal=False, probe=crafted)
    if cap >= len(crafted):
        live = K.home_window_counts(t.ref.keys(), nwin)
        assert live[nwin - 1] == 300 and live[nwin // 2] == 300 and live.max() == 300
    t.assign(flood, journal=True, probe=flood[:64])
    t.assign(flood[::-1], journal=True, probe=flood[:64])     # two journaled passes outstanding
    t.undo(NB + 5, probe=flood[:64])                          # across the pass boundary
    t.undo(-1, probe=flood[:64])
    t.assign(flood, journal=False, probe=flood[:64])

    def small_steps(steps):
        for step in range(steps):
            n = (700, NB, 2500, 5000)[step % 4]
            keys = batch(n)
            t.assign(keys, journal=True, probe=crafted[::7])
            mode = step % 3
            if mode == 1:
                t.undo(prng.randrange(1, n), probe=crafted[::7])
            elif mode == 2:
                t.undo(NB + 1 if n > NB + 1 else n - 1, probe=crafted[::7])
            t.undo(-1, probe=crafted[::7])
            t.assign(batch(n), journal=False, probe=crafted[::7])
            if step % 4 == 3:
                t.maintain()

    small_steps(6)
    for _ in range(12):
        if t.ctr.rebuilds and t.ctr.compactions:
            break
        t.assign(batch(MAX_KEYS, 0.2), journal=False, probe=crafted)
        t.assign(batch(3000), journal=True, probe=crafted)
        t.undo(1025, probe=crafted)
        t.undo(-1, probe=crafted)
    assert t.ctr.rebuilds >= 1 and t.ctr.compactions >= 1, (t.ctr.rebuilds, t.ctr.compactions)
    small_steps(6)




def _colliding_stream(cap, seed):
    nwin = K.table_windows(cap)
    rng = np.random.default_rng(seed)
    prng = random.Random(seed)
    crafted = K.keys_in_window(nwin - 1, nwin, 200, rng) + K.keys_in_window(3, nwin, 200, rng)

    def batch(n):
        return [prng.choice(crafted) if prng.random() < 0.3 else prng.randrange(4 * cap + 4096) for _ in range(n)]
    return crafted, batch


@pytest.mark.parametrize('which', ['table', 'ring'])
@pytest.mark.parametrize('cap', [64, 1 << 17])
def test_maintenance_thresholds(cap, which):
    """Passes sized so that the host counters land exactly on the rebuild (2n + used + 2*1024 == T/2) or compaction
    (n + used + 2*1024 == RC) threshold, where nothing is maintained, then the smallest pass past it, which rebuilds or compacts
    first; chains of colliding keys are live throughout."""
    crafted, batch = _colliding_stream(cap, cap + 3)
    t = Twin(cap, journal_capacity=1 << 17)
    c = t.ctr
    if which == 'table':
        room = lambda: c.T // 2 - 2 * NB - c.ht          # a pass of n keys rebuilds the table first iff 2n > room
        while room() // 2 > MAX_KEYS:
            t.assign(batch(MAX_KEYS), journal=False, probe=crafted)
        r = c.rebuilds
        t.assign(batch(room() // 2), journal=False, probe=crafted)
        assert c.rebuilds == r
        t.assign(batch(room() // 2 + 1), journal=False, probe=crafted)
        assert c.rebuilds == r + 1
    else:
        room = lambda: c.RC - 2 * NB - c.ring            # ... compacts the ring first iff n > room
        while room() > MAX_KEYS:
            t.assign(batch(MAX_KEYS), journal=False, probe=crafted)
        k = c.compactions
        t.assign(batch(room()), journal=False, probe=crafted)
        assert c.compactions == k and room() == 0
        t.assign(batch(1), journal=False, probe=crafted)
        assert c.compactions == k + 1
    t.assign(batch(3000), journal=True, probe=crafted)
    t.undo(1500, probe=crafted)
    t.undo(-1, probe=crafted)
    t.assign(batch(3000), journal=False, probe=crafted)


# ------------------------------------------------------------------------------------------------------------------------
# the resolve CTA's shared-memory hashes
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cap', [300, 1000, 2000])
def test_crowded_local_hash(cap):
    """Batches of 1024 distinct keys that all share the local hash's last cell (the probe wraps to cell 0), then the same keys with
    in-batch duplicates: above the distinct count (cap 2000, the closed form) and below it (the replay, evicting in-batch entries and
    refilling candidates).  Then 3000-key passes in which colliding keys recur across the 1024-key chunk boundaries."""
    rng = np.random.default_rng(cap + 11)
    prng = random.Random(cap + 11)
    crowd = K.keys_in_local_cell(K.LHSZ - 1, 3 * NB, rng)
    a, b = crowd[:NB], crowd[NB:2 * NB]
    t = Twin(cap)
    for keys in (a, b, a[::-1]):
        t.assign(keys, journal=True)
        t.undo(prng.randrange(1, NB))
        t.undo(-1)
        t.assign(keys, journal=False)
    few = a[:400] + b[:300] + crowd[2 * NB:2 * NB + 200]
    for step in range(4):
        keys = [prng.choice(few) for _ in range(NB)]
        t.assign(keys, journal=step % 2 == 0)
        if step % 2 == 0:
            t.undo(-1)
    for step in range(4):
        keys = [prng.choice(crowd) for _ in range(3000)]
        for p in (NB - 1, 2 * NB - 1):          # the same colliding key on both sides of a chunk boundary, and in the next chunk
            keys[p] = keys[p + 1] = keys[p + 2] = keys[p - 700]
        t.assign(keys, journal=step % 2 == 0)
        if step % 2 == 0:
            t.undo(NB + 1 + step)
            t.undo(-1)


# ------------------------------------------------------------------------------------------------------------------------
# path boundaries
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('extra', [0, 1])
@pytest.mark.parametrize('cap', [1023, 1024, 1025, 5000])
def test_misses_at_free_slots(cap, extra):
    """Batches whose distinct new keys equal the free slots (the closed form, with no eviction) or exceed them by one (the replay),
    in chunk 0 of a batch and in chunk 1 of a 2048-key batch."""
    prng = random.Random(cap * 2 + extra)
    nxt = iter(range(10 ** 6, 10 ** 7))
    for chunk in (0, 1):
        t = Twin(cap)
        t.assign([next(nxt) for _ in range(cap - 300)], journal=False)
        for journal in (True, False):
            free = cap - t.ref.cur_idx
            resident = list(t.ref.keys())
            new = [next(nxt) for _ in range(free + extra)]
            body = new + [prng.choice(resident) for _ in range(NB - len(new) - 150)] + [prng.choice(new) for _ in range(150)]
            first = body[:len(new)]                 # every new key's first occurrence stays inside the chunk
            rest = body[len(new):]
            prng.shuffle(rest)
            keys = first + rest
            if chunk:
                keys = [prng.choice(resident) for _ in range(NB)] + keys     # chunk 0: hits only
            t.assign(keys, journal=journal)
            if journal:
                t.undo(-1)


@pytest.mark.parametrize('cap', [1023, 1024, 1025])
def test_capacity_around_the_chunk(cap):
    prng = random.Random(cap)
    t = Twin(cap)
    nxt = iter(range(-10 ** 7, 0))
    for n in (NB, NB, NB + 1, 2 * NB, 3 * NB + 7):
        fresh = [next(nxt) for _ in range(n)]
        t.assign(fresh, journal=True)
        t.undo(n - NB if n > NB else 1)
        t.undo(-1)
        t.assign(fresh, journal=False)
        old = list(t.ref.keys())
        mixed = [prng.choice(old) if prng.random() < 0.5 else next(nxt) for _ in range(n)]
        t.assign(mixed, journal=False)


@pytest.mark.parametrize('n', [3000, 8192])
def test_partial_undo_of_multichunk_pass(n):
    """Journaled passes over several 1024-key chunks undone in two parts, the first of 1, 1023, 1025 and n - 1 accesses; and two
    outstanding passes undone across their boundary."""
    cap = 2000
    prng = random.Random(n)
    t = Twin(cap)
    universe = 3 * cap
    t.assign([prng.randrange(universe) for _ in range(2 * cap)], journal=False)
    for part in (1, NB - 1, NB + 1, n - 1):
        t.assign([prng.randrange(universe) for _ in range(n)], journal=True)
        t.undo(part)
        t.undo(-1)
        t.assign([prng.randrange(universe) for _ in range(n)], journal=False)
    t.assign([prng.randrange(universe) for _ in range(n)], journal=True)
    t.assign([prng.randrange(universe) for _ in range(n)], journal=True)
    t.undo(n + NB + 3)
    t.undo(-1)


def test_device_key_count_with_journal_then_undo_all():
    """assign(n_dev) journals only the keys [0, *n_dev); undo(-1) then rolls back what the device journal holds, not the n the host
    counted."""
    cap, n = 3000, 8192
    prng = random.Random(31)
    t = Twin(cap)
    t.assign([prng.randrange(5 * cap) for _ in range(2 * cap)], journal=False)
    for n_eff in (1100, 0, 1024, 2500, 8192, 1):
        keys = [prng.randrange(5 * cap) for _ in range(n)]
        cols = torch.full((n,), -7, dtype=torch.int32, device=t.dev)
        nd = torch.tensor([n_eff], dtype=torch.int32, device=t.dev)
        before = t.ref.state_dict()
        t.lru.assign(t.tensor(keys), journal=True, qpos=t.qpos, cols=cols, n_dev=nd)
        t.ctr.assign(n, True)
        r_cols = ref_batch(t.ref, t.ref_qpos, keys[:n_eff], True, t.qlog)[1]
        got = cols.tolist()
        _eq(got[:n_eff], r_cols, 'cols')
        assert all(v == -7 for v in got[n_eff:])
        assert t.lru.journal_len == n_eff
        t.undo(-1, probe=keys[:64])
        assert t.lru.state_dict() == before and t.lru.journal_len == 0
        t.lru.assign(t.tensor(keys), qpos=t.qpos, cols=cols, n_dev=nd)
        t.ctr.assign(n, False)
        _eq(cols.tolist()[:n_eff], ref_batch(t.ref, t.ref_qpos, keys[:n_eff], False)[1], 'cols')
        t.check(keys[:64])


def test_view_batch_sizes():
    cap = 7409
    prng = random.Random(5)
    t = Twin(cap)
    for _ in range(3):
        t.assign([prng.randrange(3 * cap) for _ in range(8192)], journal=False)
    for n in (1, NB + 1, MAX_KEYS + 1):
        probe = [prng.randrange(-10, 3 * cap) for _ in range(n)]
        probe[-1] = INT64_MAX
        t.check(probe)


# ------------------------------------------------------------------------------------------------------------------------
# key values
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cap', [64, 5000])
def test_extreme_key_values(cap):
    """INT64_MAX, INT64_MIN + 2, -1 and other negatives, keys that differ only in bit 63, keys that differ only in low bits."""
    prng = random.Random(cap + 17)
    pool = [INT64_MAX, INT64_MAX - 1, K.KEY_TOMB + 1, K.KEY_TOMB + 2, -1, -2, -3, 0, 1, 2, 3, -(1 << 62), 1 << 62, -(1 << 32), 1 << 32]
    for _ in range(200):
        k = prng.randrange(2, 1 << 63)
        pool += [k, k - (1 << 63)]                       # same low 63 bits, bit 63 differs
    for _ in range(150):
        k = prng.randrange(-(1 << 62), 1 << 62) & ~7
        pool += [k, k ^ 1, k ^ 2, k ^ 3, k ^ 4]
    t = Twin(cap)
    for step in range(8):
        keys = [prng.choice(pool) if prng.random() < 0.8 else -prng.randrange(1, 10 * cap) for _ in range(1500)]
        t.assign(keys, journal=True, probe=pool[:15])
        t.undo(prng.randrange(1, 1500), probe=pool[:15])
        t.undo(-1, probe=pool[:15])
        t.assign(keys[::-1], journal=False, probe=pool)


def test_reserved_keys():
    """INT64_MIN and INT64_MIN + 1 are the table's sentinels: view reports them absent; assign refuses the chunk that holds one
    (device flag 5: neither a hit nor a miss, cols -1 from that chunk on), the next host-synchronising call raises and names the
    flag, and clear() or restore() recovers."""
    from ffc_b200._capi import FFCError
    cap = 1000
    prng = random.Random(41)
    t = Twin(cap)
    # tombstones and empty cells in the table: the sentinels must match neither
    t.assign([prng.randrange(3 * cap) for _ in range(4000)], journal=False)
    probe = [K.KEY_EMPTY, K.KEY_TOMB, K.KEY_TOMB + 1, INT64_MAX] + list(t.ref.keys())[:50]
    t.check(probe)
    assert t.lru.view_batch(t.tensor([K.KEY_EMPTY, K.KEY_TOMB])).tolist() == [-1, -1]
    for bad in K.KEY_EMPTY, K.KEY_TOMB:
        with pytest.raises(ValueError):
            t.lru.get(bad)
    for i, (pos, n, journal, bad) in enumerate([(0, 10, False, K.KEY_EMPTY), (700, NB, True, K.KEY_TOMB),
                                                (2500, 3000, False, K.KEY_TOMB), (NB, 3000, True, K.KEY_EMPTY)]):
        sd = t.ref.state_dict()
        keys = [prng.randrange(3 * cap) for _ in range(n)]
        keys[pos] = bad
        cols = torch.full((n,), -7, dtype=torch.int32, device=t.dev)
        t.lru.assign(t.tensor(keys), journal=journal, cols=cols)
        got = cols.tolist()
        refused = pos // NB * NB
        assert all(v == -1 for v in got[refused:]), i
        assert all(v != -7 for v in got[:refused]), i
        for call in (lambda: t.lru.cur_idx, t.lru.state_dict, lambda: t.lru.journal_len):
            with pytest.raises(FFCError, match=r'flag 5 .*5=reserved key'):
                call()
        if i % 2 == 0:
            t.lru.clear()
            t.ref = RefLRU(cap)
            t.ctr = Counters(cap)
        else:
            t.lru.restore(sd)                         # over a flagged cache that is not empty
            t.ref = RefLRU(cap)
            t.ref.restore(sd)
            t.ctr = Counters(cap)
            t.ctr.ring, t.ctr.ht = len(sd), cap
        t.qlog = []
        t.check(probe)
        keys = [prng.randrange(3 * cap) for _ in range(2000)]
        t.assign(keys, journal=True, probe=probe)
        t.undo(-1, probe=probe)
        t.assign(keys, journal=False, probe=probe)
