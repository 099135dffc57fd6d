"""CPU restatement of the reference LRU id->slot cache.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this module; the product path
(``ffc_b200``) never does.

Follows /root/reference/lru.py:
  * ``get``                 lru.py:44-89   (hit -> move to front; miss -> next fresh
                                            slot while cur_idx < capacity, else evict
                                            the least-recently-used entry and reuse
                                            its slot)
  * ``try_get``             lru.py:157-204 (same as ``get`` plus an undo record)
  * ``rollback_one_step``   lru.py:210-248 (exact inverse of the newest undo record)
  * ``rollback_steps``      lru.py:252-255
  * ``view``/``__contains__`` lru.py:145-151 (never touch recency)
  * ``state_dict``/``restore``/``__iter__``/``keys``/``clear``  lru.py:94-153

Data layout differs from the reference on purpose (this is a restatement, not a
copy): recency is a doubly linked list threaded through two integer arrays that
are indexed by *slot*, with two sentinel indices, instead of heap-allocated node
objects.  A slot holds at most one key at any time, so slot ids can stand in
for nodes.  Parity is pinned by tests/test_oracle_lru.py against golden traces
generated from the reference itself (tests/golden/make_golden.py).
"""
from __future__ import annotations

_GET, _ADD, _OVERFLOW = 0, 1, 2


class LRU:
    def __init__(self, capacity: int):
        self.capacity = int(capacity)
        self.cur_idx = 0
        self._slot_of = {}                      # key -> slot
        n = self.capacity
        self._H, self._T = n, n + 1             # sentinel "slots": head (MRU side), tail (LRU side)
        self._prev = [-1] * (n + 2)
        self._next = [-1] * (n + 2)
        self._key = [None] * n
        self._next[self._H] = self._T
        self._prev[self._T] = self._H
        self.op_stack = []

    # -- list surgery ------------------------------------------------------------
    def _unlink(self, s):
        p, n = self._prev[s], self._next[s]
        self._next[p] = n
        self._prev[n] = p
        return p, n

    def _link_between(self, s, p, n):
        self._prev[s], self._next[s] = p, n
        self._next[p] = s
        self._prev[n] = s

    def _push_front(self, s):
        self._link_between(s, self._H, self._next[self._H])

    # -- lru.py:44-89 / 157-204 ---------------------------------------------------
    def _access(self, key, log):
        s = self._slot_of.get(key)
        if s is not None:                                   # hit
            p, n = self._unlink(s)
            if log:
                self.op_stack.append((_GET, p, n, None))
            self._push_front(s)
            return s
        if self.cur_idx < self.capacity:                    # fresh slot
            s = self.cur_idx
            self.cur_idx += 1
            self._slot_of[key] = s
            self._key[s] = key
            self._push_front(s)
            if log:
                self.op_stack.append((_ADD, s, None, None))
            return s
        s = self._prev[self._T]                             # evict LRU tail, reuse its slot
        p, n = self._unlink(s)
        old_key = self._key[s]
        del self._slot_of[old_key]
        if log:
            self.op_stack.append((_OVERFLOW, p, n, old_key))
        self._slot_of[key] = s
        self._key[s] = key
        self._push_front(s)
        return s

    def get(self, key):
        return self._access(key, False)

    def try_get(self, key):
        return self._access(key, True)

    # -- lru.py:210-255 -----------------------------------------------------------
    def rollback_one_step(self):
        if not self.op_stack:
            return
        kind, a, b, c = self.op_stack.pop()
        s = self._next[self._H]                             # the entry the undone op left at the front
        if kind == _GET:
            self._unlink(s)
            self._link_between(s, a, b)
        elif kind == _ADD:
            assert s == a
            self._unlink(s)
            del self._slot_of[self._key[s]]
            self._key[s] = None
            self.cur_idx -= 1
        else:
            self._unlink(s)
            del self._slot_of[self._key[s]]
            assert c not in self._slot_of
            self._key[s] = c
            self._slot_of[c] = s
            self._link_between(s, a, b)

    def rollback_steps(self, steps):
        for _ in range(min(steps, len(self.op_stack))):
            self.rollback_one_step()

    # -- lru.py:94-153 ------------------------------------------------------------
    def __iter__(self):
        s = self._next[self._H]
        while s != self._T:
            yield self._key[s], s
            s = self._next[s]

    def state_dict(self):
        return list(iter(self))

    def restore(self, kvs):
        assert len(kvs) <= self.capacity
        assert self.cur_idx == 0
        last = self._H
        for k, s in kvs:
            assert k not in self._slot_of
            self._slot_of[k] = s
            self._key[s] = k
            self._prev[s] = last
            self._next[last] = s
            last = s
            self.cur_idx += 1
        self._next[last] = self._T
        self._prev[self._T] = last

    def clear(self):
        # lru.py:132-141 -- note: like the reference, does NOT reset cur_idx.
        self._slot_of.clear()
        self._key = [None] * self.capacity
        self._next[self._H] = self._T
        self._prev[self._T] = self._H

    def __contains__(self, key):
        return key in self._slot_of

    def view(self, key):
        return self._slot_of.get(key, -1)

    def keys(self):
        return self._slot_of.keys()


def ref_batch(ref, qpos, keys, journal, qlog=None):
    """ffc.py:166-177 over the oracle LRU: returns rows, cols, hits, ones (set); updates qpos (a list) in place.
    With ``qlog`` (a list), appends (slot, qpos before) per access, so that undoing the last m accesses restores
    qpos by popping m entries."""
    rows, cols, hits, ones = [], [], [], set()
    for k in keys:
        known = k in ref
        s = ref.try_get(k) if journal else ref.get(k)
        if qlog is not None:
            qlog.append((s, qpos[s]))
        if known:
            rows.append(qpos[s]); ones.add(s); qpos[s] ^= 1
        else:
            rows.append(0); qpos[s] = 1
        cols.append(s); hits.append(1 if known else 0)
    return rows, cols, hits, ones
