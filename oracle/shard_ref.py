"""fp64 oracle of the column-sharded head (ffc_b200.dist.ShardedFFCHead): the dense HeadOracle with its LRU / queue positions
partitioned like the shards (SURVEY.md 8(e)).

Rank r of R owns the contiguous slot range [offs[r], offs[r] + Qls[r]) -- the first Q % R ranks one slot more -- and the identities
with key mod R == r; its LRU is the reference LRU(Qls[r]) fed the keys it owns in global batch order, and global slot = offs[r] +
local slot.  Loss and gradients are those of the dense head on the concatenated global batch.
"""
from .head_ref import HeadOracle
from .lru_ref import LRU


class ShardedOracle(HeadOracle):
    """HeadOracle whose LRU / queue positions are partitioned like ffc_b200.dist (SURVEY.md 8(e))."""

    def __init__(self, R, *a, **k):
        super().__init__(*a, **k)
        self.R = R
        base, rem = divmod(self.Q, R)
        self.Qls = [base + (1 if r < rem else 0) for r in range(R)]            # ffc_b200/dist.py: the first Q % R shards one slot longer
        self.offs = [r * base + min(r, rem) for r in range(R)]
        self.Ql = self.Qls[0]
        self.lrus = [LRU(ql) for ql in self.Qls]
        self.lru = self

    # the subset of the LRU surface HeadOracle uses, routed by identity
    def _route(self, key):
        r = key % self.R
        return r, self.lrus[r]

    def __contains__(self, key):
        return key in self._route(key)[1]

    def get(self, key):
        r, l = self._route(key)
        return self.offs[r] + l.get(key)

    def try_get(self, key):
        r, l = self._route(key)
        self._log.append(r)
        return self.offs[r] + l.try_get(key)

    def view(self, key):
        r, l = self._route(key)
        v = l.view(key)
        return v if v < 0 else self.offs[r] + v

    def rollback_steps(self, n):
        for r in reversed(self._log[-n:]):
            self.lrus[r].rollback_one_step()
        del self._log[-n:]

    def head_pass(self, *a, **k):
        if not hasattr(self, '_log'):
            self._log = []
        return super().head_pass(*a, **k)
