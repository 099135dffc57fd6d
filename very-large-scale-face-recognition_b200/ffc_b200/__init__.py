"""ffc_b200: B200-native FFC classification head (drop-in for the reference ffc.py / lru.py)."""
from ._capi import FFCError, lib  # noqa: F401
from .ffc import FFC, FFCHead, NormalizeNet, hard_neg_k  # noqa: F401
from .identify import Identification, cmc  # noqa: F401
from .lru import LRU  # noqa: F401
from .tail import FFCTail, NormalizeTail, fuse_tail, l2_normalize  # noqa: F401
