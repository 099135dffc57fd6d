"""Keys with a chosen hash, for the device LRU's tables.  TEST INFRASTRUCTURE ONLY.

The device LRU (csrc/lru.cu) places key k by ``mix64(k)``, murmur3's fmix64 (csrc/ffc_common.cuh):
  * the global table: T cells in 32-cell windows, home window ``mix64(k) & (T/32 - 1)``, linear probing over windows;
  * the resolve CTA's shared-memory dedupe hash: LHSZ cells, home cell ``mix64(k) & (LHSZ - 1)``, linear probing.
fmix64 is a bijection of the 64-bit integers, so inverting it builds keys for any home window or cell: random keys
almost never share one, and the probing past a full window or cell never runs without such keys.
"""
from __future__ import annotations

import numpy as np

M64 = (1 << 64) - 1
C1, C2 = 0xff51afd7ed558ccd, 0xc4ceb9fe1a85ec53
C1_INV, C2_INV = pow(C1, -1, 1 << 64), pow(C2, -1, 1 << 64)
KEY_EMPTY, KEY_TOMB = -(1 << 63), -(1 << 63) + 1     # reserved: hash-table sentinels
LHSZ = 4096                                          # cells of the resolve CTA's local hash (lru.cu)
WINDOW = 32                                          # cells per window of the global table


def mix64(x: int) -> int:
    """fmix64 of the key's two's-complement bits (uint64 in, uint64 out)."""
    x &= M64
    x ^= x >> 33
    x = (x * C1) & M64
    x ^= x >> 33
    x = (x * C2) & M64
    x ^= x >> 33
    return x


def unmix64(h: int) -> int:
    """Inverse of mix64: x ^= x >> 33 is its own inverse on 64 bits, and the multiplications are undone by the
    constants' inverses mod 2^64."""
    h &= M64
    h ^= h >> 33
    h = (h * C2_INV) & M64
    h ^= h >> 33
    h = (h * C1_INV) & M64
    h ^= h >> 33
    return h


def mix64_np(keys: np.ndarray) -> np.ndarray:
    """mix64 over an int64 array (uint64 arithmetic wraps mod 2^64)."""
    x = keys.astype(np.int64).view(np.uint64).copy()
    x ^= x >> np.uint64(33)
    x *= np.uint64(C1)
    x ^= x >> np.uint64(33)
    x *= np.uint64(C2)
    x ^= x >> np.uint64(33)
    return x


def to_signed(u: int) -> int:
    return u - (1 << 64) if u >= (1 << 63) else u


def next_pow2(v: int) -> int:
    p = 1
    while p < v:
        p <<= 1
    return p


def table_cells(capacity: int) -> int:
    """T of ffc_lru_create: 4x the capacity rounded up to a power of two, never less than 2^18."""
    return max(next_pow2(4 * capacity), 1 << 18)


def table_windows(capacity: int) -> int:
    return table_cells(capacity) // WINDOW


def keys_with_low_hash(low: int, bits: int, n: int, rng: np.random.Generator) -> list:
    """n distinct keys k (never a reserved value) with mix64(k) & (2^bits - 1) == low."""
    assert 0 <= low < (1 << bits)
    out, seen = [], set()
    while len(out) < n:
        hi = int(rng.integers(0, 1 << (64 - bits), dtype=np.uint64))
        k = to_signed(unmix64((hi << bits) | low))
        if k in (KEY_EMPTY, KEY_TOMB) or k in seen:
            continue
        seen.add(k)
        out.append(k)
    return out


def keys_in_window(w: int, nwin: int, n: int, rng: np.random.Generator) -> list:
    """n distinct keys whose home window in a table of nwin windows is w."""
    assert nwin & (nwin - 1) == 0
    return keys_with_low_hash(w, nwin.bit_length() - 1, n, rng)


def keys_in_local_cell(c: int, n: int, rng: np.random.Generator) -> list:
    """n distinct keys whose home cell in the resolve CTA's local hash is c."""
    return keys_with_low_hash(c, LHSZ.bit_length() - 1, n, rng)


def home_window_counts(keys, nwin: int) -> np.ndarray:
    """Number of the given keys whose home window is w, for every w."""
    k = np.asarray(list(keys), dtype=np.int64)
    w = (mix64_np(k) & np.uint64(nwin - 1)).astype(np.int64)
    return np.bincount(w, minlength=nwin)
