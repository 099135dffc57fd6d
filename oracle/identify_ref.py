"""fp64 numpy oracle of 1:N identification (ffc_identify / FFCHead.identify).

Gallery: row queue[0][s] of every resident slot, i.e. the slots of the LRU state ([(key, slot)] pairs, as LRU.state_dict()
returns them); [0, cur_idx) is exactly that set.  Score: cosine of the L2-normalised query with the stored prototype (fp64).
Result per row: k entries ordered by score descending, ties by smaller global slot (= col_offset + slot); missing entries
(fewer than k resident) are slot -1, label INT64_MIN, score -inf.
"""
import numpy as np

LABEL_NONE = np.iinfo(np.int64).min


def normalize(x):
    x = np.asarray(x, dtype=np.float64)
    return x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-12)


def gallery(lru_state, queue0, col_offset=0):
    """(prototypes [G, D] fp64, labels [G] int64, global slots [G] int64) of the resident slots, in slot order"""
    pairs = sorted((int(s), int(k)) for k, s in lru_state)
    slots = np.array([s for s, _ in pairs], dtype=np.int64)
    labels = np.array([k for _, k in pairs], dtype=np.int64)
    W = np.asarray(queue0, dtype=np.float64)[slots] if len(slots) else np.zeros((0, np.asarray(queue0).shape[1]))
    return W, labels, slots + col_offset


def identify(x, lru_state, queue0, k, col_offset=0, normalized=False):
    """-> (scores [N, k] fp64, labels [N, k] int64, slots [N, k] int64, cos [N, G] fp64, gallery slots [G])"""
    xn = np.asarray(x, dtype=np.float64) if normalized else normalize(x)
    W, labels, gslots = gallery(lru_state, queue0, col_offset)
    n = xn.shape[0]
    cos = xn @ W.T
    scores = np.full((n, k), -np.inf)
    lab = np.full((n, k), LABEL_NONE, dtype=np.int64)
    slo = np.full((n, k), -1, dtype=np.int64)
    m = min(k, W.shape[0])
    if m:
        order = np.lexsort((np.broadcast_to(gslots, cos.shape), -cos), axis=1)[:, :m]     # score desc, then slot asc
        scores[:, :m] = np.take_along_axis(cos, order, 1)
        lab[:, :m] = labels[order]
        slo[:, :m] = gslots[order]
    return scores, lab, slo, cos, gslots


def union_state(states_offsets):
    """LRU states of several shards -> one state over global slots (for the sharded search)"""
    return [(k, s + off) for st, off in states_offsets for k, s in st]
