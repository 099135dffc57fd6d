"""1:N identification on the B200 (csrc/identify_sm100.cu): parity with the fp64 oracle in both precisions, planted identities,
the gallery after training with evictions, padding / negative cosines, no side effects, determinism, emulated shards, full size."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import ffc_b200
from ffc_b200 import _capi
from ffc_b200.identify import LABEL_NONE, merge
from oracle import identify_ref

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)
NEAR = 8e-3          # bf16 operand rounding: candidates whose fp64 cosines lie this close to the row's k-th value may swap


def _head(D, Q, n_res, precision, seed=0):
    """FFCHead whose queue holds random unit rows and whose LRU has slots [0, n_res) resident (keys 10 * slot + 7, shuffled recency)"""
    g = torch.Generator().manual_seed(seed)
    m = ffc_b200.FFCHead(D, Q, precision=precision, max_batch=64).to(DEV)
    with torch.no_grad():
        m.queue.copy_(F.normalize(torch.randn(2, Q, D, generator=g), dim=2).to(DEV))
    slots = torch.randperm(n_res, generator=g).int()
    m.lru.restore_arrays(slots.long() * 10 + 7, slots)
    return m


def _check(res, x, state, q0, k, precision):
    """res against the fp64 oracle (on the GPU for speed: same definition as oracle/identify_ref.py)"""
    xn = F.normalize(x.double().to(DEV), dim=1)
    n = x.shape[0]
    res_slots, res_scores, res_labels = res.slots.cpu(), res.scores.cpu().double(), res.labels.cpu()
    key_of = dict((s, kk) for kk, s in state)
    n_res = len(state)
    if n_res == 0:
        assert (res_slots == -1).all() and (res_labels == LABEL_NONE).all() and torch.isneginf(res_scores).all()
        return
    W = q0[:n_res].double().to(DEV)
    cos = (xn @ W.t()).cpu()
    m = min(k, n_res)
    assert (res_slots[:, m:] == -1).all() and (res_labels[:, m:] == LABEL_NONE).all() and torch.isneginf(res_scores[:, m:]).all()
    got = res_slots[:, :m].long()
    assert ((got >= 0) & (got < n_res)).all()
    got_cos = torch.gather(cos, 1, got)
    assert (res_scores[:, :m] - got_cos).abs().max() <= 1e-5                     # rescored in fp32 (fp64 accumulation)
    assert res_labels[:, :m].tolist() == [[key_of[int(s)] for s in row] for row in got]
    # order: score descending, ties by slot
    d = res_scores[:, 1:m] - res_scores[:, :m - 1]
    assert (d <= 0).all() and ((d < 0) | (got[:, 1:] > got[:, :m - 1])).all()
    if precision == 'fp32':
        if n <= 1000 and n_res <= 4096:
            _, _, want, _, _ = identify_ref.identify(xn.cpu().numpy(), state, q0.double().cpu().numpy(), k, normalized=True)
            assert got.tolist() == want[:, :m].tolist()
        else:
            want_v, want_i = torch.topk(cos, m, dim=1)
            assert got.tolist() == want_i.tolist()
        return
    kth = torch.topk(cos, m, dim=1).values[:, -1:]
    for i in range(n):
        gs, ws = set(got[i].tolist()), set(torch.topk(cos[i], m).indices.tolist())
        for s in gs - ws:
            assert cos[i, s] >= kth[i, 0] - NEAR, (i, s)
        for s in ws - gs:
            assert cos[i, s] <= kth[i, 0] + NEAR, (i, s)


CASES = [(1, 4096, 1000, 1), (127, 4096, 1000, 5), (1000, 4096, 4096, 10), (4097, 65536, 40000, 5), (1000, 65536, 40000, 10)]


@pytest.mark.parametrize('precision', ['bf16', 'fp32'])
@pytest.mark.parametrize('D', [64, 128, 256, 512])
def test_parity_with_fp64_oracle(D, precision):
    for ci, (N, Q, n_res, k) in enumerate(CASES):
        m = _head(D, Q, n_res, precision, seed=ci)
        x = torch.randn(N, D, generator=torch.Generator().manual_seed(100 + ci))
        x[: N // 2] += 3.0 * m.queue[0, torch.randint(0, n_res, (N // 2,))].cpu()    # half of the rows near a prototype
        res = m.identify(x, k=k)
        assert res.scores.shape == (N, k) and res.scores.dtype == torch.float32 and res.labels.dtype == torch.int64 and res.slots.dtype == torch.int32
        _check(res, x, m.lru.state_dict(), m.queue[0], k, precision)


@pytest.mark.parametrize('precision', ['bf16', 'fp32'])
def test_planted_identities_rank1(precision):
    D, Q, n_res = 512, 8192, 5000
    m = _head(D, Q, n_res, precision)
    g = torch.Generator().manual_seed(3)
    slots = torch.randint(0, n_res, (2000,), generator=g)
    x = m.queue[0, slots].cpu() + 0.03 * torch.randn(2000, D, generator=g)
    res = m.identify(x.to(torch.bfloat16), k=5)           # bf16 input on the device path
    assert res.labels[:, 0].cpu().tolist() == (slots * 10 + 7).tolist()
    assert ffc_b200.cmc(res.labels, slots * 10 + 7, ranks=(1, 5))[1] == 1.0


def test_after_training_with_evictions():
    """C4 regime in miniature: identities = 10 x queue, Zipf labels; every answer is a resident identity at its slot"""
    D, Q, B = 128, 512, 64
    torch.manual_seed(0)
    m = ffc_b200.FFC('identity', D, queue_size=Q, loss_type='AM', max_batch=B).to(DEV)
    rng = np.random.default_rng(0)
    n_ids = 10 * Q
    seen = set()
    for _ in range(40):
        lab = torch.from_numpy((rng.zipf(1.2, size=B) - 1) % n_ids)
        seen.update(lab.tolist())
        x = F.normalize(torch.randn(B, D)).to(DEV)
        m(x, x.clone(), lab, lab).backward()
    state = dict((s, k) for k, s in m.lru.state_dict())
    cur = m.lru.cur_idx
    assert cur == Q and len(seen) > Q                       # full, with evictions
    res = m.identify(torch.randn(3000, D), k=10)
    slots, labels = res.slots.cpu(), res.labels.cpu()
    assert ((slots >= 0) & (slots < cur)).all()
    for s, l in zip(slots.flatten().tolist(), labels.flatten().tolist()):
        assert state[s] == l                                # resident at that slot: no evicted identity is returned


@pytest.mark.parametrize('precision', ['bf16', 'fp32'])
def test_padding_and_negative_cosines(precision):
    D, Q = 128, 1024
    m = _head(D, Q, 0, precision)
    r = m.identify(torch.randn(5, D), k=3)                  # empty LRU
    assert (r.slots == -1).all() and (r.labels == LABEL_NONE).all() and torch.isneginf(r.scores).all()
    m = _head(D, Q, 4, precision)
    r = m.identify(torch.randn(5, D), k=7)                  # fewer than k resident
    assert (r.slots[:, :4] >= 0).all() and (r.slots[:, 4:] == -1).all() and (r.labels[:, 4:] == LABEL_NONE).all()
    assert sorted(r.slots[0, :4].tolist()) == [0, 1, 2, 3]
    m = _head(D, Q, 900, precision)
    with torch.no_grad():
        m.queue[0].abs_()
        m.queue[0] /= m.queue[0].norm(dim=1, keepdim=True)
    x = -torch.rand(33, D) - 0.01                            # every cosine negative
    r = m.identify(x, k=10)
    assert (r.scores < 0).all()
    _check(r, x, m.lru.state_dict(), m.queue[0], 10, precision)
    z = m.identify(torch.randn(0, D), k=2)
    assert z.slots.shape == (0, 2)


def test_no_side_effects_and_prefetch():
    D, Q, B = 128, 1024, 32
    torch.manual_seed(1)

    def run(with_identify):
        torch.manual_seed(2)
        m = ffc_b200.FFC('identity', D, queue_size=Q, max_batch=B).to(DEV)
        g = torch.Generator().manual_seed(4)
        out = []
        for step in range(4):
            xl, yl = torch.randint(0, 3000, (B,), generator=g), torch.randint(0, 3000, (B,), generator=g)
            x, y = F.normalize(torch.randn(B, D, generator=g)).to(DEV), F.normalize(torch.randn(B, D, generator=g)).to(DEV)
            m.prefetch_labels(xl, yl)
            if with_identify:
                before = (m.queue.clone(), m.queue_bf16.clone(), m.lru.state_dict(), m.qpos.clone()) if step == 2 else None
                m.identify(torch.randn(50, D), k=5)
                if before is not None:
                    torch.cuda.synchronize()
                    assert torch.equal(before[0], m.queue) and torch.equal(before[1], m.queue_bf16)
                    assert before[2] == m.lru.state_dict() and torch.equal(before[3], m.qpos)
            loss, dx, dy = m.forward_pair(x, y, x, y, xl, yl)
            out.append((loss.cpu(), dx.cpu(), dy.cpu()))
        return out, m.prefetch_hits, m.lru.state_dict()

    a, hits_a, st_a = run(False)
    b, hits_b, st_b = run(True)
    assert hits_a == hits_b == 4 and st_a == st_b
    for (la, xa, ya), (lb, xb, yb) in zip(a, b):
        assert torch.equal(la, lb) and torch.equal(xa, xb) and torch.equal(ya, yb)


@pytest.mark.parametrize('precision', ['bf16', 'fp32'])
def test_deterministic_and_fixed_launch_count(precision):
    m = _head(256, 65536, 60000, precision)
    lib = _capi.lib()
    x = torch.randn(3000, 256).to(DEV)
    counts, results = [], []
    for n in (3000, 17, 3000):
        torch.cuda.synchronize()
        c0 = lib.ffc_launch_count()
        r = m.identify(x[:n], k=10)
        torch.cuda.synchronize()
        counts.append(lib.ffc_launch_count() - c0)
        results.append(r)
    assert counts == [3, 3, 3]                               # tail normalisation + search + merge, whatever N
    assert all(torch.equal(getattr(results[0], f), getattr(results[2], f)) for f in ('scores', 'labels', 'slots'))


@pytest.mark.parametrize('R', [2, 4])
def test_emulated_shards_equal_unsharded(R):
    """per-shard CudaShardBackend.identify_local + the (score, slot) merge == the one-GPU search over the union"""
    from ffc_b200.dist import CudaShardBackend
    D, Q, N, k = 512, 20000, 700, 10
    full = _head(D, Q, Q, 'bf16', seed=5)
    base, rem = divmod(Q, R)
    parts = []
    x = torch.randn(N, D, generator=torch.Generator().manual_seed(9))
    for r in range(R):
        ql, off = base + (1 if r < rem else 0), r * base + min(r, rem)
        be = CudaShardBackend(D, ql, Q, off, 64, 32.0, 'AM', 0.4, 10, 'bf16', DEV)
        be.set_queue(full.queue[:, off:off + ql])
        n_here = ql if r != R - 1 else ql - 123                  # last shard only partly resident
        be.lru.restore_arrays(torch.arange(n_here) * 10 + 7 + 10 * off, torch.arange(n_here).int())
        parts.append(be.identify_local(x.to(DEV), k))
    cat = lambda f: torch.cat([getattr(p, f) for p in parts], dim=1)
    got = merge(cat('scores'), cat('labels'), cat('slots'), k)
    # the union: global slot s resident unless it is among the last shard's unfilled 123
    state = [(10 * s + 7, s) for s in range(Q - 123)]
    _check(got, x, state, full.queue[0], k, 'bf16')


def test_full_size_1m():
    D, Q, N = 512, 1 << 20, 1024
    m = ffc_b200.FFCHead(D, Q, max_batch=64).to(DEV)
    m.lru.restore_arrays(torch.arange(Q) * 3, torch.arange(Q).int())
    x = torch.randn(N, D)
    res = m.identify(x, k=10)
    rows = torch.randperm(N, generator=torch.Generator().manual_seed(0))[:64]
    xs = F.normalize(x[rows].double().to(DEV), dim=1)
    cos = xs @ m.queue[0].double().t()
    kth = torch.topk(cos, 10, dim=1).values[:, -1]
    for j, i in enumerate(rows.tolist()):
        got = res.slots[i].long()
        assert (res.scores[i].double() - cos[j, got]).abs().max() <= 1e-5
        want = set(torch.topk(cos[j], 10).indices.tolist())
        for s in set(got.tolist()) ^ want:
            assert abs(float(cos[j, s]) - float(kth[j])) <= NEAR
