"""Full-size (BASELINE.json C3: queue 1,048,576 x D=512, 1024 rows) checks through size-independent properties:
the tcgen05 path against the fp64 check mode on the same state, rollback idempotence, gradient linearity, and the
LRU slot for slot against the oracle, with its defining property (the resident set is the most recently used `capacity` distinct keys)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

Q, D, B = 1 << 20, 512, 1024


def _rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-30))


def test_bf16_vs_check_mode_full_size():
    import ffc_b200
    dev = torch.device('cuda')
    torch.manual_seed(0)
    hb = ffc_b200.FFCHead(D, Q, 32.0, 'Arc', 0.5, precision='bf16', max_batch=B, device=dev)
    hc = ffc_b200.FFCHead(D, Q, 32.0, 'Arc', 0.5, precision='fp32', max_batch=B, device=dev)
    hc.queue.copy_(hb.queue)
    for h in (hb, hc):
        h._ensure()
        h.sync_mirror()
        # 3/4 of the slots resident, so the batch mixes hits, fresh inserts and (probe-side) outliers
        n0 = 3 * Q // 4
        h._lru.restore_arrays(torch.arange(n0, dtype=torch.int64), torch.arange(n0, dtype=torch.int32))
    gen = torch.Generator().manual_seed(1)
    for step in range(2):
        xl = torch.randint(0, Q + Q // 8, (B,), generator=gen)
        yl = torch.cat([xl[:B // 2], torch.randint(0, Q + Q // 8, (B - B // 2,), generator=gen)])
        x = F.normalize(torch.randn(B, D, generator=gen)).to(dev)
        y = F.normalize(torch.randn(B, D, generator=gen)).to(dev)
        out = []
        for h in (hb, hc):
            q_before = h.queue[:, :4096].clone()
            sd_before = h._lru.cur_idx
            l2, d2 = h._pass(x, y, xl, yl, False)
            # rollback pass is the identity on the head state (ffc.py:255-259)
            assert torch.equal(h.queue[:, :4096], q_before) and h._lru.cur_idx == sd_before and h._lru.journal_len == 0
            bk2 = (h.rows[:B].clone(), h.cols[:B].clone(), h.label[:B].clone())
            l1, d1 = h._pass(y, x, yl, xl, True)
            out.append((l1 + l2, d1, d2, bk2, (h.rows[:B].clone(), h.cols[:B].clone(), h.label[:B].clone())))
        (lb, d1b, d2b, rb_b, cm_b), (lc, d1c, d2c, rb_c, cm_c) = out
        for a, b in zip(rb_b + cm_b, rb_c + cm_c):
            assert torch.equal(a, b)                      # bookkeeping is precision independent and deterministic
        assert abs(float(lb) - float(lc)) <= 1e-2 * abs(float(lc)), (float(lb), float(lc))
        assert _rel(d1b, d1c) <= 1e-2 and _rel(d2b, d2c) <= 1e-2, (_rel(d1b, d1c), _rel(d2b, d2c))
        assert int((cm_b[2] < 0).sum()) > 0 and int((cm_b[2] >= 0).sum()) > 0     # both outliers and positives exercised
    # gradient linearity in the upstream gradient (GradScaler contract)
    p = F.normalize(torch.randn(B, D, generator=gen)).to(dev).requires_grad_(True)
    g = F.normalize(torch.randn(B, D, generator=gen)).to(dev)
    loss = hb.head(p, g, xl, yl, commit=False)
    (g1,) = torch.autograd.grad(loss * 1.0, p, retain_graph=True)
    (g2,) = torch.autograd.grad(loss * 65536.0, p)
    assert torch.allclose(g2, g1 * 65536.0, rtol=1e-6, atol=0)


def test_lru_full_size_property():
    """The 2^20-slot LRU against the oracle, slot for slot: cols and rows of every pass, qpos, view() of every key of the pass,
    and state_dict.  About 1.2 M accesses: random keys plus 1/16 keys homed in 48 crafted windows of the 2^17-window table, in
    committed passes and journaled ones that are undone.  Then the defining property on the committed stream: the resident set is
    the `capacity` most recently used distinct keys, every key maps to a unique slot.  The test also counts the home windows that
    held more than 32 live keys (a chain into the next window) at the end of some pass, and requires at least one."""
    import ffc_b200
    from oracle import lru_keys as K
    from oracle.lru_ref import LRU as RefLRU
    from oracle.lru_ref import ref_batch
    dev = torch.device('cuda')
    cap = 1 << 20
    nwin = K.table_windows(cap)
    lru = ffc_b200.LRU(cap, journal_capacity=1 << 17)
    ref = RefLRU(cap)
    qpos = torch.zeros(cap, dtype=torch.uint8, device=dev)
    ref_qpos = [0] * cap
    rng = np.random.default_rng(0)
    wins = rng.choice(nwin, size=48, replace=False)
    crafted = np.array([k for w in wins for k in K.keys_in_window(int(w), nwin, 80, rng)], dtype=np.int64)
    n_batches, bs = 12, 1024 * 96
    stream = []
    crowded = set()
    for b in range(n_batches):
        keys = rng.integers(0, 3 * cap, size=bs, dtype=np.int64)
        pick = rng.choice(bs, size=bs // 16, replace=False)
        keys[pick] = rng.choice(crafted, size=bs // 16)
        journal = b % 3 == 1
        kl = keys.tolist()
        kt = torch.from_numpy(keys).to(dev)
        rows = torch.empty(bs, dtype=torch.int32, device=dev)
        cols = lru.assign(kt, journal=journal, qpos=qpos, rows=rows)
        qlog = []
        r_rows, r_cols, _, _ = ref_batch(ref, ref_qpos, kl, journal, qlog)
        assert np.array_equal(cols.cpu().numpy(), np.array(r_cols)), b
        assert np.array_equal(rows.cpu().numpy(), np.array(r_rows)), b
        got = lru.view_batch(kt).cpu().numpy()
        assert np.array_equal(got, np.array([ref.view(k) for k in kl])), b
        crowded.update(np.flatnonzero(K.home_window_counts(ref.keys(), nwin) > 32).tolist())
        if journal:
            lru.undo(-1, qpos)
            ref.rollback_steps(len(qlog))
            for s, q in reversed(qlog):
                ref_qpos[s] = q
            assert lru.journal_len == 0
        else:
            stream.append(keys)
        if b in (4, n_batches - 1):
            assert lru.state_dict() == ref.state_dict(), b
            assert qpos.cpu().tolist() == ref_qpos, b
    print(f'home windows that held more than 32 live keys at the end of some pass: {len(crowded)}')
    assert len(crowded) > 0
    allk = np.concatenate(stream)
    # most recent occurrence index of every distinct key
    rev = allk[::-1]
    uniq, first_rev = np.unique(rev, return_index=True)
    order = np.argsort(first_rev)                   # most recently used first
    mru = uniq[order]
    expect_resident = mru[:cap]
    expect_absent = mru[cap:cap + 50000]
    v_res = lru.view_batch(torch.from_numpy(np.ascontiguousarray(expect_resident)).to(dev)).cpu().numpy()
    assert (v_res >= 0).all()
    assert len(np.unique(v_res)) == len(v_res) and v_res.max() < cap
    if len(expect_absent):
        v_abs = lru.view_batch(torch.from_numpy(np.ascontiguousarray(expect_absent)).to(dev)).cpu().numpy()
        assert (v_abs == -1).all()
    assert lru.cur_idx == min(cap, len(uniq))
    sd = lru.state_dict()
    assert [k for k, _ in sd[:2000]] == mru[:2000].tolist()      # recency order of state_dict (lru.py:102-108)
