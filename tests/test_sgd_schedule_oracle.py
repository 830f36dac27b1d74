"""CPU checks of oracle/sgd_schedule_ref.py, the one-warp restatement of the Hogwild epoch kernels that
tests/test_sgd_epoch_schedule_gpu.py compares the kernels with: its planner against the host's rules, its blocked
schedule against oracle/bpr_blk_ref.py and the serial loop, its APR arithmetic against oracle/apr_ref.py."""
import numpy as np
import pytest

from oracle import apr_ref, bpr_blk_ref, bpr_ref
from oracle import sgd_schedule_ref as sr


def rel_err(a, b):
    return float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64)) / (np.abs(b.astype(np.float64)) + 1e-3)))


def _triplets(m, n, max_per, seed):
    rng = np.random.default_rng(seed)
    per = 1 + rng.integers(0, max_per, m)
    u = np.repeat(np.arange(m, dtype=np.int32), per)
    i = rng.integers(0, n, len(u)).astype(np.int32)
    j = ((i + 1 + rng.integers(0, n - 1, len(u))) % n).astype(np.int32)
    return u, i, j


def _factors(m, n, d, seed, scale=0.1):
    rng = np.random.default_rng(seed)
    return (rng.random((m, d)) * scale).astype(np.float32), (rng.random((n, d)) * scale).astype(np.float32)


@pytest.mark.parametrize("item_segs,group_segs,max_items", [(32, 1, 1 << 30), (2, 1, 1 << 30), (3, 4, 1 << 30), (2, 1, 3)])
def test_planner_places_every_event_once_in_stream_order(item_segs, group_segs, max_items):
    rng = np.random.default_rng(item_segs * 10 + group_segs)
    deg = rng.integers(0, 260, 80)
    deg[[3, 40]] = [1100, 0]
    ev_indptr = np.concatenate([[0], np.cumsum(deg)])
    segs, items = sr.plan_epoch(ev_indptr, item_segs, group_segs=group_segs, max_items=max_items)
    # the segments of the items, in order, tile [0, T) in 1..32-event pieces of one user each
    order = [segs[s] for (a, b) in items for s in range(a, b)]
    assert [s for (a, b) in items for s in range(a, b)] == list(range(len(segs)))
    ends = [0] + [e for (_, _, e, _) in order]
    assert [b for (_, b, _, _) in order] == ends[:-1] and ends[-1] == ev_indptr[-1]
    for (u, b, e, shared) in order:
        assert 1 <= e - b <= 32 and ev_indptr[u] <= b < e <= ev_indptr[u + 1]
        assert (b - ev_indptr[u]) % 32 == 0
        assert shared == (-(-deg[u] // 32) > item_segs)
    for (a, b) in items:
        users = {segs[s][0] for s in range(a, b)}
        if segs[a][3]:                               # a heavy user's item: that user alone, the split size of the rule
            nsegs = -(-deg[segs[a][0]] // 32)
            per = max(item_segs, -(-nsegs // max_items))
            assert len(users) == 1 and (b - a == per or b == max(s for s in range(len(segs)) if segs[s][0] == segs[a][0]) + 1)
        else:                                        # light users grouped until group_segs segments
            assert all(not segs[s][3] for s in range(a, b))
            assert b - a - len([s for s in range(a, b) if segs[s][0] == segs[b - 1][0]]) < group_segs
    assert sr.default_item_segs(4000, sr.default_n_warps(4000)) == 32
    assert sr.default_item_segs(30000, 1) == 234 and sr.default_item_segs(5 * 10 ** 7, 1776) == 219
    assert sr.resync_mask(4) == 0 and sr.resync_mask(8) == 1 and sr.resync_mask(32) == 7


@pytest.mark.parametrize("d,n", [(64, 7), (20, 40), (128, 12)])
def test_blocked_epoch_equals_sgd_apply_blocked(d, n):
    """Explicit triplets, no heavy user: the epoch oracle is oracle/bpr_blk_ref.py bit for bit, except that P[u] is
    published as P0 + fl32(pu - P0) where bpr_blk_ref stores pu."""
    m = 60
    u, i, j = _triplets(m, n, 70, d + n)
    P, Q = _factors(m, n, d, d)
    Pa, Qa = P.copy(), Q.copy()
    la = bpr_blk_ref.sgd_apply_blocked(Pa, Qa, u, i, j, 0.05, 0.01, 0.02)
    Pb, Qb = P.copy(), Q.copy()
    lb = sr.blocked_epoch(Pb, Qb, sr.plan_triplets(u), i, j, 0.05, 0.01, 0.02)
    assert np.array_equal(Qa, Qb) and la == lb
    assert np.array_equal((P + (Pa - P).astype(np.float32)).astype(np.float32), Pb)


def test_lag0_is_the_serial_loop():
    m, n, d = 50, 30, 32
    u, i, j = _triplets(m, n, 60, 1)
    P, Q = _factors(m, n, d, 2)
    Pa, Qa = P.copy(), Q.copy()
    la = bpr_ref.sgd_epoch(Pa, Qa, u, i, j, 0.05, 0.01, 0.02)
    Pb, Qb = P.copy(), Q.copy()
    lb = sr.blocked_epoch(Pb, Qb, sr.plan_triplets(u), i, j, 0.05, 0.01, 0.02, lag=0)
    assert rel_err(Pb, Pa) < 1e-5 and rel_err(Qb, Qa) < 1e-5 and lb == pytest.approx(la, rel=1e-6)
    # ... and float64 at lag 0 is the float64 serial loop
    P64, Q64 = P.astype(np.float64), Q.astype(np.float64)
    lc = sr.blocked_epoch(P64, Q64, sr.plan_triplets(u), i, j, 0.05, 0.01, 0.02, lag=0)
    Pd, Qd = P.astype(np.float64), Q.astype(np.float64)
    ld = bpr_ref.sgd_epoch(Pd, Qd, u, i, j, 0.05, 0.01, 0.02, mode="float64")
    assert np.allclose(P64, Pd, rtol=1e-12, atol=1e-14) and np.allclose(Q64, Qd, rtol=1e-12, atol=1e-14)
    assert lc == pytest.approx(ld, rel=1e-12)


def test_apr_blocked_lag0_float64_is_apr_ref():
    m, n, d = 30, 25, 16
    u, i, j = _triplets(m, n, 40, 3)
    rng = np.random.default_rng(4)
    P, Q = rng.normal(0, 0.3, (m, d)), rng.normal(0, 0.3, (n, d))
    Pa, Qa = P.copy(), Q.copy()
    la = apr_ref.apr_epoch(Pa, Qa, u, i, j, 0.01, 0.002, 0.01, 0.5, 2.0)
    Pb, Qb = P.copy(), Q.copy()
    lb = sr.blocked_epoch(Pb, Qb, sr.plan_triplets(u), i, j, 0.01, 0.002, 0.01, apr=(0.5, 2.0), lag=0)
    assert np.allclose(Pb, Pa, rtol=1e-11, atol=1e-13) and np.allclose(Qb, Qa, rtol=1e-11, atol=1e-13)
    assert lb == pytest.approx(la, rel=1e-12)


def test_per_triplet_float64_matches_blocked_float64_when_rows_never_repeat():
    """Disjoint rows: no read schedule matters, and both kernels' arithmetic is the reference update."""
    m, d = 40, 24
    u, _, _ = _triplets(m, 2, 50, 5)
    T = len(u)
    i, j = np.arange(0, 2 * T, 2, dtype=np.int32), np.arange(1, 2 * T, 2, dtype=np.int32)
    P, Q = _factors(m, 2 * T, d, 6)
    P1, Q1 = P.astype(np.float64), Q.astype(np.float64)
    P2, Q2 = P1.copy(), Q1.copy()
    plan = sr.plan_triplets(u)
    l1 = sr.blocked_epoch(P1, Q1, plan, i, j, 0.05, 0.01, 0.02)
    l2 = sr.per_triplet_epoch(P2, Q2, plan, i, j, 0.05, 0.01, 0.02, pf=4)
    assert np.allclose(P1, P2, rtol=1e-12, atol=1e-14) and np.allclose(Q1, Q2, rtol=1e-12, atol=1e-14)
    assert l1 == pytest.approx(l2, rel=1e-12)
