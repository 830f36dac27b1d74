"""The ranking path (K3 exact / K3-TC + K5, K6) where it can be wrong unnoticed on random tables: the tf32 bound at its worst
case, max|q| cached across writers of Q, masks that change the answer, widths above 128, N at every instantiation switch,
every ballot word of the metrics, and ranking while the hot rows are shared.  Reference: oracle/topn.py (ids and scores bit
for bit) and oracle/metrics.py."""
import numpy as np
import pytest

from oracle import metrics, record_ref, topn
from test_rank_edges_oracle import CASES, tf32_bound_case
from yue_b200 import synth
from yue_b200.engine import MODE_HOGWILD, MODE_SERIAL, RANK_AUTO, RANK_EXACT, RANK_TC, YueError

pytestmark = pytest.mark.gpu


def csr(rows):
    rows = [np.unique(np.asarray(r, np.int32)) for r in rows]
    return np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64), \
        (np.concatenate(rows) if rows else np.zeros(0, np.int32)).astype(np.int32)


def load(engine, P, Q, uq_indptr=None, uq_items=None):
    m, n = P.shape[0], Q.shape[0]
    if uq_indptr is None:
        uq_indptr, uq_items = np.zeros(m + 1, np.int64), np.zeros(0, np.int32)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), uq_indptr, uq_items)
    engine.set_factors(P, Q)
    return uq_indptr, uq_items


def check(engine, P, Q, users, N, uq_indptr, uq_items, algo):
    ids, sc = engine.rank_topn(users, N, algo)
    rid, rsc = topn.topn_exact(P, Q, users, N, uq_indptr, uq_items)
    assert np.array_equal(ids, rid), np.argwhere(ids != rid)[:5]
    assert np.array_equal(sc, rsc)
    return ids, sc


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def exact_split(B, N, n):
    """(catalog splits, tracks per split) of the exact kernel (yue_rank_exact_device)."""
    BU = 128 if N <= 32 else 64
    BI = 16384 // BU
    row_blocks, ntiles = -(-B // BU), -(-n // BI)
    sm = sm_count()
    splits = max(1, min(ntiles // 8, 2 * sm // row_blocks)) if row_blocks < sm else 1
    return splits, -(-ntiles // splits) * BI


# ---- A. the tf32 bound at its worst case ---------------------------------------------------------------------------------
@pytest.mark.parametrize("d,form,N", CASES)
def test_tc_tf32_bound_worst_case(engine, d, form, N):
    """Track A is the exact top-1 with the lowest tf32 score of the top group (tests/test_rank_edges_oracle.py proves it
    for the matching rounding).  The TC candidate pass itself must answer every row: no spill, no fallback."""
    case = tf32_bound_case(d, form, N)
    P, Q = case["P"], case["Q"]
    ind, uq = load(engine, P, Q)
    ids, _ = check(engine, P, Q, case["users"], N, ind, uq, RANK_TC)
    assert engine.rank_stats() == (0, 0)
    assert (ids[:, 0] == case["a_id"]).all()


# ---- B. max|q| is cached: every writer of Q must invalidate it -----------------------------------------------------------
# Writers of Q in yue_b200.cu that mark RankTcState::q_dirty: yue_set_factors, run_sgd (BPR / APR epochs and apply),
# yue_cune_epoch, the GCN steps and yue_gcn_finalize, yue_bpr_adam_steps / _apply, the WRMF track sweep, yue_q_delta_apply,
# yue_hot_pull and yue_q_exchange_finish.  A new writer belongs in this list and in the tests below.
def test_qmax_follows_set_factors_and_q_delta_apply(engine):
    import torch
    from yue_b200 import sharding
    from yue_b200._lib import BUF_Q_DELTA, BUF_Q_SNAPSHOT
    case = tf32_bound_case(64, "rn", 10)
    P, Q = case["P"], case["Q"]
    small = (Q * np.float32(1e-3)).astype(np.float32)
    ind, uq = load(engine, P, small)
    check(engine, P, small, case["users"], 10, ind, uq, RANK_TC)          # caches max|q| of the small table
    engine.set_factors(P, Q)
    check(engine, P, Q, case["users"], 10, ind, uq, RANK_TC)
    assert engine.rank_stats() == (0, 0)

    engine.set_factors(P, small)
    check(engine, P, small, case["users"], 10, ind, uq, RANK_TC)
    engine.q_snapshot()
    for which, val in ((BUF_Q_SNAPSHOT, np.zeros_like(Q)), (BUF_Q_DELTA, Q)):   # snapshot + delta = Q exactly
        ptr, nbytes = engine.device_buffer(which)
        t = torch.as_tensor(sharding._DevAlias(ptr, nbytes), device="cuda:0")
        t.copy_(torch.from_numpy(val.reshape(-1)))
        torch.cuda.synchronize()
    engine.q_delta_apply()
    assert np.array_equal(engine.get_factors()[1], Q)
    check(engine, P, Q, case["users"], 10, ind, uq, RANK_TC)
    assert engine.rank_stats() == (0, 0)


def _writer_log():
    log = synth.power_law_log(600, 3000, 30000, seed=21)
    rng = np.random.default_rng(21)
    P = rng.normal(size=(log.m, 64)).astype(np.float32)
    Q = (rng.normal(size=(log.n, 64)) * 1e-4).astype(np.float32)          # tiny: the cached max|q| is far too small after
    return log, P, Q


WRITERS = ["bpr_epoch", "apr_epoch", "bpr_apply", "apr_apply", "cune_epoch", "wrmf_tracks", "gcn_finalize", "bpr_adam"]


@pytest.mark.parametrize("writer", WRITERS)
def test_qmax_follows_every_trainer(engine, writer):
    log, P, Q = _writer_log()
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    users = np.arange(log.m, dtype=np.int32)
    engine.rank_topn(users, 10, RANK_TC)
    ev_user = record_ref.ev_users(log.ev_indptr)
    rng = np.random.default_rng(3)
    sel = rng.choice(len(log.ev_items), 4000, replace=False)
    u, i, j = ev_user[sel].astype(np.int32), log.ev_items[sel], rng.integers(0, log.n, 4000).astype(np.int32)
    if writer == "bpr_epoch":
        engine.bpr_epoch(0.05, 0.01, 0.01, 5, 0, MODE_HOGWILD)
    elif writer == "apr_epoch":
        engine.apr_epoch(0.05, 0.01, 0.01, 0.5, 1.0, 5, 0)
    elif writer == "bpr_apply":
        engine.bpr_apply(u, i, j, 0.05, 0.01, 0.01, MODE_SERIAL)
    elif writer == "apr_apply":
        engine.apr_apply(u, i, j, 0.05, 0.01, 0.01, 0.5, 1.0, MODE_SERIAL)
    elif writer == "cune_epoch":
        rows = []
        for x in range(log.m):
            played = log.uq_items[log.uq_indptr[x]:log.uq_indptr[x + 1]]
            rows.append(np.setdiff1d(rng.integers(0, log.n, 20), played))
        engine.cune_set_implicit(*csr(rows))
        engine.cune_epoch(0.05, 0.01, 0.01, 1.0, 5, 0, MODE_HOGWILD)
    elif writer == "wrmf_tracks":
        engine.wrmf_sweep(1, 0.1, 10.0)
    elif writer == "gcn_finalize":
        engine.gcn_set_events(ev_user, log.ev_items)
        engine.gcn_finalize(3)
    elif writer == "bpr_adam":
        engine.bpr_adam_steps(512, 100, 0.01, 0.01, 5, 0, 1)
    Pg, Qg = engine.get_factors()
    assert np.abs(Qg).max() > 10 * np.abs(Q).max()
    it, st = engine.rank_topn(users, 10, RANK_TC)
    ie, se = engine.rank_topn(users, 10, RANK_EXACT)
    assert np.array_equal(it, ie) and np.array_equal(st, se)
    rid, rsc = topn.topn_exact(Pg, Qg, users, 10, log.uq_indptr, log.uq_items)
    assert np.array_equal(it, rid) and np.array_equal(st, rsc)


# ---- C. masks that change the answer, short rows -------------------------------------------------------------------------
def _mask_table(n, d=64, seed=4):
    rng = np.random.default_rng(seed)
    P = rng.normal(size=(8, d)).astype(np.float32)
    Q = rng.normal(size=(n, d)).astype(np.float32)
    return P, Q, topn.scores_fma32(P, Q), rng


@pytest.mark.parametrize("algo", [RANK_EXACT, RANK_TC])
@pytest.mark.parametrize("N", [10, 32])
def test_masks_that_change_the_answer(engine, algo, N):
    n = 3000
    P, Q, S, rng = _mask_table(n)
    order = [np.lexsort((np.arange(n), -S[u].astype(np.float64))) for u in range(8)]
    rows = [order[u][:k] for u, k in enumerate((1, 31, 32, 33, 500))]       # exactly the k best tracks
    rows.append(np.setdiff1d(np.arange(n), rng.choice(n, N - 3, replace=False)))   # all but N - 3
    rows.append(np.arange(n))                                               # everything
    rows.append([])
    ind, uq = load(engine, P, Q, *csr(rows))
    users = np.array([0, 1, 2, 3, 4, 5, 6, 7, 3, 3, 0, 7, 6, 5], np.int32)     # repeated users in one batch
    ids, sc = check(engine, P, Q, users, N, ind, uq, algo)
    assert (ids[5, N - 3:] == -1).all() and (ids[5, :N - 3] >= 0).all() and np.isneginf(sc[5, N - 3:]).all()
    assert (ids[6] == -1).all() and np.isneginf(sc[6]).all()
    for b, u in enumerate(users[:5]):
        assert not np.isin(ids[b], rows[u]).any()
    if algo == RANK_TC:
        for u in range(8):                                                  # B = 1
            check(engine, P, Q, np.array([u], np.int32), N, ind, uq, algo)


@pytest.mark.parametrize("algo", [RANK_EXACT, RANK_TC, RANK_AUTO])
@pytest.mark.parametrize("n", [100, 20])
def test_catalog_smaller_than_a_tile_or_than_N(engine, algo, n):
    P, Q, S, rng = _mask_table(n, seed=n)
    top = np.argsort(-S[0].astype(np.float64), kind="stable")
    rows = [top[:5], np.arange(0, n, 3), [], np.arange(n)[:-2], [], [], [], []]
    ind, uq = load(engine, P, Q, *csr(rows))
    users = np.array([0, 1, 2, 3, 2, 0], np.int32)
    ids, sc = check(engine, P, Q, users, 32, ind, uq, algo)
    assert (ids < n).all() and (ids[3, 2:] == -1).all()
    if n == 20:
        assert (ids[2, 20:] == -1).all() and np.isneginf(sc[2, 20:]).all()
    if algo == RANK_TC:
        check(engine, P, Q, np.array([2], np.int32), 32, ind, uq, algo)
        assert engine.rank_stats() == (0, 0)


# ---- D. widths above 128 -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [129, 130, 200, 256])
@pytest.mark.parametrize("N", [10, 100])
@pytest.mark.parametrize("n", [5000, 900])
def test_widths_above_128(engine, d, N, n):
    m = 40
    indptr, uq = synth.mask_csr(m, n, 30, seed=d)
    rng = np.random.default_rng(d + N)
    P = rng.normal(size=(m, d)).astype(np.float32)
    Q = rng.normal(size=(n, d)).astype(np.float32)
    load(engine, P, Q, indptr, uq)
    users = np.concatenate([np.arange(m), [3, 3, 7]]).astype(np.int32)
    assert (exact_split(len(users), N, n)[0] > 1) == (n == 5000)
    for algo in (RANK_AUTO, RANK_EXACT):
        check(engine, P, Q, users, N, indptr, uq, algo)
    with pytest.raises(YueError):
        engine.rank_topn(users, min(N, 32), RANK_TC)
    for u in (0, m - 1):
        assert np.array_equal(engine.predict(u), topn.scores_fma32(P[u:u + 1], Q)[0])


# ---- E. N at every instantiation switch, tie runs across catalog splits --------------------------------------------------
def _tie_run_table(n, N, split, d=32, seed=6):
    m = 40
    rng = np.random.default_rng(seed + N)
    P = np.abs(rng.normal(size=(m, d))).astype(np.float32) + 0.1
    Q = (rng.random((n, d)) * 0.5).astype(np.float32)
    if split:
        splits, per = exact_split(m, N, n)
        assert splits > 1
        start = per - max(1, N // 2)                     # the first N of the run straddle the first split boundary
    else:
        start = n // 3
    Q[start:start + N + 40] = 1.0                        # identical rows: one exact-score tie run at the top of every row
    Q[start + N + 60] = 0.9                              # and a lone runner-up
    return P, Q, start


@pytest.mark.parametrize("split", [True, False])
@pytest.mark.parametrize("algo,N", [(RANK_EXACT, N) for N in (1, 32, 33, 64, 127, 128)] + [(RANK_TC, N) for N in (1, 12, 13, 32)])
def test_N_at_every_switch_with_a_tie_run(engine, algo, N, split):
    n = 70000 if split else 1500
    P, Q, start = _tie_run_table(n, N, split)
    ind, uq = load(engine, P, Q)
    users = np.concatenate([np.arange(40), [5, 5]]).astype(np.int32)
    ids, _ = check(engine, P, Q, users, N, ind, uq, algo)
    assert ids[0].tolist() == list(range(start, start + N))


# ---- F. K6 at every ballot word ------------------------------------------------------------------------------------------
def _metrics_oracle(origin, ids, cuts):
    """Sums over the rows of hits, recall, AP, NDCG, and the distinct count, per cut.  A row with an empty test set adds 0
    to every sum (the device's convention; evaluation/measure.py never sees such a user)."""
    out = []
    ne = [b for b, o in enumerate(origin) if len(o)]
    for n in cuts:
        rec = [[t for t in row[:n] if t >= 0] for row in ids.tolist()]
        o_ne, r_ne = [origin[b] for b in ne], [rec[b] for b in ne]
        h = metrics.hits(origin, rec)
        out.append(dict(hits=sum(h), precision=metrics.precision(h, n),
                        recall=metrics.recall(metrics.hits(o_ne, r_ne), o_ne) * len(ne),
                        map=metrics.mean_ap(o_ne, r_ne, n) * len(ne), ndcg=metrics.ndcg(o_ne, r_ne, n) * len(ne),
                        distinct=len(set(t for r in rec for t in r))))
    return out


def _compare_metrics(engine, origin, ids, cuts):
    sums, distinct = engine.rank_metrics(cuts)
    ref = _metrics_oracle(origin, ids, cuts)
    B = len(ids)
    for k, n in enumerate(cuts):
        assert sums[k, 0] == ref[k]["hits"] and distinct[k] == ref[k]["distinct"], (n, sums[k], distinct[k], ref[k])
        assert sums[k, 0] / (B * n) == pytest.approx(ref[k]["precision"], rel=1e-13)
        for c, key in ((1, "recall"), (2, "map"), (3, "ndcg")):
            assert sums[k, c] == pytest.approx(ref[k][key], rel=1e-12, abs=1e-12), (n, key)
    return ref


def test_metrics_at_every_word(engine):
    m, n, d, N = 300, 1_000_003, 16, 128
    rng = np.random.default_rng(17)
    P = np.abs(rng.normal(size=(m, d))).astype(np.float32)
    Q = (rng.random((n, d)) * 0.1).astype(np.float32)
    Q[n - 40:] = (rng.random((40, d)) + 1.0).astype(np.float32)             # the best tracks sit in the bitmap's last words
    load(engine, P, Q)
    users = np.concatenate([np.arange(m), [0, 0, 17, 299]]).astype(np.int32)   # repeated users
    ids, _ = engine.rank_topn(users, N, RANK_EXACT)
    assert (ids >= 0).all()
    edges = [0, 30, 31, 32, 33, 63, 64, 65, 95, 96, 97, 126, 127]
    rows = []
    for u in range(m):
        mine = ids[u]
        pick = mine[rng.choice(edges, rng.integers(1, len(edges)), replace=False)]
        extra = rng.integers(0, n, 200 if u % 7 == 0 else rng.integers(0, 10))   # rows longer than 128 too
        rows.append(np.union1d(pick, extra))
    rows[1] = []                                                            # an empty test row
    rows[2] = [int(ids[2][127])]                                            # one hit, at the last rank
    t_ind, t_items = csr(rows)
    engine.set_test_set(t_ind, t_items)
    origin = [t_items[t_ind[u]:t_ind[u + 1]].tolist() for u in users]
    cuts = [1, 31, 32, 33, 64, 65, 97, 128]
    ref = _compare_metrics(engine, origin, ids, cuts)
    assert ref[-1]["hits"] > ref[-2]["hits"] > ref[-3]["hits"] > 0           # the fourth word decides something


def test_metrics_of_tc_lists_with_fallback_rows(engine):
    """The tie flood of test_rank_gpu: some rows of the TC call are written by the exact-kernel fallback's scatter."""
    m, n, d, N = 140, 6000, 64, 10
    rng = np.random.default_rng(9)
    P = np.abs(rng.normal(size=(m, d))).astype(np.float32)
    Q = np.tile(np.abs(rng.normal(size=(1, d))).astype(np.float32), (n, 1))
    Q[::7] *= 0.5
    ind, uq = load(engine, P, Q)
    users = np.concatenate([np.arange(m), [4, 4]]).astype(np.int32)
    ids, _ = check(engine, P, Q, users, N, ind, uq, RANK_TC)
    assert engine.rank_stats()[0] > 0
    rows = [rng.integers(0, 14, rng.integers(0, 6)) for _ in range(m)]
    t_ind, t_items = csr(rows)
    engine.set_test_set(t_ind, t_items)
    origin = [t_items[t_ind[u]:t_ind[u + 1]].tolist() for u in users]
    ref = _compare_metrics(engine, origin, ids, [1, 5, 10])
    assert ref[-1]["hits"] > 0


# ---- G. ranking while the hot rows are shared ----------------------------------------------------------------------------
def test_ranking_while_hot_rows_are_shared():
    """After a shared epoch Q's hot rows are stale until hot_pull: rank_topn, predict and get_factors refuse until then,
    and after it they see the trained rows (SharedHotTrainer.finalize is what the class API calls)."""
    from yue_b200 import sharding
    from yue_b200.engine import Engine
    d = 64
    rng = np.random.default_rng(d)
    ev, uq = [], []
    for k in [900] * 22 + [30] * 40:                                        # track 0 above the trainer's hot threshold
        items = np.where(rng.random(k) < 0.85, 0, rng.integers(1, 40, k)).astype(np.int32)
        ev.append(items)
        uq.append(np.unique(items))
    ev_items = np.concatenate(ev).astype(np.int32)
    ev_ind = np.concatenate([[0], np.cumsum([len(r) for r in ev])]).astype(np.int64)
    uq_ind, uq_items = csr(uq)
    m, n = len(ev), 60
    P, Q = synth.init_factors(m, n, d, seed=d)
    eng = Engine(0)
    try:
        eng.set_interactions(m, n, ev_ind, ev_items, uq_ind, uq_items)
        eng.set_factors(P, Q)
        ctl = sharding.ThreadCtl(sharding.ThreadCtl.Shared(1), 0)
        tr = sharding.SharedHotTrainer(eng, ctl, np.bincount(ev_items, minlength=n), sub_epochs=2)
        assert len(tr.hot_tracks) > 0
        users = np.arange(m, dtype=np.int32)
        eng.rank_topn(users, 10, RANK_EXACT)                                 # before any shared epoch Q is current
        tr.epoch(0.05, 0.01, 0.01, 5, 0)
        early = []
        for call in (lambda: eng.rank_topn(users, 10, RANK_EXACT), lambda: eng.rank_topn(users, 10, RANK_TC),
                     lambda: eng.predict(0), lambda: eng.get_factors()):
            try:
                early.append(call())
            except YueError:
                early.append(None)
        tr.finalize()
        Pg, Qg = eng.get_factors()
        ids, sc = eng.rank_topn(users, 10, RANK_EXACT)
        rid, rsc = topn.topn_exact(Pg, Qg, users, 10, uq_ind, uq_items)
        assert np.array_equal(ids, rid) and np.array_equal(sc, rsc)
        late = [(ids, sc), eng.rank_topn(users, 10, RANK_TC), eng.predict(0), (Pg, Qg)]
        assert np.array_equal(late[2], topn.scores_fma32(Pg[:1], Qg)[0])
        for a, b in zip(early, late):                                       # refused, or what they return after the pull
            if a is not None:
                assert all(np.array_equal(x, y) for x, y in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)))
        tr.epoch(0.05, 0.01, 0.01, 5, 1, finalize=True)                     # the class API's order keeps working
        eng.rank_topn(users, 10, RANK_AUTO)
        eng.frob2()
        tr.close()
        eng.rank_topn(users, 10, RANK_AUTO)
    finally:
        eng.close()
