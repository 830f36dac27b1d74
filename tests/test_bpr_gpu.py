"""GPU parity of the sampler (K1) and the triplet update (K2) against the oracle and the golden
vectors of the reference's own loop.  Everything goes through the C ABI (yue_b200.engine)."""
import os

import numpy as np
import pytest

from oracle import bpr_ref, philox, record_ref
from yue_b200 import synth
from yue_b200.engine import MODE_HOGWILD, MODE_HOGWILD_STORE, MODE_SERIAL, YueError

pytestmark = pytest.mark.gpu
REL = 1e-5          # north_star: factor updates match the reference loop to 1e-5 relative


def rel_err(a, b):
    return float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64)) / (np.abs(b.astype(np.float64)) + 1e-3)))


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "sgd_small.npz"))


def load_golden(engine, g):
    m, n = g["P0"].shape[0], g["Q0"].shape[0]
    engine.set_interactions(m, n, g["ev_indptr"], g["ev_items"], g["uq_indptr"], g["uq_items"])
    engine.set_factors(g["P0"], g["Q0"])
    return m, n


def test_sampler_bit_exact_vs_golden_stream(engine, golden):
    g = golden
    load_golden(engine, g)
    for ep in range(g["neg"].shape[0]):
        j = engine.sample_negatives(int(g["seed"]), ep)
        assert np.array_equal(j, g["neg"][ep])


def test_sampler_bit_exact_power_law_and_shard(engine):
    log = synth.power_law_log(3000, 800, 120000, seed=11)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    ev_user = record_ref.ev_users(log.ev_indptr)
    for seed, ep, slot in [(1, 0, 0), (2**40 + 5, 7, 2)]:
        ref = philox.sample_negatives(seed, ep, ev_user, log.n, log.uq_indptr, log.uq_items, slot=slot)
        assert np.array_equal(engine.sample_negatives(seed, ep, slot), ref)
    # a user shard with a global event offset draws the same negatives
    u0, u1 = 1000, 2200
    e0, e1 = int(log.ev_indptr[u0]), int(log.ev_indptr[u1])
    q0, q1 = int(log.uq_indptr[u0]), int(log.uq_indptr[u1])
    engine.set_interactions(u1 - u0, log.n, log.ev_indptr[u0:u1 + 1] - e0, log.ev_items[e0:e1],
                            log.uq_indptr[u0:u1 + 1] - q0, log.uq_items[q0:q1], user_begin=u0, event_base=e0)
    ref = philox.sample_negatives(1, 0, ev_user, log.n, log.uq_indptr, log.uq_items)
    assert np.array_equal(engine.sample_negatives(1, 0), ref[e0:e1])


def test_serial_epochs_match_reference_loop(engine, golden):
    """3 epochs incl. the lr schedule: GPU serial-order mode vs the reference's own loop output."""
    g = golden
    load_golden(engine, g)
    sched = bpr_ref.LearningRate(float(g["lr_init"]), float(g["max_lr"]))
    regU, regI = float(g["regU"]), float(g["regI"])
    for ep in range(3):
        assert sched.lRate == pytest.approx(float(g["lr_used"][ep]), rel=1e-12)
        loss = engine.bpr_epoch(sched.lRate, regU, regI, int(g["seed"]), ep, MODE_SERIAL)
        p2, q2 = engine.frob2()
        loss += regU * p2 + regI * q2
        P, Q = engine.get_factors()
        assert rel_err(P, g["P"][ep]) < REL and rel_err(Q, g["Q"][ep]) < REL
        assert loss == pytest.approx(float(g["loss"][ep]), rel=2e-6)
        sched.is_converged(ep + 1, loss)
    assert sched.lRate == pytest.approx(float(g["lr_final"]), rel=1e-12)


@pytest.mark.parametrize("d", [10, 64, 128, 200])
def test_apply_given_triplets_serial(engine, d):
    """Same triplet stream, conflict-free serial order, every supported row width."""
    rng = np.random.default_rng(d)
    m, n, T = 50, 90, 3000
    log = synth.power_law_log(m, n, 2000, seed=5)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    P, Q = synth.init_factors(m, n, d, seed=d)
    engine.set_factors(P, Q)
    u = np.sort(rng.integers(0, m, T)).astype(np.int32)
    i = rng.integers(0, n, T).astype(np.int32)
    j = ((i + 1 + rng.integers(0, n - 1, T)) % n).astype(np.int32)
    loss = engine.bpr_apply(u, i, j, 0.05, 0.01, 0.02, MODE_SERIAL)
    Pr, Qr = P.copy(), Q.copy()
    ref_loss = bpr_ref.sgd_epoch(Pr, Qr, u, i, j, 0.05, 0.01, 0.02)
    Pg, Qg = engine.get_factors()
    assert rel_err(Pg, Pr) < REL and rel_err(Qg, Qr) < REL
    assert loss == pytest.approx(ref_loss, rel=1e-6)


def test_hogwild_equals_serial_when_conflict_free(engine):
    """Disjoint users AND disjoint items per triplet run: the throughput kernels must then give the
    serial result (up to fp32 rounding of fma vs mul+add), whatever the scheduling."""
    m, n, d = 4000, 8200, 64
    log = synth.power_law_log(m, n, 9000, seed=3)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    P, Q = synth.init_factors(m, n, d, seed=1)
    u = np.arange(m, dtype=np.int32)
    i = (2 * np.arange(m)).astype(np.int32)
    j = (2 * np.arange(m) + 1).astype(np.int32)
    Pr, Qr = P.copy(), Q.copy()
    ref_loss = bpr_ref.sgd_epoch(Pr, Qr, u, i, j, 0.05, 0.01, 0.02)
    for mode in (MODE_HOGWILD, MODE_HOGWILD_STORE):
        engine.set_factors(P, Q)
        loss = engine.bpr_apply(u, i, j, 0.05, 0.01, 0.02, mode)
        Pg, Qg = engine.get_factors()
        assert rel_err(Pg, Pr) < REL and rel_err(Qg, Qr) < REL
        assert loss == pytest.approx(ref_loss, rel=1e-5)


def test_hogwild_epoch_statistical_parity(engine):
    """A real epoch with conflicts: loss and factors stay close to the serial oracle."""
    log = synth.power_law_log(2000, 3000, 60000, seed=21)
    d = 64
    P, Q = synth.init_factors(log.m, log.n, d, seed=2)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    ls = engine.bpr_epoch(0.05, 0.01, 0.01, 77, 0, MODE_SERIAL)
    Ps, Qs = engine.get_factors()
    engine.set_factors(P, Q)
    lh = engine.bpr_epoch(0.05, 0.01, 0.01, 77, 0, MODE_HOGWILD)
    Ph, Qh = engine.get_factors()
    # the first-epoch loss is measured while learning: fewer sequential steps -> slightly higher
    assert lh == pytest.approx(ls, rel=0.10)
    # movement away from the initial point correlates strongly with the serial movement
    ds, dh = (Qs - Q).ravel(), (Qh - Q).ravel()
    assert np.dot(ds, dh) / (np.linalg.norm(ds) * np.linalg.norm(dh)) > 0.9
    assert np.isfinite(Ph).all() and np.isfinite(Qh).all()


def test_epoch_linearity_of_event_count(engine):
    """Size-independent property at a larger size: loss at lr=0 is the sum over events of
    softplus(-(x_ui - x_uj)) and factors do not move."""
    log = synth.power_law_log(20000, 5000, 400000, seed=8)
    P, Q = synth.init_factors(log.m, log.n, 64, seed=4)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    loss = engine.bpr_epoch(0.0, 0.0, 0.0, 5, 0, MODE_HOGWILD)
    Pg, Qg = engine.get_factors()
    assert np.array_equal(Pg, P) and np.array_equal(Qg, Q)
    neg = engine.sample_negatives(5, 0)
    ev_user = record_ref.ev_users(log.ev_indptr)
    x = np.einsum("ij,ij->i", P[ev_user].astype(np.float64), (Q[log.ev_items] - Q[neg]).astype(np.float64))
    assert loss == pytest.approx(float(np.logaddexp(0.0, -x).sum()), rel=1e-5)
    assert not (neg == log.ev_items).any()


def test_edge_cases(engine):
    # empty log
    engine.set_interactions(3, 5, np.zeros(4, np.int64), np.zeros(0, np.int32), np.zeros(4, np.int64), np.zeros(0, np.int32))
    P, Q = synth.init_factors(3, 5, 10, seed=1)
    engine.set_factors(P, Q)
    assert engine.bpr_epoch(0.02, 0.01, 0.01, 1, 0, MODE_HOGWILD) == 0.0
    assert np.array_equal(engine.get_factors()[0], P)
    # ragged: users without events, a user with exactly 32 and 33 events (segment boundary)
    ev_indptr = np.array([0, 0, 32, 32, 65, 66], dtype=np.int64)
    rng = np.random.default_rng(0)
    ev_items = rng.integers(0, 40, 66).astype(np.int32)
    uq_rows = [np.unique(ev_items[ev_indptr[u]:ev_indptr[u + 1]]) for u in range(5)]
    uq_indptr = np.concatenate([[0], np.cumsum([len(r) for r in uq_rows])]).astype(np.int64)
    uq_items = np.concatenate(uq_rows).astype(np.int32)
    engine.set_interactions(5, 40, ev_indptr, ev_items, uq_indptr, uq_items)
    P, Q = synth.init_factors(5, 40, 10, seed=2)
    engine.set_factors(P, Q)
    loss = engine.bpr_epoch(0.02, 0.01, 0.01, 9, 0, MODE_SERIAL)
    ev_user = record_ref.ev_users(ev_indptr)
    neg = philox.sample_negatives(9, 0, ev_user, 40, uq_indptr, uq_items)
    Pr, Qr = P.copy(), Q.copy()
    ref = bpr_ref.sgd_epoch(Pr, Qr, ev_user, ev_items, neg, 0.02, 0.01, 0.01)
    Pg, Qg = engine.get_factors()
    assert rel_err(Pg, Pr) < REL and rel_err(Qg, Qr) < REL and loss == pytest.approx(ref, rel=1e-6)
    # a user who played the whole catalog has no negative: refused up front
    with pytest.raises(YueError):
        engine.set_interactions(1, 3, np.array([0, 3]), np.array([0, 1, 2], np.int32), np.array([0, 3]), np.array([0, 1, 2], np.int32))
    # NaN factors -> numeric error, like the reference's NaN guard (IterativeRecommender.py:63-66)
    engine.set_interactions(5, 40, ev_indptr, ev_items, uq_indptr, uq_items)
    Pn = P.copy(); Pn[1, 0] = np.nan
    engine.set_factors(Pn, Q)
    with pytest.raises(YueError) as ei:
        engine.bpr_epoch(0.02, 0.01, 0.01, 9, 0, MODE_SERIAL)
    assert ei.value.code == 4


def _train_and_eval(eng, log, P, Q, mode, epochs, lr, seed):
    from oracle import metrics
    from yue_b200.engine import RANK_EXACT
    eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    eng.set_factors(P, Q)
    for ep in range(epochs):
        eng.bpr_epoch(lr, 0.01, 0.01, seed, ep, mode)
    users = log.test_users()
    ids, _ = eng.rank_topn(users, 10, RANK_EXACT)
    origin = [log.test_items[log.test_indptr[u]:log.test_indptr[u + 1]].tolist() for u in users]
    rec = ids.tolist()
    h = metrics.hits(origin, rec)
    return metrics.recall(h, origin), metrics.ndcg(origin, rec, 10)


def test_quality_gate_hogwild_vs_serial(monkeypatch):
    """north_star: end-to-end Recall@10 and NDCG@10 within 0.5% absolute of the reference order on
    the same synthetic log.  The serial-order mode (proven equal to the reference loop above) is
    the reference trainer; the throughput mode runs with the engine's default schedule (>= 16 K
    events per warp, like config C2 on a full B200) and the shared-memory hot-row path forced on.
    tools/quality_study.py repeats this at 5 M events and at the full C2 size
    (profiles/quality_study_r1.md)."""
    from yue_b200.engine import Engine
    monkeypatch.setenv("YUE_SGD_HOT_MIN_COUNT", "4096")
    eng = Engine(0)
    try:
        log = synth.power_law_log(40000, 8000, 2500000, seed=33)
        P, Q = synth.init_factors(log.m, log.n, 32, seed=5)
        rs, ns = _train_and_eval(eng, log, P, Q, MODE_SERIAL, 8, 0.02, 99)
        rh, nh = _train_and_eval(eng, log, P, Q, MODE_HOGWILD, 8, 0.02, 99)
    finally:
        eng.close()
    print("\nrecall@10 serial %.4f hogwild %.4f | ndcg@10 %.4f %.4f" % (rs, rh, ns, nh))
    assert rs > 0.05                       # the model actually learned something
    assert abs(rh - rs) < 0.005 and abs(nh - ns) < 0.005


def test_hot_row_path_conserves_updates(monkeypatch):
    """The shared-memory hot path must neither lose nor duplicate deltas.  With a tiny learning
    rate the epoch is in the linear regime (row movement independent of update order), so the
    movement of P and Q must agree between the direct path and the hot path on a conflict-heavy
    log where the 64 hottest tracks carry most plays."""
    from yue_b200.engine import Engine
    log = synth.power_law_log(1500, 400, 150000, seed=4)         # few tracks: the 64 hottest carry most plays
    P, Q = synth.init_factors(log.m, log.n, 64, seed=6)
    out = {}
    for name, min_count in (("direct", "1000000000"), ("hot", "1")):
        monkeypatch.setenv("YUE_SGD_HOT_MIN_COUNT", min_count)
        monkeypatch.setenv("YUE_SGD_HOT_FLUSH", "8")
        eng = Engine(0)
        try:
            eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
            eng.set_factors(P, Q)
            loss = eng.bpr_epoch(1e-5, 0.0, 0.0, 3, 0, MODE_HOGWILD)     # tiny lr: updates ~ linear, order-free
            out[name] = (loss, eng.get_factors())
        finally:
            eng.close()
    (l0, (P0, Q0)), (l1, (P1, Q1)) = out["direct"], out["hot"]
    assert l1 == pytest.approx(l0, rel=1e-4)
    # movements of ~1e-3 built from ~1e-7-sized fp32 increments: compare against the largest movement
    assert np.abs((Q1 - Q) - (Q0 - Q)).max() < 2e-3 * np.abs(Q0 - Q).max()
    assert np.abs((P1 - P) - (P0 - P)).max() < 5e-2 * np.abs(P0 - P).max()
    assert np.linalg.norm(Q1 - Q) == pytest.approx(np.linalg.norm(Q0 - Q), rel=1e-3)


# ---- the blocked kernel (bpr_sgd_blk.cuh): full rows (32/64/128) and masked ones (config/BPR.conf ships num.factors=10,
# CUNE.conf 20, LightGCN.conf 50), hot-row table, second rows ----------
@pytest.mark.parametrize("d", [10, 20, 32, 50, 64, 100, 128])
def test_blocked_kernel_conflict_free_all_widths(engine, d):
    """Disjoint rows per triplet: the blocked kernel (4 triplets per block, scores from the Gram
    recurrence) must give the serial loop's factors -- several triplets per user so that the
    recurrence, partial last blocks and segment boundaries are all exercised."""
    m, n = 300, 300 * 2 * 37
    log = synth.power_law_log(m, n, 9000, seed=3)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    P, Q = synth.init_factors(m, n, d, seed=1)
    per = 1 + np.arange(m) % 37                      # 1..37 triplets per user: blocks of 1-4, up to 2 segments
    u = np.repeat(np.arange(m, dtype=np.int32), per)
    T = len(u)
    i = (2 * np.arange(T)).astype(np.int32)
    j = (2 * np.arange(T) + 1).astype(np.int32)
    Pr, Qr = P.copy(), Q.copy()
    ref_loss = bpr_ref.sgd_epoch(Pr, Qr, u, i, j, 0.05, 0.01, 0.02)
    engine.set_factors(P, Q)
    loss = engine.bpr_apply(u, i, j, 0.05, 0.01, 0.02, MODE_HOGWILD)
    Pg, Qg = engine.get_factors()
    assert rel_err(Pg, Pr) < REL and rel_err(Qg, Qr) < REL
    assert loss == pytest.approx(ref_loss, rel=1e-5)


@pytest.mark.parametrize("d,n", [(64, 40), (64, 7), (32, 12), (128, 25), (20, 9)])
def test_blocked_kernel_read_schedule_is_pinned_when_tracks_repeat(engine, d, n):
    """What the throughput kernel does when a track REPEATS inside a block of 4 triplets or in the next block -- the case
    the conflict-free test avoids and the quality checks only see statistically.  One warp (the log is far below a second
    warp's share), tiny catalogs (7-40 tracks: repeats in nearly every block), users with 1..70 triplets: the tables must
    equal oracle/bpr_blk_ref.py -- the reference's arithmetic per triplet, rows of block k read before block k-1's changes
    are added, every change added -- to 1e-4 (a row of a 7-track catalog takes ~600 float32 adds; the kernel's scores come
    from the Gram recurrence and the oracle's from a float64 dot, so the roundings differ; measured 4e-6 on P, 2e-5 on Q),
    the loss to 1e-5; the serial order is 100x further.  At one warp the epoch is deterministic: one lane adds every
    float in program order, and the same epoch run twice gives the same bits (tests/test_sgd_epoch_schedule_gpu.py)."""
    from oracle import bpr_blk_ref
    m = 60
    rng = np.random.default_rng(d * 100 + n)
    per = 1 + rng.integers(0, 70, m)
    u = np.repeat(np.arange(m, dtype=np.int32), per)
    T = len(u)
    i = rng.integers(0, n, T).astype(np.int32)
    j = ((i + 1 + rng.integers(0, n - 1, T)) % n).astype(np.int32)            # any track but the positive
    assert (i != j).all()
    log = synth.power_law_log(m, max(n, 300), 3000, seed=3)                   # only fixes m for the handle; triplets are explicit
    P, Q = synth.init_factors(m, max(n, 300), d, seed=2)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    loss = engine.bpr_apply(u, i, j, 0.05, 0.01, 0.02, MODE_HOGWILD)
    Pg, Qg = engine.get_factors()
    Pr, Qr = P.copy(), Q.copy()
    ref_loss = bpr_blk_ref.sgd_apply_blocked(Pr, Qr, u, i, j, 0.05, 0.01, 0.02)
    eP, eQ = rel_err(Pg, Pr), rel_err(Qg, Qr)
    assert eP < 1e-4 and eQ < 1e-4
    assert loss == pytest.approx(ref_loss, rel=1e-5)
    # and it is NOT the serial order: the schedule is a real, pinned deviation
    Ps, Qs = P.copy(), Q.copy()
    bpr_ref.sgd_epoch(Ps, Qs, u, i, j, 0.05, 0.01, 0.02)
    assert rel_err(Qg, Qs) > 20 * max(eQ, REL)


@pytest.mark.parametrize("d", [10, 32, 50, 64, 100, 128])
def test_blocked_kernel_hot_table_lr0_and_conservation(monkeypatch, d):
    """Hot-row table with second rows, every track of a small catalog hot.  (1) lr = 0: the epoch must
    leave P and Q bit-identical (rows travel Q -> table -> Q) and the loss is the sum of softplus;
    (2) tiny lr (linear regime, order-free): row movements agree with the per-triplet kernel's direct
    path, i.e. the table neither loses nor duplicates an update, negatives that hit hot tracks included."""
    from yue_b200.engine import Engine
    log = synth.power_law_log(1500, 400, 150000, seed=4)
    P, Q = synth.init_factors(log.m, log.n, d, seed=6)
    ev_user = record_ref.ev_users(log.ev_indptr)
    out = {}
    for name, env in (("direct", dict(YUE_SGD_KERNEL="1", YUE_SGD_HOT_MAX="0")),
                      ("table", dict(YUE_SGD_KERNEL="2", YUE_SGD_HOT_MIN_COUNT="1", YUE_SGD_HOT_DIV="1000000", YUE_SGD_HOT_SHARD_DIV="50"))):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        eng = Engine(0)
        try:
            eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
            if name == "table":
                eng.set_factors(P, Q)
                loss0 = eng.bpr_epoch(0.0, 0.0, 0.0, 3, 0, MODE_HOGWILD)
                P0, Q0 = eng.get_factors()
                assert np.array_equal(P0, P) and np.array_equal(Q0, Q)
                neg = eng.sample_negatives(3, 0)
                x = np.einsum("ij,ij->i", P[ev_user].astype(np.float64), (Q[log.ev_items] - Q[neg]).astype(np.float64))
                assert loss0 == pytest.approx(float(np.logaddexp(0.0, -x).sum()), rel=1e-5)
            eng.set_factors(P, Q)
            loss = eng.bpr_epoch(1e-5, 0.0, 0.0, 3, 0, MODE_HOGWILD)
            out[name] = (loss, eng.get_factors())
        finally:
            eng.close()
        for k in env:
            monkeypatch.delenv(k)
    (l0, (Pd, Qd)), (l1, (Pt, Qt)) = out["direct"], out["table"]
    assert l1 == pytest.approx(l0, rel=1e-4)
    assert np.abs((Qt - Q) - (Qd - Q)).max() < 2e-3 * np.abs(Qd - Q).max()
    assert np.abs((Pt - P) - (Pd - P)).max() < 5e-2 * np.abs(Pd - P).max()
    assert np.linalg.norm(Qt - Q) == pytest.approx(np.linalg.norm(Qd - Q), rel=1e-3)


def test_sub_epochs_compose_to_the_epoch(engine):
    """yue_bpr_epoch_part: parts 0..S-1 in turn are the epoch -- bit-identical in the serial order, and
    in the throughput mode every event is applied exactly once (lr = 0 loss is the full sum)."""
    log = synth.power_law_log(900, 700, 30000, seed=9)
    P, Q = synth.init_factors(log.m, log.n, 64, seed=4)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    full = engine.bpr_epoch(0.05, 0.01, 0.01, 3, 0, MODE_SERIAL)
    Pf, Qf = engine.get_factors()
    for S in (2, 7):
        engine.set_factors(P, Q)
        parts = [engine.bpr_epoch_part(0.05, 0.01, 0.01, 3, 0, k, S, MODE_SERIAL) for k in range(S)]
        Pp, Qp = engine.get_factors()
        assert np.array_equal(Pp, Pf) and np.array_equal(Qp, Qf)
        assert sum(parts) == pytest.approx(full, rel=1e-12)
    engine.set_factors(P, Q)
    l0 = engine.bpr_epoch(0.0, 0.0, 0.0, 3, 0, MODE_HOGWILD)
    lp = sum(engine.bpr_epoch_part(0.0, 0.0, 0.0, 3, 0, k, 5, MODE_HOGWILD) for k in range(5))
    assert lp == pytest.approx(l0, rel=1e-6)
    with pytest.raises(YueError):
        engine.bpr_epoch_part(0.05, 0.01, 0.01, 3, 0, 2, 2, MODE_SERIAL)


def test_sampler_invariant_under_interleaved_sharding(engine):
    """Users r, r+G, r+2G, ... on rank r with per-user event offsets: every rank draws, for its events, exactly the
    negatives the unsharded log gets (the sampler is a function of the GLOBAL event index)."""
    from yue_b200 import sharding
    log = synth.power_law_log(700, 500, 30000, seed=5)
    ev_user = record_ref.ev_users(log.ev_indptr)
    ref = philox.sample_negatives(11, 2, ev_user, log.n, log.uq_indptr, log.uq_items)
    for world in (2, 3):
        for rank in range(world):
            users = sharding.interleaved_users(log.m, world, rank)
            sh = sharding.local_shard_of_users(log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, users)
            engine.set_interactions(sh["m_local"], log.n, sh["ev_indptr"], sh["ev_items"], sh["uq_indptr"], sh["uq_items"])
            engine.set_event_offsets(sh["event_offsets"])
            got = engine.sample_negatives(11, 2)
            want = np.concatenate([ref[log.ev_indptr[u]:log.ev_indptr[u + 1]] for u in users])
            assert np.array_equal(got, want)
    # and the epoch kernels use the same stream: a serial epoch on rank 0's shard with explicit negatives == in-kernel sampling
    users = sharding.interleaved_users(log.m, 2, 0)
    sh = sharding.local_shard_of_users(log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, users)
    P, Q = synth.init_factors(sh["m_local"], log.n, 64, seed=2)
    engine.set_interactions(sh["m_local"], log.n, sh["ev_indptr"], sh["ev_items"], sh["uq_indptr"], sh["uq_items"])
    engine.set_event_offsets(sh["event_offsets"])
    engine.set_factors(P, Q)
    la = engine.bpr_epoch(0.05, 0.01, 0.01, 11, 2, MODE_SERIAL)
    Pa, Qa = engine.get_factors()
    engine.set_factors(P, Q)
    neg = engine.sample_negatives(11, 2)
    lb = engine.bpr_apply(record_ref.ev_users(sh["ev_indptr"]), sh["ev_items"], neg, 0.05, 0.01, 0.01, MODE_SERIAL)
    Pb, Qb = engine.get_factors()
    assert np.array_equal(Pa, Pb) and np.array_equal(Qa, Qb) and la == pytest.approx(lb, rel=1e-12)
