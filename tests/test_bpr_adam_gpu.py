"""K10 (BPR's shipped Adam training, recommender/cf/BPR.py:65-129; csrc/bpr_adam.cuh) on the GPU against oracle/bpr_adam_ref.py.

Tolerances (float32 kernel against the float64 restatement) are LightGCN's (tests/test_lightgcn.py): the loss of a step 2e-5
relative; the first step's gradient (read back from Adam's first moment, m_1 = 0.1 g) 2e-4 of the largest row gradient; after
several steps an entry whose gradient is rounding noise may move by a full step (Adam divides by |g|), so the tables are
compared entry-wise: at least 99.5 % within 2 % of the distance moved, none further than 2.5 lr per step."""
import numpy as np
import pytest

from oracle import bpr_adam_ref as ba
from yue_b200 import synth
from yue_b200.lightgcn import truncated_normal

pytestmark = pytest.mark.gpu


def upload(engine, log):
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)


def tables(log, d, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    return truncated_normal((log.m, d), 0.005 * scale, rng), truncated_normal((log.n, d), 0.005 * scale, rng)


def hot_log():
    """A log with a hot track (re-labelled on the device) and a user who has played all tracks but three."""
    m, n = 40, 300
    rng = np.random.default_rng(3)
    items = [np.concatenate([np.zeros(600, np.int64), rng.integers(0, n, 20)]) for _ in range(m - 1)]
    items.append(np.concatenate([np.arange(n - 3), [0] * 10]))
    ev_indptr = np.concatenate([[0], np.cumsum([len(x) for x in items])]).astype(np.int64)
    ev_items = np.concatenate(items).astype(np.int32)
    rows = [np.unique(x) for x in items]
    uq_indptr = np.concatenate([[0], np.cumsum([len(x) for x in rows])]).astype(np.int64)
    return synth.PlayLog(m, n, ev_indptr, ev_items, uq_indptr, np.concatenate(rows).astype(np.int32),
                         np.zeros(m + 1, np.int64), np.zeros(0, np.int32))


def test_sampler_is_the_oracle_bit_for_bit(engine):
    log = hot_log()
    upload(engine, log)
    assert len(engine.hot_tracks()) > 0 and 0 in engine.hot_tracks()
    full = []                                                 # negatives of the user who left three tracks unplayed
    for seed, step, B, K in ((11, 0, 512, 100), (11, 1, 512, 100), (2 ** 40 + 3, 77, 300, 7)):
        ev, neg = engine.bpr_adam_sample(seed, step, B, K)
        e, u, i, rneg = ba.sample_batch(seed, step, B, K, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, log.n)
        assert np.array_equal(ev, e) and np.array_equal(neg, rneg)
        assert (i == 0).mean() > 0.5                          # the hot track is a positive of most rows
        full.append(rneg[u == log.m - 1].ravel())
    full = np.concatenate(full)
    assert len(full) > 0 and np.isin(full, np.arange(log.n - 3, log.n)).all()
    big = synth.power_law_log(500, 700, 20000, seed=5)
    upload(engine, big)
    ev, neg = engine.bpr_adam_sample(9, 3)
    e, _, _, rneg = ba.sample_batch(9, 3, 512, 100, big.ev_indptr, big.ev_items, big.uq_indptr, big.uq_items, big.n)
    assert np.array_equal(ev, e) and np.array_equal(neg, rneg)


@pytest.mark.parametrize("d", [10, 32, 64, 100, 128, 130])
def test_one_step_gradient_loss_and_update_match_the_oracle(engine, d):
    log = synth.power_law_log(200, 300, 6000, seed=41)
    upload(engine, log)
    U, V = tables(log, d, d, scale=40.0)                      # larger rows: sigmoid away from 1/2
    engine.set_factors(U, V)
    _, u, i, neg = ba.sample_batch(5, 0, 64, 6, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, log.n)
    u, i, j = (x.astype(np.int32) for x in ba.triplets(u, i, neg))
    u[7], i[7] = u[3], i[3]                                   # a repeated user and positive
    j[11] = i[20]                                             # a negative that is another row's positive
    j[12] = j[13] = j[40]                                     # a repeated negative
    U64, V64 = U.astype(np.float64), V.astype(np.float64)
    ref_loss, gU, gV = ba.loss_and_grad(U64, V64, u, i, j, 0.01)
    loss = engine.bpr_adam_apply(u, i, j, 0.002, 0.01)
    assert abs(loss - ref_loss) <= 2e-5 * abs(ref_loss)
    mu, mt, vu, vt, steps = engine.bpr_adam_moments()
    assert steps == 1
    g = np.concatenate([gU, gV])
    got = np.concatenate([mu, mt]).astype(np.float64) / 0.1
    scale = np.linalg.norm(g, axis=1).max()
    assert np.linalg.norm(got - g, axis=1).max() <= 2e-4 * scale
    assert np.allclose(np.concatenate([vu, vt]), 0.001 * g * g, rtol=2e-3, atol=1e-7 * scale * scale)
    P1, Q1 = engine.get_factors()
    moved = np.concatenate([P1, Q1]).astype(np.float64) - np.concatenate([U64, V64])
    want = -0.002 * g / (np.abs(g) + 1e-8 / np.sqrt(0.001))
    sure = np.abs(g) > 1e-3 * scale
    assert np.allclose(moved[sure], want[sure], rtol=1e-3, atol=1e-7)
    assert np.array_equal(moved[g == 0], np.zeros(int((g == 0).sum())))     # rows the batch did not touch stay put


def run_engine(engine, log, U, V, steps, split, batch=128, K=20, lr=0.01, reg=0.01, seed=20261020):
    engine.set_factors(U, V)
    loss = np.concatenate([engine.bpr_adam_steps(batch, K, lr, reg, seed, a, b) for a, b in zip(split[:-1], split[1:])])
    P, Q = engine.get_factors()
    return loss, P, Q, engine.bpr_adam_moments()


def test_fused_steps_follow_the_oracle_and_are_deterministic(engine):
    log = synth.power_law_log(400, 500, 12000, seed=43)
    upload(engine, log)
    U, V = tables(log, 24, 9)
    batch, K, lr, reg, seed, steps = 128, 20, 0.01, 0.01, 20261020, 12
    rU, rV, rloss, _ = ba.train(U, V, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, batch, K, lr, reg, seed, steps)
    loss, P, Q, mom = run_engine(engine, log, U, V, steps, [0, 5, steps])
    assert mom[4] == steps
    assert np.allclose(loss, rloss, rtol=5e-4)
    got, ref, start = np.concatenate([P, Q]).astype(np.float64), np.concatenate([rU, rV]), np.concatenate([U, V]).astype(np.float64)
    ok = np.abs(got - ref) <= 0.02 * np.abs(ref - start) + 1e-9
    assert ok.mean() >= 0.995
    assert np.abs(got - ref).max() <= 2.5 * lr * steps
    # the same bits again, and in one call instead of 5 + 7
    for split in ([0, 5, steps], [0, steps]):
        loss2, P2, Q2, mom2 = run_engine(engine, log, U, V, steps, split)
        assert np.array_equal(loss2, loss) and np.array_equal(P2, P) and np.array_equal(Q2, Q)
        assert all(np.array_equal(a, b) for a, b in zip(mom2[:4], mom[:4])) and mom2[4] == steps
    engine.set_factors(U, V)                                   # restarts Adam
    assert engine.bpr_adam_moments()[4] == 0
    first = engine.bpr_adam_steps(batch, K, lr, reg, seed, 0, 1)
    assert first[0] == loss[0] and engine.bpr_adam_moments()[4] == 1


def test_other_paths_see_the_tables_after_adam_steps(engine):
    from yue_b200.engine import MODE_SERIAL, RANK_EXACT, RANK_TC
    from oracle import topn
    log = synth.power_law_log(300, 2000, 9000, seed=47)
    upload(engine, log)
    U, V = tables(log, 64, 2, scale=20.0)
    engine.set_factors(U, V)
    engine.rank_topn(np.arange(50, dtype=np.int32), 10, RANK_TC)          # derived copies of Q exist before the steps
    engine.bpr_adam_steps(256, 30, 0.05, 0.01, 4, 0, 3)
    P, Q = engine.get_factors()
    assert np.abs(Q - V).max() > 0.05
    assert np.allclose(engine.predict(5), Q @ P[5], rtol=1e-5, atol=1e-6)
    users = np.arange(log.m, dtype=np.int32)
    rid, _ = topn.topn_exact(P, Q, users, 10, log.uq_indptr, log.uq_items)
    for algo in (RANK_EXACT, RANK_TC):
        ids, _ = engine.rank_topn(users, 10, algo)
        assert (ids == rid).mean() > 0.99
    before = engine.get_factors()
    engine.bpr_epoch(0.05, 0.01, 0.01, 3, 0, MODE_SERIAL)                 # SGD goes on from the Adam tables
    after = engine.get_factors()
    assert np.abs(after[1] - before[1]).max() > 0 and np.abs(after[1] - before[1]).max() < 1.0


def test_refusals(engine):
    from yue_b200.engine import YueError
    log = synth.power_law_log(50, 60, 600, seed=3)
    upload(engine, log)
    with pytest.raises(YueError):
        engine.bpr_adam_steps(512, 100, 0.01, 0.01, 1, 0, 1)             # no factors yet
    U, V = tables(log, 16, 1)
    engine.set_factors(U, V)
    for args in ((0, 100), (512, 0), (512, 4096), (1 << 17, 1)):
        with pytest.raises(YueError):
            engine.bpr_adam_steps(args[0], args[1], 0.01, 0.01, 1, 0, 1)
        with pytest.raises(YueError):
            engine.bpr_adam_sample(1, 0, *args)
    with pytest.raises(YueError):
        engine.bpr_adam_steps(512, 100, 0.01, 0.01, 1, 3, 2)              # empty range backwards
    with pytest.raises(YueError):
        engine.bpr_adam_apply(np.array([0]), np.array([0]), np.array([log.n]), 0.01, 0.01)
    with pytest.raises(YueError):
        engine.bpr_adam_apply(np.array([log.m]), np.array([0]), np.array([1]), 0.01, 0.01)
    with pytest.raises(YueError):
        engine.bpr_adam_steps(64, 4, 1e30, 0.01, 1, 0, 2)                  # the tables blow up: non-finite loss
    engine.set_factors(U, V)
    assert len(engine.bpr_adam_steps(64, 4, 0.01, 0.01, 1, 0, 2)) == 2


def test_class_trains_like_the_engine(tmp_path, golden_dir):
    import io
    import json
    import os
    from contextlib import redirect_stdout
    from yue_b200.bpr import BPR
    from yue_b200.engine import Engine
    from yue_b200.host.config import Config
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    test = [e for e, h in zip(g["events"], g["held"]) if h]
    vals = {"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
            "recommender": "BPR", "evaluation.setup": "-target track -ap 0.2", "item.ranking": "-topN 5,10",
            "num.factors": "10", "num.max.iter": "3", "learnRate": "-init 0.01 -max 1",
            "reg.lambda": "-u 0.01 -i 0.01 -b 0.2 -s 0.2", "output.setup": "on -dir %s/" % tmp_path,
            "yue.train": "adam", "yue.seed": "123"}
    out = io.StringIO()
    with redirect_stdout(out):
        rec = BPR(Config(values=vals), train, test)
        rec.readConfiguration()
        rec.initModel()
        np.random.seed(17)
        hooks = []
        hook = rec.ranking_performance
        rec.ranking_performance = lambda: hooks.append(hook())
        rec.buildModel()
        rec.evalRanking()
    assert len(hooks) == 3 and text_losses(out.getvalue()) == 3
    np.random.seed(17)
    U0, V0 = truncated_normal((rec.m, 10), 0.005), truncated_normal((rec.n, 10), 0.005)
    eng = Engine(0)
    try:
        eng.set_interactions(rec.m, rec.n, *rec._engine.get_interactions())
        eng.set_factors(U0, V0)
        loss = eng.bpr_adam_steps(512, 100, 0.01, 0.01, 123, 0, 3)
        P, Q = eng.get_factors()
    finally:
        eng.close()
    assert np.array_equal(rec.P, P) and np.array_equal(rec.Q, Q) and rec.loss == loss[-1]
    assert any("-measure" in f for f in os.listdir(str(tmp_path)))


def text_losses(text):
    return sum(1 for line in text.splitlines() if line.startswith('iteration:') and 'loss:' in line)
