"""K10 (BPR's shipped Adam training, recommender/cf/BPR.py:65-129): CPU checks of oracle/bpr_adam_ref.py -- its gradient
against a numerical one, its steps against the same graph built from oracle/tf1_shim.py's TF ops, its sampler -- and of the
class's yue.train key."""
import numpy as np
import pytest

from oracle import bpr_adam_ref as ba
from oracle import tf1_shim as tf
from yue_b200 import synth


def small_log(seed=5):
    return synth.power_law_log(60, 80, 1500, seed=seed)


def test_loss_and_grad_is_the_numerical_gradient():
    rng = np.random.default_rng(0)
    m, n, k = 20, 30, 6
    U, V = rng.normal(0, 0.5, (m, k)), rng.normal(0, 0.5, (n, k))
    u, i, j = rng.integers(0, m, 64), rng.integers(0, n, 64), rng.integers(0, n, 64)
    u[3], j[5] = u[2], i[4]                                       # repeated rows on both sides
    _, gU, gV = ba.loss_and_grad(U, V, u, i, j, 0.05)
    for tab, g in ((0, gU), (1, gV)):
        for r, c in zip(rng.integers(0, (m, n)[tab], 20), rng.integers(0, k, 20)):
            Xp, Xm = [U.copy(), V.copy()], [U.copy(), V.copy()]
            Xp[tab][r, c] += 1e-6
            Xm[tab][r, c] -= 1e-6
            num = (ba.loss_of(*Xp, u, i, j, 0.05) - ba.loss_of(*Xm, u, i, j, 0.05)) / 2e-6
            assert abs(num - g[r, c]) <= 1e-6 * max(1.0, abs(num))


def test_steps_are_the_graph_built_from_tf_ops():
    """BPR.py:93-116 written with the shim's embedding_lookup / softplus / l2_loss / AdamOptimizer.minimize: five steps on the
    oracle's batches give the oracle's losses and tables to 1e-12."""
    log = small_log()
    m, n, k, lr, reg, seed, B, K = log.m, log.n, 8, 0.01, 0.01, 77, 16, 5
    rng = np.random.default_rng(1)
    U0, V0 = (0.1 * rng.standard_normal((m, k))).astype(np.float32), (0.1 * rng.standard_normal((n, k))).astype(np.float32)
    tf.reset()
    U, V = tf.Variable(U0, name='U'), tf.Variable(V0, name='V')
    u_idx, i_idx, j_idx = tf.placeholder(tf.int32, name='u'), tf.placeholder(tf.int32, name='i'), tf.placeholder(tf.int32, name='j')
    Uu, Vi, Vj = tf.nn.embedding_lookup(U, u_idx), tf.nn.embedding_lookup(V, i_idx), tf.nn.embedding_lookup(V, j_idx)
    y = tf.reduce_sum(tf.multiply(Uu, Vi), 1) - tf.reduce_sum(tf.multiply(Uu, Vj), 1)
    loss = tf.reduce_sum(tf.nn.softplus(-y)) + reg * (tf.nn.l2_loss(Uu) + tf.nn.l2_loss(Vi) + tf.nn.l2_loss(Vj))
    train = tf.train.AdamOptimizer(lr).minimize(loss)
    shim_losses = []
    with tf.Session() as sess:
        for s in range(5):
            _, u, i, neg = ba.sample_batch(seed, s, B, K, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, n)
            tu, ti, tj = ba.triplets(u, i, neg)
            _, lv = sess.run([train, loss], feed_dict={u_idx: tu, i_idx: ti, j_idx: tj})
            shim_losses.append(float(lv))
    tf.reset()
    rU, rV, losses, (aU, _) = ba.train(U0, V0, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, B, K, lr, reg, seed, 5)
    assert aU.t == 5 and np.abs(rU - U0).max() > 2 * lr          # the tables moved
    assert np.allclose(losses, shim_losses, rtol=1e-12, atol=0)
    assert np.abs(rU - U.tensor.detach().numpy()).max() < 1e-12 and np.abs(rV - V.tensor.detach().numpy()).max() < 1e-12


def test_sampler_draws_unplayed_negatives_and_is_reproducible():
    log = small_log(9)
    for seed, step in ((3, 0), (3, 1), (2 ** 40 + 7, 12345)):
        e, u, i, neg = ba.sample_batch(seed, step, 64, 30, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, log.n)
        assert ((0 <= e) & (e < log.ev_indptr[-1])).all() and ((0 <= neg) & (neg < log.n)).all()
        assert np.array_equal(u, np.searchsorted(log.ev_indptr, e, side='right') - 1) and np.array_equal(i, log.ev_items[e])
        for b in range(64):
            played = set(log.uq_items[log.uq_indptr[u[b]]:log.uq_indptr[u[b] + 1]].tolist())
            assert not played & set(neg[b].tolist())
        again = ba.sample_batch(seed, step, 64, 30, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, log.n)
        assert all(np.array_equal(x, y) for x, y in zip((e, u, i, neg), again))
    other = ba.sample_batch(3, 2, 64, 30, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, log.n)
    assert not np.array_equal(other[3], ba.sample_batch(3, 0, 64, 30, log.ev_indptr, log.ev_items, log.uq_indptr,
                                                         log.uq_items, log.n)[3])
    # rejection against a play row that leaves five of 40 tracks
    ev_indptr, ev_items = np.array([0, 3], np.int64), np.array([0, 1, 2], np.int32)
    uq_indptr, uq_items = np.array([0, 35], np.int64), np.arange(35, dtype=np.int32)
    _, _, _, neg = ba.sample_batch(1, 0, 8, 50, ev_indptr, ev_items, uq_indptr, uq_items, 40)
    assert ((neg >= 35) & (neg < 40)).all() and len(set(neg.ravel().tolist())) == 5


def test_class_rejects_an_unknown_training_mode_before_touching_a_gpu(golden_dir, tmp_path):
    import json
    import os
    from yue_b200.bpr import BPR
    from yue_b200.host.config import Config
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    vals = {"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
            "recommender": "BPR", "evaluation.setup": "-target track -ap 0.2", "item.ranking": "-topN 5,10",
            "num.factors": "10", "num.max.iter": "1", "learnRate": "-init 0.01 -max 1",
            "reg.lambda": "-u 0.01 -i 0.01 -b 0.2 -s 0.2", "output.setup": "on -dir %s/" % tmp_path, "yue.train": "adagrad"}
    rec = BPR(Config(values=vals), train, [])
    rec.readConfiguration()
    rec.initModel()
    with pytest.raises(ValueError, match="yue.train"):
        rec.buildModel()
    assert rec._engine is None
