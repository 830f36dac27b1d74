"""K9 (LightGCN, SURVEY.md 8f row 4): oracle/lightgcn_ref.py restates recommender/advanced/LightGCN.py:27-98.  The reference's
module needs TensorFlow 1 and a base file without `.py`, so it is pinned the way the SGD loop and CUNE are: its OWN text, both
files unmodified, was executed in the build container over a stand-in for the TF calls it makes (oracle/tf1_shim.py on torch
autograd, oracle/make_golden_lightgcn.py) and its losses, variables and propagated tables after 60 Adam steps are the golden
run tests/golden/lightgcn_small.npz -- the oracle reproduces them to 1e-12, the kernel to float32 accuracy.  (What the shim
cannot pin is the meaning of each TF op, restated from TF's documentation in its header.)  The CPU tests also check the
restatement's gradient numerically; the GPU tests compare csrc/lightgcn.cuh (yue_gcn_apply / _epoch / _finalize) with it.

Tolerances (float32 kernel against the float64 restatement): the loss of a step 2e-5 relative; the gradient of the first
step (read back from Adam's first moment, m_1 = 0.1 g) 2e-4 of the largest row gradient, per row; the propagated tables
1e-5 per row.  After several Adam steps a table entry whose gradient is rounding noise may differ by a full step (Adam
divides by |g|), so the tables after a run are compared entry-wise: at least 99.5 % within 2 % of the distance moved."""
import os

import numpy as np
import pytest

from oracle import lightgcn_ref as lg
from oracle import philox
from yue_b200 import synth

REF = os.environ.get("YUE_REFERENCE", "")          # a checkout of 0411tony/Yue; the shim test skips without one


def file_order(log, seed):
    """The log's training events in a shuffled 'file' order (any order with the same events per user is a valid file)."""
    users = np.repeat(np.arange(log.m, dtype=np.int32), np.diff(log.ev_indptr))
    perm = np.random.default_rng(seed).permutation(len(users))
    return users[perm], log.ev_items[perm].astype(np.int32)


def test_oracle_gradient_is_the_numerical_gradient():
    rng = np.random.default_rng(0)
    m, n, T, k = 30, 40, 300, 6
    eu, ei = rng.integers(0, m, T), rng.zipf(1.5, T) % n
    A = lg.adjacency(m, n, eu, ei)
    U, V = lg.init_tables(m, n, k, 1)
    E0 = np.concatenate([U, V]).astype(np.float64) * 20
    u, i, j = eu[:16], ei[:16], rng.integers(0, n, 16)
    _, g = lg.loss_and_grad(A, E0, m, u, i, j, 0.01)
    for r, c in zip(rng.integers(0, m + n, 30), rng.integers(0, k, 30)):
        Ep, Em = E0.copy(), E0.copy()
        Ep[r, c] += 1e-6
        Em[r, c] -= 1e-6
        num = (lg.loss_of(A, Ep, m, u, i, j, 0.01) - lg.loss_of(A, Em, m, u, i, j, 0.01)) / 2e-6
        assert abs(num - g[r, c]) <= 1e-6 * max(1.0, abs(num))


def test_oracle_reproduces_the_reference_graph_run_over_the_tf_shim(golden_dir):
    """tests/golden/lightgcn_small.npz is the output of the reference's own LightGCN.py + base/DeepRecommender (unmodified) over
    oracle/tf1_shim.py, its sampler fed the Philox attempt stream (consumed exactly: asserted by the generator).  The
    restatement gives the same 60 losses, the same U and V after two passes and the same propagated tables."""
    import os
    g = np.load(os.path.join(golden_dir, "lightgcn_small.npz"))
    m, n = int(g["m"]), int(g["n"])
    A = lg.adjacency(m, n, g["ev_user"], g["ev_item"])
    for ep in range(int(g["iters"])):                               # the kept negative = the fifth draw, Philox slot 4
        assert np.array_equal(lg.batch_negatives(int(g["seed"]), ep, g["ev_user"], n, g["uq_indptr"], g["uq_items"]), g["neg"][ep])
    U, V, losses, _ = lg.train(A, g["U0"], g["V0"], g["ev_user"], g["ev_item"], g["uq_indptr"], g["uq_items"], int(g["batch"]),
                               float(g["lr"]), float(g["reg"]), int(g["seed"]), epochs=int(g["iters"]))
    assert len(losses) == len(g["losses"]) == 60 and np.allclose(losses, g["losses"], rtol=1e-12)
    assert np.abs(g["U"] - g["U0"]).max() > 0.01                    # the variables moved ...
    assert np.abs(U - g["U"]).max() < 1e-12 and np.abs(V - g["V"]).max() < 1e-12      # ... to the same place
    FU, FV = lg.embeddings(A, U, V)
    assert np.abs(FU - g["FU"]).max() < 1e-11 and np.abs(FV - g["FV"]).max() < 1e-11
    assert np.allclose(FU[g["pred_users"]] @ FV.T, g["preds"], rtol=1e-10)


def test_oracle_adjacency_weighs_a_pair_by_its_squared_count():
    """LightGCN.py:29-33: one entry of value count per EVENT; duplicate entries add up in the sparse product."""
    eu, ei = np.array([0, 0, 0, 1, 1]), np.array([2, 2, 1, 2, 0])
    A = lg.adjacency(2, 3, eu, ei).toarray()
    assert A[0, 2 + 2] == 4 and A[0, 2 + 1] == 1 and A[1, 2 + 2] == 1 and A[1, 2 + 0] == 1
    assert np.array_equal(A, A.T) and A[:2, :2].sum() == 0 and A[2:, 2:].sum() == 0


def test_truncated_normal_init_and_class_config(tmp_path):
    from yue_b200.lightgcn import truncated_normal
    x = truncated_normal((2000, 8), 0.005, np.random.default_rng(3))
    assert x.dtype == np.float32 and np.abs(x).max() <= 0.01 + 1e-9 and 0.004 < x.std() < 0.0048


def test_class_trains_on_the_training_split_in_file_order(golden_dir, tmp_path):
    """Under -byTime (config/LightGCN.conf) Record keeps the UNSPLIT log in trainingData (data/record.py:37 before 47-48):
    the class takes the entries of the training split, in the file's order, and reads batch_size like DeepRecommender."""
    import io
    import json
    import os
    from contextlib import redirect_stdout
    from yue_b200.host.config import Config
    from yue_b200.lightgcn import LightGCN
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    test = [e for e, h in zip(g["events"], g["held"]) if h]
    vals = {"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
            "recommender": "LightGCN", "evaluation.setup": "-target track -byTime 0.2", "item.ranking": "-topN 5,10",
            "num.factors": "50", "num.max.iter": "3", "batch_size": "128", "learnRate": "-init 0.002 -max 1",
            "reg.lambda": "-u 0.001 -i 0.001 -b 0.2 -s 0.2", "output.setup": "on -dir %s/" % tmp_path}
    with redirect_stdout(io.StringIO()):
        rec = LightGCN(Config(values=vals), train, test)
        rec.readConfiguration()
        rec.initModel()
    assert rec.batch_size == 128 and rec.U.shape == (rec.m, 50) and np.abs(rec.U).max() <= 0.01
    eu, ei = rec._file_order_events()
    n_train = sum(len(v) for v in rec.data.userRecord.values())
    assert len(rec.data.trainingData) > n_train == len(eu) == len(ei)
    uid, tid = rec.data.name2id['user'], rec.data.name2id['track']
    kept = set(id(e) for evs in rec.data.userRecord.values() for e in evs)
    want = [(uid[e['user']], tid[e['track']]) for e in rec.data.trainingData if id(e) in kept]
    assert list(zip(eu.tolist(), ei.tolist())) == want
    with redirect_stdout(io.StringIO()):
        vals["evaluation.setup"] = "-target track -ap 0.2"
        rec2 = LightGCN(Config(values=vals), train, test)
        rec2.readConfiguration()
        rec2.initModel()
    eu2, _ = rec2._file_order_events()
    assert len(eu2) == len(train) and eu2.tolist() == [rec2.data.name2id['user'][e['user']] for e in train]


def test_both_ingest_modes_give_the_class_the_same_batches(golden_dir, tmp_path):
    """-byTime (config/LightGCN.conf): the dict Record and the array ingest (yue.ingest=arrays, ArrayLog with the events' file
    positions) number users and tracks alike and hand LightGCN the SAME training events in the SAME (file) order."""
    pytest.importorskip("pyarrow")
    import io
    import json
    import os
    from contextlib import redirect_stdout
    from yue_b200 import ingest
    from yue_b200.host.config import Config, LineConfig
    from yue_b200.lightgcn import LightGCN
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    events = g["events"][:2500]
    path = os.path.join(str(tmp_path), "log.txt")
    with open(path, "w") as f:
        f.write("".join("%s,%s,%s,%s\n" % (e["time"], e["user"], e["track"], e["artist"]) for e in events))
    vals = {"record": path, "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,", "recommender": "LightGCN",
            "evaluation.setup": "-target track -byTime 0.2", "item.ranking": "-topN 5,10", "num.factors": "8", "num.max.iter": "1",
            "batch_size": "128", "learnRate": "-init 0.002 -max 1", "reg.lambda": "-u 0.001 -i 0.001 -b 0.2 -s 0.2",
            "output.setup": "on -dir %s/" % tmp_path}
    columns = dict([("user", 1), ("track", 2), ("artist", 3), ("time", 0)])
    log = ingest.load_numbered(path, columns, ",", LineConfig(vals["evaluation.setup"]), "track")
    with redirect_stdout(io.StringIO()):
        a = LightGCN(Config(values=vals), log, [])
        b = LightGCN(Config(values=vals), [dict(e) for e in events], [])
        for mdl in (a, b):
            mdl.readConfiguration()
            mdl.initModel()
    assert (a.m, a.n, a.train_size) == (b.m, b.n, sum(len(v) for v in b.data.userRecord.values()))
    ua, ia = a._file_order_events()
    ub, ib = b._file_order_events()
    assert np.array_equal(ua, ub) and np.array_equal(ia, ib)
    names = np.asarray(log.names["user"], dtype=object)
    assert names[ua[:20]].tolist() == [b.data.id2name["user"][int(x)] for x in ub[:20]]


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the Yue reference: set YUE_REFERENCE to its directory")
def test_dropin_shim_on_top_of_the_reference_tree(golden_dir, tmp_path):
    """dropin/recommender/advanced/LightGCN.py shadows the reference's module (TF-1, unimportable base), derives from the
    REFERENCE's own base.IterativeRecommender and Record (under -byTime: the reference's own time split), and drives the
    engine with the calls INTEGRATION.md lists -- checked with a recording engine in place of the CUDA one."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    conf = {"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
            "recommender": "LightGCN", "evaluation.setup": "-target track -byTime 0.2", "item.ranking": "-topN 5,10",
            "num.factors": "50", "num.max.iter": "2", "batch_size": "128", "learnRate": "-init 0.002 -max 1",
            "reg.lambda": "-u 0.001 -i 0.001 -b 0.2 -s 0.2", "output.setup": "on -dir %s/" % tmp_path, "yue.seed": "11"}
    code = r'''
import io, json, sys
import numpy as np
from contextlib import redirect_stdout
sys.path[:0] = [%(dropin)r, %(ref)r, %(root)r]
from tool.config import Config
from recommender.advanced.LightGCN import LightGCN
import base.IterativeRecommender as ref_base
import recommender.advanced.LightGCN as mod
assert mod.__file__.startswith(%(dropin)r) and LightGCN.__mro__[3] is ref_base.IterativeRecommender, LightGCN.__mro__
g = json.load(open(%(gold)r + "/record_small.json"))
events = g["events"]
open(%(tmp)r + "/c.conf", "w").write("\n".join(k + "=" + v for k, v in %(conf)r.items()))
calls = []
class Rec(object):
    def set_factors(self, U, V): calls.append(("set_factors", U.shape, V.shape, float(np.abs(U).max())))
    def gcn_set_events(self, eu, ei): calls.append(("events", len(eu))); self.T = len(eu)
    def gcn_epoch(self, batch, lr, reg, seed, it, L): calls.append(("epoch", batch, lr, reg, seed, it, L)); return np.arange(3.0) + it
    def get_factors(self): return np.zeros((2, 50), np.float32), np.ones((3, 50), np.float32)
    def gcn_finalize(self, L): calls.append(("finalize", L))
with redirect_stdout(io.StringIO()) as out:
    m = LightGCN(Config(%(tmp)r + "/c.conf"), events, [])
    m.readConfiguration()
    m.initModel()
    eng = Rec()
    m._get_engine = lambda: eng
    m._engine = eng
    m.buildModel()
n_train = sum(len(v) for v in m.data.userRecord.values())
assert 0 < n_train < len(events) and m.data.testSet                      # the reference's own -byTime split
assert calls[0][0] == "set_factors" and calls[0][1] == (m.m, 50) and calls[0][3] <= 0.01
assert calls[1] == ("events", n_train)
assert calls[2] == ("epoch", 128, 0.002, 0.001, 11, 0, 3) and calls[3] == ("epoch", 128, 0.002, 0.001, 11, 1, 3)
assert calls[4] == ("finalize", 3) and m.loss == 3.0
assert m.multi_item_embeddings.shape == (3, 50) and "training: 2 batch 2 loss: 3.0" in out.getvalue()
print("shim ok")
''' % dict(dropin=os.path.join(root, "dropin"), ref=REF, root=root, gold=golden_dir, tmp=str(tmp_path), conf=conf)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "shim ok" in res.stdout, res.stdout + res.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("d", [8, 50, 100, 130])
def test_one_step_gradient_loss_and_update_match_the_oracle(engine, d):
    log = synth.power_law_log(300, 200, 9000, seed=41)
    eu, ei = file_order(log, 1)
    assert np.bincount(ei, minlength=log.n).max() > 64                  # a row a whole CTA works on
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    U, V = lg.init_tables(log.m, log.n, d, 7)
    U, V = U * 20, V * 20                                                # larger rows: sigmoid away from 1/2
    engine.set_factors(U, V)
    rng = np.random.default_rng(d)
    B = 96
    u, i = eu[:B].copy(), ei[:B].copy()
    j = rng.integers(0, log.n, B).astype(np.int32)
    u[5], i[5], j[6] = u[4], i[4], i[4]                                  # repeated rows inside the batch, on both sides
    A = lg.adjacency(log.m, log.n, eu, ei)
    E0 = np.concatenate([U, V]).astype(np.float64)
    ref_loss, g = lg.loss_and_grad(A, E0, log.m, u, i, j, 0.001)
    loss = engine.gcn_apply(u, i, j, 0.002, 0.001)
    assert abs(loss - ref_loss) <= 2e-5 * abs(ref_loss)
    mu, mt, vu, vt, steps = engine.gcn_moments()
    assert steps == 1
    got = np.concatenate([mu, mt]).astype(np.float64) / 0.1
    scale = np.linalg.norm(g, axis=1).max()
    assert np.linalg.norm(got - g, axis=1).max() <= 2e-4 * scale
    assert np.allclose(np.concatenate([vu, vt]), 0.001 * g * g, rtol=2e-3, atol=1e-7 * scale * scale)
    # the first Adam step moves every entry with a gradient by lr * g / (|g| + 1e-8 / sqrt(0.001)) ...
    P1, Q1 = engine.get_factors()
    moved = np.concatenate([P1, Q1]).astype(np.float64) - E0
    want = -0.002 * g / (np.abs(g) + 1e-8 / np.sqrt(0.001))
    sure = np.abs(g) > 1e-3 * scale
    assert np.allclose(moved[sure], want[sure], rtol=1e-3, atol=1e-7)
    assert np.array_equal(moved[g == 0], np.zeros(int((g == 0).sum())))  # ... and leaves the others where they were


@pytest.mark.gpu
def test_steps_with_the_fused_sampler_follow_the_oracle_and_finalize_gives_the_ranking_tables(engine):
    log = synth.power_law_log(400, 300, 6000, seed=43)
    eu, ei = file_order(log, 2)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    d, batch, lr, reg, seed, steps = 50, 128, 0.002, 0.001, 20260107, 12
    U, V = lg.init_tables(log.m, log.n, d, 9)
    engine.set_factors(U, V)
    engine.gcn_set_events(eu, ei)
    neg = philox.sample_negatives(seed, 0, eu, log.n, log.uq_indptr, log.uq_items, slot=lg.NEG_SLOT)
    assert not any(neg[e] in log.uq_items[log.uq_indptr[eu[e]]:log.uq_indptr[eu[e] + 1]] for e in range(0, len(eu), 37))
    A = lg.adjacency(log.m, log.n, eu, ei)
    rU, rV, rloss, _ = lg.train(A, U, V, eu, ei, log.uq_indptr, log.uq_items, batch, lr, reg, seed, epochs=1, max_steps=steps)
    # two launches (5 + 7 steps): Adam's state and the step counter carry over
    loss = np.concatenate([engine.gcn_epoch(batch, lr, reg, seed, 0, step_begin=0, step_end=5),
                           engine.gcn_epoch(batch, lr, reg, seed, 0, step_begin=5, step_end=steps)])
    assert np.allclose(loss, rloss, rtol=5e-4)
    P, Q = engine.get_factors()
    got, ref, start = np.concatenate([P, Q]).astype(np.float64), np.concatenate([rU, rV]), np.concatenate([U, V]).astype(np.float64)
    moved = np.abs(ref - start)
    ok = np.abs(got - ref) <= 0.02 * moved + 1e-9
    assert ok.mean() >= 0.995
    assert np.abs(got - ref).max() <= 2.5 * lr * steps
    # the tables predict() ranks with: F of the kernel's own variables against the oracle's propagation of the same variables
    engine.gcn_finalize()
    FU, FV = engine.get_factors()
    wU, wV = lg.embeddings(A, P, Q)
    rel = np.linalg.norm(np.concatenate([FU, FV]) - np.concatenate([wU, wV]), axis=1) / np.linalg.norm(np.concatenate([wU, wV]), axis=1)
    assert rel.max() <= 1e-5
    scores = engine.predict(3)
    assert np.allclose(scores, FV @ FU[3], rtol=1e-5, atol=1e-6)
    # training goes on from the variables, not from F
    more = engine.gcn_epoch(batch, lr, reg, seed, 0, step_begin=steps, step_end=steps + 1)
    P2, _ = engine.get_factors()
    assert np.isfinite(more).all() and np.abs(P2 - P).max() <= 3 * lr


@pytest.mark.gpu
def test_whole_pass_with_a_partial_last_batch_and_two_layers(engine):
    """ceil(T / batch) steps, the last one shorter; n_layers = 2; rows without any neighbour (tracks nobody played) in the graph."""
    log = synth.power_law_log(120, 400, 1500, seed=47)
    eu, ei = file_order(log, 5)
    assert len(eu) % 128 != 0 and (np.bincount(ei, minlength=log.n) == 0).sum() > 50
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    U, V = lg.init_tables(log.m, log.n, 20, 13)
    U, V = U * 10, V * 10
    engine.set_factors(U, V)
    engine.gcn_set_events(eu, ei)
    A = lg.adjacency(log.m, log.n, eu, ei)
    rU, rV, rloss, _ = lg.train(A, U, V, eu, ei, log.uq_indptr, log.uq_items, 128, 0.002, 0.001, 77, epochs=1, n_layers=2)
    loss = engine.gcn_epoch(128, 0.002, 0.001, 77, 0, n_layers=2)
    assert len(loss) == len(rloss) == (len(eu) + 127) // 128
    assert np.allclose(loss, rloss, rtol=5e-4)
    P, Q = engine.get_factors()
    got, ref, start = np.concatenate([P, Q]).astype(np.float64), np.concatenate([rU, rV]), np.concatenate([U, V]).astype(np.float64)
    assert (np.abs(got - ref) <= 0.02 * np.abs(ref - start) + 1e-9).mean() >= 0.995
    engine.gcn_finalize(2)
    FU, FV = engine.get_factors()
    wU, wV = lg.embeddings(A, P, Q, n_layers=2)
    assert np.abs(np.concatenate([FU, FV]) - np.concatenate([wU, wV])).max() <= 1e-5 * np.abs(np.concatenate([wU, wV])).max()


@pytest.mark.gpu
def test_kernel_follows_the_reference_graph_golden_run(engine, golden_dir):
    """The CUDA path against the golden run of the reference's own LightGCN text (tests/golden/lightgcn_small.npz): the same
    log, initial variables and sampler seed, two passes of 30 steps through yue_gcn_epoch: every step's loss within 5e-4,
    >= 99.5 % of the table entries within 2 % of the distance they moved, the propagated tables the golden ones."""
    import os
    g = np.load(os.path.join(golden_dir, "lightgcn_small.npz"))
    m, n = int(g["m"]), int(g["n"])
    engine.set_interactions(m, n, g["ev_indptr"], g["ev_items"], g["uq_indptr"], g["uq_items"])
    engine.set_factors(g["U0"].astype(np.float32), g["V0"].astype(np.float32))
    engine.gcn_set_events(g["ev_user"], g["ev_item"])
    loss = np.concatenate([engine.gcn_epoch(int(g["batch"]), float(g["lr"]), float(g["reg"]), int(g["seed"]), ep) for ep in range(int(g["iters"]))])
    assert np.allclose(loss, g["losses"], rtol=5e-4)
    P, Q = engine.get_factors()
    got, ref = np.concatenate([P, Q]).astype(np.float64), np.concatenate([g["U"], g["V"]])
    moved = np.abs(ref - np.concatenate([g["U0"], g["V0"]]))
    assert (np.abs(got - ref) <= 0.02 * moved + 1e-9).mean() >= 0.995
    engine.gcn_finalize()
    FU, FV = engine.get_factors()
    ref_f = np.concatenate([g["FU"], g["FV"]])
    assert np.abs(np.concatenate([FU, FV]) - ref_f).max() <= 2e-3 * np.abs(ref_f).max()


@pytest.mark.gpu
def test_refusals(engine):
    from yue_b200.engine import YueError
    log = synth.power_law_log(50, 60, 600, seed=3)
    eu, ei = file_order(log, 3)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    U, V = lg.init_tables(log.m, log.n, 16, 1)
    engine.set_factors(U, V)
    with pytest.raises(YueError):
        engine.gcn_epoch(128, 0.002, 0.001, 1, 0)                        # events not set
    with pytest.raises(YueError):
        engine.gcn_set_events(eu[:-1], ei[:-1])                          # not the resident log
    bad = eu.copy()
    bad[0] = (bad[0] + 1) % log.m
    with pytest.raises(YueError):
        engine.gcn_set_events(bad, ei)                                   # another user's event
    engine.gcn_set_events(eu, ei)
    with pytest.raises(YueError):
        engine.gcn_epoch(5000, 0.002, 0.001, 1, 0)                       # batch beyond the scratch
    with pytest.raises(YueError):
        engine.gcn_apply(np.array([0]), np.array([0]), np.array([log.n]), 0.002, 0.001)
    assert len(engine.gcn_epoch(128, 0.002, 0.001, 1, 0)) == (len(eu) + 127) // 128


@pytest.mark.gpu
def test_class_api_trains_and_ranks_with_the_propagated_tables(tmp_path, golden_dir):
    """Yue -> LightGCN.execute() on the golden log: the losses of a pass fall, predict() is F_items . F_user, the measure
    list has the reference's layout."""
    import io
    import json
    import os
    from contextlib import redirect_stdout
    from yue_b200.host.config import Config
    from yue_b200.lightgcn import LightGCN
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    test = [e for e, h in zip(g["events"], g["held"]) if h]
    conf = Config(values={"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
                          "recommender": "LightGCN", "evaluation.setup": "-target track -byTime 0.2", "item.ranking": "-topN 5,10",
                          "num.factors": "50", "num.max.iter": "3", "batch_size": "128", "learnRate": "-init 0.002 -max 1",
                          "reg.lambda": "-u 0.001 -i 0.001 -b 0.2 -s 0.2", "output.setup": "on -dir %s/" % tmp_path,
                          "yue.seed": "5"})
    out = io.StringIO()
    with redirect_stdout(out):
        rec = LightGCN(conf, train, test)
        measure = rec.execute()
    text = out.getvalue()
    first = [float(l.split('loss:')[1]) for l in text.splitlines() if l.startswith('training:') and ' batch 0 ' in l]
    assert len(first) == 3 and first[2] < first[0]
    assert measure[0] == 'Top 5\n' and measure[1].startswith('Precision:')
    u = next(iter(rec.data.testSet))
    uid = rec.data.getId(u, 'user')
    assert np.allclose(rec.predict(u), rec.multi_item_embeddings @ rec.multi_user_embeddings[uid], rtol=1e-5, atol=1e-6)
    assert rec.U.shape == (rec.m, 50) and not np.array_equal(rec.U, rec.multi_user_embeddings)
