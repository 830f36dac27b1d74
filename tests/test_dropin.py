"""The recommender class layer (yue_b200/bpr.py): CPU checks of the host logic with the engine
replaced by the oracle, and a GPU end-to-end run of config C1 through the reference-shaped API."""
import io
import json
import os
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import bpr_ref, philox, record_ref, topn
from yue_b200.host.config import Config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("YUE_REFERENCE", "")          # a checkout of 0411tony/Yue; the tests that import it skip without one
NO_REF = "needs a checkout of the Yue reference: set YUE_REFERENCE to its directory"


def conf_values(out_dir, eval_setup="-target track -ap 0.2", extra=None):
    v = {"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
         "recommender": "BPR", "evaluation.setup": eval_setup, "item.ranking": "-topN 5,10",
         "num.factors": "10", "num.max.iter": "3", "learnRate": "-init 0.02 -max 1",
         "reg.lambda": "-u 0.01 -i 0.01 -b 0.2 -s 0.2", "output.setup": "on -dir %s/" % out_dir}
    v.update(extra or {})
    return v


class OracleEngine:
    """Stands in for yue_b200.engine.Engine on a CPU-only box (tests only)."""

    def __init__(self, model):
        self.m = model
        self.arr = model.data.interaction_arrays(model.recType) if hasattr(model.data, "interaction_arrays") else None

    def rank_topn(self, users, N, algo):
        ev_indptr, ev_items, uq_indptr, uq_items = self.arr
        return topn.topn_exact(self.m.P, self.m.Q, users, N, uq_indptr, uq_items)


def golden_split(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    test = [e for e, h in zip(g["events"], g["held"]) if h]
    return g, train, test


def test_evalranking_host_logic_matches_reference_measure(golden_dir, tmp_path):
    """Same P, Q as the golden run -> the class's evalRanking (ids -> names -> result lines ->
    Measure) reproduces the reference's Measure output on exact top-N lists, and writes the two
    result files the reference writes (IterativeRecommender.py:156-173)."""
    from yue_b200.bpr import BPR
    g, train, test = golden_split(golden_dir)
    e = np.load(os.path.join(golden_dir, "eval_small.npz"))
    mj = json.load(open(os.path.join(golden_dir, "measure_small.json")))
    with redirect_stdout(io.StringIO()):
        model = BPR(Config(values=conf_values(tmp_path)), train, test)
        model.readConfiguration()
        model.initModel()
        assert model.P.dtype == np.float32 and model.P.shape == (model.m, 10) and model.Q.shape == (model.n, 10)
        assert model.P.min() >= 0 and model.P.max() < 0.1
        model.P, model.Q = e["P"], e["Q"]
        oe = OracleEngine(model)
        model._push_factors = lambda: oe
        model.evalRanking()
    assert model.measure == mj["measure_exact"]
    files = sorted(os.listdir(tmp_path))
    assert len(files) == 2 and "-measure[1].txt" in files[0] and "-top-5,10items[1].txt" in files[1]
    lines = open(os.path.join(tmp_path, files[1])).read().splitlines()
    assert lines[0].startswith("userId: recommendations in (itemId, ranking score) pairs")
    assert len(lines) == 1 + len(model.data.testSet) and "*" in "".join(lines)
    assert set(model.ndcg) == {5, 10} and 0 < model.ndcg[10] < 1


@pytest.mark.skipif(not os.path.isdir(REF), reason=NO_REF)
def test_dropin_shim_on_top_of_the_reference_tree(golden_dir, tmp_path):
    """dropin/recommender/cf/BPR.py imports against the REFERENCE's own base classes, Record and
    Measure, and produces the reference's measure strings."""
    import subprocess
    code = r'''
import io, json, os, sys
import numpy as np
from contextlib import redirect_stdout
sys.path[:0] = [%(dropin)r, %(ref)r, %(root)r]
from tool.config import Config
from recommender.cf.BPR import BPR
import base.IterativeRecommender as ref_base
assert BPR.__mro__[2] is ref_base.IterativeRecommender
from oracle import topn
g = json.load(open(%(gold)r + "/record_small.json"))
train = [e for e, h in zip(g["events"], g["held"]) if not h]
test = [e for e, h in zip(g["events"], g["held"]) if h]
open(%(tmp)r + "/c.conf", "w").write("\n".join(k + "=" + v for k, v in %(conf)r.items()))
e = np.load(%(gold)r + "/eval_small.npz")
mj = json.load(open(%(gold)r + "/measure_small.json"))
with redirect_stdout(io.StringIO()):
    m = BPR(Config(%(tmp)r + "/c.conf"), train, test)
    m.readConfiguration(); m.initModel()
    m.P, m.Q = e["P"], e["Q"]
    from yue_b200.host.record import interaction_arrays
    arr = interaction_arrays(m.data.name2id, m.data.userRecord, m.recType)
    class E:
        def rank_topn(self, users, N, algo): return topn.topn_exact(m.P, m.Q, users, N, arr[2], arr[3])
    m._push_factors = lambda: E()
    m.evalRanking()
assert m.measure == mj["measure_exact"], m.measure[:3]
print("OK")
''' % dict(dropin=os.path.join(ROOT, "dropin"), ref=REF, root=ROOT, gold=golden_dir, tmp=str(tmp_path),
           conf=conf_values(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


@pytest.mark.gpu
def test_c1_end_to_end_through_the_class_api(tmp_path):
    """Config C1 (Xiami-100K-shaped log, d = 10, config/BPR.conf hyper-parameters, -ap 0.2) from a
    CSV file through Yue -> BPR.execute() on the GPU; the serial-order run is compared with the
    oracle trained from the same initial factors, the default (Hogwild) run with the serial one."""
    from yue_b200 import synth
    from yue_b200.host.driver import Yue
    import random
    log_path = tmp_path / "log.txt"
    synth.write_csv_log(str(log_path), 4000, 50000, 100000, seed=20260101)
    results = {}
    for mode in ("serial", "hogwild", "serial-device-metrics"):
        vals = conf_values(tmp_path / mode, extra={"record": str(log_path), "yue.sgd": mode.split("-")[0], "yue.seed": "77",
                                                   "num.max.iter": "2",
                                                   "yue.metrics": "device" if mode.endswith("metrics") else "host",
                                                   "yue.ingest": "device" if mode.endswith("metrics") else "host"})
        random.seed(5)                       # DataSplit uses the global stream (tool/dataSplit.py:15)
        np.random.seed(11)                   # initModel uses the global numpy stream
        with redirect_stdout(io.StringIO()):
            y = Yue(Config(values=vals))
            from yue_b200.bpr import BPR
            model = BPR(y.config, y.trainingData, y.testData)
            measure = model.execute()
        results[mode] = (model, measure)
    ms, meas = results["serial"]
    # oracle: same split (same seed), same init stream, same sampler seed
    ev_indptr, ev_items, uq_indptr, uq_items = ms.data.interaction_arrays()
    np.random.seed(11)
    P = np.random.rand(ms.m, 10).astype(np.float32) / 10
    Q = np.random.rand(ms.n, 10).astype(np.float32) / 10
    hist = bpr_ref.train(P, Q, record_ref.ev_users(ev_indptr), ev_items, ms.n, uq_indptr, uq_items, 2, 0.02, 1.0,
                         0.01, 0.01, 77)
    assert np.allclose(ms.P, P, rtol=1e-5, atol=1e-7) and np.allclose(ms.Q, Q, rtol=1e-5, atol=1e-7)
    assert ms.loss == pytest.approx(hist[-1][0], rel=1e-5)
    assert meas[0] == "Top 5\n" and meas[6] == "Top 10\n" and meas[1].startswith("Precision:")
    # metrics computed on the device (K6): same numbers as the reference's Measure on the same lists
    md, meas_d = results["serial-device-metrics"]
    assert len(meas_d) == len(meas)
    for a, b in zip(meas, meas_d):
        if ":" in a:
            assert a.split(":")[0] == b.split(":")[0]
            assert float(b.split(":")[1]) == pytest.approx(float(a.split(":")[1]), rel=1e-12, abs=1e-15)
        else:
            assert a == b
    assert meas_d[1] == meas[1] and meas_d[5] == meas[5]          # Precision and Coverage: integer sums, same strings
    assert md.ndcg[10] == pytest.approx(ms.ndcg[10], rel=1e-12)
    mh, _ = results["hogwild"]
    rec = lambda m: float(m.measure[8].split(":")[1])       # Recall@10
    assert abs(rec(mh) - rec(ms)) < 0.005


@pytest.mark.gpu
def test_class_api_on_several_devices(tmp_path):
    """yue.devices=a,b through Yue -> BPR.execute() (yue.py:59-131, base/recommender.py:152-174): evalRanking ranks a block
    of the test users per device and must produce the lists and measures of ONE device bit for bit; buildModel shards the
    users over the devices (hot rows shared over peer memory, tail summed over peer memory, no NCCL) and must stay within
    the 0.5-point gate of the serial-order run.  On a one-GPU box the two "devices" are two handles on device 0 -- the
    same code, threads and peer pointers included."""
    from yue_b200 import synth
    from yue_b200.engine import device_count
    from yue_b200.host.driver import Yue
    from yue_b200.bpr import BPR
    from yue_b200.apr import APR
    import random
    devs = "0,1" if device_count() >= 2 else "0,0"
    log_path = tmp_path / "log.txt"
    synth.write_csv_log(str(log_path), 6000, 3000, 400000, seed=20260102)
    runs = {}
    for name, extra in (("serial", {"yue.sgd": "serial"}), ("one", {}), ("two", {"yue.devices": devs, "yue.sub_epochs": "16"})):
        vals = conf_values(tmp_path / name, extra=dict({"record": str(log_path), "yue.seed": "77", "num.max.iter": "4", "num.factors": "64",
                                                        "item.ranking": "-topN 10"}, **extra))
        random.seed(5)
        np.random.seed(11)
        with redirect_stdout(io.StringIO()):
            y = Yue(Config(values=vals))
            model = BPR(y.config, y.trainingData, y.testData)
            model.execute()
        runs[name] = model
    rec = lambda m: float(m.measure[2].split(":")[1])          # Recall@10
    ser, one, two = runs["serial"], runs["one"], runs["two"]
    assert two.P.shape == ser.P.shape and two.Q.shape == ser.Q.shape and np.isfinite(two.P).all() and np.isfinite(two.Q).all()
    assert abs(rec(one) - rec(ser)) < 0.005 and abs(one.ndcg[10] - ser.ndcg[10]) < 0.005
    assert abs(rec(two) - rec(ser)) < 0.005 and abs(two.ndcg[10] - ser.ndcg[10]) < 0.005
    assert two.loss == pytest.approx(ser.loss, rel=0.02)
    # ranking on two devices = ranking on one, given the same tables
    users = list(two.data.testSet.keys())
    with redirect_stdout(io.StringIO()):
        lists2, ids2, sc2 = two._topn_lists(users, 10)
        one.P, one.Q = two.P, two.Q
        lists1, ids1, sc1 = one._topn_lists(users, 10)
    assert np.array_equal(ids1, ids2) and np.array_equal(sc1, sc2) and lists1 == lists2
    # APR (recommender/advanced/APR.py:113-137) through the same sharded session: trains, stays finite, ranks
    vals = conf_values(tmp_path / "apr", extra={"record": str(log_path), "recommender": "APR", "yue.seed": "77", "num.max.iter": "2",
                                                "num.factors": "64", "item.ranking": "-topN 10", "yue.devices": devs, "yue.sub_epochs": "16",
                                                "batch_size": "512", "APR": "-eps 0.5 -regA 2 -advEpoch 1"})
    random.seed(5)
    np.random.seed(11)
    with redirect_stdout(io.StringIO()):
        y = Yue(Config(values=vals))
        apr = APR(y.config, y.trainingData, y.testData)
        apr.execute()
    assert np.isfinite(apr.P).all() and np.isfinite(apr.Q).all() and np.isfinite(apr.loss)
    assert rec(apr) > 0.5 * rec(ser)


@pytest.mark.gpu
def test_cv_folds_and_progress_hook(tmp_path):
    """SURVEY 8f row 3.  `-cv 3` through the driver (yue.py:72-123): every fold trains and ranks in its own process
    (serially, and under `-p` on device fold % device_count), the fold measures are averaged label by label and the
    k-fold file is written.  `ranking_performance` (IterativeRecommender.py:175-235): top-10 of the first 300 test
    users, with the TRAINING tracks masked, equals Measure on the exact lists of the oracle."""
    from yue_b200 import synth
    from yue_b200.host.driver import Yue
    from yue_b200.host.measure import Measure
    import random
    log_path = tmp_path / "log.txt"
    synth.write_csv_log(str(log_path), 800, 3000, 20000, seed=3)
    out = {}
    for flag in ("", " -p", "arrays"):                   # "arrays": the folds numbered from ONE coded read of the file (ingest.cv_folds)
        extra = {"record": str(log_path), "yue.sgd": "serial", "yue.seed": "5", "num.max.iter": "2"}
        if flag == "arrays":
            extra["yue.ingest"] = "arrays"
        vals = conf_values(tmp_path / ("cv" + flag.strip()), eval_setup="-target track -cv 3" + (flag if flag != "arrays" else ""), extra=extra)
        random.seed(9)
        with redirect_stdout(io.StringIO()):
            res = Yue(Config(values=vals)).execute()
        assert [r.split(":")[0] for r in res[:6]] == ["Top 5\n", "Precision", "Recall", "F1", "MAP", "Coverage"]
        files = os.listdir(tmp_path / ("cv" + flag.strip()))
        assert sum("-3-fold-cv" in f for f in files) == 1
        assert sum("-measure[%d]" % i in f for f in files for i in (1, 2, 3)) == 3
        out[flag] = res
    # same folds (same `random` seed), same sampler seed, serial order: the two schedules give the same averages up to
    # the unseeded factor init in the child processes -- so only the structure and the ranges are compared
    for a, b, c in zip(out[""], out[" -p"], out["arrays"]):
        assert a.split(":")[0] == b.split(":")[0] == c.split(":")[0]
        if ":" in a:
            assert all(0.0 <= float(x.split(":")[1]) <= 1.0 for x in (a, b, c))

    # the progress hook
    vals = conf_values(tmp_path / "hook", extra={"record": str(log_path), "yue.seed": "5", "num.max.iter": "1"})
    random.seed(9)
    np.random.seed(3)
    with redirect_stdout(io.StringIO()):
        y = Yue(Config(values=vals))
        from yue_b200.bpr import BPR
        model = BPR(y.config, y.trainingData, y.testData)
        model.readConfiguration()
        model.initModel()
        model.buildModel()
        got = model.ranking_performance()
    sample = dict(list(model.data.testSet.items())[:300])
    ev_indptr, ev_items, uq_indptr, uq_items = model.data.interaction_arrays()
    uid = np.array([model.data.getId(u, "user") for u in sample], dtype=np.int32)
    ids, _ = topn.topn_exact(model.P, model.Q, uid, 10, uq_indptr, uq_items)
    id2name = model.data.id2name[model.recType]
    rec = {u: [id2name[int(t)] for t in row if t >= 0] for u, row in zip(sample, ids)}
    itemcount = 0
    for k, u in enumerate(model.data.testSet):           # the reference counts one user past the sample (176-181)
        itemcount += len(model.data.testSet[u])
        if k == 300:
            break
    assert got == Measure.rankingMeasure(sample, rec, [10], itemcount)


def test_wrmf_class_host_logic_reproduces_the_reference_class(golden_dir, tmp_path):
    """yue_b200.wrmf.WRMF on the log of the golden run, the same seeded init stream, with the oracle standing in for the
    CUDA sweeps (CPU box): X = P*10 / Y = Q*10, exactly num.max.iter iterations, reg.lambda -u on both sweeps, the loss of
    the user sweep -- the tables equal the output of the REFERENCE's own WRMF class (tests/golden/wrmf_small.npz) bit for
    bit, and predict() its scores."""
    from oracle import wrmf_ref
    from yue_b200.wrmf import WRMF
    g, train, test = golden_split(golden_dir)
    w = np.load(os.path.join(golden_dir, "wrmf_small.npz"))
    vals = conf_values(tmp_path, extra={"recommender": "WRMF", "num.factors": "20", "num.max.iter": "2",
                                        "reg.lambda": "-u 1 -i 0.1 -b 0.2 -s 0.2"})

    class OracleSweeps:
        def __init__(self, model):
            self.m = model
            ev_indptr, ev_items, self.up, self.ui = model.data.interaction_arrays(model.recType)
            self.cnt = wrmf_ref.pair_counts(ev_indptr, ev_items, self.up, self.ui)
            self.tp, self.tu, self.tc = wrmf_ref.transpose(model.m, model.n, self.up, self.ui, self.cnt)
            self.calls = []

        def wrmf_sweep(self, side, reg, alpha=10.0, want_loss=False):
            self.calls.append((side, reg, alpha))
            if side == 0:
                return wrmf_ref.half_sweep(self.m.X, self.m.Y, self.up, self.ui, self.cnt, reg, "f32", want_loss, alpha)
            return wrmf_ref.half_sweep(self.m.Y, self.m.X, self.tp, self.tu, self.tc, reg, "f32", want_loss, alpha)

        def predict(self, u):
            return self.m.Y.dot(self.m.X[u])

    with redirect_stdout(io.StringIO()):
        model = WRMF(Config(values=vals), train, test)
        model.readConfiguration()
        np.random.seed(4321)
        model.initModel()
        assert np.array_equal(model.X, w["X0"]) and np.array_equal(model.Y, w["Y0"])
        oe = OracleSweeps(model)
        model._push_factors = lambda: oe
        model._pull_factors = lambda: None
        model.buildModel()
    assert oe.calls == [(0, 1.0, 10.0), (1, 1.0, 10.0)] * 2
    assert np.array_equal(model.X, w["X"][-1]) and np.array_equal(model.Y, w["Y"][-1])
    assert model.loss == pytest.approx(float(w["loss"][-1]), rel=1e-7)
    id2u = {v: k for k, v in model.data.name2id["user"].items()}
    for u, s in zip(w["score_users"][:5], w["scores"][:5]):
        assert np.allclose(model.predict(id2u[int(u)]), s, rtol=1e-6, atol=1e-7)


@pytest.mark.skipif(not os.path.isdir(REF), reason=NO_REF)
def test_wrmf_dropin_shim_on_top_of_the_reference_tree(golden_dir, tmp_path):
    """dropin/recommender/cf/WRMF.py shadows the reference's module, derives from the REFERENCE's own
    base.IterativeRecommender, and with the oracle in place of the CUDA sweeps reproduces the tables of the reference's
    WRMF class (the golden run) bit for bit."""
    import subprocess
    code = r'''
import io, json, os, sys
import numpy as np
from contextlib import redirect_stdout
sys.path[:0] = [%(dropin)r, %(ref)r, %(root)r]
from tool.config import Config
from recommender.cf.WRMF import WRMF
import base.IterativeRecommender as ref_base
import recommender.cf.WRMF as mod
assert mod.__file__.startswith(%(dropin)r) and WRMF.__mro__[3] is ref_base.IterativeRecommender, WRMF.__mro__
from oracle import wrmf_ref
from yue_b200.host.record import interaction_arrays
g = json.load(open(%(gold)r + "/record_small.json"))
train = [e for e, h in zip(g["events"], g["held"]) if not h]
test = [e for e, h in zip(g["events"], g["held"]) if h]
open(%(tmp)r + "/c.conf", "w").write("\n".join(k + "=" + v for k, v in %(conf)r.items()))
w = np.load(%(gold)r + "/wrmf_small.npz")
with redirect_stdout(io.StringIO()):
    m = WRMF(Config(%(tmp)r + "/c.conf"), train, test)
    m.readConfiguration()
    np.random.seed(4321)
    m.initModel()
    ev_indptr, ev_items, up, ui = interaction_arrays(m.data.name2id, m.data.userRecord, m.recType)
    cnt = wrmf_ref.pair_counts(ev_indptr, ev_items, up, ui)
    tp, tu, tc = wrmf_ref.transpose(m.m, m.n, up, ui, cnt)
    class E:
        def wrmf_sweep(self, side, reg, alpha=10.0, want_loss=False):
            if side == 0: return wrmf_ref.half_sweep(m.X, m.Y, up, ui, cnt, reg, "f32", want_loss, alpha)
            return wrmf_ref.half_sweep(m.Y, m.X, tp, tu, tc, reg, "f32", want_loss, alpha)
    m._push_factors = lambda: E()
    m._pull_factors = lambda: None
    m.buildModel()
assert np.array_equal(m.X, w["X"][-1]) and np.array_equal(m.Y, w["Y"][-1])
print("OK")
''' % dict(dropin=os.path.join(ROOT, "dropin"), ref=REF, root=ROOT, gold=golden_dir, tmp=str(tmp_path),
           conf=conf_values(tmp_path, extra={"recommender": "WRMF", "num.factors": "20", "num.max.iter": "2",
                                             "reg.lambda": "-u 1 -i 0.1 -b 0.2 -s 0.2"}))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]
