"""yue_b200/ingest.py (SURVEY 8f rows 1-2): the log as numbered events without a Python object per event, and the result
lines / measures without a Python loop per item -- against the goldens of the reference's own Record (tests/golden/
record_small.json, produced by oracle/make_golden.py from data/record.py) and against the reference-pinned host classes."""
import io
import json
import os
import random
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import record_ref
from yue_b200 import ingest
from yue_b200.host.config import Config, LineConfig
from yue_b200.host.fileio import DataSplit
from yue_b200.host.measure import Measure

REF = os.environ.get("YUE_REFERENCE", "")          # a checkout of 0411tony/Yue: when set, one more comparison
COLUMNS = {"user": 1, "track": 2, "artist": 3, "time": 0}          # record.setup of config/BPR.conf: -columns user:1,track:2,artist:3,time:0


def _write_csv(path, events):
    with open(path, "w") as f:
        for e in events:
            f.write("%s,%s,%s,%s\n" % (e["time"], e["user"], e["track"], e["artist"]))


def _csr_from_numbered(log):
    """What K0 builds on the device, in numpy: events grouped by user (stable), sorted-unique play rows."""
    tr = log.is_test == 0
    u, it = log.ev_user[tr].astype(np.int64), log.ev_item[tr]
    order = np.argsort(u, kind="stable")
    ev_indptr = np.zeros(log.m + 1, np.int64)
    np.cumsum(np.bincount(u, minlength=log.m), out=ev_indptr[1:])
    key = np.unique(u * log.n + it)
    uq_indptr = np.zeros(log.m + 1, np.int64)
    np.cumsum(np.bincount(key // log.n, minlength=log.m), out=uq_indptr[1:])
    return ev_indptr, it[order].astype(np.int32), uq_indptr, (key % log.n).astype(np.int32)


def test_numbered_events_reproduce_the_reference_records_ids_and_arrays(golden_dir, tmp_path):
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    path = str(tmp_path / "log.txt")
    _write_csv(path, g["events"])
    cols = ingest.read_columns(path, COLUMNS, ",")
    assert list(cols.keys()) == ["user", "track", "artist", "time"] and len(cols["user"]) == len(g["events"])
    assert cols["track"][0] == g["events"][0]["track"] and cols["time"][1] == g["events"][1]["time"]
    held = np.array(g["held"], dtype=bool)
    log = ingest.number_events({k: v[~held] for k, v in cols.items()}, {k: v[held] for k, v in cols.items()}, "track", list(COLUMNS))
    # ids: the reference's Record, key by key (data/record.py:138-146, 182-188)
    for kind in ("user", "track", "artist"):
        assert {name: i for i, name in enumerate(log.names[kind])} == g["name2id"][kind]
    assert log.train_size == g["recordCount"]
    # arrays: the oracle's restatement of BPR.py:32-45 on the reference-shaped dicts
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    test = [e for e, h in zip(g["events"], g["held"]) if h]
    name2id, user_record, test_set = record_ref.preprocess(train, test)
    want = record_ref.interaction_arrays(name2id, user_record)
    for a, b in zip(_csr_from_numbered(log), want):
        assert np.array_equal(a, b)
    # the Record facade
    rec = ingest.ArrayRecord(log)
    assert rec.getSize("user") == len(g["name2id"]["user"]) and rec.getId("u15", "user") == g["name2id"]["user"]["u15"]
    assert rec.id2name["track"][g["name2id"]["track"]["t5"]] == "t5" and len(rec.trainingData) == g["recordCount"]
    # test set: held-out pairs minus training pairs, as a CSR (what K0 returns) -> the dict view equals the reference's
    te = log.is_test == 1
    tr_key = np.unique(log.ev_user[~te].astype(np.int64) * log.n + log.ev_item[~te])
    te_key = np.unique(log.ev_user[te].astype(np.int64) * log.n + log.ev_item[te])
    te_key = te_key[~np.isin(te_key, tr_key)]
    rec.test_indptr = np.zeros(log.m + 1, np.int64)
    np.cumsum(np.bincount(te_key // log.n, minlength=log.m), out=rec.test_indptr[1:])
    rec.test_items = (te_key % log.n).astype(np.int32)
    assert {u: set(d) for u, d in rec.testSet.items()} == {u: set(d) for u, d in g["testSet"].items()}


def test_splits_follow_the_reference(golden_dir, tmp_path):
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    # -ap: one random() per event in file order (tool/dataSplit.py:9-23)
    random.seed(5)
    held = ingest.split_ap(len(g["events"]), 0.2)
    random.seed(5)
    train, test = DataSplit.dataSplit(g["events"], test_ratio=0.2)
    assert [e for e, h in zip(g["events"], held) if not h] == train and int(held.sum()) == len(test)
    # -byTime: the reference's own Record on the first events (golden), ids and per-user training rows
    bt = g["byTime"]
    events = g["events"][:bt["n_events"]]
    path = str(tmp_path / "log.txt")
    _write_csv(path, events)
    ev = LineConfig("-target track -byTime 0.2")
    log = ingest.load_numbered(path, COLUMNS, ",", ev, "track")
    for kind in ("user", "track"):
        assert {name: i for i, name in enumerate(log.names[kind])} == bt["name2id"][kind]
    assert log.train_size == bt["recordCount"]
    ev_indptr, ev_items, _, _ = _csr_from_numbered(log)
    for user, tracks in bt["userRecord"].items():
        u = bt["name2id"]["user"][user]
        assert [log.names["track"][t] for t in ev_items[ev_indptr[u]:ev_indptr[u + 1]]] == tracks


def test_arrow_coded_path_equals_the_object_path(golden_dir, tmp_path):
    """load_numbered's fast path (Arrow CSV reader + dictionary codes, ids re-assigned by integer work only) gives exactly
    the numbered events and name tables of the object path (which the tests above pin to the reference's Record)."""
    pytest.importorskip("pyarrow")
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    path = str(tmp_path / "log.txt")
    _write_csv(path, g["events"])
    assert ingest.read_coded(path, COLUMNS, ",") is not None and ingest.read_coded(path, COLUMNS, "") is None
    for ev in ("-target track -ap 0.2", "-target track"):
        random.seed(5)
        a = ingest.load_numbered(path, COLUMNS, ",", LineConfig(ev), "track")
        random.seed(5)
        cols = ingest.read_columns(path, COLUMNS, ",")
        if "-ap" in ev:
            held = ingest.split_ap(len(cols["user"]), 0.2)
            b = ingest.number_events({k: v[~held] for k, v in cols.items()}, {k: v[held] for k, v in cols.items()}, "track", list(COLUMNS))
        else:
            b = ingest.number_events(cols, None, "track", list(COLUMNS))
        assert np.array_equal(a.ev_user, b.ev_user) and np.array_equal(a.ev_item, b.ev_item) and np.array_equal(a.is_test, b.is_test)
        for kind in ("user", "track", "artist"):
            assert list(a.names[kind]) == list(b.names[kind])


@pytest.mark.parametrize("times", ["golden", "epoch", "ragged"])
def test_coded_by_time_split_equals_the_object_path(golden_dir, tmp_path, times):
    """-byTime (config/BPR.conf's own evaluation.setup): the coded path -- user codes + the time column as one Arrow array,
    numeric sort when every time field is a run of digits of one length, Arrow's string sort otherwise -- gives the training
    and test events of the object path (data/record.py:108-123 restated on Python strings, pinned to the reference above):
    users by first appearance, inside a user by the time STRING, ties in file order."""
    pytest.importorskip("pyarrow")
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    events = [dict(e) for e in g["events"]]
    rng = np.random.default_rng(11)
    if times == "epoch":                                         # ten digits, many ties
        for e in events:
            e["time"] = str(1500000000 + int(rng.integers(0, 400)))
    elif times == "ragged":                                      # strings of different lengths and non-digits: "10" < "9", "2a" > "2"
        pool = ["9", "10", "2", "2a", "100", "x1", "", "07", "7", "1e3"]
        for e in events:
            e["time"] = pool[int(rng.integers(0, len(pool)))]
    path = str(tmp_path / "log.txt")
    _write_csv(path, events)
    ev = LineConfig("-target track -byTime 0.2")
    coded = ingest.read_coded(path, COLUMNS, ",", want_time=True)
    assert coded is not None and len(coded["time"]) == len(events)
    a = ingest.load_numbered(path, COLUMNS, ",", ev, "track")
    cols = ingest.read_columns(path, COLUMNS, ",")
    tr, te = ingest.by_time(cols, 0.2)
    tr2, te2 = ingest.by_time_coded(coded["user"][0], coded["time"], 0.2)
    assert np.array_equal(tr, tr2) and np.array_equal(te, te2)
    b = ingest.number_events({k: v[tr] for k, v in cols.items()}, {k: v[te] for k, v in cols.items()}, "track", list(COLUMNS))
    assert np.array_equal(a.ev_user, b.ev_user) and np.array_equal(a.ev_item, b.ev_item) and np.array_equal(a.is_test, b.is_test)
    for kind in ("user", "track", "artist"):
        assert list(a.names[kind]) == list(b.names[kind])
    # the position of every numbered event in the file (LightGCN's batches walk the training events in file order)
    assert np.array_equal(a.file_pos, np.concatenate([tr, te])) and sorted(a.file_pos.tolist()) == list(range(len(events)))
    names = np.asarray(a.names["user"], dtype=object)
    assert [events[p]["user"] for p in a.file_pos[:50].tolist()] == names[a.ev_user[:50]].tolist()


def test_cv_folds_equal_the_reference_split_numbered_fold_by_fold(golden_dir, tmp_path):
    """-cv k: tool/dataSplit.py:26-38 holds out the events at positions i modulo k; every fold is numbered like the Record the
    reference builds from the two lists.  cv_folds (one read of the file, coded columns) against crossValidation + the object
    path; k outside 2..10 means 3 (dataSplit.py:27-28)."""
    pytest.importorskip("pyarrow")
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    events = g["events"][:1500]
    path = str(tmp_path / "log.txt")
    _write_csv(path, events)
    cols = ingest.read_columns(path, COLUMNS, ",")
    for k in (4, 1):
        kk = 3 if k <= 1 else k
        folds = list(ingest.cv_folds(path, COLUMNS, ",", k, "track"))
        assert len(folds) == kk
        for i, a in enumerate(folds):
            held = np.arange(len(events)) % kk == i
            b = ingest.number_events({c: v[~held] for c, v in cols.items()}, {c: v[held] for c, v in cols.items()}, "track", list(COLUMNS))
            assert np.array_equal(a.ev_user, b.ev_user) and np.array_equal(a.ev_item, b.ev_item) and np.array_equal(a.is_test, b.is_test)
            assert list(a.names["user"]) == list(b.names["user"]) and list(a.names["track"]) == list(b.names["track"])
            assert int(a.is_test.sum()) == int(held.sum())


@pytest.mark.parametrize("ev", ["-target track -ap 0.2 -cold 3", "-target track -ap 0.2 -sample", "-target track -ap 0.2 -cold 5 -sample"])
def test_cold_and_sample_edit_the_test_csr_like_the_dict_form(golden_dir, tmp_path, ev):
    """base/recommender.py:22-49 (-cold t, -sample) on the CSR form of the test set (ingest.filter_test_rows) against the
    dict form the Recommender base class edits -- and, given a checkout of the reference, against its own base class."""
    from yue_b200.host.recommender import Recommender
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    test = [e for e, h in zip(g["events"], g["held"]) if h]
    vals = {"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,", "recommender": "BPR",
            "evaluation.setup": ev, "item.ranking": "-topN 5,10", "num.factors": "8", "num.max.iter": "1",
            "learnRate": "-init 0.02 -max 0.1", "reg.lambda": "-u 0.01 -i 0.01 -b 0.01 -s 0.2", "output.setup": "off"}
    with redirect_stdout(io.StringIO()):
        ref = Recommender(Config(values=vals), train, test)
    want = {u: sorted(t) for u, t in ref.data.testSet.items()}
    if os.path.isdir(REF):                         # the reference's own base class says the same
        import subprocess
        import sys
        code = ("import sys, json, io\nfrom contextlib import redirect_stdout\nsys.path.insert(0, %r)\n"
                "from tool.config import Config\nfrom base.recommender import Recommender\n"
                "g = json.load(open(%r))\ntrain = [e for e, h in zip(g['events'], g['held']) if not h]\n"
                "test = [e for e, h in zip(g['events'], g['held']) if h]\nopen(%r, 'w').write(%r)\n"
                "with redirect_stdout(io.StringIO()):\n    r = Recommender(Config(%r), train, test)\n"
                "print(json.dumps({u: sorted(t) for u, t in r.data.testSet.items()}))\n"
                % (REF, os.path.join(golden_dir, "record_small.json"), str(tmp_path / "c.conf"),
                   "\n".join(k + "=" + v for k, v in vals.items()), str(tmp_path / "c.conf")))
        res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
        assert res.returncode == 0, res.stderr
        assert json.loads(res.stdout.strip().splitlines()[-1]) == want
    # the array form: numbered events -> the test CSR K0 would build (unique held-out pairs minus training pairs) -> the edits
    cols = {k: np.array([e[k] for e in train + test], dtype=object) for k in ("user", "track", "artist")}
    nt = len(train)
    log = ingest.number_events({k: v[:nt] for k, v in cols.items()}, {k: v[nt:] for k, v in cols.items()}, "track", ["user", "track", "artist"])
    tr = log.is_test == 0
    tr_key = np.unique(log.ev_user[tr].astype(np.int64) * log.n + log.ev_item[tr])
    te_key = np.unique(log.ev_user[~tr].astype(np.int64) * log.n + log.ev_item[~tr])
    te_key = te_key[~np.isin(te_key, tr_key)]
    indptr = np.zeros(log.m + 1, np.int64)
    np.cumsum(np.bincount(te_key // log.n, minlength=log.m), out=indptr[1:])
    items = (te_key % log.n).astype(np.int32)
    line = LineConfig(ev)
    ip, it = ingest.filter_test_rows(log, indptr, items, cold=int(line["-cold"]) if line.contains("-cold") else None, sample=line.contains("-sample"))
    un, tn = log.names["user"], log.names["track"]
    got = {un[u]: sorted(tn[t] for t in it[ip[u]:ip[u + 1]]) for u in np.flatnonzero(np.diff(ip) > 0)}
    assert got == want and 0 < len(got) < len(np.flatnonzero(np.diff(indptr) > 0)) + (0 if "-sample" in ev else 1)


def test_coded_test_set_file_equals_the_object_path(golden_dir, tmp_path):
    """-testSet file: the log and the test file are read by the coded reader into ONE names table per column, then numbered
    like the object path (training events first, the test file's events extend the maps: data/record.py:138-146, 182-188)."""
    pytest.importorskip("pyarrow")
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    train = [e for e, h in zip(g["events"], g["held"]) if not h]
    test = [e for e, h in zip(g["events"], g["held"]) if h]
    p_train, p_test = str(tmp_path / "train.txt"), str(tmp_path / "test.txt")
    _write_csv(p_train, train)
    _write_csv(p_test, test)
    ev = LineConfig("-target track -testSet " + p_test)
    a = ingest.load_numbered(p_train, COLUMNS, ",", ev, "track")
    b = ingest.number_events(ingest.read_columns(p_train, COLUMNS, ","), ingest.read_columns(p_test, COLUMNS, ","), "track", list(COLUMNS))
    both = ingest.read_coded([p_train, p_test], COLUMNS, ",")
    assert len(both) == 2 and both[0]["user"][1] is both[1]["user"][1] and len(both[1]["user"][0]) == len(test)
    assert np.array_equal(a.ev_user, b.ev_user) and np.array_equal(a.ev_item, b.ev_item) and np.array_equal(a.is_test, b.is_test)
    for kind in ("user", "track", "artist"):
        assert list(a.names[kind]) == list(b.names[kind])


def test_result_lines_and_measures_match_the_loops():
    rng = np.random.default_rng(3)
    m, n, N = 300, 500, 10
    users = np.sort(rng.choice(m, 200, replace=False)).astype(np.int32)
    ids = np.stack([rng.choice(n, N, replace=False) for _ in users]).astype(np.int32)
    ids[5, 7:] = -1                                           # a short list (fewer than N unmasked tracks)
    deg = np.zeros(m, np.int64)
    deg[users] = rng.integers(1, 8, len(users))
    test_indptr = np.zeros(m + 1, np.int64)
    np.cumsum(deg, out=test_indptr[1:])
    test_items = np.concatenate([np.sort(rng.choice(n, d, replace=False)) for d in deg]).astype(np.int32)
    for b, u in enumerate(users[:50]):                        # plant hits (exact top-N lists never repeat a track)
        t = test_items[test_indptr[u]]
        if t not in ids[b]:
            ids[b, rng.integers(0, 5)] = t
    un = np.array(["u%d" % i for i in range(m)], dtype=object)
    tn = np.array(["t%d" % i for i in range(n)], dtype=object)
    hits = ingest.hit_mask(users, ids, n, test_indptr, test_items)
    origin = {un[u]: {tn[t]: 1 for t in test_items[test_indptr[u]:test_indptr[u + 1]]} for u in users}
    rec = {un[u]: [tn[t] for t in row if t >= 0] for u, row in zip(users, ids)}
    want_hits = np.array([[t >= 0 and tn[t] in origin[un[u]] for t in row] for u, row in zip(users, ids)])
    assert np.array_equal(hits, want_hits) and hits.sum() >= 40
    # IterativeRecommender.py:145-155
    want_lines = [un[u] + ":" + "".join(item + ("*" if item in origin[un[u]] else "") for item in rec[un[u]]) + "\n" for u in users]
    assert ingest.result_lines(un[users], tn, ids, hits) == want_lines
    # the same lines from the library's host code (yue_result_lines, what the class API uses): one string, all cores
    ub, uo = ingest.name_blob(un[users])
    tb, to = ingest.name_blob(tn)
    assert ingest.result_text(ub, uo, tb, to, ids, hits) == "".join(want_lines)
    big = np.tile(ids, (30, 1))                               # > 4096 rows: the multi-threaded path
    bh = np.tile(hits, (30, 1))
    bub, buo = ingest.name_blob(np.tile(un[users], 30))
    assert ingest.result_text(bub, buo, tb, to, big, bh) == "".join(want_lines * 30)
    bad = ids.copy(); bad[3, 2] = n                           # an id outside the catalog is refused, not read
    with pytest.raises(Exception):
        ingest.result_text(ub, uo, tb, to, bad, hits)
    # evaluation/measure.py:16-41 (+ NDCG)
    with redirect_stdout(io.StringIO()):
        want = Measure.rankingMeasure(origin, rec, [5, 10], n)
        got, ndcg = ingest.ranking_measure(ids, hits, np.diff(test_indptr)[users], [5, 10], n)
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert a.split(":")[0] == b.split(":")[0]
        if ":" in a:
            assert float(a.split(":")[1]) == pytest.approx(float(b.split(":")[1]), rel=1e-12, abs=1e-15)
    for k in (5, 10):
        assert ndcg[k] == pytest.approx(Measure.NDCG(origin, rec, k), rel=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("ev", ["-target track -ap 0.2", "-target track -byTime 0.2 -sample"])
def test_class_api_with_array_ingest_equals_the_dict_path(tmp_path, ev):
    """Yue -> BPR.execute() with yue.ingest=arrays (C parser, column-wise ids, K0 on the device, array result lines) against
    the default path (lists of dicts, Record, Python loops): same split (same `random` seed; or config/WRMF.conf's -byTime
    with -sample), same initial tables, same sampler seed, serial order -> the same tables bit for bit, the same measures
    and the same result lines."""
    from yue_b200 import synth
    from yue_b200.bpr import BPR
    from yue_b200.host.driver import Yue
    log_path = tmp_path / "log.txt"
    synth.write_csv_log(str(log_path), 1500, 4000, 60000, seed=20260101)
    out = {}
    for name in ("dicts", "arrays"):
        vals = {"record": str(log_path), "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,", "recommender": "BPR",
                "evaluation.setup": ev, "item.ranking": "-topN 5,10", "num.factors": "10", "num.max.iter": "2",
                "learnRate": "-init 0.02 -max 1", "reg.lambda": "-u 0.01 -i 0.01 -b 0.2 -s 0.2", "output.setup": "on -dir %s/" % (tmp_path / name),
                "yue.sgd": "serial", "yue.seed": "77"}
        if name == "arrays":
            vals["yue.ingest"] = "arrays"
        random.seed(5)
        np.random.seed(11)
        with redirect_stdout(io.StringIO()):
            y = Yue(Config(values=vals))
            model = BPR(y.config, y.trainingData, y.testData)
            measure = model.execute()
        files = sorted(os.listdir(tmp_path / name))
        top = [f for f in files if "-top-" in f][0]
        out[name] = (model, measure, open(tmp_path / name / top).read().splitlines())
    (md, meas_d, lines_d), (ma, meas_a, lines_a) = out["dicts"], out["arrays"]
    assert ma.m == md.m and ma.n == md.n and np.array_equal(ma.P, md.P) and np.array_equal(ma.Q, md.Q)
    assert len(meas_a) == len(meas_d)
    for a, b in zip(meas_a, meas_d):
        assert a.split(":")[0] == b.split(":")[0]
        if ":" in a:
            assert float(a.split(":")[1]) == pytest.approx(float(b.split(":")[1]), rel=1e-12, abs=1e-15)
    # the dict path lists the test users in the order of the test events, the array path in id order: same set of lines
    assert lines_a[0] == lines_d[0] and sorted(lines_a[1:]) == sorted(lines_d[1:])


def test_global_randoms_is_the_random_module_stream_bit_for_bit():
    """ingest.global_randoms(n) == [random.random() for _ in range(n)] on the SAME global generator, and the generator
    continues where the loop would have left it (tool/dataSplit.py:15 draws from it, and so does whatever runs next)."""
    import random
    from yue_b200 import ingest
    for seed in (1, 20260101):
        for n in (0, 1, 311, 312, 313, 50001):                  # around the 624-word refill of the twister
            random.seed(seed)
            ref = [random.random() for _ in range(n)]
            after = (random.random(), random.randint(0, 10 ** 9), random.getrandbits(63))
            random.seed(seed)
            got = ingest.global_randoms(n)
            assert got.dtype == np.float64 and np.array_equal(got, np.array(ref, dtype=np.float64))
            assert (random.random(), random.randint(0, 10 ** 9), random.getrandbits(63)) == after
    random.seed(7)
    held = ingest.split_ap(1000, 0.2)
    random.seed(7)
    assert held.tolist() == [random.random() < 0.2 for _ in range(1000)]


def test_read_coded_blocks_merge_to_the_same_numbering(tmp_path):
    """A file larger than the reader's block: the per-block dictionaries are merged and number_coded assigns the ids of
    the one-pass dict reader (first appearance over the training events, then the test events)."""
    from yue_b200 import ingest
    rng = np.random.default_rng(4)
    n = 700_000                                                  # ~ 20 MB of text: three 8 MB blocks
    users = rng.zipf(1.3, n) % 50_000
    tracks = rng.zipf(1.2, n) % 30_000
    path = os.path.join(str(tmp_path), "log.csv")
    with open(path, "w") as f:
        f.write("".join("%d,user_%d,track_%d,a%d\n" % (1500000000 + k, u, t, t % 97) for k, (u, t) in enumerate(zip(users, tracks))))
    assert os.path.getsize(path) > (16 << 20)
    cols = dict([('user', 1), ('track', 2), ('artist', 3), ('time', 0)])
    coded = ingest.read_coded(path, cols, ',')
    log = ingest.number_coded(coded, None, 'track', list(cols))
    first_u, first_t = {}, {}
    for u, t in zip(users.tolist(), tracks.tolist()):
        first_u.setdefault(u, len(first_u))
        first_t.setdefault(t, len(first_t))
    assert log.m == len(first_u) and log.n == len(first_t)
    assert np.array_equal(log.ev_user, np.array([first_u[u] for u in users.tolist()], dtype=np.int32))
    assert np.array_equal(log.ev_item, np.array([first_t[t] for t in tracks.tolist()], dtype=np.int32))
    assert log.names['user'][log.ev_user[12345]] == "user_%d" % users[12345]
