"""Host-side mirror of the reference interface (yue_b200/host) against golden outputs of the
reference's own modules (tests/golden, made by oracle/make_golden.py).  CPU only."""
import io
import json
import os
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import record_ref
from yue_b200.host.config import Config, LineConfig
from yue_b200.host.fileio import DataSplit, FileIO
from yue_b200.host.measure import Measure
from yue_b200.host.record import Record


@pytest.fixture(scope="module")
def gcfg(golden_dir):
    return json.load(open(os.path.join(golden_dir, "config_cases.json")))


@pytest.fixture(scope="module")
def grec(golden_dir):
    return json.load(open(os.path.join(golden_dir, "record_small.json")))


def base_conf(eval_setup="-target track -ap 0.2"):
    return Config(values={"record": "./dataset/log.txt",
                          "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
                          "recommender": "BPR", "evaluation.setup": eval_setup,
                          "item.ranking": "-topN 5,10", "num.factors": "10", "num.max.iter": "3",
                          "learnRate": "-init 0.02 -max 1", "reg.lambda": "-u 0.01 -i 0.01 -b 0.2 -s 0.2",
                          "output.setup": "off -dir ./results/"})


def test_lineconfig_matches_reference(gcfg):
    for case in gcfg["line_cases"]:
        lc = LineConfig(case["line"])
        assert lc.options == case["options"], case["line"]
        assert lc.isMainOn() == case["main"]


def test_config_file_matches_reference(gcfg, tmp_path):
    p = tmp_path / "c.conf"
    p.write_text(gcfg["conf_text"])
    with redirect_stdout(io.StringIO()) as out:
        cfg = Config(str(p))
    assert cfg.config == gcfg["conf"]
    assert "not in the correct format" in out.getvalue()
    with pytest.raises(IOError):
        with redirect_stdout(io.StringIO()):
            Config(str(tmp_path / "missing.conf"))


def test_invalid_key_exits_like_reference():
    with redirect_stdout(io.StringIO()) as out:
        with pytest.raises(SystemExit) as e:
            LineConfig("-a 1")["-b"]
    assert e.value.code == -1 and "parameter -b is invalid!" in out.getvalue()


def test_record_matches_reference(grec):
    train = [e for e, h in zip(grec["events"], grec["held"]) if not h]
    test = [e for e, h in zip(grec["events"], grec["held"]) if h]
    rec = Record(base_conf(), train, test)
    assert {k: dict(v) for k, v in rec.name2id.items()} == grec["name2id"]
    assert list(rec.userRecord.keys()) == grec["userRecord_order"]
    assert [len(v) for v in rec.userRecord.values()] == grec["userRecord_len"]
    assert list(rec.testSet.keys()) == grec["testSet_order"]
    assert {u: dict(d) for u, d in rec.testSet.items()} == grec["testSet"]
    assert rec.recordCount == grec["recordCount"]
    for kind in rec.name2id:
        assert all(rec.id2name[kind][i] == name for name, i in rec.name2id[kind].items())
    # array form == the oracle's
    got = rec.interaction_arrays()
    ref = record_ref.interaction_arrays(grec["name2id"], rec.userRecord)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)


def test_record_bytime_matches_reference(grec):
    bt = grec["byTime"]
    rec = Record(base_conf("-target track -byTime 0.2"), grec["events"][:bt["n_events"]], [])
    assert {k: dict(v) for k, v in rec.name2id.items()} == bt["name2id"]
    assert {u: [e["track"] for e in v] for u, v in rec.userRecord.items()} == bt["userRecord"]
    assert list(rec.testSet.keys()) == bt["testSet_order"]
    assert {u: dict(d) for u, d in rec.testSet.items()} == bt["testSet"]
    assert rec.recordCount == bt["recordCount"]


def test_measure_matches_reference(golden_dir, grec):
    e = np.load(os.path.join(golden_dir, "eval_small.npz"))
    mj = json.load(open(os.path.join(golden_dir, "measure_small.json")))
    i2t = {v: k for k, v in grec["name2id"]["track"].items()}
    i2u = {v: k for k, v in grec["name2id"]["user"].items()}
    users = [i2u[int(u)] for u in e["test_users"]]
    origin = {u: grec["testSet"][u] for u in users}
    with redirect_stdout(io.StringIO()):
        exact = Measure.rankingMeasure(origin, {u: [i2t[t] for t in row] for u, row in zip(users, mj["exact_ids"])},
                                       [5, 10], mj["item_count"])
        quirk = Measure.rankingMeasure(origin, {u: [i2t[int(t)] for t in row] for u, row in zip(users, e["quirk_ids"])},
                                       [5, 10], mj["item_count"])
    assert exact == mj["measure_exact"] and quirk == mj["measure_quirk"]


def test_loader_and_splitters(tmp_path):
    p = tmp_path / "log.txt"
    p.write_text("10,u1,t1,a1\n11,u2,t2,a1\n12,u1,t3,a2\n")
    with redirect_stdout(io.StringIO()):
        data = FileIO.loadDataSet(str(p), {"user": 1, "track": 2, "artist": 3, "time": 0}, delim=",")
    assert data[2] == {"user": "u1", "track": "t3", "artist": "a2", "time": "12"}
    assert list(data[0].keys()) == ["user", "track", "artist", "time"]
    folds = list(DataSplit.crossValidation(list(range(10)), 5))
    assert len(folds) == 5 and folds[1][1] == [1, 6] and len(folds[0][0]) == 8
    tr, te = DataSplit.dataSplit(list(range(1000)), 0.2)
    assert len(tr) + len(te) == 1000 and 120 < len(te) < 280


def test_bench_clock_sampler_windows_on_the_timed_region():
    """bench.py's clock sampler: lines that arrive inside the timed region are the ones reported; a region shorter than a
    sampling period falls back to everything since the start and says so; throttle reasons are collected by name."""
    import importlib.util
    import os
    import time
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_for_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class FakeProc(object):
        def terminate(self):
            pass

    class FakeThread(object):
        def join(self, timeout=None):
            pass

    def sampler(rows, mark_at):
        c = bench.ClockSampler(0)
        c.proc, c.thread = FakeProc(), FakeThread()
        now = time.monotonic()
        c.rows = [(now + dt, r) for dt, r in rows]
        c.t_mark = now + mark_at
        return c

    idle = ["0", "210", "1965", "140", "0x0", "Not Active", "Not Active", "Not Active", "Not Active"]
    busy = ["0", "1965", "1965", "900", "0x4", "Not Active", "Not Active", "Not Active", "Active"]
    out = sampler([(-1.0, idle), (-0.5, idle), (-0.02, busy), (-0.01, busy)], mark_at=-0.05).stop()
    assert out["samples"] == 2 and out["sm_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"] and out["window"] == "timed region"
    out = sampler([(-1.0, idle), (-0.5, busy)], mark_at=-0.05).stop()
    assert out["samples"] == 2 and out["window"].startswith("warm-up + timed region")
    assert bench.ClockSampler(0).stop()["reasons"] == ["nvidia-smi unavailable"]


def test_bench_dump_tables_keeps_small_tables_and_samples_large_ones_by_a_fixed_seed(tmp_path):
    """bench.py --dump-outputs: float32 .npy per table, a table within the budget whole, a larger one as the same sorted
    sample of its rows on every call, and both files together within 2 x the per-table budget."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_for_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    bench.DUMP_TABLE_BYTES = 64 * 4 * 1000                       # 1000 rows of d = 64
    P = np.arange(5000 * 64, dtype=np.float64).reshape(5000, 64)
    Q = np.random.default_rng(1).random((700, 64), dtype=np.float32)
    got = []
    for run in ("a", "b"):
        bench.dump_tables(str(tmp_path / run), P, Q)
        got.append({n: np.load(str(tmp_path / run / (n + ".npy"))) for n in ("P", "Q")})
    p, q = got[0]["P"], got[0]["Q"]
    assert p.dtype == np.float32 and q.dtype == np.float32 and p.shape == (1000, 64)
    rows = p[:, 0].astype(np.int64) // 64
    assert np.all(np.diff(rows) > 0) and np.array_equal(p, P[rows].astype(np.float32))
    assert np.array_equal(q, Q)
    assert np.array_equal(got[1]["P"], p) and np.array_equal(got[1]["Q"], q)
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))) <= 2 * bench.DUMP_TABLE_BYTES + 512
