"""CUNE's two-level BPR (SURVEY 8f row 4): host logic of yue_b200/cune.py on CPU with the oracle standing in for the
CUDA epoch, and the kernel (csrc/cune_sgd.cuh through yue_cune_epoch) against the golden run of the reference's own loop
text (tests/golden/cune_small.npz, oracle/make_golden_cune.py)."""
import io
import json
import os
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import cune_ref, philox, record_ref
from yue_b200.host.config import Config

REF = os.environ.get("YUE_REFERENCE", "")          # a checkout of 0411tony/Yue; the shim test skips without one


def _golden_slice(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "record_small.json")))
    keep = set('u%d' % x for x in range(60))                  # the slice make_golden_cune.py trains on
    train = [e for e, h in zip(g["events"], g["held"]) if not h and e['user'] in keep]
    test = [e for e, h in zip(g["events"], g["held"]) if h and e['user'] in keep]
    return train, test


def _conf(out_dir):
    return {"record": "./dataset/log.txt", "record.setup": "-columns user:1,track:2,artist:3,time:0 -delim ,",
            "recommender": "CUNE", "evaluation.setup": "-target track -ap 0.2", "item.ranking": "-topN 5,10",
            "num.factors": "12", "num.max.iter": "2", "CUNE": "-T 20 -L 10 -l 20 -w 5 -k 50 -s 2 -ep 10",
            "learnRate": "-init 0.02 -max 0.1", "reg.lambda": "-u 0.01 -i 0.01 -b 0.01 -s 0.2",
            "output.setup": "on -dir %s/" % out_dir, "yue.sgd": "serial", "yue.seed": "20260105"}


def test_implicit_positive_lists_follow_the_reference_statement():
    """CUNE.py:111-113: per similar user, its tracks minus the user's own; contributions concatenated, duplicates kept."""
    from yue_b200.cune import implicit_positive_lists
    rng = np.random.default_rng(5)
    m, n = 30, 40
    rows = [np.unique(rng.integers(0, n, rng.integers(1, 12))) for _ in range(m)]
    uq_indptr = np.zeros(m + 1, np.int64)
    np.cumsum([len(r) for r in rows], out=uq_indptr[1:])
    uq_items = np.concatenate(rows).astype(np.int32)
    top = {u: [int(f) for f in rng.choice([x for x in range(m) if x != u], 3, replace=False)] for u in range(m) if u % 4}
    indptr, items = implicit_positive_lists(m, uq_indptr, uq_items, top)
    for u in range(m):
        want = []
        for f in top.get(u, ()):
            want += sorted(set(rows[f].tolist()).difference(rows[u].tolist()))
        assert items[indptr[u]:indptr[u + 1]].tolist() == want
        assert not set(want) & set(rows[u].tolist())
    assert indptr[-1] == len(items) and (np.diff(indptr)[::4] == 0).all()


def test_cune_class_host_logic_reproduces_the_reference_loop(golden_dir, tmp_path):
    """yue_b200.cune.CUNE on the log slice of the golden run, the same seeded init, similar users supplied (the embedding
    stage needs gensim), the oracle standing in for yue_cune_epoch: the implicit-positive lists equal the golden run's and
    the tables after two iterations equal the output of the REFERENCE's loop text bit for bit."""
    from yue_b200.cune import CUNE
    from yue_b200.engine import MODE_SERIAL
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    train, test = _golden_slice(golden_dir)

    class OracleEpochs:
        def __init__(self, model):
            self.m = model
            self.arr = model.data.interaction_arrays(model.recType)
            self.calls = []

        def get_interactions(self):
            return self.arr

        def cune_set_implicit(self, ip_indptr, ip_items):
            self.ip = (np.asarray(ip_indptr), np.asarray(ip_items))

        def cune_epoch(self, lr, regU, regI, s, seed, epoch, mode):
            self.calls.append((lr, regU, regI, s, seed, epoch, mode))
            ev_indptr, ev_items, uq_indptr, uq_items = self.arr
            ev_user = record_ref.ev_users(ev_indptr)
            kp = [cune_ref.sample_implicit(seed, epoch, nn, ev_user, self.ip[0]) for nn in range(3)]
            neg = [philox.sample_negatives(seed, epoch, ev_user, self.m.n, uq_indptr, uq_items, slot=nn) for nn in range(3)]
            return cune_ref.epoch(self.m.P, self.m.Q, ev_indptr, ev_items, self.ip[0], self.ip[1], kp, neg, lr, regU, regI, s)

    with redirect_stdout(io.StringIO()):
        model = CUNE(Config(values=_conf(tmp_path)), train, test)
        model.readConfiguration()
        np.random.seed(99)
        model.initModel()
        assert (model.walkCount, model.walkLength, model.walkDim, model.winSize, model.topK, model.s, model.epoch) == \
            (20, 10, 20, 5, 50, 2.0, 10)
        assert np.array_equal(model.P, g["P0"]) and np.array_equal(model.Q, g["Q0"])
        # the similar users of the golden run (make_golden_cune.py): two fixed others, none for every fifth user
        u2i = model.data.name2id['user']
        by_id = {v: k for k, v in u2i.items()}
        m = len(u2i)
        model.topKSim = {}
        for name, uid in u2i.items():
            if name in model.data.userRecord and uid % 5 != 0:
                fr = [by_id[f] for f in ((uid * 7 + 3) % m, (uid * 11 + 5) % m)]
                model.topKSim[name] = [(f, 1.0) for f in fr if f in model.data.userRecord and f != name]
        oe = OracleEpochs(model)
        model._push_factors = lambda: oe
        model._pull_factors = lambda: None
        model.isConverged = lambda it: False                   # the golden run does exactly num.max.iter iterations
        model.buildModel()
    assert np.array_equal(oe.ip[0], g["ip_indptr"]) and np.array_equal(oe.ip[1], g["ip_items"])
    assert [c[5:] for c in oe.calls] == [(0, MODE_SERIAL), (1, MODE_SERIAL)] and oe.calls[0][:5] == (0.02, 0.01, 0.01, 2.0, 20260105)
    assert np.array_equal(model.P, g["P"][-1]) and np.array_equal(model.Q, g["Q"][-1])
    assert float(model.loss) == pytest.approx(float(g["loss"][-1]), rel=1e-9)


# ---- GPU: K8 against the golden run ------------------------------------------------------------------------------------
# Round 2, first hardware run (profiles/cune_r2.md): the serial kernel reproduced the reference loop at every width on the
# first try; the Hogwild kernel with EVERY user of these tiny logs in flight at once (64 warps, 60 users) landed a whole
# P[u] norm away from the serial tables -- not a fault of the kernel (one warp taking the same work items in order gives
# the serial tables to 1e-6) but a schedule that is not a window sliding over the reference's user stream.  The C-ABI
# now gives a small log few warps, like K2; the tests pin the Hogwild text with ONE warp (deterministic: the serial order
# through the atomic / fast-math path, shared users published and re-read) and check many warps for sanity only.
import contextlib


@contextlib.contextmanager
def _env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    try:
        for k, v in kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = str(v)
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _row_err(a, b):
    return float((np.linalg.norm(a.astype(np.float64) - b, axis=1) / np.maximum(np.linalg.norm(b.astype(np.float64), axis=1), 1e-12)).max())


def _load(engine, g):
    m, n = g["P0"].shape[0], g["Q0"].shape[0]
    engine.set_interactions(m, n, g["ev_indptr"], g["ev_items"], g["uq_indptr"], g["uq_items"])
    engine.set_factors(g["P0"].copy(), g["Q0"].copy())
    engine.cune_set_implicit(g["ip_indptr"], g["ip_items"])
    return m, n


@pytest.mark.gpu
def test_cune_serial_epochs_match_the_reference_loop(engine, golden_dir):
    """Two serial-order iterations from the golden start: tables within 1e-5 relative of the reference loop's float32
    tables (north_star's serial-order tolerance; the float32 dots sum in a different order), loss within 1e-4 (the
    reference's loss turns float32 after the first user under numpy 2, the kernel's is float64)."""
    from yue_b200.engine import MODE_SERIAL
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    _load(engine, g)
    for it in range(len(g["loss"])):
        loss = engine.cune_epoch(float(g["lr"]), float(g["regU"]), float(g["regI"]), float(g["s"]), int(g["seed"]), it, MODE_SERIAL)
        P, Q = engine.get_factors()
        for a, b in ((P, g["P"][it]), (Q, g["Q"][it])):
            d = np.linalg.norm(a.astype(np.float64) - b, axis=1) / np.maximum(np.linalg.norm(b.astype(np.float64), axis=1), 1e-12)
            assert d.max() < 1e-5
        assert loss == pytest.approx(float(g["loss"][it]), rel=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [None, 32])
def test_cune_hogwild_kernel_in_stream_order_reproduces_the_serial_tables(engine, golden_dir, chunk):
    """The Hogwild kernel on the golden log.  3 347 events are far below one warp's minimum share, so the C-ABI launches
    ONE warp: the work items in stream order through the atomic path (float adds, fast sigmoid, fused multiply-adds).
    Same draws, same order -> the serial tables to 1e-4 and the -log part of the loss to 1e-3.  With 32-event items the
    heavy users (up to 494 events) are SHARED items: P[u] published as adds and re-read every 8 events."""
    from yue_b200.engine import MODE_HOGWILD
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    lr, s_, seed = float(g["lr"]), float(g["s"]), int(g["seed"])
    for regU, regI in ((0.0, 0.0), (float(g["regU"]), float(g["regI"]))):
        _load(engine, g)
        with _env(YUE_CUNE_CHUNK=chunk, YUE_CUNE_WARPS=None):
            loss = engine.cune_epoch(lr, regU, regI, s_, seed, 0, MODE_HOGWILD)
        P, Q = engine.get_factors()
        Pr, Qr = g["P0"].copy(), g["Q0"].copy()
        ref = cune_ref.epoch(Pr, Qr, g["ev_indptr"], g["ev_items"], g["ip_indptr"], g["ip_items"], g["kpos"][0], g["neg"][0],
                             lr, regU, regI, s_)
        assert _row_err(P, Pr) < 1e-4 and _row_err(Q, Qr) < 1e-4
        if regU == 0.0:                                         # with a regulariser the two modes define the loss differently
            assert loss == pytest.approx(float(ref), rel=1e-3)


@pytest.mark.gpu
def test_cune_hogwild_with_every_user_in_flight_stays_sane(engine, golden_dir):
    """64 warps forced onto the 60 users of the golden log: NOT the serial order (every user trains against tables that
    all the others are changing), so only sanity is asserted -- finite tables, no lost padding, the epoch loss within 15 %
    of the serial one (measured on a B200: +2.9 % whole users, +5.4 % with 32-event shared items)."""
    from yue_b200.engine import MODE_HOGWILD
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    Pr, Qr = g["P0"].copy(), g["Q0"].copy()
    ref = cune_ref.epoch(Pr, Qr, g["ev_indptr"], g["ev_items"], g["ip_indptr"], g["ip_items"], g["kpos"][0], g["neg"][0],
                         float(g["lr"]), 0.0, 0.0, float(g["s"]))
    for chunk in (None, 32):
        _load(engine, g)
        with _env(YUE_CUNE_CHUNK=chunk, YUE_CUNE_WARPS=64):
            loss = engine.cune_epoch(float(g["lr"]), 0.0, 0.0, float(g["s"]), int(g["seed"]), 0, MODE_HOGWILD)
        P, Q = engine.get_factors()
        assert np.isfinite(P).all() and np.isfinite(Q).all()
        assert np.abs(P).max() < 2.0 and np.abs(Q).max() < 2.0
        assert loss == pytest.approx(float(ref), rel=0.15)


@pytest.mark.gpu
def test_cune_refusals(engine, golden_dir):
    from yue_b200.engine import MODE_SERIAL, YueError
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    m, n = g["P0"].shape[0], g["Q0"].shape[0]
    engine.set_interactions(m, n, g["ev_indptr"], g["ev_items"], g["uq_indptr"], g["uq_items"])
    engine.set_factors(g["P0"].copy(), g["Q0"].copy())
    with pytest.raises(YueError):                               # no implicit positives yet
        engine.cune_epoch(0.02, 0.01, 0.01, 2.0, 1, 0, MODE_SERIAL)
    bad = g["ip_items"].copy()
    u = int(np.nonzero(np.diff(g["ip_indptr"]) > 0)[0][0])
    bad[g["ip_indptr"][u]] = g["uq_items"][g["uq_indptr"][u]]  # a track the user has played
    with pytest.raises(YueError):
        engine.cune_set_implicit(g["ip_indptr"], bad)
    engine.cune_set_implicit(g["ip_indptr"], g["ip_items"])
    with pytest.raises(YueError):                               # s must be positive
        engine.cune_epoch(0.02, 0.01, 0.01, 0.0, 1, 0, MODE_SERIAL)


# ---- CPU: the kernel's text, compiled for the host ---------------------------------------------------------------------
def test_cune_kernel_text_on_the_host_reproduces_the_reference_loop(golden_dir, tmp_path):
    """tests/emul/cune_emul.cpp compiles csrc/cune_sgd.cuh itself with g++ as a one-lane warp (shuffles are identities):
    the kernel's statement order, j == k aliasing, fused Philox draws of k and j, padding columns and loss -- everything
    but the 32-lane reductions and the launch -- against the golden run of the reference's own loop text, without a GPU."""
    import ctypes as C
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = str(tmp_path / "libcune_emul.so")
    subprocess.run(["g++", "-O1", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", "-Wl,-Bsymbolic", "-I" + os.path.join(root, "tests", "emul", "stub"),
                    "-o", so, os.path.join(root, "tests", "emul", "cune_emul.cpp")], check=True, capture_output=True)
    lib = C.CDLL(so)
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    (m, k), n = g["P0"].shape, g["Q0"].shape[0]
    csr = [np.ascontiguousarray(g[x], dtype=d) for x, d in (("ev_indptr", np.int64), ("ev_items", np.int32), ("uq_indptr", np.int64),
                                                           ("uq_items", np.int32), ("ip_indptr", np.int64), ("ip_items", np.int32))]
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    # the golden draws contain repeats whose negative IS the implicit positive (one row updated under two names)
    ev_user = record_ref.ev_users(g["ev_indptr"])
    alias = 0
    for it in range(len(g["loss"])):
        for nn in range(3):
            has = g["kpos"][it][nn] >= 0
            assert has.any() and (~has).any()                  # both branches of the loop
            alias += int((g["ip_items"][g["ip_indptr"][ev_user[has]] + g["kpos"][it][nn][has]] == g["neg"][it][nn][has]).sum())
    assert alias > 0
    err = lambda a, b: float((np.linalg.norm(a.astype(np.float64) - b, axis=1) / np.maximum(np.linalg.norm(b.astype(np.float64), axis=1), 1e-12)).max())
    # chunk: Hogwild cuts users with more events into work items that publish and re-read P[u] (0 = whole users); run one
    # after the other they are still the serial order, so the bookkeeping of the shared row is checked here
    assert int(np.diff(g["ev_indptr"]).max()) > 16
    for ld, serial, chunk, tol in ((12, 1, 0, 1e-5), (16, 1, 0, 1e-5), (16, 0, 0, 1e-4), (16, 0, 16, 1e-4)):
        P, Q = np.zeros((m, ld), np.float32), np.zeros((n, ld), np.float32)
        P[:, :k], Q[:, :k] = g["P0"], g["Q0"]
        for it in range(len(g["loss"])):
            loss, users = C.c_double(), C.c_uint64()
            rc = lib.cune_emul_epoch(ptr(P), ptr(Q), ld, k, C.c_int64(m), C.c_int64(n), *[ptr(a) for a in csr], C.c_uint64(int(g["seed"])),
                                     C.c_uint32(it), C.c_double(float(g["lr"])), C.c_double(float(g["regU"])), C.c_double(float(g["regI"])),
                                     C.c_double(float(g["s"])), serial, C.byref(loss), C.byref(users), None, C.c_int64(0), None, C.c_int64(chunk))
            assert rc == 0 and users.value == int((np.diff(g["ev_indptr"]) > 0).sum())
            assert err(P[:, :k], g["P"][it]) < tol and err(Q[:, :k], g["Q"][it]) < tol
            assert not P[:, k:].any() and not Q[:, k:].any()
            if serial:
                assert loss.value == pytest.approx(float(g["loss"][it]), rel=1e-5)
    # The device-side log conventions the kernel shares with K2: hot positives stored re-labelled as -slot-1, and a log
    # held as two user shards (local user indices, event_base / per-user offsets giving the global event index the draws
    # are keyed on).  Shard 0 then shard 1 on the same Q table is the serial epoch.
    ev_indptr, ev_items = csr[0], csr[1].copy()
    hot = np.bincount(ev_items).argsort()[::-1][:3].astype(np.int32)
    for slot, t in enumerate(hot):
        ev_items[ev_items == t] = -slot - 1
    assert (ev_items < 0).any()
    cut = m // 2
    for use_delta in (False, True):
        P, Q = np.zeros((m, 16), np.float32), np.zeros((n, 16), np.float32)
        P[:, :k], Q[:, :k] = g["P0"], g["Q0"]
        for lo, hi in ((0, cut), (cut, m)):
            e0 = int(ev_indptr[lo])
            loc = [np.ascontiguousarray(x) for x in (ev_indptr[lo:hi + 1] - e0, ev_items[e0:int(ev_indptr[hi])],
                                                     csr[2][lo:hi + 1] - csr[2][lo], csr[3][int(csr[2][lo]):int(csr[2][hi])],
                                                     csr[4][lo:hi + 1] - csr[4][lo], csr[5][int(csr[4][lo]):int(csr[4][hi])])]
            Ploc = np.ascontiguousarray(P[lo:hi])
            delta = np.full(hi - lo, e0, np.int64)
            loss, users = C.c_double(), C.c_uint64()
            rc = lib.cune_emul_epoch(ptr(Ploc), ptr(Q), 16, k, C.c_int64(hi - lo), C.c_int64(n), *[ptr(a) for a in loc],
                                     C.c_uint64(int(g["seed"])), C.c_uint32(0), C.c_double(float(g["lr"])), C.c_double(float(g["regU"])),
                                     C.c_double(float(g["regI"])), C.c_double(float(g["s"])), 1, C.byref(loss), C.byref(users),
                                     ptr(hot), C.c_int64(0 if use_delta else e0), ptr(delta) if use_delta else None, C.c_int64(0))
            assert rc == 0
            P[lo:hi] = Ploc
        assert err(P[:, :k], g["P"][0]) < 1e-5 and err(Q[:, :k], g["Q"][0]) < 1e-5


def test_cune_kernel_text_as_an_eight_lane_warp_in_lockstep(golden_dir, tmp_path):
    """The same header with -DEMUL_LANES=8: eight host threads in lockstep, a shuffle = an exchange between two barriers.
    Runs the warp-level text as written -- xor butterflies, one lane per event drawing k and j and the broadcast of its
    draws, lane-owned 16-byte chunks (three of them at 12 columns: most lanes hold none), the barrier before the per-user norms that
    read other lanes' columns, lane 0's cursor and loss -- against the golden run, serial and Hogwild with shared items."""
    import ctypes as C
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = str(tmp_path / "libcune_emul8.so")
    subprocess.run(["g++", "-O1", "-ffp-contract=off", "-std=c++20", "-pthread", "-DEMUL_LANES=8", "-shared", "-fPIC", "-fvisibility=hidden", "-Wl,-Bsymbolic",
                    "-I" + os.path.join(root, "tests", "emul", "stub"), "-o", so, os.path.join(root, "tests", "emul", "cune_emul.cpp")],
                   check=True, capture_output=True)
    lib = C.CDLL(so)
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    (m, k), n = g["P0"].shape, g["Q0"].shape[0]
    csr = [np.ascontiguousarray(g[x], dtype=d) for x, d in (("ev_indptr", np.int64), ("ev_items", np.int32), ("uq_indptr", np.int64),
                                                           ("uq_items", np.int32), ("ip_indptr", np.int64), ("ip_items", np.int32))]
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    err = lambda a, b: float((np.linalg.norm(a.astype(np.float64) - b, axis=1) / np.maximum(np.linalg.norm(b.astype(np.float64), axis=1), 1e-12)).max())
    for ld, serial, chunk, tol in ((12, 1, 0, 1e-5), (16, 0, 16, 1e-4)):
        P, Q = np.zeros((m, ld), np.float32), np.zeros((n, ld), np.float32)
        P[:, :k], Q[:, :k] = g["P0"], g["Q0"]
        loss, users = C.c_double(), C.c_uint64()
        rc = lib.cune_emul_epoch(ptr(P), ptr(Q), ld, k, C.c_int64(m), C.c_int64(n), *[ptr(a) for a in csr], C.c_uint64(int(g["seed"])),
                                 C.c_uint32(0), C.c_double(float(g["lr"])), C.c_double(float(g["regU"])), C.c_double(float(g["regI"])),
                                 C.c_double(float(g["s"])), serial, C.byref(loss), C.byref(users), None, C.c_int64(0), None, C.c_int64(chunk))
        assert rc == 0 and users.value == int((np.diff(g["ev_indptr"]) > 0).sum())
        assert err(P[:, :k], g["P"][0]) < tol and err(Q[:, :k], g["Q"][0]) < tol
        assert not P[:, k:].any() and not Q[:, k:].any()
        if serial:
            assert loss.value == pytest.approx(float(g["loss"][0]), rel=1e-5)


def test_cune_kernel_text_at_the_device_warp_width(golden_dir, tmp_path):
    """-DEMUL_LANES=32: the instantiation the C-ABI launches for num.factors <= 128 (one 16-byte chunk per lane, 32-event
    batches of draws), as 32 host threads in lockstep, on the first users of the golden log (one of them has 203 events:
    seven batches) against the oracle loop fed the golden draws; serial, and Hogwild with 32-event shared items."""
    import ctypes as C
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = str(tmp_path / "libcune_emul32.so")
    subprocess.run(["g++", "-O1", "-ffp-contract=off", "-std=c++20", "-pthread", "-DEMUL_LANES=32", "-shared", "-fPIC", "-fvisibility=hidden", "-Wl,-Bsymbolic",
                    "-I" + os.path.join(root, "tests", "emul", "stub"), "-o", so, os.path.join(root, "tests", "emul", "cune_emul.cpp")],
                   check=True, capture_output=True)
    lib = C.CDLL(so)
    g = np.load(os.path.join(golden_dir, "cune_small.npz"))
    mm, k, n = 6, g["P0"].shape[1], g["Q0"].shape[0]
    E = int(g["ev_indptr"][mm])
    csr = [np.ascontiguousarray(x) for x in (g["ev_indptr"][:mm + 1], g["ev_items"][:E], g["uq_indptr"][:mm + 1],
                                             g["uq_items"][:int(g["uq_indptr"][mm])], g["ip_indptr"][:mm + 1],
                                             g["ip_items"][:int(g["ip_indptr"][mm])])]
    assert int(np.diff(csr[0]).max()) > 64 and (np.diff(csr[4]) == 0).any() and (np.diff(csr[4]) > 0).any()
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    err = lambda a, b: float((np.linalg.norm(a.astype(np.float64) - b, axis=1) / np.maximum(np.linalg.norm(b.astype(np.float64), axis=1), 1e-12)).max())
    for serial, chunk, reg, tol in ((1, 0, float(g["regU"]), 1e-5), (0, 32, 0.0, 1e-4)):
        P, Q = np.zeros((mm, 16), np.float32), np.zeros((n, 16), np.float32)
        P[:, :k], Q[:, :k] = g["P0"][:mm], g["Q0"]
        loss, users = C.c_double(), C.c_uint64()
        rc = lib.cune_emul_epoch(ptr(P), ptr(Q), 16, k, C.c_int64(mm), C.c_int64(n), *[ptr(a) for a in csr], C.c_uint64(int(g["seed"])),
                                 C.c_uint32(0), C.c_double(float(g["lr"])), C.c_double(reg), C.c_double(reg), C.c_double(float(g["s"])),
                                 serial, C.byref(loss), C.byref(users), None, C.c_int64(0), None, C.c_int64(chunk))
        Pr, Qr = g["P0"][:mm].copy(), g["Q0"].copy()
        ref = cune_ref.epoch(Pr, Qr, csr[0], csr[1], csr[4], csr[5], [x[:E] for x in g["kpos"][0]], [x[:E] for x in g["neg"][0]],
                             float(g["lr"]), reg, reg, float(g["s"]))
        assert rc == 0 and users.value == mm
        assert err(P[:, :k], Pr) < tol and err(Q[:, :k], Qr) < tol
        assert loss.value == pytest.approx(float(ref), rel=1e-5 if serial else 1e-3)


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the Yue reference: set YUE_REFERENCE to its directory")
def test_cune_dropin_shim_on_top_of_the_reference_tree(golden_dir, tmp_path):
    """dropin/recommender/advanced/CUNE.py shadows the reference's module (which needs gensim at import), derives from the
    REFERENCE's own base.IterativeRecommender and Record, and with the oracle in place of yue_cune_epoch reproduces the
    golden tables of the reference's loop text bit for bit."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r'''
import io, json, os, sys
import numpy as np
from contextlib import redirect_stdout
sys.path[:0] = [%(dropin)r, %(ref)r, %(root)r]
from tool.config import Config
from recommender.advanced.CUNE import CUNE
import base.IterativeRecommender as ref_base
import recommender.advanced.CUNE as mod
assert mod.__file__.startswith(%(dropin)r) and CUNE.__mro__[3] is ref_base.IterativeRecommender, CUNE.__mro__
from oracle import cune_ref, philox, record_ref
from yue_b200.host.record import interaction_arrays
g = json.load(open(%(gold)r + "/record_small.json"))
keep = set('u%%d' %% x for x in range(60))
train = [e for e, h in zip(g["events"], g["held"]) if not h and e['user'] in keep]
test = [e for e, h in zip(g["events"], g["held"]) if h and e['user'] in keep]
open(%(tmp)r + "/c.conf", "w").write("\n".join(k + "=" + v for k, v in %(conf)r.items()))
w = np.load(%(gold)r + "/cune_small.npz")
with redirect_stdout(io.StringIO()):
    m = CUNE(Config(%(tmp)r + "/c.conf"), train, test)
    m.readConfiguration()
    np.random.seed(99)
    m.initModel()
    arr = interaction_arrays(m.data.name2id, m.data.userRecord, m.recType)
    u2i = m.data.name2id['user']; by_id = {v: k for k, v in u2i.items()}; M = len(u2i)
    m.topKSim = {}
    for name, uid in u2i.items():
        if name in m.data.userRecord and uid %% 5 != 0:
            fr = [by_id[f] for f in ((uid * 7 + 3) %% M, (uid * 11 + 5) %% M)]
            m.topKSim[name] = [(f, 1.0) for f in fr if f in m.data.userRecord and f != name]
    class E:
        def get_interactions(self): return arr
        def cune_set_implicit(self, a, b): self.ip = (np.asarray(a), np.asarray(b))
        def cune_epoch(self, lr, regU, regI, s, seed, epoch, mode):
            evu = record_ref.ev_users(arr[0])
            kp = [cune_ref.sample_implicit(seed, epoch, nn, evu, self.ip[0]) for nn in range(3)]
            neg = [philox.sample_negatives(seed, epoch, evu, m.n, arr[2], arr[3], slot=nn) for nn in range(3)]
            return cune_ref.epoch(m.P, m.Q, arr[0], arr[1], self.ip[0], self.ip[1], kp, neg, lr, regU, regI, s)
    e = E()
    m._push_factors = lambda: e
    m._pull_factors = lambda: None
    m.isConverged = lambda it: False
    m.buildModel()
assert np.array_equal(e.ip[1], w["ip_items"])
assert np.array_equal(m.P, w["P"][-1]) and np.array_equal(m.Q, w["Q"][-1])
print("OK")
''' % dict(dropin=os.path.join(root, "dropin"), ref=REF, root=root, gold=golden_dir, tmp=str(tmp_path), conf=_conf(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 128, 200])
def test_cune_serial_epoch_matches_oracle_at_bench_widths(engine, d):
    """Row widths the golden run does not have (one 16-byte chunk per lane on 16 / 32 lanes, two chunks at d = 200) on a
    synthetic power-law log with synthetic similar users: serial kernel (fused draws) against the oracle loop fed the
    oracle's draws; then the Hogwild kernel with heavy users cut into 32-event items stays close to it."""
    from yue_b200 import synth
    from yue_b200.cune import implicit_positive_lists
    from yue_b200.engine import MODE_HOGWILD, MODE_SERIAL
    log = synth.power_law_log(80, 150, 1500, seed=11, test_ratio=0.0)
    m, n = log.m, log.n
    top = {u: [f for f in ((u * 7 + 3) % m, (u * 11 + 5) % m) if f != u] for u in range(m) if u % 5}
    ip_indptr, ip_items = implicit_positive_lists(m, log.uq_indptr, log.uq_items, top)
    rng = np.random.default_rng(d)
    P0 = rng.uniform(0, 0.1, (m, d)).astype(np.float32)
    Q0 = rng.uniform(0, 0.1, (n, d)).astype(np.float32)
    engine.set_interactions(m, n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P0.copy(), Q0.copy())
    engine.cune_set_implicit(ip_indptr, ip_items)
    loss = engine.cune_epoch(0.02, 0.01, 0.01, 2.0, 5, 0, MODE_SERIAL)
    P, Q = engine.get_factors()
    ev_user = record_ref.ev_users(log.ev_indptr)
    kp = [cune_ref.sample_implicit(5, 0, nn, ev_user, ip_indptr) for nn in range(3)]
    neg = [philox.sample_negatives(5, 0, ev_user, n, log.uq_indptr, log.uq_items, slot=nn) for nn in range(3)]
    Pr, Qr = P0.copy(), Q0.copy()
    ref = cune_ref.epoch(Pr, Qr, log.ev_indptr, log.ev_items, ip_indptr, ip_items, kp, neg, 0.02, 0.01, 0.01, 2.0)
    err = lambda a, b: float((np.linalg.norm(a.astype(np.float64) - b, axis=1) / np.maximum(np.linalg.norm(b.astype(np.float64), axis=1), 1e-12)).max())
    assert err(P, Pr) < 1e-5 and err(Q, Qr) < 1e-5
    assert loss == pytest.approx(float(ref), rel=1e-4)
    # the Hogwild kernel, one warp (what the C-ABI gives a log this small), heavy users cut into 32-event shared items
    with _env(YUE_CUNE_CHUNK=32, YUE_CUNE_WARPS=None):
        engine.set_factors(P0.copy(), Q0.copy())
        lh = engine.cune_epoch(0.02, 0.0, 0.0, 2.0, 5, 0, MODE_HOGWILD)
    Ph, Qh = engine.get_factors()
    Pr, Qr = P0.copy(), Q0.copy()
    ref0 = cune_ref.epoch(Pr, Qr, log.ev_indptr, log.ev_items, ip_indptr, ip_items, kp, neg, 0.02, 0.0, 0.0, 2.0)
    assert err(Ph, Pr) < 1e-4 and err(Qh, Qr) < 1e-4
    assert lh == pytest.approx(float(ref0), rel=1e-3)
    # and with all 80 users in flight on 64 warps: a different schedule, sanity only (measured: loss within 2 %)
    with _env(YUE_CUNE_CHUNK=32, YUE_CUNE_WARPS=64):
        engine.set_factors(P0.copy(), Q0.copy())
        lw = engine.cune_epoch(0.02, 0.0, 0.0, 2.0, 5, 0, MODE_HOGWILD)
    Pw, Qw = engine.get_factors()
    assert np.isfinite(Pw).all() and np.isfinite(Qw).all()
    assert lw == pytest.approx(float(ref0), rel=0.1)
