"""The Hogwild SGD epoch kernels, one warp at a time, against oracle/sgd_schedule_ref.py.

yue_set_sgd_concurrency(h, 1, 1) runs an epoch on one warp: what it reads and when is then fixed by the code, and the
oracle restates it -- the host's work plan (segments, heavy users cut into shared items), the in-kernel sampler at the
global event index, the blocked kernel's read schedule (block k read before block k-1 is added, P[u] published and
re-read at user switches, shared segments and resync points) and the per-triplet kernel's (rows PF events ahead).
The epoch path of bench.py (yue_bpr_epoch in MODE_HOGWILD) and of APR is pinned here by exact-schedule comparisons:
the kernel's tables may be no further from the float64 run of the schedule than 3x the float32 oracle is (floor 2e-5
in rel_err), the loss within 1e-5 of the float32 oracle's; switches that must not change the result are bit-identity
checks.  The CPU tests at the bottom show, at every GPU case's own shape, that a wrong schedule -- the serial order, a
lag of two blocks, a resync that drops P[u]'s changes, negatives drawn at the local event index -- is at least 20x that
tolerance away."""
import collections

import numpy as np
import pytest

from oracle import sgd_schedule_ref as sr
from yue_b200 import synth
from yue_b200.engine import MODE_HOGWILD, MODE_HOGWILD_STORE

REG_U, REG_I, SEED = 0.01, 0.02, 17
EPS, REG_A = 0.5, 2.0
BPR_EPOCHS = ((0.05, 0, 0), (0.02, 3, 0))          # (lr, epoch index, slot)
APR_EPOCHS = ((0.005, 1, 0), (0.005, 1, 1), (0.005, 1, 2))
HOT_ON = dict(YUE_SGD_HOT_MIN_COUNT="1", YUE_SGD_HOT_DIV="1000000", YUE_SGD_HOT_SHARD_DIV="50")
HOT_OFF = dict(YUE_SGD_HOT_MAX="0")

Log = collections.namedtuple("Log", "m n ev_indptr ev_items uq_indptr uq_items")


def rel_err(a, b):
    return float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64)) / (np.abs(b.astype(np.float64)) + 1e-3)))


def make_log(deg, n, seed):
    """Users with the given event counts on a catalog of n tracks, zipf-like plays (the top tracks repeat inside and
    across blocks); every user leaves at least one track unplayed (a negative exists)."""
    rng = np.random.default_rng(seed)
    w = 1.0 / np.arange(1, n + 1) ** 0.8
    ev, uq = [], []
    for k in deg:
        allowed = np.ones(n, bool)
        allowed[rng.integers(0, n)] = False
        p = np.where(allowed, w, 0.0)
        items = rng.choice(n, size=int(k), p=p / p.sum()).astype(np.int32)
        ev.append(items)
        uq.append(np.unique(items).astype(np.int32))
    indptr = lambda rows: np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)   # noqa: E731
    return Log(len(deg), n, indptr(ev), np.concatenate(ev), indptr(uq), np.concatenate(uq))


def light(m, seed, hi=70):
    return list(1 + np.random.default_rng(seed).integers(0, hi, m))


# ---- the cases: every GPU test and its discrimination check run the same shape -------------------------------------
# heavy users: ragged last segment and block (97 = 3 x 32 + 1, 70 = 2 x 32 + 4 + 2, 250 = 7 x 32 + 4 x 6 + 2)
HEAVY_DEG = [97, 70, 250, 133]
CASES = {}
for d, n in ((10, 7), (20, 12), (32, 25), (50, 40), (64, 60), (100, 200), (128, 400)):
    CASES["bpr_d%d" % d] = dict(d=d, n=n, deg=light(120, d), epochs=BPR_EPOCHS)
for segs in (2, 3):
    for rs in (4, 8, 32):
        CASES["heavy_s%d_r%d" % (segs, rs)] = dict(d=32 if segs == 2 else 64, n=30, deg=light(40, segs * rs)[:20] + HEAVY_DEG + light(20, rs),
                                                   epochs=BPR_EPOCHS, env=dict(YUE_SGD_ITEM_SEGS=str(segs), YUE_SGD_RESYNC_EVENTS=str(rs)))
# default settings: one warp's log of ~4 K events gives item_segs = 32, a user of 1 100 events is cut into items of 32 segments
CASES["heavy_default"] = dict(d=64, n=50, deg=light(80, 5)[:40] + [1100] + light(80, 6)[:40], epochs=BPR_EPOCHS)
for d in (10, 64, 128):
    CASES["hot_d%d" % d] = dict(d=d, n=20, deg=light(60, d)[:30] + [300] + light(60, d + 1)[:30], epochs=BPR_EPOCHS,
                                env=dict(HOT_ON, YUE_SGD_ITEM_SEGS="3"))
for d, n in ((10, 9), (20, 15), (50, 30), (64, 40), (100, 120), (128, 300)):
    CASES["apr_d%d" % d] = dict(d=d, n=n, deg=light(60, 3 * d) + [140], epochs=APR_EPOCHS, apr=True, env=dict(YUE_SGD_ITEM_SEGS="3"))
CASES["shard_contiguous"] = dict(d=64, n=30, deg=light(140, 7), epochs=BPR_EPOCHS, shard="contiguous")
CASES["shard_interleaved"] = dict(d=64, n=30, deg=light(140, 8), epochs=BPR_EPOCHS, shard="interleaved")
CASES["parts"] = dict(d=64, n=25, deg=light(30, 9) + [700] + light(30, 10), epochs=BPR_EPOCHS[:1], env=dict(HOT_ON, YUE_SGD_ITEM_SEGS="2"))
CASES["pt_d200"] = dict(d=200, n=40, deg=light(70, 11) + [160], epochs=BPR_EPOCHS, kernel="pt", pf=2,
                        env=dict(YUE_SGD_ITEM_SEGS="3"))
for name, store in (("pt_d64", False), ("pt_d64_store", True)):
    CASES[name] = dict(d=64, n=30, deg=light(70, 12) + [160], epochs=BPR_EPOCHS, kernel="pt", pf=4, store=store,
                       env=dict(YUE_SGD_KERNEL="1", YUE_SGD_ITEM_SEGS="3"))


def case_data(name):
    c = CASES[name]
    log = make_log(c["deg"], c["n"], seed=len(name) * 7 + c["d"])
    if c.get("apr"):
        rng = np.random.default_rng(c["d"])
        P = rng.normal(0, 0.3, (log.m, c["d"])).astype(np.float32)       # norms well away from 0: APR divides by |P|, |d|
        Q = rng.normal(0, 0.3, (log.n, c["d"])).astype(np.float32)
    else:
        P, Q = synth.init_factors(log.m, log.n, c["d"], seed=c["d"])
    return c, log, P, Q


def item_segs_of(c, T):
    env = c.get("env", {})
    return int(env["YUE_SGD_ITEM_SEGS"]) if "YUE_SGD_ITEM_SEGS" in env else sr.default_item_segs(T, sr.default_n_warps(T))


def shard_of(log, how):
    """(local log, event_base, per-user offsets or None, user_begin) of the shard a case trains."""
    if how == "contiguous":
        u0, u1 = 40, 110
        e0, e1, q0, q1 = log.ev_indptr[u0], log.ev_indptr[u1], log.uq_indptr[u0], log.uq_indptr[u1]
        sub = Log(u1 - u0, log.n, log.ev_indptr[u0:u1 + 1] - e0, log.ev_items[e0:e1], log.uq_indptr[u0:u1 + 1] - q0, log.uq_items[q0:q1])
        return sub, int(e0), None, u0
    from yue_b200 import sharding
    users = sharding.interleaved_users(log.m, 3, 1)
    sh = sharding.local_shard_of_users(log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, users)
    sub = Log(sh["m_local"], log.n, sh["ev_indptr"], sh["ev_items"], sh["uq_indptr"], sh["uq_items"])
    return sub, 0, sh["event_offsets"], 0


def run_oracle(name, f32=True, lag=1, resync="publish", local_index=False):
    """The case's epochs on the oracle; returns (losses, P, Q) of the trained (local) tables."""
    c, log, P, Q = case_data(name)
    base, delta = 0, None
    if c.get("shard"):
        log, base, delta, u0 = shard_of(log, c["shard"])
        P = P[u0:u0 + log.m] if delta is None else P[1::3]
    dt = np.float32 if f32 else np.float64
    P, Q = P.astype(dt), Q.astype(dt)
    env = c.get("env", {})
    rs = int(env.get("YUE_SGD_RESYNC_EVENTS", 8))
    plan = sr.plan_epoch(log.ev_indptr, item_segs_of(c, len(log.ev_items)))
    losses = []
    for (lr, ep, slot) in c["epochs"]:
        neg = sr.epoch_negatives(SEED, ep, log.ev_indptr, log.n, log.uq_indptr, log.uq_items, slot,
                                 event_base=0 if local_index else base, ev_delta=None if local_index else delta)
        if c.get("kernel") == "pt":
            losses.append(sr.per_triplet_epoch(P, Q, plan, log.ev_items, neg, lr, REG_U, REG_I, c["pf"], rs, c.get("store", False)))
        else:
            losses.append(sr.blocked_epoch(P, Q, plan, log.ev_items, neg, lr, REG_U, REG_I, apr=(EPS, REG_A) if c.get("apr") else None,
                                           resync_events=rs, lag=lag, resync=resync))
    return losses, P, Q


def tolerance(name):
    """The case's yardstick: (float64 run, float32 run, tolerance)."""
    o64, o32 = run_oracle(name, f32=False), run_oracle(name)
    return o64, o32, max(3 * max(rel_err(o32[1], o64[1]), rel_err(o32[2], o64[2])), 2e-5)


def run_gpu(monkeypatch, name, env=None, parts=None, repeat=1, shared_trainer=False):
    """The case's epochs on a fresh handle (switches are read when it is created) at one warp; returns
    (losses, P, Q, hot tracks).  parts = S: every epoch as S sub-epochs, the losses summed.  repeat: run the epochs
    again from the initial tables (the results of every run)."""
    from yue_b200.engine import Engine
    c, log, P, Q = case_data(name)
    env = dict(c.get("env", {}), **(env or {}))
    base, delta, u0 = 0, None, 0
    if c.get("shard"):
        log, base, delta, u0 = shard_of(log, c["shard"])
        P = np.ascontiguousarray(P[u0:u0 + log.m] if delta is None else P[1::3])
    out = []
    with monkeypatch.context() as mp:
        for k, v in env.items():
            mp.setenv(k, v)
        eng = Engine(0)
        try:
            eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items, user_begin=u0, event_base=base)
            if delta is not None:
                eng.set_event_offsets(delta)
            for _ in range(repeat):
                eng.set_factors(P, Q)
                eng.set_sgd_concurrency(1, 1)
                mode = MODE_HOGWILD_STORE if c.get("store") else MODE_HOGWILD
                losses = []
                for (lr, ep, slot) in c["epochs"]:
                    if c.get("apr"):
                        if parts:
                            losses.append(sum(eng.apr_epoch_part(lr, REG_U, REG_I, EPS, REG_A, SEED, ep, k, parts, slot, mode) for k in range(parts)))
                        else:
                            losses.append(eng.apr_epoch(lr, REG_U, REG_I, EPS, REG_A, SEED, ep, slot, mode))
                    elif parts:
                        losses.append(sum(eng.bpr_epoch_part(lr, REG_U, REG_I, SEED, ep, k, parts, mode) for k in range(parts)))
                    else:
                        losses.append(eng.bpr_epoch(lr, REG_U, REG_I, SEED, ep, mode))
                out.append((losses,) + eng.get_factors() + (eng.hot_tracks(),))
        finally:
            eng.close()
    return out if repeat > 1 else out[0]


def check_against_oracle(name, got):
    (l64, P64, Q64), (l32, _, _), tol = tolerance(name)
    losses, Pg, Qg = got[:3]
    assert tol < 1e-3, (name, tol)
    assert rel_err(Pg, P64) < tol and rel_err(Qg, Q64) < tol, (name, rel_err(Pg, P64), rel_err(Qg, Q64), tol)
    for lg, lr in zip(losses, l32):
        assert lg == pytest.approx(lr, rel=1e-5)


def same_bits(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a[1:3], b[1:3])) and a[0] == b[0]


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", [k for k in CASES if k.startswith("bpr_d")])
def test_blocked_bpr_epochs_follow_the_schedule(monkeypatch, name):
    check_against_oracle(name, run_gpu(monkeypatch, name))


@pytest.mark.gpu
@pytest.mark.parametrize("name", [k for k in CASES if k.startswith("heavy_")])
def test_heavy_users_shared_items_and_resync(monkeypatch, name):
    c, log, _, _ = case_data(name)
    segs, _ = sr.plan_epoch(log.ev_indptr, item_segs_of(c, len(log.ev_items)))
    assert any(s[3] for s in segs)                           # the case has shared segments
    check_against_oracle(name, run_gpu(monkeypatch, name))


@pytest.mark.gpu
@pytest.mark.parametrize("name", [k for k in CASES if k.startswith("hot_")])
def test_hot_table_is_transparent_at_one_warp_and_deterministic(monkeypatch, name):
    """At one warp every change goes to a hot track's first row (warp 0), the second rows stay zero and a hot negative
    read through the table is the row itself: the tables equal the epoch without the table bit for bit.  The same
    epoch twice gives the same bits (one lane adds every float, in program order)."""
    c, log, _, _ = case_data(name)
    counts = np.bincount(log.ev_items, minlength=log.n)
    assert (counts * 50 > len(log.ev_items)).any()           # tracks above 1 / HOT_SHARD_DIV of the plays: second rows exist
    a, b = run_gpu(monkeypatch, name, repeat=2)
    assert len(a[3]) > 0 and same_bits(a, b)
    off = run_gpu(monkeypatch, name, env=HOT_OFF)
    assert len(off[3]) == 0 and same_bits(a, off)
    check_against_oracle(name, a)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [k for k in CASES if k.startswith("apr_")])
def test_blocked_apr_epochs_follow_the_schedule(monkeypatch, name):
    off = run_gpu(monkeypatch, name)
    check_against_oracle(name, off)
    on = run_gpu(monkeypatch, name, env=HOT_ON)
    assert len(on[3]) > 0 and same_bits(on, off)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["shard_contiguous", "shard_interleaved"])
def test_shards_draw_global_negatives(monkeypatch, name):
    check_against_oracle(name, run_gpu(monkeypatch, name))


@pytest.mark.gpu
@pytest.mark.parametrize("apr", [False, True])
def test_sub_epochs_are_the_epoch_bit_for_bit(monkeypatch, apr):
    name = "parts"
    c, log, _, _ = case_data(name)
    _, items = sr.plan_epoch(log.ev_indptr, item_segs_of(c, len(log.ev_items)))
    segs, _ = sr.plan_epoch(log.ev_indptr, item_segs_of(c, len(log.ev_items)))
    heavy = [k for k, (s0, _) in enumerate(items) if segs[s0][3]]
    if apr:
        CASES[name] = dict(c, apr=True, epochs=APR_EPOCHS[:2])
    try:
        whole = run_gpu(monkeypatch, name)
        assert len(whole[3]) > 0
        for S in (2, 5):
            cuts = [a for (a, _) in sr.plan_parts(items, S)[1:]]
            assert any(heavy[0] < x <= heavy[-1] for x in cuts)      # a part boundary inside the heavy user
            got = run_gpu(monkeypatch, name, parts=S)
            assert np.array_equal(got[1], whole[1]) and np.array_equal(got[2], whole[2])
            for a, b in zip(got[0], whole[0]):
                assert a == pytest.approx(b, rel=1e-12)
        check_against_oracle(name, whole)
    finally:
        CASES[name] = c


@pytest.mark.gpu
def test_per_triplet_kernel_d200_hot_shards_transparent(monkeypatch):
    off = run_gpu(monkeypatch, "pt_d200", env=HOT_OFF)
    check_against_oracle("pt_d200", off)
    on = run_gpu(monkeypatch, "pt_d200", env=HOT_ON)
    assert len(on[3]) > 0 and same_bits(on, off)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pt_d64", "pt_d64_store"])
def test_per_triplet_kernel_hogwild_modes(monkeypatch, name):
    check_against_oracle(name, run_gpu(monkeypatch, name))


@pytest.mark.gpu
def test_switches_that_do_not_change_results(monkeypatch):
    base = run_gpu(monkeypatch, "bpr_d64")
    assert same_bits(run_gpu(monkeypatch, "bpr_d64", env=dict(YUE_SGD_L2_PREFETCH="32")), base)
    pt = run_gpu(monkeypatch, "pt_d64")
    assert same_bits(run_gpu(monkeypatch, "pt_d64", env=dict(YUE_SGD_Q_INTERLEAVE="1")), pt)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 64, 128])
def test_shared_hot_table_at_world_1_is_the_plain_epoch(monkeypatch, d):
    """sharding.SharedHotTrainer on one rank: the hot rows live in the shared table across the sub-epochs (SHARED
    instantiation: system-scope loads and adds); at one warp that is the plain epoch bit for bit."""
    from yue_b200 import sharding
    from yue_b200.engine import Engine
    deg = [900] * 22 + light(40, d)                          # ~20 K events, track 0 above the trainer's 16 384 plays
    rng = np.random.default_rng(d)
    ev, uq = [], []
    for k in deg:
        items = np.where(rng.random(k) < 0.85, 0, rng.integers(1, 40, k)).astype(np.int32)
        ev.append(items)
        uq.append(np.unique(items))
    ind = lambda rows: np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)   # noqa: E731
    log = Log(len(deg), 60, ind(ev), np.concatenate(ev), ind(uq), np.concatenate(uq).astype(np.int32))
    P, Q = synth.init_factors(log.m, log.n, d, seed=d)
    out = []
    for shared in (False, True):
        eng = Engine(0)
        try:
            eng.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
            eng.set_factors(P, Q)
            if shared:
                ctl = sharding.ThreadCtl(sharding.ThreadCtl.Shared(1), 0)
                tr = sharding.SharedHotTrainer(eng, ctl, np.bincount(log.ev_items, minlength=log.n), sub_epochs=4)
                assert len(tr.hot_tracks) > 0
                eng.set_sgd_concurrency(1, 1)
                losses = [tr.epoch(lr, REG_U, REG_I, SEED, ep, want_loss=True) for (lr, ep, _) in BPR_EPOCHS]
                tr.finalize()
                res = (losses,) + eng.get_factors()
                tr.close()
            else:
                eng.set_sgd_concurrency(1, 1)
                losses = [eng.bpr_epoch(lr, REG_U, REG_I, SEED, ep, MODE_HOGWILD) for (lr, ep, _) in BPR_EPOCHS]
                res = (losses,) + eng.get_factors()
            out.append(res)
        finally:
            eng.close()
    (la, Pa, Qa), (lb, Pb, Qb) = out
    assert np.array_equal(Pa, Pb) and np.array_equal(Qa, Qb)
    for a, b in zip(la, lb):
        assert a == pytest.approx(b, rel=1e-12)


# ---- CPU: the tolerances above can see a wrong kernel --------------------------------------------------------------
def _variants(name):
    c = CASES[name]
    v = {"serial order": dict(lag=0), "lag of 2 blocks": dict(lag=2)}
    if c.get("kernel") == "pt":
        v = {"serial order": None}                           # the per-triplet oracle's variants below
    log = case_data(name)[1]
    segs = sr.plan_epoch(log.ev_indptr, item_segs_of(c, len(log.ev_items)))[0]
    if c.get("kernel") != "pt" and any(s[3] for s in segs):
        v["resync without publish"] = dict(resync="lose")
    if c.get("shard"):
        v["local event index"] = dict(local_index=True)
    return v


@pytest.mark.parametrize("name", sorted(CASES))
def test_wrong_schedules_are_20x_the_tolerance_away(name):
    (_, P64, Q64), _, tol = tolerance(name)
    assert tol < 1e-3
    for what, kw in _variants(name).items():
        if kw is None:                                       # per-triplet: the blocked schedule's serial order (lag 0)
            c = CASES[name]
            CASES[name] = dict(c, kernel="blk")
            try:
                _, Pv, Qv = run_oracle(name, lag=0)
            finally:
                CASES[name] = c
        else:
            _, Pv, Qv = run_oracle(name, **kw)
        dist = max(rel_err(Pv, P64), rel_err(Qv, Q64))
        assert dist > 20 * tol, (name, what, dist, tol)
