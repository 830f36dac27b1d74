"""GPU parity of full-catalog scoring + masked top-N (K3/K5) against the oracle: ids bit-exact
(ties broken by track id), scores bit-exact for the canonical FMA chain and within 1e-3 relative
of numpy's dot."""
import json
import os

import numpy as np
import pytest

from oracle import topn
from yue_b200 import synth
from yue_b200.engine import RANK_EXACT

pytestmark = pytest.mark.gpu


def check(engine, P, Q, users, N, uq_indptr, uq_items, algo):
    ids, sc = engine.rank_topn(users, N, algo)
    rid, rsc = topn.topn_exact(P, Q, users, N, uq_indptr, uq_items)
    assert np.array_equal(ids, rid)
    assert np.array_equal(sc, rsc)
    return ids, sc


def test_golden_eval_ids(engine, golden_dir):
    e = np.load(os.path.join(golden_dir, "eval_small.npz"))
    mj = json.load(open(os.path.join(golden_dir, "measure_small.json")))
    m, n = e["P"].shape[0], e["Q"].shape[0]
    z = np.zeros(m + 1, np.int64)
    engine.set_interactions(m, n, z, np.zeros(0, np.int32), e["uq_indptr"], e["uq_items"])
    engine.set_factors(e["P"], e["Q"])
    ids, sc = engine.rank_topn(e["test_users"], 10, RANK_EXACT)
    assert ids.tolist() == mj["exact_ids"]
    blas = e["blas_scores"]
    for b in range(40):
        assert np.allclose(sc[b], blas[b][ids[b]], rtol=1e-3, atol=1e-7)
    s0 = engine.predict(int(e["test_users"][0]))
    assert np.array_equal(s0, topn.scores_fma32(e["P"][e["test_users"][:1]], e["Q"])[0])


@pytest.mark.parametrize("d,N,n", [(10, 5, 777), (64, 10, 5000), (64, 20, 3001), (128, 32, 1500), (36, 100, 1200)])
def test_exact_topn_shapes(engine, d, N, n):
    m = 300
    log = synth.power_law_log(m, n, 12000, seed=d + N)
    P, Q = synth.init_factors(m, n, d, seed=N)
    rng = np.random.default_rng(1)
    P = (P - 0.05) * rng.uniform(0.5, 3.0, (m, 1)).astype(np.float32)     # mixed signs and scales
    Q = (Q - 0.05).astype(np.float32)
    engine.set_interactions(m, n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    users = rng.permutation(m)[:211].astype(np.int32)                      # ragged last block
    check(engine, P, Q, users, N, log.uq_indptr, log.uq_items, RANK_EXACT)


def test_ties_break_by_track_id_and_padding(engine):
    m, n, d, N = 4, 40, 8, 10
    P = np.ones((m, d), np.float32)
    Q = np.zeros((n, d), np.float32)
    Q[:, 0] = np.repeat(np.arange(8), 5)[::-1]          # 5-way ties, descending blocks
    uq_rows = [np.array([], np.int32), np.arange(0, 35, dtype=np.int32), np.arange(n, dtype=np.int32)[:-3], np.array([0, 1, 2], np.int32)]
    uq_indptr = np.concatenate([[0], np.cumsum([len(r) for r in uq_rows])]).astype(np.int64)
    uq_items = np.concatenate(uq_rows).astype(np.int32)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), uq_indptr, uq_items)
    engine.set_factors(P, Q)
    ids, sc = check(engine, P, Q, np.arange(m, dtype=np.int32), N, uq_indptr, uq_items, RANK_EXACT)
    assert ids[0].tolist() == list(range(10))            # ties -> ascending id
    assert ids[1].tolist() == [35, 36, 37, 38, 39, -1, -1, -1, -1, -1]
    assert ids[2].tolist()[:3] == [37, 38, 39] and (ids[2][3:] == -1).all() and np.isneginf(sc[2][3:]).all()


def test_adversarial_orders(engine):
    """Ascending scores make every new tile beat the running threshold (worst case for the buffers)."""
    m, n, d, N = 130, 4000, 16, 20
    rng = np.random.default_rng(3)
    P = np.abs(rng.normal(size=(m, d))).astype(np.float32)
    base = np.abs(rng.normal(size=d)).astype(np.float32)
    Q = (base[None, :] * (1.0 + np.arange(n)[:, None] * 1e-3)).astype(np.float32)
    uq_indptr = np.zeros(m + 1, np.int64)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), uq_indptr, np.zeros(0, np.int32))
    engine.set_factors(P, Q)
    check(engine, P, Q, np.arange(m, dtype=np.int32), N, uq_indptr, np.zeros(0, np.int32), RANK_EXACT)
    Qd = np.ascontiguousarray(Q[::-1])
    engine.set_factors(P, Qd)
    check(engine, P, Qd, np.arange(m, dtype=np.int32), N, uq_indptr, np.zeros(0, np.int32), RANK_EXACT)


def test_rank_block_sharding_concatenates(engine):
    """Ranking shards by user block: any split of the user list gives the same rows."""
    m, n, d, N = 500, 2500, 64, 10
    log = synth.power_law_log(m, n, 20000, seed=9)
    P, Q = synth.init_factors(m, n, d, seed=9)
    engine.set_interactions(m, n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    users = np.arange(m, dtype=np.int32)
    full, fs = engine.rank_topn(users, N, RANK_EXACT)
    parts = [engine.rank_topn(users[a:b], N, RANK_EXACT) for a, b in [(0, 130), (130, 131), (131, 500)]]
    assert np.array_equal(np.concatenate([p[0] for p in parts]), full)
    assert np.array_equal(np.concatenate([p[1] for p in parts]), fs)


# ---- tcgen05 flavour: must return exactly what the exact kernel / the oracle return -----------
from yue_b200.engine import RANK_TC  # noqa: E402


@pytest.mark.parametrize("d,N,n,B", [(64, 10, 5000, 300), (64, 20, 20011, 257), (32, 5, 3000, 128),
                                     (10, 10, 777, 50), (48, 32, 9000, 130), (128, 10, 6000, 200), (96, 20, 5003, 129), (72, 5, 900, 40)])
def test_tc_topn_matches_oracle(engine, d, N, n, B):
    m = max(B, 300)
    log = synth.power_law_log(m, n, 15000, seed=d + N)
    P, Q = synth.init_factors(m, n, d, seed=N)
    rng = np.random.default_rng(2)
    P = ((P - 0.03) * rng.uniform(0.5, 4.0, (m, 1))).astype(np.float32)       # mixed signs and scales
    Q = ((Q - 0.04) * rng.uniform(0.2, 3.0, (n, 1))).astype(np.float32)
    engine.set_interactions(m, n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    users = rng.permutation(m)[:B].astype(np.int32)
    check(engine, P, Q, users, N, log.uq_indptr, log.uq_items, RANK_TC)


@pytest.mark.parametrize("d,N", [(64, 10), (64, 20), (128, 10)])
def test_tc_equals_exact_kernel_at_the_catalog_of_config_c4(engine, d, N):
    """Config C4's catalog (2 M tracks, ~50 masked tracks per user; BASELINE.json configs[3]) on a block of users: the
    tensor-core flavour (15 625 tiles per row, spill pool and exact-kernel fallback included) returns the exact kernel's
    ids and scores bit for bit; uniform U[0, 0.1) tables like bench.py's -- the near-tie-heavy case."""
    m, n = 640, 2_000_000
    indptr, uq = synth.mask_csr(m, n, 50, seed=8)
    P, Q = synth.init_factors(m, n, d, seed=9)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), indptr, uq)
    engine.set_factors(P, Q)
    users = np.arange(m, dtype=np.int32)
    ie, se = engine.rank_topn(users, N, RANK_EXACT)
    it, st = engine.rank_topn(users, N, RANK_TC)
    assert np.array_equal(ie, it) and np.array_equal(se, st)
    assert (ie >= 0).all() and (np.diff(se, axis=1) <= 0).all()
    for b in (0, 77, m - 1):
        assert not np.isin(it[b], uq[indptr[b]:indptr[b + 1]]).any()


def test_tc_equals_exact_kernel_at_scale(engine):
    """Bigger than the oracle likes: the tensor-core flavour against the exact kernel, trained-like
    factors (heavy-tailed norms), 100 K tracks."""
    m, n, d, N = 3000, 100_000, 64, 10
    rng = np.random.default_rng(5)
    P = (rng.normal(size=(m, d)) * rng.lognormal(0, 0.5, (m, 1))).astype(np.float32)
    Q = (rng.normal(size=(n, d)) * rng.lognormal(0, 0.7, (n, 1)) * 0.3).astype(np.float32)
    indptr, uq = synth.mask_csr(m, n, 50, seed=3)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), indptr, uq)
    engine.set_factors(P, Q)
    users = np.arange(m, dtype=np.int32)
    ie, se = engine.rank_topn(users, N, RANK_EXACT)
    it, st = engine.rank_topn(users, N, RANK_TC)
    assert np.array_equal(ie, it) and np.array_equal(se, st)
    for b in (0, 1, m - 1):                     # and never a masked track
        assert not np.isin(it[b], uq[indptr[b]:indptr[b + 1]]).any()


def test_tc_tie_flood_falls_back_exactly(engine):
    """Thousands of identical rows: more near-ties than a candidate buffer holds -> those users are
    re-run through the exact kernel and the answer is still (score desc, id asc)."""
    m, n, d, N = 140, 6000, 64, 10
    rng = np.random.default_rng(9)
    P = np.abs(rng.normal(size=(m, d))).astype(np.float32)
    Q = np.tile(np.abs(rng.normal(size=(1, d))).astype(np.float32), (n, 1))    # every track identical
    Q[::7] *= 0.5
    uq_indptr = np.zeros(m + 1, np.int64)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), uq_indptr, np.zeros(0, np.int32))
    engine.set_factors(P, Q)
    ids, sc = check(engine, P, Q, np.arange(m, dtype=np.int32), N, uq_indptr, np.zeros(0, np.int32), RANK_TC)
    assert ids[0].tolist() == [1, 2, 3, 4, 5, 6, 8, 9, 10, 11]


def test_tc_overflow_pool_keeps_exactness(engine):
    """~150 tracks share the top score of every user: more near-ties than the 32 a shared-memory row
    buffer keeps, few enough for the global overflow pool -- no exact-kernel fallback needed and the
    ids are still (score desc, id asc)."""
    m, n, d, N = 200, 20000, 64, 10
    rng = np.random.default_rng(11)
    P = np.abs(rng.normal(size=(m, d))).astype(np.float32)
    Q = (np.abs(rng.normal(size=(n, d))) * 0.1).astype(np.float32)
    top = np.abs(rng.normal(size=(1, d))).astype(np.float32) * 2.0
    dup = rng.choice(n, 150, replace=False)
    Q[dup] = top                                          # identical rows -> identical exact scores
    uq_indptr = np.zeros(m + 1, np.int64)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), uq_indptr, np.zeros(0, np.int32))
    engine.set_factors(P, Q)
    ids, sc = check(engine, P, Q, np.arange(m, dtype=np.int32), N, uq_indptr, np.zeros(0, np.int32), RANK_TC)
    assert ids[0].tolist() == sorted(dup.tolist())[:10]


def test_exact_kernel_catalog_split_and_stats(engine):
    """Few rows against a big catalog: the exact kernel splits the catalog over CTAs and merges the
    partial lists -- ids and scores must still be the oracle's, bit for bit; rank_stats is callable."""
    from oracle import topn
    from yue_b200.engine import RANK_EXACT, RANK_TC
    m, n, d = 40, 70000, 64
    indptr, uq = synth.mask_csr(m, n, 30, seed=5)
    P, Q = synth.init_factors(m, n, d, seed=9)
    Q[1000:1040] = Q[999]                           # exact ties across a run of ids: order must be id ascending
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), indptr, uq)
    engine.set_factors(P, Q)
    users = np.arange(m, dtype=np.int32)
    for N in (10, 50):
        ids, sc = engine.rank_topn(users, N, RANK_EXACT)
        rid, rsc = topn.topn_exact(P, Q, users, N, indptr, uq)
        assert np.array_equal(ids, rid) and np.array_equal(sc, rsc)
    rep = np.arange(m, dtype=np.int32).repeat(8)        # every user eight times in one batch
    ids, sc = engine.rank_topn(rep, 10, RANK_TC)
    rid, rsc = topn.topn_exact(P, Q, rep, 10, indptr, uq)
    assert np.array_equal(ids, rid) and np.array_equal(sc, rsc)
    fb, spilled = engine.rank_stats()
    assert fb >= 0 and spilled >= 0


def test_tc_refuses_what_it_cannot_hold(engine):
    """N > 32 does not fit the tcgen05 kernel's per-row buffer: RANK_TC says so, RANK_AUTO takes the exact kernel."""
    from oracle import topn
    from yue_b200.engine import RANK_AUTO, YueError
    m, n = 300, 4000
    indptr, uq = synth.mask_csr(m, n, 20, seed=1)
    P, Q = synth.init_factors(m, n, 64, seed=2)
    engine.set_interactions(m, n, np.zeros(m + 1, np.int64), np.zeros(0, np.int32), indptr, uq)
    engine.set_factors(P, Q)
    users = np.arange(m, dtype=np.int32)
    with pytest.raises(YueError):
        engine.rank_topn(users, 40, RANK_TC)
    ids, sc = engine.rank_topn(users, 40, RANK_AUTO)
    rid, rsc = topn.topn_exact(P, Q, users, 40, indptr, uq)
    assert np.array_equal(ids, rid) and np.array_equal(sc, rsc)
