"""K9 (csrc/lightgcn.cuh, gcn_steps_kernel) at the switches tests/test_lightgcn.py does not reach.

Each test names the switch it pins and asserts, through oracle/lightgcn_ref.plan / gcn_hash or the batch's shape, that its
input takes it.  First-step gradients are read back through Adam's first moment (m_1 = 0.1 g) and compared row by row with
the float64 oracle under oracle/lightgcn_cases.row_bound, calibrated in tests/test_lightgcn_edges_oracle.py.  The kernel sums
every value in a fixed order (a light row in CSR order, a heavy row in chunk order, a graph row's slots in slot order, the
loss per group), so results that must not depend on the CTA count, on how a step range is split into launches or on where
the negatives come from are compared bit for bit."""
import numpy as np
import pytest

from oracle import lightgcn_cases as lc
from oracle import lightgcn_ref as lg
from oracle import philox

pytestmark = pytest.mark.gpu
LR = 0.002


@pytest.fixture(scope="module")
def edge():
    return lc.edge_graph()


@pytest.fixture(scope="module")
def inv():
    return lc.invariant_graph()


def _first_step(engine, g, L, d, u, i, j):
    """One gcn_apply from fresh tables; loss and every row of the gradient against the oracle."""
    U, V = lc.edge_tables(g, d)
    engine.set_factors(U, V)
    E0 = np.concatenate([U, V]).astype(np.float64)
    ref_loss, g64 = lg.loss_and_grad(g.A, E0, g.m, u, i, j, lc.REG, L)
    bound = lc.row_bound(g.A, E0, g.m, u, i, j, lc.REG, L)
    loss = engine.gcn_apply(u, i, j, LR, lc.REG, n_layers=L)
    assert abs(loss - ref_loss) <= 2e-5 * abs(ref_loss)
    mu, mt, _, _, steps = engine.gcn_moments()
    assert steps == 1
    got = np.concatenate([mu, mt]).astype(np.float64) / 0.1
    dev = np.linalg.norm(got - g64, axis=1)
    assert lc.excess(dev, bound) <= 1.0, (np.argmax(dev / np.maximum(bound, 1e-300)), lc.excess(dev, bound))
    return E0, g64


@pytest.mark.parametrize("L,d,pad", lc.FIRST_STEP_CASES, ids=["L%d-d%d%s" % (L, d, "" if p else "-unpadded") for L, d, p in lc.FIRST_STEP_CASES])
def test_first_step_gradient_per_row(engine, edge, monkeypatch, L, d, pad):
    """n_layers 1..4 (at L = 1 the Adam phase reads the stamped source; at L = 4 E[3] and the last phase slots), every
    instantiation: ld <= 32 G = 8, <= 64 G = 16, <= 128 G = 32, above NC = 2 (d = 129: one lane of the second chunk; d = 256:
    every lane, two chunks), d = 4 (one lane), d = 100 padded to 128 and unpadded (YUE_LD_PAD128=0: 25 of 32 lanes).  On a
    graph with a row of > 4096 neighbours (chunks of 72), a heavy user, rows of degree exactly 64 (a light segment of 64
    edges) and 65 (chunks of 64 and 1), padded empty chunks, a two-row segment of exactly 64 edges; a batch with repeated
    rows and a connected user whose layers 1 and 3 are exactly zero (l2_normalize's clamp: its NB_k is 1e6 g)."""
    g, m = edge, edge.m
    assert g.deg[m + lc.BIG_TRACK] > 4096 and [c[2] for c in g.chunks if c[0] == m + lc.DEG65_TRACK] == [64, 1]
    assert (m + lc.DEG64_TRACK, 1) in g.segs and (lc.SEG64_USERS[0], 2) in g.segs and lc.HEAVY_USER in g.heavy
    assert any(c[5] == lg.PAD_CHUNK for c in g.chunks)
    if not pad:
        monkeypatch.setenv("YUE_LD_PAD128", "0")
    g.set_on(engine)
    u, i, j = lc.edge_batch(g, 96)
    assert u[8] == u[7] and i[8] == i[7] and j[9] == i[7]
    E0, g64 = _first_step(engine, g, L, d, u, i, j)
    _, layers, _ = lg.propagate(g.A, E0, L)
    assert lc.ZERO_USER in u and g.deg[lc.ZERO_USER] > 0 and not layers[1][lc.ZERO_USER].any()
    assert np.abs(g64[m + lc.ZERO_TRACK]).max() > 1e4 * np.abs(g64[lc.HEAVY_USER]).max()     # the clamp's 1e6


def test_hash_probe_chains_collide_and_wrap(engine, edge):
    """The stamped rows' shared-memory hash (batches of <= 1024): three rows in bucket 8191, the last bucket, so the
    probes of two of them wrap to bucket 0, where rows 0, 4181 and 10946 also land.  Every one of them has neighbours, so a
    lookup that stops early loses a row of NB_L in the first backward product.  L = 1 (the hash feeds the Adam phase) and
    L = 3."""
    g, m = edge, edge.m
    rows = [lc.HASH_0[0], lc.HASH_0[1], lc.HASH_8191[0], lc.HASH_8191[1], lc.HASH_8191[2], lc.HASH_0[2]]
    u = np.array([rows[0], rows[1], rows[0]], np.int32)
    i = np.array([rows[2] - m, rows[4] - m, lc.BIG_TRACK], np.int32)
    j = np.array([rows[3] - m, rows[5] - m, rows[4] - m], np.int32)
    stamped = set(u.tolist()) | set((m + i).tolist()) | set((m + j).tolist())
    assert [lg.gcn_hash(r) for r in lc.HASH_8191] == [8191] * 3 and [lg.gcn_hash(r) for r in lc.HASH_0] == [0] * 3
    assert set(lc.HASH_ROWS) <= stamped and all(g.deg[r] > 0 for r in stamped) and 3 * len(u) <= lg.SMEM_SLOTS
    g.set_on(engine)
    for L in (1, 3):
        _first_step(engine, g, L, 16, u, i, j)


@pytest.mark.parametrize("B", lc.SLOT_BATCHES)
def test_batches_around_the_shared_slot_list(engine, edge, B):
    """3 B slots against the 3072 kept in shared memory: B = 1 and 1024 take the shared list and the hash, B = 1025 and
    4096 (the largest batch) read the slot list from global memory and look stamped rows up by their stamps."""
    g = edge
    assert (3 * B <= lg.SMEM_SLOTS) == (B <= 1024)
    g.set_on(engine)
    u, i, j = lc.edge_batch(g, B)
    _first_step(engine, g, 3, 32, u, i, j)


@pytest.mark.parametrize("batch", [1024, 1025])
def test_epoch_step_with_the_fused_sampler_around_the_slot_list(engine, edge, batch):
    """gcn_epoch's first step at batch 1024 (3072 slots: shared) and 1025 (global), negatives drawn in the kernel."""
    g = edge
    g.set_on(engine)
    U, V = lc.edge_tables(g, 32)
    engine.set_factors(U, V)
    engine.gcn_set_events(g.eu, g.ei)
    seed = 99
    neg = philox.sample_negatives(seed, 0, g.eu, g.n, g.log.uq_indptr, g.log.uq_items, slot=lg.NEG_SLOT)
    u, i, j = g.eu[:batch], g.ei[:batch], neg[:batch]
    E0 = np.concatenate([U, V]).astype(np.float64)
    ref_loss, g64 = lg.loss_and_grad(g.A, E0, g.m, u, i, j, lc.REG, 3)
    loss = engine.gcn_epoch(batch, LR, lc.REG, seed, 0, n_layers=3, step_begin=0, step_end=1)
    assert abs(loss[0] - ref_loss) <= 2e-5 * abs(ref_loss)
    mu, mt, _, _, _ = engine.gcn_moments()
    dev = np.linalg.norm(np.concatenate([mu, mt]).astype(np.float64) / 0.1 - g64, axis=1)
    assert lc.excess(dev, lc.row_bound(g.A, E0, g.m, u, i, j, lc.REG, 3)) <= 1.0


def _tables_follow(P, Q, rU, rV, U, V):
    """tests/test_lightgcn.py's criterion after several Adam steps: >= 99.5 % of the entries within 2 % of the distance moved."""
    got, ref = np.concatenate([P, Q]).astype(np.float64), np.concatenate([rU, rV])
    moved = np.abs(ref - np.concatenate([U, V]).astype(np.float64))
    assert (np.abs(got - ref) <= 0.02 * moved + 1e-9).mean() >= 0.995


def _state(engine):
    P, Q = engine.get_factors()
    mu, mt, vu, vt, steps = engine.gcn_moments()
    return [P, Q, mu, mt, vu, vt, np.array([steps])]


def _same_bits(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def test_mixed_launch_alternates_global_and_shared_slot_lists(engine):
    """One launch over T = 2700 events at batch 1100: steps of 1100, 1100 (3300 slots: global) and 500 (1500: shared, the
    hash) triplets.  Losses and tables follow the oracle; the launch gives the bits of launches [0, 2) + [2, 3)."""
    g = lc.mixed_graph()
    assert len(g.eu) == 2700 and [min(1100, 2700 - s * 1100) * 3 > lg.SMEM_SLOTS for s in range(3)] == [True, True, False]
    assert g.heavy
    g.set_on(engine)
    U, V = lg.init_tables(g.m, g.n, 20, 5)
    U, V = U * 10, V * 10
    seed = 31
    rU, rV, rloss, _ = lg.train(g.A, U, V, g.eu, g.ei, g.log.uq_indptr, g.log.uq_items, 1100, LR, lc.REG, seed)
    engine.set_factors(U, V)
    engine.gcn_set_events(g.eu, g.ei)
    loss = engine.gcn_epoch(1100, LR, lc.REG, seed, 0)
    assert len(loss) == len(rloss) == 3 and np.allclose(loss, rloss, rtol=5e-4)
    whole = _state(engine) + [loss]
    _tables_follow(whole[0], whole[1], rU, rV, U, V)
    engine.set_factors(U, V)
    split = np.concatenate([engine.gcn_epoch(1100, LR, lc.REG, seed, 0, step_begin=0, step_end=2),
                            engine.gcn_epoch(1100, LR, lc.REG, seed, 0, step_begin=2, step_end=3)])
    assert _same_bits(whole, _state(engine) + [split])


@pytest.mark.parametrize("d", [20, 50, 100, 160], ids=["G8", "G16", "G32", "NC2"])
def test_bits_do_not_depend_on_ctas_launch_split_or_negative_source(engine, inv, monkeypatch, d):
    """Exact invariants of a whole pass (11 batches of 128 and one of 50) over a log with a 200-user track (4 chunks), a
    100-track user (2) and other heavy tracks, at every instantiation: P, Q, both moments and the losses are the same bits with YUE_GCN_CTAS 1,
    7, 148 and unset; as one launch and as 5 + 7; gcn_apply on the sampler's negatives gives gcn_epoch's step 0; and the
    same call twice after set_factors gives the same bits."""
    g = inv
    m = g.m
    assert len(g.eu) == 11 * 128 + 50 and m - 1 in g.heavy and [c[2] for c in g.chunks if c[0] == m] == [64, 64, 64, 8]
    g.set_on(engine)
    U, V = lg.init_tables(g.m, g.n, d, 3)
    U, V = U * 10, V * 10
    seed = 17

    def run(**kw):
        engine.set_factors(U, V)
        engine.gcn_set_events(g.eu, g.ei)
        if "split" in kw:
            loss = np.concatenate([engine.gcn_epoch(128, LR, lc.REG, seed, 0, step_begin=0, step_end=5),
                                   engine.gcn_epoch(128, LR, lc.REG, seed, 0, step_begin=5, step_end=12)])
        else:
            loss = engine.gcn_epoch(128, LR, lc.REG, seed, 0, step_end=kw.get("end", -1))
        return _state(engine) + [loss]
    base = run()
    assert len(base[-1]) == 12 and base[-2][0] == 12
    for ctas in ("1", "7", "148"):
        monkeypatch.setenv("YUE_GCN_CTAS", ctas)
        assert _same_bits(base, run()), ctas
    monkeypatch.delenv("YUE_GCN_CTAS")
    assert _same_bits(base, run(split=True))
    first = run(end=1)
    neg = philox.sample_negatives(seed, 0, g.eu, g.n, g.log.uq_indptr, g.log.uq_items, slot=4)
    for _ in range(2):
        engine.set_factors(U, V)
        loss = engine.gcn_apply(g.eu[:128], g.ei[:128], neg[:128], LR, lc.REG)
        assert _same_bits(first, _state(engine) + [np.array([loss])])


@pytest.mark.parametrize("L", [1, 4])
def test_multi_step_runs_and_finalize_at_one_and_four_layers(engine, inv, L):
    """12 steps (the last a partial batch) at n_layers 1 and 4 against lg.train, then gcn_finalize(L) against lg.embeddings
    row by row."""
    g = inv
    g.set_on(engine)
    U, V = lg.init_tables(g.m, g.n, 50, 9)
    seed = 23
    rU, rV, rloss, _ = lg.train(g.A, U, V, g.eu, g.ei, g.log.uq_indptr, g.log.uq_items, 128, LR, lc.REG, seed, n_layers=L)
    engine.set_factors(U, V)
    engine.gcn_set_events(g.eu, g.ei)
    loss = engine.gcn_epoch(128, LR, lc.REG, seed, 0, n_layers=L)
    assert len(loss) == 12 and np.allclose(loss, rloss, rtol=5e-4)
    P, Q = engine.get_factors()
    _tables_follow(P, Q, rU, rV, U, V)
    engine.gcn_finalize(L)
    FU, FV = engine.get_factors()
    wU, wV = lg.embeddings(g.A, P, Q, n_layers=L)
    want = np.concatenate([wU, wV])
    rel = np.linalg.norm(np.concatenate([FU, FV]) - want, axis=1) / np.linalg.norm(want, axis=1)
    assert rel.max() <= 1e-5


def test_refusals_of_layers_and_batch(engine, inv):
    """n_layers 0 and 5 on every entry point; a batch of 4097 triplets on gcn_apply."""
    from yue_b200.engine import YueError
    g = inv
    g.set_on(engine)
    U, V = lg.init_tables(g.m, g.n, 8, 1)
    engine.set_factors(U, V)
    engine.gcn_set_events(g.eu, g.ei)
    for L in (0, 5):
        with pytest.raises(YueError):
            engine.gcn_epoch(128, LR, lc.REG, 1, 0, n_layers=L)
        with pytest.raises(YueError):
            engine.gcn_apply(g.eu[:4], g.ei[:4], g.ei[:4], LR, lc.REG, n_layers=L)
        with pytest.raises(YueError):
            engine.gcn_finalize(L)
    idx = np.arange(4097) % len(g.eu)
    with pytest.raises(YueError):
        engine.gcn_apply(g.eu[idx], g.ei[idx], g.ei[idx], LR, lc.REG)
    assert engine.gcn_moments()[4] == 0                        # nothing ran
    engine.gcn_apply(g.eu[:4], g.ei[:4], g.ei[:4], LR, lc.REG, n_layers=4)
    assert engine.gcn_moments()[4] == 1
