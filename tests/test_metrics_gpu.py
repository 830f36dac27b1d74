"""K6: ranking metrics on the device against the oracle's restatement of evaluation/measure.py."""
import numpy as np
import pytest

from oracle import metrics
from yue_b200 import synth
from yue_b200.engine import MODE_HOGWILD, RANK_AUTO, RANK_EXACT, YueError

pytestmark = pytest.mark.gpu


def _oracle(log, users, ids, cuts):
    origin = [log.test_items[log.test_indptr[u]:log.test_indptr[u + 1]].tolist() for u in users]
    out = []
    for n in cuts:
        rec = [[t for t in row[:n] if t >= 0] for row in ids.tolist()]
        h = metrics.hits(origin, rec)
        out.append(dict(hits=sum(h), precision=metrics.precision(h, n), recall=metrics.recall(h, origin),
                        map=metrics.mean_ap(origin, rec, n), ndcg=metrics.ndcg(origin, rec, n),
                        distinct=len(set(t for r in rec for t in r))))
    return out


@pytest.mark.parametrize("N,cuts", [(10, [5, 10]), (100, [1, 20, 33, 64, 100])])
def test_device_metrics_match_measure(engine, N, cuts):
    log = synth.power_law_log(3000, 900, 150000, seed=11)
    P, Q = synth.init_factors(log.m, log.n, 32, seed=3)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    for ep in range(3):
        engine.bpr_epoch(0.05, 0.01, 0.01, 5, ep, MODE_HOGWILD)
    engine.set_test_set(log.test_indptr, log.test_items)
    users = log.test_users()
    ids, _ = engine.rank_topn(users, N, RANK_EXACT)
    sums, distinct = engine.rank_metrics(cuts)
    ref = _oracle(log, users, ids, cuts)
    B = len(users)
    for k, n in enumerate(cuts):
        assert sums[k, 0] == ref[k]["hits"]                                    # integer: exact
        assert distinct[k] == ref[k]["distinct"]
        assert sums[k, 0] / (B * n) == pytest.approx(ref[k]["precision"], rel=1e-13)
        assert sums[k, 1] / B == pytest.approx(ref[k]["recall"], rel=1e-12)
        assert sums[k, 2] / B == pytest.approx(ref[k]["map"], rel=1e-12)
        assert sums[k, 3] / B == pytest.approx(ref[k]["ndcg"], rel=1e-12)
    assert ref[-1]["hits"] > 0
    # the sums are reduced in a fixed order: a second call returns the same bits
    sums2, distinct2 = engine.rank_metrics(cuts)
    assert np.array_equal(sums, sums2) and np.array_equal(distinct, distinct2)


def test_device_metrics_edge_cases(engine):
    log = synth.power_law_log(200, 50, 6000, seed=2)             # tiny catalog: rows shorter than N get -1 padding
    P, Q = synth.init_factors(log.m, log.n, 10, seed=3)
    engine.set_interactions(log.m, log.n, log.ev_indptr, log.ev_items, log.uq_indptr, log.uq_items)
    engine.set_factors(P, Q)
    engine.set_test_set(log.test_indptr, log.test_items)
    users = np.arange(log.m, dtype=np.int32)                       # includes users with an empty test row
    ids, _ = engine.rank_topn(users, 40, RANK_AUTO)
    assert (ids < 0).any()
    sums, distinct = engine.rank_metrics([10, 40])
    origin = [log.test_items[log.test_indptr[u]:log.test_indptr[u + 1]].tolist() for u in users]
    ne = [b for b, o in enumerate(origin) if len(o)]                # an empty test row adds 0 to every sum on the device
    assert len(ne) < len(origin)
    for k, n in enumerate((10, 40)):
        rec = [[t for t in row[:n] if t >= 0] for row in ids.tolist()]
        assert sums[k, 0] == sum(metrics.hits(origin, rec))
        assert distinct[k] == len(set(t for r in rec for t in r))
        o_ne, r_ne = [origin[b] for b in ne], [rec[b] for b in ne]
        assert sums[k, 1] == pytest.approx(metrics.recall(metrics.hits(o_ne, r_ne), o_ne) * len(ne), rel=1e-12)
        assert sums[k, 2] == pytest.approx(metrics.mean_ap(o_ne, r_ne, n) * len(ne), rel=1e-12)
        assert sums[k, 3] == pytest.approx(metrics.ndcg(o_ne, r_ne, n) * len(ne), rel=1e-12)
    with pytest.raises(YueError):
        engine.rank_metrics([41])                                  # beyond the N of the last ranking call
