"""K9's work plan and the first-step gradient tolerance of tests/test_lightgcn_edges_gpu.py, on the CPU.

The plan: oracle/lightgcn_ref.plan restates gcn_plan's rules (segments, heavy rows, chunks, padding); here it is held to
lists worked out by hand for a small log, so that the GPU tests can use it to show which path their inputs take.

The tolerance (oracle/lightgcn_cases.row_bound): per row, BOUND_K * EPS32 * |row of the magnitude pass|, with BOUND_K = 1024.
It is calibrated at every shape the GPU file holds the kernel to (the 13 first-step cases and the 4 batch sizes around the
slot list, on the 36 000-row edge graph):
  * the float32 restatement of the gradient, once in CSR order and once with every neighbour list reversed, stays within
    a quarter of the bound on every row (measured: at most 0.17 of it, at B = 1; 0.01-0.07 elsewhere);
  * each kernel mistake below, written as a float64 variant of the gradient, moves some row by at least 20 bounds at every
    shape (each margin is printed with -s; the smallest measured is 21, a hash miss at B = 1024, the next 78):
      a layer's norm-backward NB_k dropped (every k); the projection n (n . g) of NB_k dropped (every k); one stamped row
      missing from the first backward product, as a hash miss would, at the batches that build the hash (each of the
      batch's rows on the colliding probe chains and its heavy rows, the least visible one counts -- among thousands of
      stamped rows some are too faint to see one by one; a row whose NB_L vanishes is left out: at L = 1 the zero pair's
      track has a gradient parallel to its layer, and a miss of it changes nothing); the least visible chunk of every heavy row dropped from the row's sums; the last
      neighbour of a segment's row attributed to the segment's next row (at two segments); edge weights c instead of c^2; NB_{k+1} added in
      place of NB_k."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import lightgcn_cases as lc
from oracle import lightgcn_ref as lg


def test_plan_matches_hand_computed_lists_for_a_small_log():
    """3 users, 190 tracks.  User 0 plays tracks 0..129 (heavy: 130 > 64, chunks of max(ceil(sqrt(130) / 8) * 8, 64) = 64:
    0..63, 64..127, 128..129, then one empty chunk to a multiple of 4), user 1 plays 130..189 (60), user 2 plays 0..4 (5:
    60 + 5 > 64 closes user 1's segment).  Tracks 0..4 have 2 users, the others 1; row m = 3 opens a segment of its own."""
    m, n = 3, 190
    uq_indptr = np.array([0, 130, 190, 195])
    uq_items = np.concatenate([np.arange(130), np.arange(130, 190), np.arange(5)])
    deg, it_indptr = lg.degrees(m, n, uq_indptr, uq_items)
    assert deg[:3].tolist() == [130, 60, 5] and deg[3:8].tolist() == [2] * 5 and (deg[8:] == 1).all()
    segs, heavy, chunks = lg.plan(m, n, uq_indptr, it_indptr)
    track_segs = [(3 + 8 * s, 8) for s in range(23)] + [(187, 6)]          # 190 = 23 * 8 + 6 track rows
    assert segs == [(1, 1), (3, 8)] + track_segs[1:23] + [(187, 6), (2, 1)]    # by neighbours: 60, 13, 8 x 22, 6, 5
    assert heavy == [0]
    assert chunks == [(0, 0, 64, 0, 0, 3, 0), (0, 64, 64, 1, 0, 3, 0), (0, 128, 2, 2, 0, 3, 0),
                      (0, 0, 0, 3, 3, lg.PAD_CHUNK, 1)]


def test_plan_orders_heavy_rows_and_sizes_chunks_past_4096():
    """Two heavy rows, the lighter first in row order: the heavier is planned first.  A row of 5000 neighbours takes chunks
    of ceil(sqrt(5000) / 8) * 8 = 72 (more than 64): 70 of them, the last of 32."""
    m, n = 5000, 2
    uq_indptr = np.concatenate([[0], np.cumsum(np.r_[np.full(70, 2), np.full(4930, 1)])]).astype(np.int64)
    uq_items = np.concatenate([np.tile([0, 1], 70), np.ones(4930)]).astype(np.int32)
    deg, it_indptr = lg.degrees(m, n, uq_indptr, uq_items)
    assert deg[m] == 70 and deg[m + 1] == 5000
    segs, heavy, chunks = lg.plan(m, n, uq_indptr, it_indptr)
    assert heavy == [m + 1, m]
    big = [c for c in chunks if c[0] == m + 1]
    assert len(big) == 70 and all(c[2] == 72 for c in big[:-1]) and big[-1][1:3] == (69 * 72, 32)
    assert [c[2] for c in chunks if c[0] == m] == [64, 6] and len(chunks) == 72        # 72 % 4 == 0: no padding
    assert sum(sg[1] for sg in segs) == m and all(sg[1] == 8 for sg in segs)


def test_gcn_hash_is_the_kernels_and_the_edge_graph_takes_every_switch():
    """The rows the edge graph plants collide in the hash; the graph has every row kind the GPU file names."""
    assert [lg.gcn_hash(r) for r in lc.HASH_8191] == [8191] * 3 and [lg.gcn_hash(r) for r in lc.HASH_0] == [0] * 3
    g = lc.edge_graph()
    m = g.m
    assert g.m + g.n >= 30000 and all(g.deg[r] > 0 for r in lc.HASH_ROWS)
    assert g.deg[m + lc.BIG_TRACK] > 4096 and g.deg[lc.HEAVY_USER] > lg.HEAVY
    assert g.deg[m + lc.DEG64_TRACK] == 64 and g.deg[m + lc.DEG65_TRACK] == 65
    assert g.heavy[:1] == [m + lc.BIG_TRACK] and {lc.HEAVY_USER, m + lc.DEG65_TRACK} <= set(g.heavy)
    big = [c for c in g.chunks if c[0] == m + lc.BIG_TRACK]
    assert big[0][2] > lg.HEAVY and len(big) > 50
    assert [c[2] for c in g.chunks if c[0] == m + lc.DEG65_TRACK] == [64, 1]
    assert any(c[5] == lg.PAD_CHUNK for c in g.chunks) and len(g.chunks) % 4 == 0
    assert (m + lc.DEG64_TRACK, 1) in g.segs                                 # degree 64 is light: a segment of 64 edges
    assert (lc.SEG64_USERS[0], 2) in g.segs                                  # 30 + 34: two rows, closed at 64 edges
    assert any(nr == 8 for _, nr in g.segs)
    last = [sg for sg in g.segs if sg[0] + sg[1] == m]
    assert len(last) == 1 and last[0][1] < 8 and g.deg[last[0][0]:m + 1].sum() <= 64   # only r == m closes it
    A = g.A.tocsr()
    assert A[lc.ZERO_USER].indices.tolist() == [m + lc.ZERO_TRACK] and A[lc.ZERO_USER].data.tolist() == [4.0]


def _reversed(A):
    """A with every row's neighbour list stored in reverse (scipy's products then sum in that order)."""
    A = A.tocsr()
    idx, dat = A.indices.copy(), A.data.copy()
    for r in range(A.shape[0]):
        a, b = A.indptr[r], A.indptr[r + 1]
        idx[a:b], dat[a:b] = idx[a:b][::-1], dat[a:b][::-1]
    return sp.csr_matrix((dat, idx, A.indptr.copy()), shape=A.shape)


def grad_variant(A, E0, m, u, i, j, reg, L, walk=None, drop_nb=None, no_proj=None, nb_shift=False):
    """The float64 gradient as the kernel computes it -- every product row by row with `walk` (default A) -- with one
    mistake: NB_drop_nb = 0, NB_no_proj without its projection, or NB_{k+1} added where NB_k belongs."""
    u, i, j = (np.asarray(x, dtype=np.int64) for x in (u, i, j))
    W = A if walk is None else walk
    F, layers, rinv = lg.propagate(W, E0, L)
    Fu, Fi, Fj = F[u], F[m + i], F[m + j]
    c = 1.0 / (1.0 + np.exp((Fu * Fi).sum(1) - (Fu * Fj).sum(1)))
    G = np.zeros_like(E0)
    np.add.at(G, u, -c[:, None] * (Fi - Fj) + reg * Fu)
    np.add.at(G, m + i, -c[:, None] * Fu + reg * Fi)
    np.add.at(G, m + j, c[:, None] * Fu + reg * Fj)

    def nb(k):
        if k == 0:
            return G
        if k == drop_nb:
            return np.zeros_like(G)
        E, r = layers[k], rinv[k]
        n_ = E * r[:, None]
        out = r[:, None] * G if k == no_proj else r[:, None] * (G - n_ * (n_ * G).sum(1)[:, None])
        clamped = (E * E).sum(1) <= lg.EPS_NORM
        out[clamped] = r[clamped, None] * G[clamped]
        return out
    D = nb(L)
    for k in range(L - 1, -1, -1):
        D = W @ D + nb(k + 1 if nb_shift else k)
    return D


def _shapes():
    for L, d, pad in lc.FIRST_STEP_CASES:
        yield "L=%d d=%d%s B=96" % (L, d, "" if pad else " unpadded"), L, d, 96
    for B in lc.SLOT_BATCHES:
        yield "L=3 d=32 B=%d" % B, 3, 32, B


@pytest.fixture(scope="module")
def edge():
    return lc.edge_graph()


@pytest.mark.parametrize("name,L,d,B", list(_shapes()), ids=[s[0] for s in _shapes()])
def test_bound_holds_float32_inside_and_every_mutant_far_outside(edge, name, L, d, B):
    g, m = edge, edge.m
    A = g.A.tocsr()
    U, V = lc.edge_tables(g, d)
    E0 = np.concatenate([U, V]).astype(np.float64)
    u, i, j = lc.edge_batch(g, B)
    _, g64 = lg.loss_and_grad(A, E0, m, u, i, j, lc.REG, L)
    bound = lc.row_bound(A, E0, m, u, i, j, lc.REG, L)
    rows = np.linalg.norm

    # float32, two summation orders: well inside
    inside = 0.0
    for Ax in (A, _reversed(A)):
        _, g32 = lg.loss_and_grad(Ax, E0, m, u, i, j, lc.REG, L, dtype=np.float32)
        inside = max(inside, lc.excess(rows(g32.astype(np.float64) - g64, axis=1), bound))
    assert inside <= 0.25, (name, inside)

    def margin(gm):
        return lc.excess(rows(gm - g64, axis=1), bound)
    assert margin(grad_variant(A, E0, m, u, i, j, lc.REG, L)) <= 1e-6      # the variant without a mistake is the oracle
    got = {}
    got["drop NB_k"] = min(margin(grad_variant(A, E0, m, u, i, j, lc.REG, L, drop_nb=k)) for k in range(1, L + 1))
    got["no projection"] = min(margin(grad_variant(A, E0, m, u, i, j, lc.REG, L, no_proj=k)) for k in range(1, L + 1))
    got["NB_{k+1} for NB_k"] = margin(grad_variant(A, E0, m, u, i, j, lc.REG, L, nb_shift=True))
    W = A.copy()
    W.data = np.sqrt(W.data)
    got["c for c^2"] = margin(grad_variant(A, E0, m, u, i, j, lc.REG, L, walk=W))

    # a hash miss on stamped row s: the first backward product loses A[:, s] NB_L[s], which the remaining L - 1 products
    # carry on -- the gradient moves by (A^L)[:, s] NB_L[s] (A is symmetric)
    F, layers, rinv = lg.propagate(A, E0, L)
    stamped = np.unique(np.concatenate([u, m + i, m + j]))
    stamped = stamped[g.deg[stamped] > 0]
    c = 1.0 / (1.0 + np.exp((F[u] * F[m + i]).sum(1) - (F[u] * F[m + j]).sum(1)))
    G = np.zeros_like(E0)
    np.add.at(G, u, -c[:, None] * (F[m + i] - F[m + j]) + lc.REG * F[u])
    np.add.at(G, m + i, -c[:, None] * F[u] + lc.REG * F[m + i])
    np.add.at(G, m + j, c[:, None] * F[u] + lc.REG * F[m + j])
    n_ = layers[L] * rinv[L][:, None]
    nbL = rinv[L][:, None] * (G - n_ * (n_ * G).sum(1)[:, None])
    clamped = (layers[L] ** 2).sum(1) <= lg.EPS_NORM
    nbL[clamped] = rinv[L][clamped, None] * G[clamped]
    vanishes = rows(nbL, axis=1) <= 1e-9 * rinv[L] * rows(G, axis=1)      # the projection takes all of g
    stamped = np.intersect1d(stamped[~vanishes[stamped]], list(lc.HASH_ROWS) + g.heavy)
    P = sp.csr_matrix((np.ones(len(stamped)), (stamped, np.arange(len(stamped)))), shape=(A.shape[0], len(stamped)))
    for _ in range(L):
        P = A @ P
    P = P.toarray() * rows(nbL[stamped], axis=1)[None, :]
    if 3 * B <= lg.SMEM_SLOTS:                                                # larger batches build no hash
        got["hash miss"] = min(lc.excess(P[:, s], bound) for s in range(len(stamped)))

    # the least visible chunk of every heavy row, dropped from that row's sums in every product
    worst = np.inf
    for h in g.heavy:
        cks = [ck for ck in g.chunks if ck[0] == h]
        a, b = A.indptr[h], A.indptr[h + 1]
        cols, vals = A.indices[a:b], A.data[a:b]
        size = [rows(vals[ck[1]:ck[1] + ck[2]] @ E0[cols[ck[1]:ck[1] + ck[2]]]) for ck in cks]
        ck = cks[int(np.argmin(size))]
        Wc = A.copy()
        Wc.data[a + ck[1]:a + ck[1] + ck[2]] = 0
        worst = min(worst, margin(grad_variant(A, E0, m, u, i, j, lc.REG, L, walk=Wc)))
    got["chunk dropped"] = worst

    # at two segment boundaries (the 64-edge segment, whose rows the batch holds, and tracks 79 | 80 of the heavy user,
    # played twice | once): a row's last neighbour walked as the next row's
    Wl = A.tolil()
    for r in (lc.SEG64_USERS[0], m + 79):
        assert any(r0 <= r and r + 1 < r0 + nr for r0, nr in g.segs)
        col = A.indices[A.indptr[r + 1] - 1]
        Wl[r + 1, col] = A[r, col]
        Wl[r, col] = 0
    got["neighbour to next row"] = margin(grad_variant(A, E0, m, u, i, j, lc.REG, L, walk=Wl.tocsr()))

    print("\n%-28s float32 within %.3f of the bound; mutants, bounds away: %s" % (
        name, inside, ", ".join("%s %.3g" % kv for kv in got.items())))
    for k, v in got.items():
        assert v >= 20, (name, k, v)
