"""Inputs that drive K9 (csrc/lightgcn.cuh) down its rarely taken paths, and the per-row tolerance its first-step gradient is
held to.  Shared by tests/test_lightgcn_edges_oracle.py (which calibrates the tolerance on the CPU and shows that broken
kernels land outside it at every shape below) and tests/test_lightgcn_edges_gpu.py (which holds the kernel to it).

The tolerance.  Every float32 operation rounds by at most EPS32 of its result, and the error of a sum is bounded by the sum
of its terms' MAGNITUDES, not by the sum.  grad_magnitude() is the gradient computation with every term replaced by its
absolute value (the norm-backward's projection added instead of subtracted, |c| for the sigmoid factor), so row r of the
gradient may be wrong by about EPS32 * |row r of the magnitude pass| times a small factor for the depth of the computation.
row_bound() allows BOUND_K of that factor.  Measured by the oracle test on every case below: float32 restatements of the
same arithmetic in two summation orders stay within 0.25 of it (0.17 at worst); every broken variant it tries
lands at least 20x outside at every case.  A row the batch cannot reach has a magnitude of exactly zero: the kernel must
leave it exactly zero."""
import numpy as np

from yue_b200 import synth

from . import lightgcn_ref as lg

EPS32 = 2.0 ** -24
BOUND_K = 1024
REG = 0.001


def make_log(m, n, eu, ei):
    """A PlayLog from training events given in file order (no held-out part)."""
    eu, ei = np.asarray(eu, np.int32), np.asarray(ei, np.int32)
    order = np.argsort(eu, kind="stable")
    ev_indptr = np.zeros(m + 1, np.int64)
    np.cumsum(np.bincount(eu, minlength=m), out=ev_indptr[1:])
    uq_indptr, uq_items, _ = synth._csr_unique(eu[order], ei[order], m, n)
    return synth.PlayLog(m, n, ev_indptr, np.ascontiguousarray(ei[order]), uq_indptr, uq_items,
                         np.zeros(m + 1, np.int64), np.zeros(0, np.int32))


class Graph(object):
    """A log in file order with its adjacency, its degrees and the kernel's plan of it."""

    def __init__(self, m, n, eu, ei):
        perm = np.random.default_rng(len(eu)).permutation(len(eu))
        self.m, self.n, self.eu, self.ei = m, n, np.asarray(eu, np.int32)[perm], np.asarray(ei, np.int32)[perm]
        self.log = make_log(m, n, self.eu, self.ei)
        self.A = lg.adjacency(m, n, self.eu, self.ei)
        self.deg, self.it_indptr = lg.degrees(m, n, self.log.uq_indptr, self.log.uq_items)
        self.segs, self.heavy, self.chunks = lg.plan(m, n, self.log.uq_indptr, self.it_indptr)

    def set_on(self, engine):
        lo = self.log
        engine.set_interactions(lo.m, lo.n, lo.ev_indptr, lo.ev_items, lo.uq_indptr, lo.uq_items)


# ---- the edge graph: 36 000 rows ----
EDGE_M, EDGE_N = 6000, 30000
BIG_TRACK, DEG64_TRACK, DEG65_TRACK = 1, 2, 3          # 4200 / 64 / 65 distinct users
HEAVY_USER = 5000                                       # 200 distinct tracks: 4 chunks, 65 in all, 3 empty ones pad
SEG64_USERS = (5001, 5002)                              # 30 + 34 neighbours: one segment of exactly 64 edges
ZERO_USER, ZERO_TRACK = 5900, 290                       # a pair alone in the graph; V[ZERO_TRACK] = 0 makes e_1, e_3 of the user 0
HASH_8191 = (6765, 17711, 28657)                        # graph rows with gcn_hash == 8191
HASH_0 = (0, 4181, 10946)                               # graph rows with gcn_hash == 0
HASH_ROWS = HASH_8191 + HASH_0


def edge_graph():
    m, n = EDGE_M, EDGE_N
    rng = np.random.default_rng(2026)
    eu, ei = [], []

    def add(u, t):
        eu.extend(np.broadcast_to(u, np.shape(t)) if np.ndim(t) else [u])
        ei.extend(np.atleast_1d(t))
    special = set(SEG64_USERS) | {HEAVY_USER, ZERO_USER} | set(range(m - 6, m))
    for u in range(m):
        if u not in special:
            add(u, rng.integers(300, n, int(rng.integers(1, 7))))
    for u in range(m - 6, m):                            # the last user segment is short: only row m closes it
        add(u, rng.integers(300, n, 1))
    add_users = np.arange(4200)
    eu.extend(add_users); ei.extend([BIG_TRACK] * 4200)
    rep = rng.choice(4200, 300, replace=False)          # played twice: weight 4
    eu.extend(rep); ei.extend([BIG_TRACK] * 300)
    eu.extend(range(4200, 4264)); ei.extend([DEG64_TRACK] * 64)
    eu.extend(range(4300, 4365)); ei.extend([DEG65_TRACK] * 65)
    add(HEAVY_USER, np.arange(50, 250))
    add(HEAVY_USER, np.arange(50, 80))
    add(SEG64_USERS[0], rng.choice(np.arange(300, n), 30, replace=False))
    add(SEG64_USERS[1], rng.choice(np.arange(300, n), 34, replace=False))
    add(ZERO_USER, [ZERO_TRACK, ZERO_TRACK])
    for r in HASH_ROWS:                                  # every hashed row has neighbours
        if r >= m:
            add(10, [r - m])
    return Graph(m, n, np.asarray(eu), np.asarray(ei))


def edge_tables(g, d, seed=7):
    """Tables 20x the class's initial scale (sigmoid away from 1/2), V[ZERO_TRACK] = 0."""
    U, V = lg.init_tables(g.m, g.n, d, seed)
    U, V = U * 20, V * 20
    V[ZERO_TRACK] = 0
    return U, V


def edge_batch(g, B, seed=3):
    """B triplets: the log's first events in file order and random negatives, with the switch rows planted in front -- the
    heavy rows, the 64-edge segment, the zero-layer user, the hash rows; a repeated user, track and negative."""
    rng = np.random.default_rng(seed + B)
    idx = np.arange(B) % len(g.eu)
    u, i, j = g.eu[idx].copy(), g.ei[idx].copy(), rng.integers(0, g.n, B).astype(np.int32)
    m = g.m
    plant = [(HEAVY_USER, BIG_TRACK, DEG65_TRACK), (ZERO_USER, ZERO_TRACK, DEG64_TRACK),
             (HASH_0[0], HASH_8191[0] - m, HASH_8191[1] - m), (HASH_0[1], HASH_8191[2] - m, HASH_0[2] - m),
             (SEG64_USERS[0], BIG_TRACK, 5), (SEG64_USERS[1], 6, DEG65_TRACK)]
    for x, (a, b, c) in enumerate(plant[:B]):
        u[x], i[x], j[x] = a, b, c
    if B >= 10:
        u[8], i[8], j[9] = u[7], i[7], i[7]               # repeated rows inside the batch, on both sides
    return u, i, j


# (n_layers, d, pad d in 65..127 to 128): every instantiation (G = 8 / 16 / 32, NC = 1 / 2), 1..4 layers, idle lanes
FIRST_STEP_CASES = [(1, 32, True), (2, 32, True), (3, 32, True), (4, 32, True), (3, 4, True), (3, 33, True), (3, 64, True),
                    (3, 100, True), (3, 100, False), (3, 129, True), (3, 256, True), (1, 256, True), (4, 129, True)]
# batch sizes around the shared slot list (3 B slots against SMEM_SLOTS), at L = 3, d = 32
SLOT_BATCHES = [1, 1024, 1025, 4096]


def grad_magnitude(A, E0, m, u, i, j, reg, n_layers):
    """loss_and_grad with every term replaced by its magnitude (see the module's docstring)."""
    u, i, j = (np.asarray(x, dtype=np.int64) for x in (u, i, j))
    F, layers, rinv = lg.propagate(A, E0, n_layers)
    Fa = np.abs(E0).astype(np.float64)
    for k in range(1, n_layers + 1):
        Fa += np.abs(layers[k]) * rinv[k][:, None]
    Fu, Fi, Fj = F[u], F[m + i], F[m + j]
    c = np.abs(1.0 / (1.0 + np.exp((Fu * Fi).sum(1) - (Fu * Fj).sum(1))))[:, None]
    Ga = np.zeros_like(Fa)
    np.add.at(Ga, u, c * (Fa[m + i] + Fa[m + j]) + reg * Fa[u])
    np.add.at(Ga, m + i, c * Fa[u] + reg * Fa[m + i])
    np.add.at(Ga, m + j, c * Fa[u] + reg * Fa[m + j])

    def nb(k):
        n_ = np.abs(layers[k]) * rinv[k][:, None]
        return rinv[k][:, None] * (Ga + n_ * (n_ * Ga).sum(1)[:, None])
    D = nb(n_layers)
    for k in range(n_layers - 1, 0, -1):
        D = A @ D + nb(k)
    return A @ D + Ga


def row_bound(A, E0, m, u, i, j, reg, n_layers):
    """The largest |g_kernel - g_oracle| accepted per row (2-norm over the row's entries)."""
    return BOUND_K * EPS32 * np.linalg.norm(grad_magnitude(A, E0, m, u, i, j, reg, n_layers), axis=1)


def excess(dev, bound):
    """max over rows of dev / bound; a row the bound says must be exactly zero counts as infinitely far if it is not."""
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bound > 0, dev / np.where(bound > 0, bound, 1.0), np.where(dev > 0, np.inf, 0.0))
    return float(r.max())


# ---- logs for the multi-step runs ----
def invariant_graph():
    """1458 events = 11 batches of 128 and one of 50; a track with 200 users (4 chunks), a user with 100 tracks (2) and the
    most played of the Zipf-drawn tracks (heavy too)."""
    rng = np.random.default_rng(11)
    m, n = 400, 300
    eu = np.concatenate([np.arange(200), np.full(100, m - 1), rng.integers(0, m - 1, 1158)])
    ei = np.concatenate([np.zeros(200, np.int64), np.arange(100, 200), np.minimum(rng.zipf(1.3, 1158), n - 1)])
    return Graph(m, n, eu, ei)


def mixed_graph():
    """2700 events: batches of 1100 take steps of 1100, 1100 and 500 triplets."""
    rng = np.random.default_rng(13)
    m, n = 900, 2000
    eu = np.concatenate([np.arange(300), rng.integers(0, m, 2400)])
    ei = np.concatenate([np.full(300, 5), np.minimum(rng.zipf(1.2, 2400), n - 1)])
    return Graph(m, n, eu, ei)
