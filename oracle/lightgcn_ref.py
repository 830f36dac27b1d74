"""Oracle (test infrastructure) for LightGCN as the reference ships it: recommender/advanced/LightGCN.py:15-100 on
base/DeepRecommender:22-35 (SURVEY.md 8f row 4).

PINNED BY THE REFERENCE'S OWN TEXT, up to the meaning of the TensorFlow ops: the module imports TensorFlow 1.x and
`base.DeepRecommender`, a file without the `.py` extension (SURVEY R7), so it cannot be imported as it stands -- but
oracle/make_golden_lightgcn.py executes both files UNMODIFIED in the build container over oracle/tf1_shim.py (a stand-in for
the TF calls they make, on torch autograd in float64) with `random.randint` fed the Philox attempt stream, and commits the
run as tests/golden/lightgcn_small.npz: 60 Adam steps, their losses, U and V, the propagated tables.  This file reproduces
that run to 1e-12 (tests/test_lightgcn.py) -- the graph wiring, the loss, the optimiser's scope, the batch loop and the
sampler are therefore the reference's; what each TF op MEANS (duplicate entries of a SparseTensor add up, l2_normalize's
epsilon, Adam's formula) is restated from TensorFlow's documentation in the shim's header and has no pin in the reference
tree.  Its hand-derived gradient is also checked against a numerical one and, through the shim, against torch's autograd.

What the text says, line by line:

* 29-33  the adjacency is a SparseTensor with ONE ENTRY PER TRAINING EVENT (and its transpose), each carrying the play
         count of its (user, track) pair.  `tf.sparse_tensor_dense_matmul` adds duplicate entries up, so a pair played c
         times weighs c * c.  `adjacency()` builds exactly that list and lets scipy sum the duplicates.  (The
         degree-normalised values are the commented line 31: not what runs.)
* 37-45  e_0 = [U; V];  e_k = A e_{k-1} (the UN-normalised product feeds the next layer);  the layers are summed, not
         averaged:  F = e_0 + sum_k l2_normalize(e_k),  l2_normalize(x) = x * rsqrt(max(|x|^2, 1e-12))  (TF's epsilon).
* 56-79  batches are consecutive slices of `trainingData` in FILE order; five negatives are drawn per event but only the
         LAST one is kept (the appends sit outside the inner loop): one triplet per event.  The fifth draw = Philox slot 4.
* 83-87  loss = -sum log sigmoid(F_u . F_i - F_u . F_j) + regU * (l2_loss(F_u) + l2_loss(F_i) + l2_loss(F_j)) over the
         batch rows (with repeats), l2_loss(x) = sum(x^2) / 2.
* 88-90  tf.train.AdamOptimizer(lRate).minimize(loss): dense gradients (they flow through the sparse product into every
         row), beta1 0.9, beta2 0.999, epsilon 1e-8, lr_t = lr sqrt(1 - beta2^t) / (1 - beta1^t),
         var -= lr_t m / (sqrt(v) + epsilon).
* 94-98  num.max.iter passes over the batches.
* 101-105  predict(u) = F_items . F_user[u] -- the PROPAGATED embeddings rank, not U and V.
* DeepRecommender:30-31  U, V ~ truncated_normal(stddev 0.005): `init_tables` (redraw beyond two sigmas).
"""
import numpy as np
import scipy.sparse as sp

from . import philox

EPS_NORM = 1e-12
BETA1, BETA2, EPS_ADAM = 0.9, 0.999, 1e-8
NEG_SLOT = 4                    # the fifth draw of LightGCN.py:72-75 is the one that is kept


def adjacency(m, n, ev_user, ev_item):
    """LightGCN.py:29-33: (m+n) x (m+n) CSR, one entry of value count(u, t) per event and per direction, duplicates summed."""
    ev_user = np.asarray(ev_user, dtype=np.int64)
    ev_item = np.asarray(ev_item, dtype=np.int64)
    key = ev_user * n + ev_item
    uniq, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    vals = cnt[inv].astype(np.float64)
    rows = np.concatenate([ev_user, m + ev_item])
    cols = np.concatenate([m + ev_item, ev_user])
    A = sp.coo_matrix((np.concatenate([vals, vals]), (rows, cols)), shape=(m + n, m + n)).tocsr()
    A.sum_duplicates()
    return A


def init_tables(m, n, k, seed):
    """truncated_normal(stddev=0.005) of DeepRecommender:30-31 (values beyond two sigmas are redrawn), float32."""
    rng = np.random.default_rng(seed)

    def draw(shape):
        x = rng.standard_normal(shape)
        bad = np.abs(x) > 2
        while bad.any():
            x[bad] = rng.standard_normal(int(bad.sum()))
            bad = np.abs(x) > 2
        return (0.005 * x).astype(np.float32)
    return draw((m, k)), draw((n, k))


def propagate(A, E0, n_layers=3, dtype=np.float64):
    """LightGCN.py:37-45.  Returns F and what the backward pass needs: the layers and their 1/norm.

    dtype=np.float32 runs every operation in float32 (A's values too; scipy's sparse product accumulates in the matrix's
    type, in the order the CSR stores a row's neighbours): a second rounding of the same arithmetic, used only to calibrate
    the tolerances the float32 kernel is held to."""
    A, E0 = A.astype(dtype), np.asarray(E0).astype(dtype)
    layers, rinv = [E0], [None]
    F = E0.copy()
    for _ in range(n_layers):
        E = A @ layers[-1]
        r = (1.0 / np.sqrt(np.maximum((E * E).sum(1), dtype(EPS_NORM)))).astype(dtype)
        layers.append(E)
        rinv.append(r)
        F += E * r[:, None]
    return F, layers, rinv


def loss_of(A, E0, m, u, i, j, reg, n_layers=3):
    F, _, _ = propagate(A, E0, n_layers)
    Fu, Fi, Fj = F[u], F[m + i], F[m + j]
    y = (Fu * Fi).sum(1) - (Fu * Fj).sum(1)
    return float(np.logaddexp(0.0, -y).sum() + 0.5 * reg * ((Fu * Fu).sum() + (Fi * Fi).sum() + (Fj * Fj).sum()))


def loss_and_grad(A, E0, m, u, i, j, reg, n_layers=3, dtype=np.float64):
    """Loss of one batch and d loss / d E0 ([m+n, k], dense).  dtype: as in propagate()."""
    u, i, j = (np.asarray(x, dtype=np.int64) for x in (u, i, j))
    A = A.astype(dtype)
    F, layers, rinv = propagate(A, E0, n_layers, dtype)
    reg = dtype(reg)
    Fu, Fi, Fj = F[u], F[m + i], F[m + j]
    y = (Fu * Fi).sum(1) - (Fu * Fj).sum(1)
    loss = float(np.logaddexp(0.0, -y).sum() + 0.5 * reg * ((Fu * Fu).sum() + (Fi * Fi).sum() + (Fj * Fj).sum()))
    c = (1.0 / (1.0 + np.exp(y))).astype(dtype)               # 1 - sigmoid(y)
    G = np.zeros_like(F)
    np.add.at(G, u, -c[:, None] * (Fi - Fj) + reg * Fu)
    np.add.at(G, m + i, -c[:, None] * Fu + reg * Fi)
    np.add.at(G, m + j, c[:, None] * Fu + reg * Fj)

    def norm_bwd(k):                                          # d/dE_k of l2_normalize(E_k), applied to G
        E, r = layers[k], rinv[k]
        nrm = E * r[:, None]
        clamped = (E * E).sum(1) <= dtype(EPS_NORM)
        out = r[:, None] * (G - nrm * (nrm * G).sum(1)[:, None])
        out[clamped] = r[clamped, None] * G[clamped]
        return out
    D = norm_bwd(n_layers)                                    # d loss / d E_L
    for k in range(n_layers - 1, 0, -1):
        D = A.T @ D + norm_bwd(k)
    return loss, A.T @ D + G


class Adam(object):
    def __init__(self, shape):
        self.m, self.v, self.t = np.zeros(shape), np.zeros(shape), 0

    def step(self, var, grad, lr):
        self.t += 1
        self.m = BETA1 * self.m + (1 - BETA1) * grad
        self.v = BETA2 * self.v + (1 - BETA2) * grad * grad
        lr_t = lr * np.sqrt(1 - BETA2 ** self.t) / (1 - BETA1 ** self.t)
        var -= lr_t * self.m / (np.sqrt(self.v) + EPS_ADAM)


def batch_negatives(seed, epoch, ev_user, n, uq_indptr, uq_items):
    """One kept negative per training event in FILE order (event index = position in trainingData)."""
    return philox.sample_negatives(seed, epoch, ev_user, n, uq_indptr, uq_items, slot=NEG_SLOT)


def train(A, U, V, ev_user, ev_item, uq_indptr, uq_items, batch_size, lr, reg, seed, epochs=1, n_layers=3, adam=None,
          max_steps=None, dtype=np.float64):
    """LightGCN.py:81-98 on copies of U, V (float64; dtype: as in propagate(), the gradient only).  Returns U, V, the
    per-step losses and the Adam state."""
    m, n = U.shape[0], V.shape[0]
    E0 = np.concatenate([U, V]).astype(np.float64)
    adam = adam or Adam(E0.shape)
    losses = []
    T = len(ev_user)
    for ep in range(epochs):
        neg = batch_negatives(seed, ep, ev_user, n, uq_indptr, uq_items)
        for b0 in range(0, T, batch_size):
            if max_steps is not None and len(losses) >= max_steps:
                break
            sl = slice(b0, min(T, b0 + batch_size))
            loss, g = loss_and_grad(A, E0, m, ev_user[sl], ev_item[sl], neg[sl], reg, n_layers, dtype)
            adam.step(E0, g.astype(np.float64), lr)
            losses.append(loss)
    return E0[:m].copy(), E0[m:].copy(), np.array(losses), adam


def embeddings(A, U, V, n_layers=3):
    """The tables predict() ranks with (LightGCN.py:45-47, 101-105)."""
    F, _, _ = propagate(A, np.concatenate([U, V]).astype(np.float64), n_layers)
    return F[:U.shape[0]], F[U.shape[0]:]


# ---- the kernel's work plan (csrc/yue_b200.cu gcn_plan), restated so tests can say which path an input takes ----
HEAVY = 64                      # kGcnHeavy: a row with more neighbours is cut into chunks
SEG_ROWS, SEG_EDGES = 8, 64     # kGcnSegRows, kGcnSegEdges
HASH_SIZE = 8192                # kGcnHashSize
SMEM_SLOTS = 3072               # kGcnSmemSlots: batches of more than 1024 triplets keep their slot list in global memory
PAD_CHUNK = 0x7fffffff          # n_chunks of the empty chunks that pad the list to a multiple of 4


def gcn_hash(r):
    """The bucket of graph row r in the stamped rows' shared-memory hash (lightgcn.cuh gcn_hash): Fibonacci hashing, 13 bits."""
    return ((int(r) * 2654435761) & 0xFFFFFFFF) >> 19


def plan(m, n, uq_indptr, it_indptr):
    """gcn_plan's rules.  Graph rows are users 0..m-1, then tracks m..m+n-1; a row's degree is its number of distinct
    neighbours.  Returns (segs, heavy, chunks):
      segs    [(first row, rows)]: runs of consecutive rows with at most HEAVY neighbours each, at most SEG_ROWS rows and
              SEG_EDGES neighbours together, never across row m; sorted by neighbours, most first (stable)
      heavy   the rows with more than HEAVY neighbours, most first (stable)
      chunks  [(row, off, len, slot, first_slot, n_chunks, hidx)]: heavy row hidx cut into chunks of
              max(ceil(sqrt(deg) / 8) * 8, HEAVY) neighbours, then empty chunks (row 0, n_chunks PAD_CHUNK, hidx = len(heavy))
              up to a multiple of 4
    This is a description of the plan for tests to assert which path an input takes, not a second implementation."""
    uq_indptr, it_indptr = np.asarray(uq_indptr, np.int64), np.asarray(it_indptr, np.int64)
    deg = np.concatenate([np.diff(uq_indptr), np.diff(it_indptr)])
    segs, heavy = [], []
    open_row, open_edges = -1, 0

    def close(r):
        nonlocal open_row, open_edges
        if open_row >= 0:
            segs.append((open_row, r - open_row))
        open_row, open_edges = -1, 0
    for r in range(m + n):
        d = int(deg[r])
        if r == m:
            close(r)
        if d > HEAVY:
            close(r)
            heavy.append(r)
            continue
        if open_row >= 0 and (r - open_row >= SEG_ROWS or open_edges + d > SEG_EDGES):
            close(r)
        if open_row < 0:
            open_row = r
        open_edges += d
    close(m + n)
    segs.sort(key=lambda sg: -int(deg[sg[0]:sg[0] + sg[1]].sum()))
    heavy.sort(key=lambda r: -int(deg[r]))
    chunks = []
    for hi, r in enumerate(heavy):
        d = int(deg[r])
        c = max(int(np.ceil(np.sqrt(d) / 8.0)) * 8, HEAVY)
        nck, first = (d + c - 1) // c, len(chunks)
        chunks += [(r, q * c, min(c, d - q * c), first + q, first, nck, hi) for q in range(nck)]
    while len(chunks) % 4:
        chunks.append((0, 0, 0, len(chunks), len(chunks), PAD_CHUNK, len(heavy)))
    return segs, heavy, chunks


def degrees(m, n, uq_indptr, uq_items):
    """Distinct neighbours of every graph row (users, then tracks) and the track side's indptr."""
    it_indptr = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(np.asarray(uq_items), minlength=n), out=it_indptr[1:])
    return np.concatenate([np.diff(np.asarray(uq_indptr, np.int64)), np.diff(it_indptr)]), it_indptr
