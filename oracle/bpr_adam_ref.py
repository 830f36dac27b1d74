"""Oracle (test infrastructure) for BPR as the reference ships it: the live TF-1 graph and loop of recommender/cf/BPR.py:65-129
(SURVEY.md 3.3, DESIGN.md row a10).  The per-triplet SGD loop of BPR.py:31-62 that the rest of the build restates is
commented out in the shipped file; this is what runs.

PINNED BY THE SURVEY'S READING OF BPR.py:65-129 AND BY TENSORFLOW'S DOCUMENTED ADAM, not by running the reference: the
reference tree is not part of this repository, and its module needs TensorFlow 1.  tests/test_bpr_adam_oracle.py builds the
same graph from oracle/tf1_shim.py's ops (embedding_lookup, softplus, l2_loss, AdamOptimizer.minimize) and checks that this
restatement gives its losses and tables to 1e-12; what each op means is restated in the shim's header.

What one step computes:
* next_batch (65-81): `batch` training events drawn uniformly with replacement, for each `negatives` unplayed tracks (uniform
  over all n tracks -- test-only tracks included, as getSize counts them -- redrawn while the user played them).  The
  reference draws with numpy's and CPython's unseeded generators; here the Philox stream of oracle/philox.py with
  epoch = the step and event = the batch row: the event is attempt 0 of slot 4095 drawn over T (e = (r T) >> 32), negative
  k is slot k with the usual attempt loop.  The batch is a pure function of (seed, step).
* graph (93-115): loss = sum over the batch x negatives triplets (repeats included) of softplus(-(U_u.V_i - U_u.V_j))
  + regU (l2_loss(U_u) + l2_loss(V_i) + l2_loss(V_j)), l2_loss(x) = |x|^2 / 2, the rows read before the step.
* AdamOptimizer(lRate).minimize (in the graph, 93-124): TF-1 hands sparse Adam IndexedSlices; it sums duplicate indices
  and decays m and v of every row, which is dense Adam on the summed gradient: beta1 0.9, beta2 0.999, epsilon 1e-8,
  lr_t = lr sqrt(1 - beta2^t) / (1 - beta1^t), var -= lr_t m / (sqrt(v) + epsilon), every row every step.
* loop (121-129): num.max.iter steps, no lr schedule, no isConverged.
Deliberate deviation: under -byTime the reference's trainingData is the unsplit log, so its batches draw held-out events;
here positives come from the training split (the event CSR) only.
"""
import numpy as np

from . import philox

BETA1, BETA2, EPS_ADAM = 0.9, 0.999, 1e-8
POS_SLOT = 4095                 # the positive's Philox slot; negatives use slots 0 .. K-1


def sample_events(seed, step, batch, T):
    """Row b's training event: attempt 0 of slot 4095 over T."""
    assert 0 < T < 1 << 32
    return philox.draw_item(seed, step, np.arange(batch, dtype=np.uint64), POS_SLOT, np.zeros(batch, np.uint64), T)


def sample_batch(seed, step, batch, negatives, ev_indptr, ev_items, uq_indptr, uq_items, n):
    """(events[batch], u[batch], i[batch], neg[batch, negatives]) of step `step`."""
    assert negatives <= POS_SLOT
    ev_indptr = np.asarray(ev_indptr, np.int64)
    T = int(ev_indptr[-1])
    e = sample_events(seed, step, batch, T)
    u = np.searchsorted(ev_indptr, e, side='right') - 1
    i = np.asarray(ev_items, np.int64)[e]
    neg = np.empty((batch, negatives), np.int64)
    for k in range(negatives):
        # sample_negatives numbers its events 0 .. batch-1: exactly the batch rows
        neg[:, k] = philox.sample_negatives(seed, step, u, n, uq_indptr, uq_items, slot=k)
    return e, u, i, neg


def triplets(u, i, neg):
    """The batch x negatives triplets, row-major: a row's u and i repeat `negatives` times."""
    K = neg.shape[1]
    return np.repeat(u, K), np.repeat(i, K), neg.reshape(-1)


def loss_of(U, V, u, i, j, reg):
    Uu, Vi, Vj = U[u], V[i], V[j]
    y = (Uu * Vi).sum(1) - (Uu * Vj).sum(1)
    return float(np.logaddexp(0.0, -y).sum() + 0.5 * reg * ((Uu * Uu).sum() + (Vi * Vi).sum() + (Vj * Vj).sum()))


def loss_and_grad(U, V, u, i, j, reg):
    """Loss of the triplets and its dense gradients d/dU [m, k], d/dV [n, k]; duplicates add up."""
    u, i, j = (np.asarray(x, dtype=np.int64) for x in (u, i, j))
    Uu, Vi, Vj = U[u], V[i], V[j]
    y = (Uu * Vi).sum(1) - (Uu * Vj).sum(1)
    loss = float(np.logaddexp(0.0, -y).sum() + 0.5 * reg * ((Uu * Uu).sum() + (Vi * Vi).sum() + (Vj * Vj).sum()))
    c = 1.0 / (1.0 + np.exp(y))                                   # 1 - sigmoid(y)
    gU, gV = np.zeros_like(U), np.zeros_like(V)
    np.add.at(gU, u, -c[:, None] * (Vi - Vj) + reg * Uu)
    np.add.at(gV, i, -c[:, None] * Uu + reg * Vi)
    np.add.at(gV, j, c[:, None] * Uu + reg * Vj)
    return loss, gU, gV


class Adam(object):
    """tf.train.AdamOptimizer's dense update on one variable."""

    def __init__(self, shape):
        self.m, self.v, self.t = np.zeros(shape), np.zeros(shape), 0

    def step(self, var, grad, lr):
        self.t += 1
        self.m = BETA1 * self.m + (1 - BETA1) * grad
        self.v = BETA2 * self.v + (1 - BETA2) * grad * grad
        lr_t = lr * np.sqrt(1 - BETA2 ** self.t) / (1 - BETA1 ** self.t)
        var -= lr_t * self.m / (np.sqrt(self.v) + EPS_ADAM)


def train(U, V, ev_indptr, ev_items, uq_indptr, uq_items, batch, negatives, lr, reg, seed, steps, step_begin=0, adam=None):
    """Steps [step_begin, step_begin + steps) in float64 on copies of U, V.  Returns U, V, the losses, the Adam states."""
    U, V = np.array(U, dtype=np.float64), np.array(V, dtype=np.float64)
    aU, aV = adam or (Adam(U.shape), Adam(V.shape))
    losses = []
    for s in range(step_begin, step_begin + steps):
        _, u, i, neg = sample_batch(seed, s, batch, negatives, ev_indptr, ev_items, uq_indptr, uq_items, V.shape[0])
        loss, gU, gV = loss_and_grad(U, V, *triplets(u, i, neg), reg)
        aU.step(U, gU, lr)
        aV.step(V, gV, lr)
        losses.append(loss)
    return U, V, np.array(losses), (aU, aV)
