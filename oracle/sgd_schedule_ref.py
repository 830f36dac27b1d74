"""Oracle (test infrastructure): a whole Hogwild SGD epoch as ONE warp runs it -- the work plan of the host
(yue_b200.cu: plan_runs), the negatives of the kernel's sampler, and the read schedule of both epoch kernels:

* blocked_epoch: bpr_sgd_blk.cuh (BPR and APR, rows of up to 128 floats, the benchmark's path);
* per_triplet_epoch: bpr_sgd.cuh in MODE_HOGWILD / MODE_HOGWILD_STORE (rows above 128 floats, YUE_SGD_KERNEL=1).

yue_set_sgd_concurrency(h, 1, 1) makes an epoch run on a single warp: every float is then added by one lane in program
order, and what the warp reads and when is fixed by the code, so the kernels' results are a deterministic function of
the plan restated here.  Every schedule runs on float32 tables (row arithmetic rounded like the kernel's, fused
multiply-adds emulated in float64) or on float64 tables (no rounding: the yardstick the float32 runs are measured from).

Blocked schedule (one warp):
* the items of the plan in order; inside an item its segments' blocks of 4 triplets form one sequence, and the rows of
  block k are read before block k-1's changes are added (`lag` = 1; the lag runs across segment and, when items group
  several light users, across user boundaries); at the start of an item everything has been added;
* P[u] lives in registers (pu) next to the value it was read as (pu0); a publish adds fl32(pu - pu0) to P[u] and the
  row is re-read at once: at a user switch (the new user's row), at each shared segment whose user is already current,
  inside a shared segment before block b when b > 0 and (b & resync_mask) == 0, and at the end of the launch.
  At one warp P[u] holds pu0 when it is published, so a publish changes pu only by the rounding of pu0 + (pu - pu0) --
  none at all while the two are within a factor of 2 (Sterbenz) -- and a missing resync cannot be seen; a resync that
  re-reads without publishing (the changes since the last publish are lost) can, and `resync="lose"` restates it.
Per-triplet schedule (one warp): inside a segment the rows of event t are read when event t - PF is processed, before its
update (the first PF events read at the segment's start); a shared segment publishes and re-reads P[u] at its start and
before every event t > 0 with t % resync_events == 0; MODE_HOGWILD adds qn - q_read, MODE_HOGWILD_STORE stores qn (and
P[u] itself), losing the changes that land inside the read-ahead window."""
import math

import numpy as np

from . import apr_ref, philox
from .bpr_blk_ref import BLOCK, SEGMENT, _sigmoid_terms


# ---- the work plan (yue_b200.cu: plan_runs, yue_set_interactions, sgd_apply) --------------------------------------
def default_n_warps(T, sm_count=148, warps_per_sm=12, min_events_per_warp=16384):
    """Warps the host gives an epoch of T events when nothing forces the concurrency."""
    return max(1, min(sm_count * warps_per_sm, T // min_events_per_warp))


def default_item_segs(T, n_warps):
    """Segments per item of a heavy user: a quarter of a warp's fair share, 32..256 (yue_set_interactions)."""
    return max(32, min(256, T // (n_warps * 4 * SEGMENT)))


def plan_runs(runs, item_segs, group_segs=1, max_items=1 << 30, allow_shared=True):
    """runs: (user, begin, end) event ranges in stream order.  Returns (segs, items): segs[s] = (user, begin, end, shared)
    with <= 32 events each, items[k] = (first segment, end segment) in the order the cursor hands them out."""
    segs, items = [], []
    open_first = -1
    for (u, b, e) in runs:
        nsegs = (e - b + SEGMENT - 1) // SEGMENT
        if nsegs == 0:
            continue
        heavy = allow_shared and nsegs > item_segs
        if heavy and open_first >= 0:
            items.append((open_first, len(segs)))
            open_first = -1
        first = len(segs)
        segs += [(int(u), int(x), int(min(e, x + SEGMENT)), heavy) for x in range(b, e, SEGMENT)]
        if heavy:
            per = max(item_segs, (nsegs + max_items - 1) // max_items)
            items += [(s, min(len(segs), s + per)) for s in range(first, len(segs), per)]
        else:
            if open_first < 0:
                open_first = first
            if len(segs) - open_first >= group_segs:
                items.append((open_first, len(segs)))
                open_first = -1
    if open_first >= 0:
        items.append((open_first, len(segs)))
    return segs, items


def plan_epoch(ev_indptr, item_segs, **kw):
    """The plan of an epoch over a CSR log: one run per user."""
    ev_indptr = np.asarray(ev_indptr, dtype=np.int64)
    return plan_runs([(u, int(ev_indptr[u]), int(ev_indptr[u + 1])) for u in range(len(ev_indptr) - 1)], item_segs, **kw)


def plan_triplets(u, item_segs=None, **kw):
    """The plan of yue_bpr_apply / yue_apr_apply in a Hogwild mode: one run per maximal run of equal users."""
    u = np.asarray(u)
    runs, t = [], 0
    while t < len(u):
        e = t
        while e < len(u) and u[e] == u[t]:
            e += 1
        runs.append((int(u[t]), t, e))
        t = e
    if item_segs is None:
        item_segs = default_item_segs(len(u), default_n_warps(len(u)))
    return plan_runs(runs, item_segs, **kw)


def plan_parts(items, n_parts):
    """Item ranges of yue_bpr_epoch_part's parts 0..n_parts-1."""
    n = len(items)
    return [(n * k // n_parts, n * (k + 1) // n_parts) for k in range(n_parts)]


def epoch_negatives(seed, epoch, ev_indptr, n_items, uq_indptr, uq_items, slot=0, event_base=0, ev_delta=None):
    """The negatives the epoch kernels draw: the sampler at the GLOBAL event index, event_base + e, or ev_delta[user] + e
    for a shard with per-user offsets."""
    ev_indptr = np.asarray(ev_indptr, dtype=np.int64)
    uq_indptr = np.asarray(uq_indptr, dtype=np.int64)
    m = len(ev_indptr) - 1
    if ev_delta is None:
        ev_user = np.repeat(np.arange(m), np.diff(ev_indptr))
        return philox.sample_negatives(seed, epoch, ev_user, n_items, uq_indptr, uq_items, slot=slot, event_base=event_base)
    out = np.empty(int(ev_indptr[-1]), dtype=np.int32)
    for u in range(m):
        b, e = int(ev_indptr[u]), int(ev_indptr[u + 1])
        if e > b:
            row = np.asarray(uq_items[uq_indptr[u]:uq_indptr[u + 1]])
            out[b:e] = philox.sample_negatives(seed, epoch, np.zeros(e - b, np.int64), n_items, np.array([0, len(row)]), row,
                                               slot=slot, event_base=int(ev_delta[u]) + b)
    return out


def resync_mask(resync_events):
    """The blocked kernel resyncs before block b when (b & mask) == 0 (yue_b200.cu: run_sgd)."""
    rb = 1
    while rb * 2 * BLOCK <= resync_events:
        rb *= 2
    return rb - 1


# ---- one triplet, as the kernels compute it ------------------------------------------------------------------------
def _round(x, f32):
    return np.float32(x) if f32 and np.isscalar(x) else (np.asarray(x).astype(np.float32) if f32 else x)


def _softplus_sigmoid(x, lr):
    """float64: g = lr * sigmoid(-x), loss term softplus(-x)."""
    return lr / (1.0 + math.exp(x)) if x < 700 else 0.0, apr_ref.softplus(-x)


def _bpr_step_blk(pu, qi, qj, lr, c_u, c_i, f32):
    """The blocked kernel's BPR arithmetic (bpr_sgd_blk.cuh): returns (new pu, change of Q[i], change of Q[j], loss)."""
    if f32:
        d = qi - qj
        g, l = _sigmoid_terms(np.float32(np.dot(pu.astype(np.float64), d.astype(np.float64))), lr)
        pn = (pu.astype(np.float64) + np.float64(g) * d.astype(np.float64)).astype(np.float32)
        gp = (g * pn).astype(np.float32)
        di = ((-np.float64(c_i)) * (qi + gp).astype(np.float32).astype(np.float64) + gp.astype(np.float64)).astype(np.float32)
        dj = ((-np.float64(c_i)) * (qj - gp).astype(np.float32).astype(np.float64) - gp.astype(np.float64)).astype(np.float32)
        pu = ((-np.float64(c_u)) * pn.astype(np.float64) + pn.astype(np.float64)).astype(np.float32)
        return pu, di, dj, float(l)
    d = qi - qj
    g, l = _softplus_sigmoid(float(pu.dot(d)), lr)
    pn = pu + g * d
    gp = g * pn
    return pn - c_u * pn, gp - c_i * (qi + gp), -gp - c_i * (qj - gp), l


def _apr_step_blk(pu, qi, qj, lr, c_u, c_i, f32, eps, regA):
    """The blocked kernel's APR arithmetic: the closed form of oracle/apr_ref.py from the rows as read,
    P <- c (alpha P + a d), alpha = 1 - 2 b / |P|;  Q[i] += a P - (b / |d|) d,  Q[j] -= the same, then the shrinks."""
    d = qi - qj
    p64, d64 = pu.astype(np.float64), d.astype(np.float64)
    r = (lambda v: float(np.float32(v))) if f32 else float
    y, np2, dd = r(p64.dot(d64)), r(p64.dot(p64)), r(d64.dot(d64))
    n_p, n_d = math.sqrt(np2), math.sqrt(dd)
    ya = apr_ref.adv_score(y, n_p, n_d, eps)
    s0 = 1.0 / (1.0 + math.exp(y)) if y < 700 else 0.0
    s1 = 1.0 / (1.0 + math.exp(ya)) if ya < 700 else 0.0
    loss = apr_ref.softplus(-y) + regA * apr_ref.softplus(-ya)
    a, b = r(lr * (s0 + regA * s1)), lr * regA * s1 * eps
    alpha = r(1.0 - 2.0 * b / n_p) if n_p > 0 else 1.0
    bd = r(b / n_d) if n_d > 0 else 0.0
    if f32:
        step = (a * p64 - bd * d64).astype(np.float32)                                  # fmaf(a, pu, -(b/|d|) d)
        pn = (alpha * p64 + np.float64(np.float32(a * d64))).astype(np.float32)        # fmaf(alpha, pu, a d)
        s64 = step.astype(np.float64)
        di = (-np.float64(c_i) * (qi + step).astype(np.float32).astype(np.float64) + s64).astype(np.float32)
        dj = (-np.float64(c_i) * (qj - step).astype(np.float32).astype(np.float64) - s64).astype(np.float32)
        pu = (-np.float64(c_u) * pn.astype(np.float64) + pn.astype(np.float64)).astype(np.float32)
        return pu, di, dj, loss
    step = a * pu - bd * d
    pn = alpha * pu + a * d
    return pn - c_u * pn, step - c_i * (qi + step), -step - c_i * (qj - step), loss


def _bpr_step_pt(pu, qi, qj, lr, c_u, c_i, f32):
    """The per-triplet kernel's BPR arithmetic (bpr_sgd.cuh, Hogwild modes): returns (new pu, new Q[i], new Q[j], loss)."""
    if f32:
        p64 = pu.astype(np.float64)
        x = np.float32(np.float32(p64.dot(qi.astype(np.float64))) - np.float32(p64.dot(qj.astype(np.float64))))
        ex = np.float32(math.exp(-abs(float(x))))
        s = np.float32(np.float32(1.0 if x >= 0 else ex) / np.float32(np.float32(1) + ex))
        g = np.float32(np.float32(lr) * np.float32(np.float32(1) - s))
        loss = float(np.float32(max(-x, np.float32(0))) + np.float32(math.log1p(float(ex))))
        d = (qi - qj).astype(np.float64)
        pn = (p64 + np.float64(g) * d).astype(np.float32)
        pn64 = pn.astype(np.float64)
        qni = (qi.astype(np.float64) + np.float64(g) * pn64).astype(np.float32)
        qnj = (qj.astype(np.float64) - np.float64(g) * pn64).astype(np.float32)
        pu = (pn64 - np.float64(c_u) * pn64).astype(np.float32)
        qni = (qni.astype(np.float64) - np.float64(c_i) * qni.astype(np.float64)).astype(np.float32)
        qnj = (qnj.astype(np.float64) - np.float64(c_i) * qnj.astype(np.float64)).astype(np.float32)
        return pu, qni, qnj, loss
    g, l = _softplus_sigmoid(float(pu.dot(qi) - pu.dot(qj)), lr)
    pn = pu + g * (qi - qj)
    qni, qnj = qi + g * pn, qj - g * pn
    return pn - c_u * pn, qni - c_i * qni, qnj - c_i * qnj, l


# ---- the schedules -------------------------------------------------------------------------------------------------
class _User:
    """P[u] in registers: pu, and pu0 = the value it was read as."""

    def __init__(self, P, f32, store=False):
        self.P, self.f32, self.store, self.cur, self.pu, self.pu0 = P, f32, store, -1, None, None

    def publish(self):
        if self.cur >= 0:
            if self.store:
                self.P[self.cur] = self.pu
            else:
                self.P[self.cur] = _round(self.P[self.cur] + _round(self.pu - self.pu0, self.f32), self.f32)

    def read(self, u):
        self.cur, self.pu = u, self.P[u].copy()
        self.pu0 = self.pu.copy()


def blocked_epoch(P, Q, plan, ev_items, ev_neg, lr, regU, regI, apr=None, resync_events=8, lag=1, resync="publish",
                  items=None):
    """The blocked kernel on one warp, in place on P and Q (both float32 or both float64); returns the loss.
    plan = (segs, items) of plan_runs; ev_items / ev_neg index the events of the segments.  apr = (eps, regA) for K2a.
    Variants, to show what the tests can tell apart: lag = 0 reads every triplet's rows when it is reached (blocks of one
    triplet, nothing pending: the serial order), lag = 2 reads block k before blocks k-1 and k-2 are added;
    resync = "lose" re-reads P[u] at a resync without publishing it first.  items: a range of the plan's items (a part)."""
    f32 = P.dtype == np.float32
    c_u, c_i = (np.float32(lr * regU), np.float32(lr * regI)) if f32 else (lr * regU, lr * regI)
    if apr is None:
        step = lambda pu, qi, qj: _bpr_step_blk(pu, qi, qj, lr, c_u, c_i, f32)           # noqa: E731
    else:
        step = lambda pu, qi, qj: _apr_step_blk(pu, qi, qj, lr, c_u, c_i, f32, apr[0], apr[1])   # noqa: E731
    segs, all_items = plan
    it0, it1 = items if items is not None else (0, len(all_items))
    block = BLOCK if lag > 0 else 1
    mask = resync_mask(resync_events)
    usr = _User(P, f32)

    def sync(u):
        if resync == "publish":
            usr.publish()
        usr.read(u)

    def add(deltas):
        for row, dv in deltas:
            Q[row] = _round(Q[row] + dv, f32)
    loss = 0.0
    for (s0, s1) in all_items[it0:it1]:
        pending = []                                 # changes of the blocks not yet added, oldest first
        for s in range(s0, s1):
            u, b, e, shared = segs[s]
            for k, b0 in enumerate(range(b, e, block)):
                if k == 0 and u != usr.cur:
                    usr.publish()
                    usr.read(u)
                elif shared and (k == 0 or (k & mask) == 0):
                    sync(u)
                while len(pending) > lag:
                    add(pending.pop(0))
                trip = range(b0, min(e, b0 + block))
                qi = [Q[ev_items[x]].copy() for x in trip]
                qj = [Q[ev_neg[x]].copy() for x in trip]
                out = []
                for a, x in enumerate(trip):
                    usr.pu, di, dj, lt = step(usr.pu, qi[a], qj[a])
                    loss += lt
                    out += [(ev_items[x], di), (ev_neg[x], dj)]
                pending.append(out)
        for blk in pending:
            add(blk)
    usr.publish()
    return loss


def per_triplet_epoch(P, Q, plan, ev_items, ev_neg, lr, regU, regI, pf, resync_events=8, store=False):
    """The per-triplet kernel on one warp (MODE_HOGWILD, or MODE_HOGWILD_STORE with store=True), in place; returns the
    loss.  pf: rows in flight, 4 when ceil(ld / 64) <= 2, else 2."""
    f32 = P.dtype == np.float32
    c_u, c_i = (np.float32(lr * regU), np.float32(lr * regI)) if f32 else (lr * regU, lr * regI)
    segs, items = plan
    usr = _User(P, f32, store)
    loss = 0.0
    for (s0, s1) in items:
        for s in range(s0, s1):
            u, b, e, shared = segs[s]
            if u != usr.cur or shared:
                usr.publish()
                usr.read(u)
            n = e - b
            rows = {t: (Q[ev_items[b + t]].copy(), Q[ev_neg[b + t]].copy()) for t in range(min(pf, n))}
            for t in range(n):
                if shared and t > 0 and t % resync_events == 0:
                    usr.publish()
                    usr.read(u)
                qi, qj = rows.pop(t)
                if t + pf < n:
                    rows[t + pf] = (Q[ev_items[b + t + pf]].copy(), Q[ev_neg[b + t + pf]].copy())
                usr.pu, qni, qnj, lt = _bpr_step_pt(usr.pu, qi, qj, lr, c_u, c_i, f32)
                loss += lt
                i, j = ev_items[b + t], ev_neg[b + t]
                if store:
                    Q[i], Q[j] = qni, qnj
                else:
                    Q[i] = _round(Q[i] + _round(qni - qi, f32), f32)
                    Q[j] = _round(Q[j] + _round(qnj - qj, f32), f32)
    usr.publish()
    return loss
