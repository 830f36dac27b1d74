"""Oracle (test infrastructure): full-catalog scoring and masked top-N.

Restates the evaluation loop of ``base/IterativeRecommender.py:77-145``:

* ``predict`` (58-60): scores = Q.dot(P[u]) over every track id;
* N = max(-topN list), reset to 10 when N > 100 or N < 0 (80-86);
* the user's training tracks are removed from the candidates (102-106);
* "find the K biggest scores" (107-145).

Two selections are provided:

``topn_exact``  what the reference's comment says it intends and what north_star requires:
    the N highest-scoring unmasked tracks ordered by (score desc, track id asc).
    The *canonical score* is the float32 FMA chain  acc = fma(P[u,k], Q[t,k], acc), k = 0..d-1
    (SURVEY.md section 8c) so that CPU and GPU agree bit for bit and ids can be compared exactly.

``topn_ref_quirk``  the selection the shipped code actually performs (seed with the first N
    candidates, then overwrite slot ind+1 instead of inserting; lines 107-145), restated so
    end-to-end numbers can be quoted against both.  Pinned by tests/golden/eval_*.npz,
    produced by running the reference's own evalRanking.
"""
import numpy as np


def clamp_topn(top):
    """IterativeRecommender.py:80-86."""
    N = max(int(t) for t in top)
    if N > 100 or N < 0:
        N = 10
    return N


def scores_fma32(P_rows, Q):
    """Canonical float32 FMA-chain scores, [B, n].

    fma(a, b, c) in float32 is emulated as float32(float64(a)*float64(b) + float64(c)): the
    product of two float32 is exact in float64; the float64 sum is rounded once more than a
    true FMA would, which can differ only when the exact sum lies within 2^-29 ulp32 of a
    float32 rounding boundary.  The C oracle (oracle/csrc/oracle.c) uses fmaf() and is the
    tie-breaker when the two disagree; tests compare both.
    """
    P_rows = np.ascontiguousarray(P_rows, dtype=np.float32)
    Q = np.ascontiguousarray(Q, dtype=np.float32)
    B, d = P_rows.shape
    acc = np.zeros((B, Q.shape[0]), dtype=np.float32)
    Q64 = Q.astype(np.float64)
    for k in range(d):
        acc = (P_rows[:, k].astype(np.float64)[:, None] * Q64[None, :, k]
               + acc.astype(np.float64)).astype(np.float32)
    return acc


def tf32_trunc(x):
    """float32 -> tf32 by truncation: the low 13 of the 23 mantissa bits cleared."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    return (b & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_rn(x):
    """float32 -> tf32 rounded to nearest, ties to even, at mantissa bit 13 (finite inputs)."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    b = (b + 0xFFF + ((b >> 13) & 1)) & 0xFFFFE000
    return b.astype(np.uint32).view(np.float32)


def topn_exact(P, Q, users, N, uq_indptr, uq_items, scores=None):
    """ids [B,N] int32 (-1 padded), scores [B,N] float32 (-inf padded)."""
    users = np.asarray(users, dtype=np.int64)
    n = Q.shape[0]
    ids = np.full((len(users), N), -1, dtype=np.int32)
    sc = np.full((len(users), N), -np.inf, dtype=np.float32)
    for b, u in enumerate(users):
        s = scores[b] if scores is not None else scores_fma32(P[u:u + 1], Q)[0]
        s = s.astype(np.float32).copy()
        mask = uq_items[uq_indptr[u]:uq_indptr[u + 1]]
        valid = np.ones(n, dtype=bool)
        valid[mask] = False
        cand = np.nonzero(valid)[0]
        # lexsort: last key is primary.  score desc, id asc.
        order = np.lexsort((cand, -s[cand].astype(np.float64)))[:N]
        top = cand[order]
        ids[b, :len(top)] = top
        sc[b, :len(top)] = s[top]
    return ids, sc


def topn_ref_quirk(score_row, masked_ids, N):
    """The shipped selection (IterativeRecommender.py:107-145) on one user's score vector.

    ``score_row[t]`` is the score of track id t; candidates are visited in id order (the
    reference iterates a dict filled in id order, 98-100) minus ``masked_ids``.  Returns the
    list of N track ids it would recommend (duplicates possible, as in the reference).
    """
    masked = set(int(x) for x in masked_ids)
    cand = [t for t in range(len(score_row)) if t not in masked]
    seed = cand[:N]
    seed.sort(key=lambda t: score_row[t], reverse=True)       # stable, like list.sort
    rec_scores = [score_row[t] for t in seed]
    rec_ids = list(seed)
    for t in cand:
        v = score_row[t]
        ind = N
        l, r = 0, N - 1
        if rec_scores[r] < v:
            while True:
                mid = (l + r) // 2
                if rec_scores[mid] >= v:
                    l = mid + 1
                elif rec_scores[mid] < v:
                    r = mid - 1
                if r < l:
                    ind = r
                    break
        if ind < N - 1:
            rec_scores[ind + 1] = v
            rec_ids[ind + 1] = t
    return rec_ids
