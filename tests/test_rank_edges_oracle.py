"""Adversarial tables for the ranking path, and CPU proofs that they are adversarial.

The tcgen05 ranking kernel (rank_tc.cuh) scores in tf32 and keeps every track whose approximate score is at least
tau - 2 eps, eps = kTf32ErrCoef * |p_u| * max_t |q_t|.  On random tables the tf32 order and the exact order differ only
by noise, so a coefficient several times too small would go unnoticed.  `tf32_bound_case` builds a table on which it
would not: track A is the exact top-1 but has the LOWEST tf32 score of the top group, and the group's tracks come first
in id order, so the row's threshold is already set from them when A's tile arrives.

Two forms, because which rounding the tensor core applies to fp32 operands is not documented here:
  "trunc"  p_k = A_k = 1 + 2^-10 - 2^-23 (tf32 by truncation: 1); competitors mix 1 and 1 + 2^-10 (tf32-exact), d - 1 of
           them at 1 + 2^-10.  Under round-to-nearest p rounds UP and the table is harmless.
  "rn"     p_k = A_k = 1 + 2^-11 - 2^-23, just below the halfway point: 1 under truncation AND under round-to-nearest;
           competitors have d/2 - 1 components at 1 + 2^-10.
A competitor's tf32 score is d + j 2^-10 > d = A's, while its exact score p (d + j 2^-10) stays below A's d p^2.
"""
import os
import re

import numpy as np
import pytest

from oracle import topn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORMS = {"trunc": (np.float32(1 + 2.0 ** -10 - 2.0 ** -23), topn.tf32_trunc),
         "rn": (np.float32(1 + 2.0 ** -11 - 2.0 ** -23), topn.tf32_rn)}
HI = np.float32(1 + 2.0 ** -10)


def tf32_err_coef():
    """kTf32ErrCoef as compiled (rank_tc.cuh)."""
    src = open(os.path.join(ROOT, "yue_b200", "csrc", "rank_tc.cuh")).read()
    return float(re.search(r"constexpr float kTf32ErrCoef = ([0-9.eE+-]+)f;", src).group(1))


def tc_cap(N):
    """Candidate slots per row of rank_tc_kernel (rank_tc_run: 64 for N <= 12, else 96)."""
    return 64 if N <= 12 else 96


def tf32_bound_case(d, form, N, n=300, seed=0):
    """One catalog, users whose rows are p scaled by powers of two (2^-10 .. 2^10, plus a few other scales).

    Tracks [0, cap): n_comp = cap - 33 competitors at random ids, fillers elsewhere.  With the threshold still at -inf
    the kernel pushes every track, so after `cap` tracks the buffer (cap - 32 slots) is compacted and the threshold set
    to tau - 2 eps from the competitors; they all stay (no spill: cap - 33 + A <= cap - 32).  A comes at id cap + 7.
    Fillers have mixed signs (score ~ 0) and norms at most the group's, so max|q| is a top-group track."""
    v, _ = FORMS[form]
    jmax = d - 1 if form == "trunc" else d // 2 - 1
    cap = tc_cap(N)
    n_comp = cap - 33
    rng = np.random.default_rng(seed + 131 * d + N)
    Q = np.empty((n, d), np.float32)
    for t in range(n):                                   # balanced signs: |score| small
        sgn = np.where(rng.permutation(d) < d // 2, 1.0, -1.0)
        Q[t] = sgn * rng.choice([1.0, float(HI), 0.5, 0.25], d)
    comp = np.sort(rng.choice(cap, n_comp, replace=False))
    for t in comp:
        row = np.ones(d, np.float32)
        row[rng.choice(d, jmax, replace=False)] = HI
        Q[t] = row
    a_id = cap + 7
    Q[a_id] = v
    scales = [2.0 ** k for k in range(-10, 11)] + [3.7, 0.013, 611.0]
    P = np.stack([np.full(d, v, np.float32) * np.float32(s) for s in scales]).astype(np.float32)
    users = np.resize(rng.permutation(len(scales)), 200).astype(np.int32)   # 200 rows: two user blocks, repeats
    return dict(P=P, Q=Q, users=users, a_id=a_id, comp=comp, cap=cap, n_comp=n_comp, N=N, d=d, form=form,
                pow2_users=np.arange(21))


def approx_scores(p, Q, rnd):
    """tf32 operands, exact products, float64 sum (the sums of the top group are exact in fp32 too: checked)."""
    return rnd(Q).astype(np.float64) @ rnd(p).astype(np.float64)


def f32(x):
    return np.float32(x)


def kernel_norms(p, Q):
    """pnorm and qmax as rank_tc.cuh computes them (sqrt of the fp32 sum of squares, times 1.0001f)."""
    pn = f32(f32(np.sqrt(np.float32(np.sum(p.astype(np.float64) ** 2)))) * f32(1.0001))
    qm = f32(f32(np.sqrt(np.float32(np.max(np.sum(Q.astype(np.float64) ** 2, axis=1))))) * f32(1.0001))
    return pn, qm


def filter_emulation(case, u, rnd):
    """(approx, tau, pnorm, qmax) of user u: tau = N-th best approximate score of the tracks before A (the row's threshold
    is set from them at the first compaction)."""
    p, Q = case["P"][u], case["Q"]
    ap = approx_scores(p, Q, rnd)
    tau = np.sort(ap[:case["cap"]])[::-1][case["N"] - 1]
    pn, qm = kernel_norms(p, Q)
    return ap, tau, pn, qm


def survives(ap, tau, pn, qm, a_id, c):
    e2 = f32(f32(f32(2.0) * f32(c)) * pn) * qm
    return f32(ap[a_id]) >= f32(f32(tau) - e2)


CASES = [(d, form, N) for d in (64, 128) for form in ("trunc", "rn") for N in (1, 10, 32)]


@pytest.mark.parametrize("d,form,N", CASES)
def test_tf32_bound_case_is_adversarial(d, form, N):
    case = tf32_bound_case(d, form, N)
    P, Q, a = case["P"], case["Q"], case["a_id"]
    _, rnd = FORMS[form]
    coef = tf32_err_coef()
    assert a >= case["cap"] and N <= case["n_comp"] <= case["cap"] - 33
    exact = topn.scores_fma32(P, Q)
    cstar_all = []
    for u in case["pow2_users"]:
        s = exact[u]
        # A is the exact top-1, strictly; every competitor beats it in tf32 and loses to it exactly
        assert s[a] > np.max(np.delete(s, a))
        ap, tau, pn, qm = filter_emulation(case, u, rnd)
        assert np.all(ap[case["comp"]] > ap[a]) and np.all(s[case["comp"]] < s[a])
        assert np.all(ap[case["comp"]] == np.float64(f32(ap[case["comp"]])))          # fp32 accumulation is exact here
        assert ap[a] < tau
        assert np.isclose(qm / f32(1.0001), np.linalg.norm(Q.astype(np.float64), axis=1).max(), rtol=1e-6)
        assert np.argmax(np.linalg.norm(Q.astype(np.float64), axis=1)) in set(case["comp"].tolist()) | {a}
        cstar = float(tau - ap[a]) / (2.0 * float(pn) * float(qm))
        assert survives(ap, tau, pn, qm, a, cstar * (1 + 1e-3))
        assert not survives(ap, tau, pn, qm, a, cstar * (1 - 1e-3))
        assert survives(ap, tau, pn, qm, a, coef)
        # the compaction that sets the threshold keeps only the competitors: no spill, no fallback
        lim = f32(f32(tau) - f32(f32(f32(2.0) * f32(coef)) * pn) * qm)
        assert np.sum(ap[:case["cap"]] >= lim) == case["n_comp"]
        assert np.sum(ap[case["cap"]:] >= lim) == 1                                      # A alone after it
        cstar_all.append(cstar)
    cstar = max(cstar_all)
    assert np.ptp(cstar_all) <= 1e-6 * cstar                                              # power-of-two scales: same c*
    print("d=%d form=%s N=%d: c* = %.3e (kTf32ErrCoef = %.2e, %.1fx slack)" % (d, form, N, cstar, coef, coef / cstar))
    assert cstar < coef
    if form == "trunc":
        assert cstar > 4e-4                        # kTf32ErrCoef = 4e-4 must lose A on a truncating device


def test_rn_form_is_adversarial_under_truncation_too():
    """The round-to-nearest form also loses A under truncation, so it bites whichever rounding the device applies."""
    case = tf32_bound_case(64, "rn", 10)
    ap, tau, pn, qm = filter_emulation(case, 0, topn.tf32_trunc)
    assert ap[case["a_id"]] < tau and not survives(ap, tau, pn, qm, case["a_id"], 0.0)


def test_tf32_helpers():
    x = np.array([1 + 2.0 ** -10 - 2.0 ** -23, 1 + 2.0 ** -11 - 2.0 ** -23, 1 + 2.0 ** -11, 1 + 3 * 2.0 ** -11,
                  -(1 + 2.0 ** -10 - 2.0 ** -23), 3.0], np.float32)
    assert topn.tf32_trunc(x).tolist() == [1.0, 1.0, 1.0, 1 + 2.0 ** -10, -1.0, 3.0]
    assert topn.tf32_rn(x).tolist() == [1 + 2.0 ** -10, 1.0, 1.0, 1 + 2.0 ** -9, -(1 + 2.0 ** -10), 3.0]   # ties to even


def test_c_oracle_agrees_on_the_constructions():
    from oracle import c_oracle
    for form in FORMS:
        case = tf32_bound_case(64, form, 10)
        P, Q = case["P"], case["Q"]
        assert np.array_equal(c_oracle.scores_fma32(P, Q), topn.scores_fma32(P, Q))
