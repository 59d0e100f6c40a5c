"""CPU pin of the panel kernel's fast path: the numpy restatement of CholeskyQR2 + Householder reconstruction
(tests/fastpath_model.py, stage by stage what k_panel does) reproduces the reference's column recurrences (oracle np_qr,
S:122-148) on well-conditioned panels, and its guards refuse the panels on which CholeskyQR2 would lose accuracy."""
import numpy as np
import pytest

import fastpath_model as F


@pytest.mark.parametrize("rows,seed", [(64, 1), (221, 2), (512, 3), (4096, 4)])
def test_fast_path_reproduces_reference_reflectors(oracle, rows, seed):
    P = oracle.np_uniform(seed, rows, 32)
    Href, aref = oracle.np_qr(P)
    H, alpha, fast = F.fast_panel(P)
    assert fast
    assert np.abs(alpha - aref).max() <= 1e-12 * np.abs(aref).max()
    assert np.abs(H - Href).max() < 1e-11
    assert oracle.qr_residual(P, np.asfortranarray(H), alpha) < 1e-13


def test_fast_path_signs_and_negative_pivots(oracle):
    # mixed-sign entries exercise both branches of the on-the-fly sign choice (alphafactor, S:8)
    P = oracle.np_uniform(7, 300, 32) - 0.5
    Href, aref = oracle.np_qr(P)
    H, alpha, fast = F.fast_panel(P)
    assert fast and (aref > 0).any() and (aref < 0).any()
    assert np.abs(alpha - aref).max() <= 1e-12 * np.abs(aref).max()
    assert np.abs(H - Href).max() < 1e-11


def test_guards_refuse_ill_conditioned_panels(oracle):
    P = oracle.np_uniform(21, 1024, 32)
    Pi = P.copy()
    Pi[:, 7] = Pi[:, 3] + 1e-9 * oracle.np_uniform(22, 1024, 1)[:, 0]       # kappa ~ 1e9
    assert F.fast_panel(Pi)[2] is False
    Pz = P.copy()
    Pz[:, 5] = 0.0                                                           # zero column: the reference yields NaN (S:131)
    assert F.fast_panel(Pz)[2] is False
    Pn = P.copy()
    Pn[10, 4] = np.nan
    assert F.fast_panel(Pn)[2] is False


def test_every_panel_the_guards_accept_is_backward_stable(oracle):
    # The blocked solves invert 8x8 diagonal blocks explicitly and lose ~5e-18 x (diagonal spread of the first factor) in
    # ||QR - A|| / ||A||; the kernel's guard (spread < 250) keeps every accepted panel within a few eps, and everything
    # beyond goes to the column-by-column path.  Sweep the conditioning through the threshold.
    accepted = refused = 0
    for eps in (1e-1, 3e-2, 1e-2, 6e-3, 3e-3, 1e-3, 3e-4, 1e-4, 1e-5, 1e-7):
        P = oracle.np_uniform(31, 2048, 32)
        P[:, 9] = P[:, 2] + eps * oracle.np_uniform(32, 2048, 1)[:, 0]
        H, alpha, fast = F.fast_panel(P)
        if not fast:
            refused += 1
            continue
        accepted += 1
        assert oracle.qr_residual(P, np.asfortranarray(H), alpha) < 3e-15
        Href, aref = oracle.np_qr(P)
        assert np.abs(alpha - aref).max() <= 1e-12 * np.abs(aref).max() / eps
    assert accepted >= 3 and refused >= 4


def test_substitution_guard_would_not_be_enough_for_blocked_solves(oracle, monkeypatch):
    # documents why the guard is tighter than row-by-row substitution would need: with a spread up to 1e5 the blocked
    # solves would accept a panel whose factorisation residual is ~1e-13
    monkeypatch.setattr(F, "SPREAD_MIN", 1e-5)
    P = oracle.np_uniform(31, 2048, 32)
    P[:, 9] = P[:, 2] + 1e-4 * oracle.np_uniform(32, 2048, 1)[:, 0]
    H, alpha, fast = F.fast_panel(P)
    assert fast and oracle.qr_residual(P, np.asfortranarray(H), alpha) > 2e-14


def test_blocked_trsm_matches_substitution():
    rng = np.random.default_rng(5)
    R = np.triu(rng.standard_normal((32, 32))) + 6.0 * np.eye(32)
    X = rng.standard_normal((100, 32))
    Y = F.blocked_trsm(X, R, 1.0 / np.diag(R))
    assert np.abs(Y @ R - X).max() < 1e-12


def test_design_study_blocked_recurrences_match_the_unblocked_ones(oracle):
    # next-round design study: 8-column blocked Cholesky and signed LU give the factors of the 32-step recurrences
    P = oracle.np_uniform(41, 1500, 32) - 0.3
    G = P.T @ P
    R, rinv, ok = F.cholesky_upper(G)
    Rb, rinvb, okb = F.cholesky_upper_blocked(G)
    assert ok and okb and np.abs(R - Rb).max() < 1e-12 * np.abs(R).max() and np.abs(rinv - rinvb).max() < 1e-12 * rinv.max()
    Q = np.linalg.qr(P)[0][:32, :]
    Wt = Q.copy()
    Sg, Ud = np.zeros(32), np.zeros(32)
    for j in range(32):
        w = Wt[j, j]
        Sg[j] = -1.0 if w > 0.0 else 1.0
        Ud[j] = 1.0 + abs(w)
        Wt[j + 1:, j + 1:] += np.outer(Sg[j] / Ud[j] * Wt[j + 1:, j], Wt[j, j + 1:])
    Wb, Sgb, Udb = F.lu_signed_blocked(Q)
    off = ~np.eye(32, dtype=bool)
    assert np.array_equal(Sg, Sgb) and np.abs(Ud - Udb).max() < 1e-13 and np.abs((Wt - Wb)[off]).max() < 1e-13


def test_kahan_like_panels_high_condition_without_a_small_pivot(oracle):
    # Kahan-type factors are ill-conditioned with a slowly decaying diagonal, so the spread guard alone does not see them;
    # accepted panels must still be backward stable and the orthogonality guard must refuse them before CholeskyQR2 breaks
    rng = np.random.default_rng(0)
    Q, _ = np.linalg.qr(rng.standard_normal((2048, 32)))
    accepted = refused = 0
    for theta in (1.5, 1.4, 1.3, 1.2, 1.1, 1.0, 0.9):
        c, s = np.cos(theta), np.sin(theta)
        R = np.diag(s ** np.arange(32)) @ (np.eye(32) - c * np.triu(np.ones((32, 32)), 1))
        P = Q @ R
        H, alpha, fast = F.fast_panel(P)
        if fast:
            accepted += 1
            assert oracle.qr_residual(P, np.asfortranarray(H), alpha) < 3e-15
        else:
            refused += 1
            assert np.linalg.cond(P) > 1e7
    assert accepted >= 4 and refused >= 1
