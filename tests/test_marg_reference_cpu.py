"""The marginalisation reference (tests/marg_reference.py) against a 40-digit computation, and the C++ oracle's
orc_marginalize_dense against the reference under the bars the device is held to (no GPU).

The 40-digit route takes the eigenpairs of Amm_s and of A_s from mpmath.eigsy and forms everything else in longdouble, so both
sides round their products in longdouble: the bars of marg_reference.check with u_ld doubled, and a refinement of at most 15
sweeps' worth of rounding (Newton-Schulz, V^T A V and the Jacobi sweeps) that stops at off <= n u_ld |A|_F."""
import numpy as np
import pytest

import marg_reference as mr

LD = mr.LD


def _mp_eigh(A):
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    n = A.shape[0]

    def mpf(v):   # a longdouble as the exact sum of two doubles
        hi = float(v)
        return mp.mpf(hi) + mp.mpf(float(v - LD(hi)))

    M = mp.matrix(n, n)
    for i in range(n):
        for j in range(n):
            M[i, j] = mpf(A[i, j])
    E, Q = mp.eigsy(M)

    def ld(x):
        hi = float(x)
        return LD(hi) + LD(float(x - hi))

    w = np.array([ld(E[i]) for i in range(n)], dtype=LD)
    V = np.array([[ld(Q[i, j]) for j in range(n)] for i in range(n)], dtype=LD)
    o = np.argsort(w, kind="stable")
    return w[o], V[:, o]


def _rows(ref):
    """J and r the way the reference code forms them, from the reference's own eigenpairs (longdouble)."""
    w, V, kept = ref["w"], ref["V"], ref["info"]["kept"]
    S = np.where(kept, w, LD(0))
    J = (np.sqrt(S)[:, None] * V.T)
    r = np.where(kept, 1 / np.sqrt(np.where(kept, w, LD(1))), LD(0)) * (V.T @ ref["b_s"])
    return J, r


SMALL = ["kappa1e+02", "kappa1e+10", "graded", "null", "gauge", "eps_sides_mm", "eps_sides_s", "negative", "repeated", "cluster", "zero", "eps0",
         "eps_large", "asymmetric", "n1"]


@pytest.mark.parametrize("name", SMALL)
def test_reference_against_mpmath(name):
    case = {c[0]: c[1:] for c in mr.edge_cases()}[name]
    A, b, m, eps = case
    if A.shape[0] > 24:   # keep the 40-digit eigensolver at n <= 24: the leading 24 x 24 of the case
        k = 24
        A, b, m = A[:k, :k], b[:k], min(m, 12)
    truth = mr.marginalize(A, b, m, eps, eigh=_mp_eigh)
    ref = mr.marginalize(A, b, m, eps)
    J, r = _rows(ref)
    n = A.shape[0] - m
    mr.check(truth, ref["A_s"], ref["b_s"], J, r, 15, ("mpmath", name), unit=2 * mr.U_LD, stop=n * mr.U_LD,
             bounded=name not in mr.UNBOUNDED)


def test_reference_reports_undecidable_threshold():
    """An eigenvalue of Amm at eps (to rounding) is reported, not assigned to a side; so is one of A_s."""
    rng = np.random.default_rng(5)
    A, b = mr.problem(rng, [1e-8, 1.0, 2.0], [1.0, 3.0, 2.0])
    assert mr.marginalize(A, b, 3, 1e-8)["Amm_info"]["undecidable"]
    assert not mr.marginalize(A, b, 3, 1e-5)["Amm_info"]["undecidable"]
    A, b = mr.problem(rng, [1.0, 3.0, 2.0], [1.0, 1e-8, 3.0])
    assert mr.marginalize(A, b, 3, 1e-8)["info"]["undecidable"]
    assert not mr.marginalize(A, b, 3, 1e-5)["info"]["undecidable"]


def test_schur_solve_matches_eigen_route():
    """The solve route of the size sweeps against the eigen route where both apply (every eigenvalue of Amm kept)."""
    rng = np.random.default_rng(3)
    for pos, m in ((17, 8), (64, 63), (130, 65)):
        A, b = mr.problem(rng, np.logspace(2, -1, m), np.logspace(1, -1, pos - m))
        ref = mr.marginalize(A, b, m, eig=False)
        As, bs = mr.schur_solve(A, b, m)
        bars = mr.schur_bars(ref, 15, 2 * mr.U_LD, m * mr.U_LD)
        assert mr._n2((As - ref["A_s"]).astype(np.float64)) <= bars["A_s"]
        assert np.linalg.norm((bs - ref["b_s"]).astype(np.float64)) <= bars["b_s"]


@pytest.mark.parametrize("name", [c[0] for c in mr.edge_cases()])
def test_oracle_against_reference(orc, name):
    """orc_marginalize_dense (serial cyclic Jacobi, at most 60 sweeps) under the bars of the device with its own sweep cap."""
    A, b, m, eps = {c[0]: c[1:] for c in mr.edge_cases()}[name]
    ref = mr.marginalize(A, b, m, eps)
    As, bs, lj, lr = orc.marginalize_dense(A, b, m, eps)
    mr.check(ref, As, bs, lj, lr, 60, ("oracle", name), bounded=name not in mr.UNBOUNDED)


def test_oracle_every_size_sample(orc):
    rng = np.random.default_rng(11)
    for pos in (1, 2, 3, 16, 17, 33, 64, 97):
        for m in sorted({0, 1, 15, pos // 2, pos - 1}):
            if m >= pos:
                continue
            A, b = mr.problem(rng, np.logspace(0, -3, m), np.logspace(0, -3, pos - m))
            ref = mr.marginalize(A, b, m)
            As, bs, lj, lr = orc.marginalize_dense(A, b, m)
            mr.check(ref, As, bs, lj, lr, 60, ("oracle sizes", pos, m))
