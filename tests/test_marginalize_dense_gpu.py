"""viml_marginalize_batch (marg_kernel: pseudo-inverse of Amm_s by cyclic Jacobi, Schur complement, Jacobi of A_s) against the
extended-precision reference of tests/marg_reference.py, at every accepted size and at the spectra where an eigen route goes
wrong.

Every bar is the error analysis of marg_reference.check / schur_bars (u = 2^-53), with the kernel's Jacobi taken as backward
stable: its pairs are exact for a matrix within |E|_F <= eps_J |A|_F, eps_J = 12 S r u + 1e-15 (S <= 40 sweeps of r = n - 1
rounds, or n for odd n, of disjoint rotations, each round perturbing A by at most 12 u |A|_F on its two sides; 1e-15 |A|_F is the
off-diagonal the stopping rule off^2 <= 1e-30 |A|_F^2 leaves), and orthogonal to eps_J.  Then:

  A_s, b_s  first-order perturbation of the kept pseudo-inverse X: 2 |E| (|Arm X| |X Amr| + (|Arm P_d| |X Amr| + |Arm X| |P_d Amr|)
            / gap), V's loss of orthogonality eps_J (|Arm| |X Amr| + |Arm X| |Amr|), and the rounding of the products
            u ((3 m + 4) | |Arm| |V| |L^+| |V|^T |Amr| | + 2 |A_s|);
  J^T J     delta = bar(A_s) + eps_J |A_s|_F moves A_s P_{>eps} by 2 delta + 4 max|l_dropped| delta / gap (Davis-Kahan for the
            rotation of P), plus 2 eps_J |A_s P| (orthogonality) and u (n + 5) | |J|^T |J| | (two roundings of sqrt(S) v, the Gram);
  J^T r     2 delta / gap |b_s| + bar(b_s) + 2 eps_J |b_s| + u (n + 4) (| |V_k| |V_k|^T |b_s| | + | |J|^T |r| |) + u |J^T r|, and per
            simple pair with gap_k >= 4 delta the same with 4 delta / gap_k;
  rows      J's rows in ascending eigenvalue order: the dropped ones (l <= eps) first and exactly +-0 with their residuals, each kept
            row's squared norm its eigenvalue to delta + l (2 eps_J + (n + 4) u), rows orthogonal to 2 eps_J + (n + 4) u.

The bars hold only in their first-order range (|E| |X| <= 1/2, |E| <= gap / 4, no eigenvalue within delta of eps); graded rows at
the realistic inertial scales and kappa(Amm) = 1e12 fall outside it, and there only finiteness is checked.  Exact structure is
checked bit for bit: m = 0 returns A and b, a diagonal input returns sqrt(l) and sqrt(1 / l) b in ascending order (ties by index)
with l == eps dropped, an exactly zero row (eps = 0) decouples, and with K > 2 x SMs (the grid-stride loop reusing a CTA's scratch)
every problem equals its own K = 1 call."""
import numpy as np
import pytest

import marg_reference as mr

pytestmark = pytest.mark.gpu

S_DEVICE = 40      # block_jacobi's sweep cap
MAX_POS = 256      # viml_marginalize_batch accepts pos <= 256
EIG_SIZES = {1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 63, 64, 65, 100, 127, 128, 129, 200, 255, 256}


def _run(ctx, A, b, m, eps=1e-8):
    got = ctx.marginalize(np.asarray(A)[None], np.asarray(b)[None], m, eps)
    return (got["A_schur"][0], got["b_schur"][0], got["linearized_jacobians"][0], got["linearized_residuals"][0])


def test_every_size(ctx):
    """pos = 1 .. 256 with m in {0, 1, 15, pos / 2, pos - 1} (n >= 1): odd and even n and m (the round robin's dummy player), n = 1,
    m > n, and m = 15 (MARGIN_OLD's pose and speed-bias).  A_s and b_s at every pair (by the reference's solve route outside
    EIG_SIZES), the eigen outputs at the sizes of EIG_SIZES.
    Spectra log-spaced over [1e-2, 1] (Amm) and [1e-3, 10] (A_s); every third problem has a skew-symmetric part of 1e-6 |A|."""
    rng = np.random.default_rng(2025)
    worst = 0.0
    for pos in range(1, MAX_POS + 1):
        for m in sorted({0, 1, 15, pos // 2, pos - 1}):
            if m >= pos:
                continue
            n = pos - m
            A, b = mr.problem(rng, np.logspace(0, -2, m), np.logspace(1, -3, n), skew=1e-6 if (pos + m) % 3 == 0 else 0.0)
            As, bs, J, r = _run(ctx, A, b, m)
            if m == 0:
                assert np.array_equal(As.view(np.uint64), A.view(np.uint64)) and np.array_equal(bs.view(np.uint64), b.view(np.uint64))
            eig = pos in EIG_SIZES
            ref = mr.marginalize(A, b, m, eig=eig, solve=not eig)
            worst = max(worst, mr.check(ref, As, bs, J if eig else None, r if eig else None, S_DEVICE, ("size", pos, m)))
    print("every size: largest error / bar", worst)


@pytest.mark.parametrize("name", [c[0] for c in mr.edge_cases()])
def test_spectrum_edges(ctx, name):
    A, b, m, eps = {c[0]: c[1:] for c in mr.edge_cases()}[name]
    ref = mr.marginalize(A, b, m, eps)
    As, bs, J, r = _run(ctx, A, b, m, eps)
    q = mr.check(ref, As, bs, J, r, S_DEVICE, ("edge", name), bounded=name not in mr.UNBOUNDED)
    print(name, "largest error / bar", q)
    if name == "zero":
        assert np.all(As == 0) and np.array_equal(bs, b[m:]) and np.all(J == 0) and np.all(r == 0)


def test_diagonal_exact(ctx):
    """A diagonal A: no rotation runs, so the outputs are exact: A_s = Arr, b_s = brr, row rank(k) of J is sqrt(l_k) e_k and
    r = sqrt(fl(1 / l_k)) b_k for l_k > eps, both +-0 otherwise; l_k == eps (both in Amm and in A_s) is dropped, ties keep index
    order, and eps = 0 with an exactly zero eigenvalue of Amm leaves every output finite (1 / 0 is never formed)."""
    rng = np.random.default_rng(4)
    for eps, mm, kk in ((1e-8, [1e-8, 2.0, -3.0, 0.0, 5.0], [3.0, 1e-8, -1.0, 3.0, 0.0, 1e-9, 7.5, 3.0]),
                        (0.0, [0.0, 4.0, 0.0], [0.0, 2.0, -0.5, 2.0, 9.0]),
                        (2.0, [], [2.0, 1.0, 2.0, 4.0, 16.0])):
        d = np.array(mm + kk)
        pos, m = len(d), len(mm)
        A = np.diag(d)
        b = rng.standard_normal(pos)
        As, bs, J, r = _run(ctx, A, b, m, eps)
        assert np.array_equal(As, A[m:, m:]) and np.array_equal(bs, b[m:]), eps
        lam = d[m:]
        rank = np.empty(len(lam), int)
        rank[np.argsort(lam, kind="stable")] = np.arange(len(lam))
        Je = np.zeros_like(J)
        re = np.zeros_like(r)
        for k, l in enumerate(lam):
            if l > eps:
                Je[rank[k], k] = np.sqrt(l)
                re[rank[k]] = np.sqrt(1.0 / l) * b[m + k]
        assert np.array_equal(J, Je) and np.array_equal(r, re), (eps, J, Je, r, re)


def test_zero_rows_decouple(ctx):
    """With eps = 0 an exactly zero row and column (one in Amm, one in the kept part) is an exactly zero eigenvalue that no rotation
    touches: it is dropped, and everything else equals the problem without those rows, to the bars."""
    rng = np.random.default_rng(8)
    pos, m, zm, zr = 40, 15, 4, 15 + 7
    A, b = mr.problem(rng, np.logspace(1, -1, m), np.logspace(1, -1, pos - m))
    for z in (zm, zr):
        A[z, :] = 0.0
        A[:, z] = 0.0
    As, bs, J, r = _run(ctx, A, b, m, 0.0)
    keep = np.array([i for i in range(pos) if i not in (zm, zr)])
    kr = np.array([i for i in range(pos - m) if i != zr - m])
    assert np.all(As[zr - m] == 0) and np.all(As[:, zr - m] == 0) and bs[zr - m] == b[zr]
    assert np.all(J[0] == 0) and r[0] == 0 and np.all(J[:, zr - m] == 0)
    ref = mr.marginalize(A[np.ix_(keep, keep)], b[keep], m - 1, 0.0)
    mr.check(ref, As[np.ix_(kr, kr)], bs[kr], J[1:][:, kr], r[1:], S_DEVICE, "zero rows")


def test_grid_stride_reuses_scratch(ctx):
    """K = 333 > 2 x 148 distinct problems (different spectra: rank-deficient, negative, clustered, so different sweep counts): the
    grid-stride loop gives a CTA several problems in its scratch slice; each must equal its own K = 1 call bit for bit (one CTA per
    problem, a fixed order of every sum)."""
    rng = np.random.default_rng(12)
    pos, m, K = 40, 15, 333
    A = np.empty((K, pos, pos))
    b = rng.standard_normal((K, pos))
    for k in range(K):
        kind = k % 4
        mm = np.logspace(0, -2, m) if kind != 1 else np.concatenate([np.zeros(3), np.logspace(0, -2, m - 3)])
        ss = np.logspace(1, -3, pos - m) if kind != 2 else np.linspace(-2, 3, pos - m)
        if kind == 3:
            ss = 1.0 + 1e-10 * np.arange(pos - m)
        A[k] = mr.problem(rng, mm, ss)[0]
    got = ctx.marginalize(A, b, m)
    for k in range(K):
        one = ctx.marginalize(A[k:k + 1], b[k:k + 1], m)
        for key in got:
            assert np.array_equal(got[key][k].view(np.uint64), one[key][0].view(np.uint64)), (k, key)
