"""The dense part of viml_gn_step and viml_reduced_from_schur against an extended-precision reference, at every accepted system size.

A step builds Sx = embed(S) + sum_k J_k^T J_k, gx = embed(g) + sum_k J_k^T r_k and solves (Sx + lambda diag Sx) dx = -gx with a tiled
Cholesky: solve_tiled_kernel<true> (the system built in shared memory) for Dx <= 200, reduced_kernel + solve_tiled_kernel<false>
for 201 <= Dx <= 232.  The systems here are built from dense factors whose Sx has a chosen spectrum; the reference forms gx and
Sx x in np.longdouble from the same factors, solves with a float64 Cholesky and three steps of iterative refinement with the
residual in longdouble, and every bar is the error analysis of the computation it checks (u = 2^-53), not a tolerance that
happens to pass:

  assembly   |Sx^ - Sx| <= gamma(k) (|J|^T |J| + |S|) entrywise, k the roundings of one entry (Higham, Accuracy and Stability of
             Numerical Algorithms, 2nd ed., eq. 3.5 for each sum of products);
  Cholesky   (M^ + dC) x^ = -g^,  |dC| <= gamma(3 Dx + 1) |R^T| |R|  (Higham Thm 10.4, factorisation and both substitutions);
  so the normwise backward error  eta = |M x^ + g| / (|M| |x^| + |g|)  measured against the exact M = Sx + lambda diag Sx is at most
  u [(3 Dx + 1) |(|R^T| |R|)| + (rows + 2)(1 + lambda) |(|J|^T |J| + |S|)|] / |M|   or   u (rows + 1) |(|J|^T |r| + |g|)| / |g|,
  whichever is larger (2-norms; for a nonnegative B >= |E| entrywise, |E|_2 <= |B|_2), and the forward error is at most
  2 kappa eta / (1 - kappa eta) (Higham Thm 7.2 with the relative perturbation eta in M and g).

A wrong tile update, a wrong padding row or a double-counted factor moves eta by many orders of magnitude; these bars stay
valid at kappa = 1e13.  Which kernel and which stage branch ran is a function of the shapes alone (see gn_kernels.cuh)."""
import ctypes as C

import numpy as np
import pytest
import scipy.linalg

from vi_helpers import Guarded

U = 2.0 ** -53
LD = np.longdouble
U_LD = float(np.finfo(LD).eps) / 2   # unit roundoff of the extended type the reference computes in
FUSED_STAGE, REDUCED_STAGE = 6656, 12288   # kFusedStage (common.cuh), gn::kReducedStage (doubles)
MAX_DX = 232


def _stage_need(n, c):
    """Doubles a factor of n rows x c columns needs in a kernel's Jacobian stage (np (cp + 4) + np)."""
    np_, cp = (n + 3) & ~3, (c + 7) & ~7
    return np_ * (cp + 4) + np_


# ---- the reference --------------------------------------------------------------------------------------------------------------
class Ref:
    """One window's system Sx = embed(S) + sum J^T J, gx = embed(g) + sum J^T r (factors: list of (r, J, col_index)), with the
    exact (longdouble) matrix-vector product and right-hand side, and the solve of (Sx + lambda diag Sx) x = -gx."""

    def __init__(self, Dx, factors, S=None, g=None):
        self.Dx, self.factors = Dx, [(np.asarray(r, float), np.asarray(J, float).reshape(len(r), len(ci)), np.asarray(ci))
                                     for r, J, ci in factors]
        self.S = None if S is None else np.asarray(S, float)
        self.D = 0 if S is None else self.S.shape[0]
        self.gS = None if g is None else np.asarray(g, float)
        gx = np.zeros(Dx, LD)
        d = np.zeros(Dx, LD)
        cnt = np.zeros((Dx, Dx), np.int64)   # rows summed into each entry
        B = np.zeros((Dx, Dx))               # |J|^T |J| + |S|
        gabs = np.zeros(Dx)                  # |J|^T |r| + |g|
        for r, J, ci in self.factors:
            Jl = J.astype(LD)
            gx[ci] += Jl.T @ r.astype(LD)
            d[ci] += (Jl * Jl).sum(axis=0)
            cnt[np.ix_(ci, ci)] += len(r)
            B[np.ix_(ci, ci)] += np.abs(J).T @ np.abs(J)
            gabs[ci] += np.abs(J).T @ np.abs(r)
        if S is not None:
            D = self.D
            gx[:D] += self.gS.astype(LD)
            d[:D] += np.diag(self.S).astype(LD)
            B[:D, :D] += np.abs(self.S)
            gabs[:D] += np.abs(self.gS)
            cnt[:D, :D] += 1
        self.gx, self.d, self.cnt, self.B, self.gabs = gx, d, cnt, B, gabs
        self.rows = int(cnt.max()) if Dx else 0

    def Sx64(self):
        """Sx summed in float64: only the Cholesky factor the refinement iterates with is built from it; the longdouble residual
        corrects its rounding."""
        A = np.zeros((self.Dx, self.Dx))
        for r, J, ci in self.factors:
            A[np.ix_(ci, ci)] += J.T @ J
        if self.S is not None:
            A[:self.D, :self.D] += self.S
        return A

    def sx_matvec(self, x):
        """Sx x, exactly up to longdouble rounding (no Sx is formed)."""
        xl = np.asarray(x).astype(LD)
        y = np.zeros(self.Dx, LD)
        for r, J, ci in self.factors:
            Jl = J.astype(LD)
            y[ci] += Jl.T @ (Jl @ xl[ci])
        if self.S is not None:
            y[:self.D] += self.S.astype(LD) @ xl[:self.D]
        return y

    def residual(self, x, lam):
        """(Sx + lambda diag Sx) x + gx in longdouble."""
        xl = np.asarray(x).astype(LD)
        return self.sx_matvec(xl) + LD(lam) * self.d * xl + self.gx

    def spectrum(self, lam):
        """(lambda_min, lambda_max) of M = Sx + lambda diag Sx from the singular values of a square root of M (accurate where an
        eigensolver on M itself would lose lambda_min below u |M|)."""
        rows = []
        for r, J, ci in self.factors:
            Z = np.zeros((len(r), self.Dx))
            Z[:, ci] = J
            rows.append(Z)
        if self.S is not None:
            e, V = np.linalg.eigh(0.5 * (self.S + self.S.T))
            Z = np.zeros((self.D, self.Dx))
            Z[:, :self.D] = np.sqrt(np.maximum(e, 0.0))[:, None] * V.T
            rows.append(Z)
        if lam:
            rows.append(np.diag(np.sqrt(lam * self.d.astype(np.float64))))
        s = np.linalg.svd(np.concatenate(rows) if rows else np.zeros((1, self.Dx)), compute_uv=False)
        return float(s[-1] ** 2) if len(s) == self.Dx else 0.0, float(s[0] ** 2)

    def solve(self, lam, steps=3):
        """x* (longdouble), |last correction| / |x*|, and the float64 Cholesky factor R (None when it breaks down)."""
        M = self.Sx64()
        M[np.diag_indices(self.Dx)] += lam * self.d.astype(np.float64)
        try:
            R, low = scipy.linalg.cho_factor(M, lower=False, check_finite=False)
        except np.linalg.LinAlgError:
            return None, None, None
        x = scipy.linalg.cho_solve((R, low), -self.gx.astype(np.float64)).astype(LD)
        corr = np.inf
        for _ in range(steps):
            dx = scipy.linalg.cho_solve((R, low), -self.residual(x, lam).astype(np.float64))
            x = x + dx.astype(LD)
            corr = float(np.linalg.norm(dx) / max(np.linalg.norm(x.astype(np.float64)), 1e-300))
        return x, corr, np.triu(R)

    def model(self, x):
        """-gx.x - 1/2 x.Sx x in longdouble."""
        xl = np.asarray(x).astype(LD)
        return -(self.gx @ xl) - LD(0.5) * (xl @ self.sx_matvec(xl))


def check_step(ref, lam, dx, solved, model, tag):
    """Holds the kernel's step of one window to the bars of the module docstring; returns eta / bar."""
    Dx = ref.Dx
    lmin, lmax = ref.spectrum(lam)
    x_star, corr, R = ref.solve(lam)
    ref_ok = x_star is not None
    if bool(solved) != ref_ok:
        # the two Cholesky factorisations may disagree only on a matrix that is singular to working precision
        assert lmin <= Dx * U * lmax, (tag, "solved", solved, ref_ok, lmin / lmax)
    if not solved:
        assert np.all(dx.view(np.uint64) == 0), tag
        assert model == 0.0 and not np.signbit(model), tag
        return 0.0
    assert np.all(np.isfinite(dx)), tag
    res = ref.residual(dx, lam).astype(np.float64)
    nM, nx, ng = lmax, np.linalg.norm(dx), np.linalg.norm(ref.gx.astype(np.float64))
    eta = np.linalg.norm(res) / (nM * nx + ng)
    # the Cholesky term with the reference's factor (the kernel's |R^T||R| agrees with it to first order); a failed reference
    # factorisation (allowed above) leaves the term to the largest it can be, n |M| (Higham Lemma 10.5 with |R|^2 <= n |M|)
    bR = np.linalg.norm(np.abs(R).T @ np.abs(R), 2) if ref_ok else Dx * nM
    bJ = np.linalg.norm(ref.B, 2)
    bar = max(U * ((3 * Dx + 1) * bR + (ref.rows + 2) * (1.0 + lam) * bJ) / nM,
              U * (ref.rows + 1) * np.linalg.norm(ref.gabs) / ng if ng > 0 else 0.0)
    assert eta <= bar, (tag, "backward error", eta, bar)
    if ref_ok:
        kappa = lmax / lmin if lmin > 0 else np.inf
        fwd = np.linalg.norm(dx - x_star.astype(np.float64)) / np.linalg.norm(x_star.astype(np.float64))
        fbar = (2 * kappa * eta / (1 - kappa * eta) if kappa * eta < 1 else np.inf) + corr
        assert fwd <= fbar, (tag, "forward error", fwd, fbar, kappa)
    # cost[2]: m(x^) in longdouble at the kernel's own x^.  With res = M x^ + g, m(x^) = -1/2 g.x^ + 1/2 lambda x^.D x^ - 1/2 x^.res
    # (what the fused kernel evaluates, res dropped); both kernels use their rounded g, diag / Sx, each off by gamma(rows + 1)
    # times |J|^T|r|, |J|^T|J|, and sum Dx + 2 terms
    ax = np.abs(dx)
    mbar = (0.5 * abs(float(dx @ res)) +
            U * (Dx + ref.rows + 2) * (ref.gabs @ ax + ax @ ref.B @ ax + lam * float(ref.d.astype(np.float64) @ (ax * ax))))
    merr = abs(model - float(ref.model(dx)))
    assert merr <= mbar, (tag, "model decrease", model, float(ref.model(dx)), merr, mbar)
    return eta / bar


# ---- systems with a known structure ---------------------------------------------------------------------------------------------
def spd_rows(rng, n, kappa, N=None, scale=1e4):
    """J (N x n, N >= n) with J^T J = Q diag(sigma) Q^T, sigma log-spaced over [scale / kappa, scale], Q random orthogonal.  N == n
    (default): the upper-triangular R of the QR factorisation of diag(sqrt(sigma)) Q^T, so row i touches columns i.. only."""
    Q = np.linalg.qr(rng.standard_normal((n, n)))[0]
    sig = scale * np.logspace(0.0, -np.log10(kappa), n)
    J0 = np.sqrt(sig)[:, None] * Q.T
    if N is None:
        return np.linalg.qr(J0, mode="r")
    Uo = np.linalg.qr(rng.standard_normal((N, n)))[0]
    return Uo @ J0


def split_rows(rng, R, cols, max_rows=24, first=None):
    """Factors (r, J, col_index) from consecutive row groups of R (columns of R -> tangent columns `cols`): a group keeps the
    columns its rows touch, in a random order (col_index unsorted; groups overlap in their columns).  The first group has `first`
    rows when given; a group of the last row of a triangular R is a 1 x 1 factor."""
    n = R.shape[0]
    fs, i = [], 0
    while i < n:
        k = first if (i == 0 and first) else int(rng.integers(1, max_rows + 1))
        k = min(k, n - i)
        blk = R[i:i + k]
        nz = np.flatnonzero(np.any(blk != 0.0, axis=0))
        order = rng.permutation(len(nz))
        fs.append((rng.standard_normal(k), blk[:, nz[order]], np.asarray(cols)[nz[order]]))
        i += k
    return fs


def structured(rng, Dx, kappa, max_rows=24):
    """Factors of one window over all Dx columns (tangent columns permuted) with Sx of condition number ~kappa; the first factor
    has one row and the last (the last row of R) one column."""
    R = spd_rows(rng, Dx, kappa)
    fs = split_rows(rng, R, rng.permutation(Dx), max_rows=max_rows, first=1)
    if len(fs[-1][0]) > 1:   # split the last group so that its last row is a 1-column factor
        r, J, ci = fs.pop()
        keep = np.flatnonzero(np.any(J[-1:] != 0.0, axis=0))
        fs += [(r[:-1], J[:-1], ci), (r[-1:], J[-1:, keep], ci[keep])]
    return fs


def pick_P(Dx, rng):
    """A pose count with D = 6 (P + 1) <= Dx (X = Dx - D extra columns), varied."""
    pmax = Dx // 6 - 1
    return int(rng.integers(1, pmax + 1)) if pmax > 1 else 1


def empty_batch(pkg, W, P, rng):
    """W windows of P poses without point / line factors or landmarks: S = 0, g = 0, so Sx is the dense factors alone."""
    q = rng.standard_normal((W, P + 1, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    x = np.concatenate([rng.standard_normal((W, P + 1, 3)), q], axis=-1)
    return pkg._abi.Batch(x[:, :P], x[:, P], np.zeros((W, 0)), np.zeros(W + 1, np.int32), np.zeros(0, np.uint32), np.zeros((0, 4)))


def dense_of(pkg, W, X, per_window):
    return pkg._abi.Dense(W, X, [(w, r, J, ci) for w, fs in enumerate(per_window) for r, J, ci in fs])


def run_step(pkg, ctx, P, X, per_window, lam, seed=0):
    rng = np.random.default_rng(seed)
    W = len(per_window)
    b = empty_batch(pkg, W, P, rng)
    extra = rng.standard_normal((W, X))
    return b, extra, ctx.gn_step(b, dense_of(pkg, W, X, per_window), extra, 0, lam=lam)


def check_batch(pkg, ctx, Dx, P, per_window, lam, tag, seed=0):
    b, extra, o = run_step(pkg, ctx, P, Dx - 6 * (P + 1), per_window, lam, seed)
    for w, fs in enumerate(per_window):
        check_step(Ref(Dx, fs), lam, o["dx"][w], o["solved"][w], o["cost"][w, 2], (tag, Dx, w, lam))
    return b, extra, o


# ---- the reference itself (CPU) -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kappa", [1e2, 1e10])
def test_reference_against_mpmath(kappa):
    """x* and m(x*) of the reference against a 40-digit solve of the same factors.  Bars: refinement with the residual in
    longdouble converges to |x* - x| / |x| <= 4 n kappa u_ld (Higham Thm 12.1 with u_r = u_ld), plus the last correction for
    what the three steps have not yet removed; m is a sum of n + n^2 terms of x*."""
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    rng = np.random.default_rng(7 if kappa < 1e5 else 8)
    n = 24 if kappa > 1e5 else 19
    fs = structured(rng, n, kappa, max_rows=5)
    ref = Ref(n, fs)
    lam = 0.25
    x, corr, _ = ref.solve(lam)
    A = mp.zeros(n, n)
    g = mp.zeros(n, 1)
    for r, J, ci in fs:
        for a in range(len(ci)):
            g[int(ci[a])] += mp.fsum(mp.mpf(float(J[q, a])) * mp.mpf(float(r[q])) for q in range(len(r)))
            for c in range(len(ci)):
                A[int(ci[a]), int(ci[c])] += mp.fsum(mp.mpf(float(J[q, a])) * mp.mpf(float(J[q, c])) for q in range(len(r)))
    M = A.copy()
    for i in range(n):
        M[i, i] = A[i, i] * (1 + mp.mpf(lam))
    xm = mp.lu_solve(M, -g)
    lmin, lmax = ref.spectrum(lam)
    def mpf(v):   # a longdouble as the exact sum of two doubles
        hi = float(v)
        return mp.mpf(hi) + mp.mpf(float(v - LD(hi)))

    xmv = np.array([float(v) for v in xm])
    err = np.linalg.norm(np.array([float(mpf(x[i]) - xm[i]) for i in range(n)])) / np.linalg.norm(xmv)
    assert err <= 4 * n * (lmax / lmin) * U_LD + corr, (err, lmax / lmin, corr)
    mm = -(g.T * xm)[0] - (xm.T * A * xm)[0] / 2
    # m(x*) - m(x): the gradient -g - Sx x is bounded by |J|^T|r| + (|J|^T|J|) |x| entrywise, |x* - x|_inf <= err |x|_2; and the
    # longdouble evaluation sums n + n^2 terms
    m = ref.model(x)
    ax = np.abs(x.astype(np.float64))
    bound = (n * n + n) * U_LD * (ref.gabs @ ax + ax @ ref.B @ ax) + np.abs(ref.gabs + ref.B @ ax).sum() * err * np.linalg.norm(ax)
    assert abs(float(mpf(m) - mm)) <= bound, (float(mpf(m) - mm), bound)
    # and the bars of check_step hold for the reference's own float64-rounded solution
    xd = x.astype(np.float64)
    check_step(ref, lam, xd, 1, float(ref.model(xd)), ("reference", kappa))


# ---- (a) every size at kappa = 1e3 ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sweep_every_size(pkg, ctx):
    """Dx = 12 .. 232: every tile residue, 2 to 29 tile columns, the fused kernel up to 200 and the unfused one from 201; two
    windows where Dx is odd, one where it is even."""
    rng = np.random.default_rng(2024)
    for Dx in range(12, MAX_DX + 1):
        P = pick_P(Dx, rng)
        per = [structured(rng, Dx, 1e3) for _ in range(1 + Dx % 2)]
        check_batch(pkg, ctx, Dx, P, per, 1e-3 if Dx % 3 == 0 else 0.0, "sweep", seed=Dx)


# ---- (b) conditioning x damping -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("Dx", [48, 171, 200, 201, 232])
def test_conditioning(pkg, ctx, Dx):
    rng = np.random.default_rng(Dx)
    P = 11 if Dx >= 72 else 3
    per = [structured(rng, Dx, kappa) for kappa in (1e6, 1e10, 1e13)]
    for lam in (0.0, 1e-4, 1.0, 1e4):
        check_batch(pkg, ctx, Dx, P, per, lam, "kappa", seed=Dx)


# ---- (c) the stage boundaries and factor shapes ---------------------------------------------------------------------------------
def boundary_window(rng, Dx, n, c):
    """One n x c factor (the shape under test) plus what makes the window's Sx positive definite: for n < c the remaining rows of
    a triangular R as small factors, for n >= c nothing (the factor is full rank)."""
    if n >= c:
        assert c == Dx
        J = spd_rows(rng, Dx, 1e3, N=n)
        order = rng.permutation(Dx)
        return [(rng.standard_normal(n), J[:, order], order)]
    assert c == Dx
    R = spd_rows(rng, Dx, 1e3)
    order = rng.permutation(Dx)
    return [(rng.standard_normal(n), R[:n][:, order], order)] + [
        (rng.standard_normal(1), R[i:i + 1, i:], np.arange(i, Dx)) for i in range(n, Dx)]


@pytest.mark.gpu
def test_stage_boundaries(pkg, ctx):
    """The Jacobian stage of each kernel just fits and just overflows:  fused 76 x 80 (6460 <= 6656) and 77 x 80 (6800);
    reduced_kernel 112 x 104 (12208 <= 12288) and 113 x 104 (12644), those two through viml_reduced_system (Sx entrywise) and
    through the step (where the fused kernel overflows with both)."""
    rng = np.random.default_rng(77)
    P = 11
    for n, c, need, cap in ((76, 80, 6460, FUSED_STAGE), (77, 80, 6800, FUSED_STAGE), (112, 104, 12208, REDUCED_STAGE),
                            (113, 104, 12644, REDUCED_STAGE)):
        Dx = c
        per = [boundary_window(rng, Dx, n, c) for _ in range(2)]
        assert _stage_need(n, c) == need and (need <= cap) == (n in (76, 112))
        for lam in (0.0, 1e-2):
            check_batch(pkg, ctx, Dx, P, per, lam, ("stage", n, c))
        b = empty_batch(pkg, 2, P, rng)
        Sx, gx = ctx.reduced_system(b, dense_of(pkg, 2, Dx - 6 * (P + 1), per), 0)
        for w in range(2):
            check_reduced(Ref(Dx, per[w]), Sx[w], gx[w], ("reduced", n, c))


@pytest.mark.gpu
@pytest.mark.parametrize("Dx", [120, 217])
def test_factor_shapes(pkg, ctx, Dx):
    """Factors of 1 row, of 1 column, of row and column counts that are not multiples of 4 or 8; a window of 200 small factors
    sharing columns; and an empty window between two windows that have factors (its Sx is 0: not solved)."""
    rng = np.random.default_rng(Dx + 1)
    P = 11
    odd = []   # row / column counts 1, 3, 5, 6, 7, 9, 13 over a triangular R
    R = spd_rows(rng, Dx, 1e4)
    cols = rng.permutation(Dx)
    i = 0
    for k in (1, 3, 5, 6, 7, 9, 13):
        blk = R[i:i + k]
        nz = np.flatnonzero(np.any(blk != 0.0, axis=0))
        odd.append((rng.standard_normal(k), blk[:, nz], cols[nz]))
        i += k
    odd += split_rows(rng, R[i:], cols, max_rows=11)
    odd.append((rng.standard_normal(5), rng.standard_normal((5, 1)), cols[:1]))                 # a 5 x 1 column
    odd.append((rng.standard_normal(1), rng.standard_normal((1, 7)), rng.permutation(Dx)[:7]))  # 1 x 7
    many = []
    for _ in range(200):
        k, c = int(rng.integers(1, 6)), int(rng.integers(1, 13))
        many.append((rng.standard_normal(k), 3.0 * rng.standard_normal((k, c)), rng.permutation(Dx)[:c]))
    cover = rng.permutation(Dx)   # every column held by a diagonal factor of 1-row pieces: Sx is positive definite
    many += [(rng.standard_normal(1), np.full((1, 1), 2.0 + rng.uniform()), cover[j:j + 1]) for j in range(Dx)]
    assert len(many) == 200 + Dx and all(len(f[2]) == len(set(f[2].tolist())) for f in many)
    per = [odd, [], many]
    for lam in (0.0, 1e-3):
        b, extra, o = check_batch(pkg, ctx, Dx, P, per, lam, ("shapes", Dx))
        assert o["solved"][1] == 0 and o["cost"][1, 2] == 0.0 and np.all(o["dx"][1].view(np.uint64) == 0)
        assert np.array_equal(o["poses"][1], b.poses[1]) and np.array_equal(o["extra"][1], extra[1])
        assert o["solved"][0] and o["solved"][2]


def check_reduced(ref, Sx, gx, tag):
    """Sx, gx of viml_reduced_system / viml_reduced_from_schur against the exact sums: entrywise within 2 (k + 1) u (|J|^T|J| + |S|)
    with k the rows summed into the entry (a DMMA step or an fma chain rounds at most twice per product, and one more rounding
    adds the factor to S); an entry no factor touches is embed(S) / embed(g) exactly."""
    Dx = ref.Dx
    A = np.zeros((Dx, Dx), LD)
    for r, J, ci in ref.factors:
        Jl = J.astype(LD)
        A[np.ix_(ci, ci)] += Jl.T @ Jl
    emb = np.zeros((Dx, Dx))
    gemb = np.zeros(Dx)
    if ref.S is not None:
        emb[:ref.D, :ref.D] = ref.S
        gemb[:ref.D] = ref.gS
    A += emb.astype(LD)
    ca = np.zeros((Dx, Dx), np.int64)
    gc = np.zeros(Dx, np.int64)
    for r, J, ci in ref.factors:
        ca[np.ix_(ci, ci)] += len(r)
        gc[ci] += len(r)
    err = np.abs((Sx.astype(LD) - A).astype(np.float64))
    bar = 2 * (ca + 1) * U * ref.B
    assert np.all(err <= bar), (tag, "Sx", float((err - bar).max()))
    assert np.array_equal(Sx[ca == 0], emb[ca == 0]), (tag, "untouched Sx entries")
    gerr = np.abs((gx.astype(LD) - ref.gx).astype(np.float64))
    assert np.all(gerr <= 2 * (gc + 1) * U * ref.gabs), (tag, "gx")
    assert np.array_equal(gx[gc == 0], gemb[gc == 0]), (tag, "untouched gx entries")


# ---- (d) realistic inertial windows ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("P", [11, 12])
def test_realistic_inertial_windows(pkg, ctx, P):
    """EuRoC noise densities (bias rows of the covariance near 1e-11) with visual factors; P = 12 has an 81 x 81 prior, which
    overflows the fused kernel's stage at Dx = 186.  S from viml_linearize_batch is an input of the reference; the step
    linearises again and sums its pose blocks through atomics, so its own S differs from that one by the rounding of its sums,
    which the assembly term bounds with |S| replaced by |H_pp| + |H_lp|^T H_ll^-1 |H_lp| and k by the factors of the window."""
    abi = pkg._abi
    batch = pkg.synth.make_windows(3, seed=300 + P, P=P, F=60)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=310 + P, realistic=True)
    dense = vi.to_dense(ctx.inertial_evaluate(batch, extra, vi))
    flags = abi.LOSS_CAUCHY
    lin = ctx.linearize(batch, abi.OUT_HB | abi.OUT_SCHUR | flags)
    Dx = batch.D + vi.X
    if P == 12:
        assert vi.n_max == 81 and _stage_need(81, 81) > FUSED_STAGE and Dx == 186
    for lam in (0.0, 1e-4):
        o = ctx.gn_step(batch, dense, extra, flags, lam=lam)
        for w in range(batch.W):
            fs = [(r, J, ci) for (ww, r, J, ci) in dense.factors if ww == w]
            ref = Ref(Dx, fs, lin["S"][w], lin["g"][w])
            Hlp, Hll = lin["H_lp"][w], lin["H_ll"][w]
            keep = Hll > 1e-8
            vis = np.abs(lin["H_pp"][w]) + np.abs(Hlp[keep]).T @ (np.abs(Hlp[keep]) / Hll[keep][:, None])
            gvis = np.abs(lin["b_p"][w]) + np.abs(Hlp[keep]).T @ (np.abs(lin["b_l"][w][keep]) / Hll[keep])
            nvis = int(np.diff(batch.pf_window_offset)[w] + np.diff(batch.lf_window_offset)[w] + batch.F)
            ref.B[:batch.D, :batch.D] += vis - np.abs(ref.S)
            ref.gabs[:batch.D] += gvis - np.abs(ref.gS)
            ref.rows = max(ref.rows, nvis)
            check_step(ref, lam, o["dx"][w], o["solved"][w], o["cost"][w, 2], ("inertial", P, w, lam))


# ---- (e) where a factorisation fails --------------------------------------------------------------------------------------------
def failing_window(rng, Dx, p):
    """A positive definite system on every column but p, which no factor touches.  Sx = embed(S) + sum J^T J is positive
    semidefinite by construction, so no input makes a pivot clearly negative; but row p of Sx is exactly 0, every update of it
    subtracts products with L[p][k] = 0, and (1 + lambda) 0 = 0: the pivot of column p is exactly 0 for every lambda, whatever the
    rounding of the rest of the factorisation."""
    rest = np.array([c for c in range(Dx) if c != p])
    return split_rows(rng, spd_rows(rng, Dx - 1, 1e3), rest[rng.permutation(len(rest))])


@pytest.mark.gpu
@pytest.mark.parametrize("Dx", [171, 227])
def test_failure_only_affects_its_window(pkg, ctx, Dx):
    """A zero pivot (a column no factor touches) in the first tile, a middle tile, the last full tile and the real rows of the padded last tile, and a NaN in one
    Jacobian entry: that window alone reports solved = 0 with dx = +0.0, its state returned bit for bit, cost[1] == cost[0] and
    cost[2] == 0; every other window is bit-identical to the same window solved alone."""
    rng = np.random.default_rng(Dx)
    P = 11
    X = Dx - 6 * (P + 1)
    NB = (Dx + 7) // 8
    assert Dx % 8 >= 2
    places = {"first tile": 2, "middle tile": 8 * (NB // 2) + 3, "last full tile": 8 * (NB - 2) + 5,
              "padded last tile": 8 * (NB - 1) + Dx % 8 - 1}
    bads = {name: failing_window(rng, Dx, p) for name, p in places.items()}
    nan = structured(rng, Dx, 1e3)
    r, J, ci = nan[len(nan) // 2]
    J = J.copy()
    J[len(r) // 2, len(ci) // 2] = np.nan
    nan[len(nan) // 2] = (r, J, ci)
    bads["NaN in a Jacobian"] = nan
    goods = [structured(rng, Dx, 1e3) for _ in range(2)]
    for name, bad in bads.items():
        b, extra, o = run_step(pkg, ctx, P, X, [goods[0], bad, goods[1]], 0.0, seed=0)
        assert o["solved"][1] == 0, name
        assert np.all(o["dx"][1].view(np.uint64) == 0), name
        assert np.array_equal(o["poses"][1].view(np.uint64), b.poses[1].view(np.uint64)), name
        assert np.array_equal(o["ex_pose"][1].view(np.uint64), b.ex_pose[1].view(np.uint64)), name
        assert np.array_equal(o["extra"][1].view(np.uint64), extra[1].view(np.uint64)), name
        assert o["cost"][1, 1] == o["cost"][1, 0] and o["cost"][1, 2] == 0.0, (name, o["cost"][1])
        for w, k in ((0, 0), (2, 1)):
            assert o["solved"][w] == 1, name
            b1 = pkg._abi.Batch(b.poses[w:w + 1], b.ex_pose[w:w + 1], np.zeros((1, 0)), np.zeros(2, np.int32), np.zeros(0, np.uint32),
                                np.zeros((0, 4)))
            one = ctx.gn_step(b1, dense_of(pkg, 1, X, [goods[k]]), extra[w:w + 1], 0, lam=0.0)
            for key in ("dx", "cost", "poses", "ex_pose", "extra", "solved"):
                assert np.array_equal(o[key][w], one[key][0]), (name, key)
    # damping does not move a zero pivot
    _, _, o = run_step(pkg, ctx, P, X, [goods[0], bads["padded last tile"], goods[1]], 1e-2)
    assert list(o["solved"]) == [1, 0, 1]


# ---- (f) viml_reduced_from_schur ------------------------------------------------------------------------------------------------
def schur_case(rng, W, D, X):
    """Random (not symmetric: a transposed copy shows) S, g and factors over ~3/4 of the columns, one of them too large for
    reduced_kernel's stage when Dx allows."""
    Dx = D + X
    S = rng.standard_normal((W, D, D))
    g = rng.standard_normal((W, D))
    per = []
    for w in range(W):
        touched = rng.permutation(Dx)[:max(1, (3 * Dx) // 4)]
        fs = []
        for _ in range(int(rng.integers(3, 9))):
            c = int(rng.integers(1, min(len(touched), 40) + 1))
            n = int(rng.integers(1, 30))
            fs.append((rng.standard_normal(n), rng.standard_normal((n, c)), rng.permutation(touched)[:c]))
        if Dx >= 100:   # all touched columns, rows enough to overflow the stage
            c = len(touched)
            n = REDUCED_STAGE // (((c + 7) & ~7) + 5) + 1
            fs.append((rng.standard_normal(n), rng.standard_normal((n, c)), rng.permutation(touched)))
            assert _stage_need(n, c) > REDUCED_STAGE
        per.append(fs)
    return S, g, per


@pytest.mark.gpu
@pytest.mark.parametrize("D,X", [(1, 11), (7, 60), (72, 99), (150, 150)])
def test_reduced_from_schur(pkg, ctx, D, X):
    abi = pkg._abi
    rng = np.random.default_rng(D * 1000 + X)
    W, Dx = 3, D + X
    S, g, per = schur_case(rng, W, D, X)
    dense = dense_of(pkg, W, X, per)
    # host pointers
    Sx, gx = np.full((W, Dx, Dx), np.nan), np.full((W, Dx), np.nan)
    ro = abi.ReducedOut()
    ro.Sx, ro.gx = abi.ptr(Sx), abi.ptr(gx)
    d = dense.struct()
    ctx._check(ctx.lib.viml_reduced_from_schur(ctx.h, W, D, abi.ptr(S), abi.ptr(g), C.byref(d), C.byref(ro), 0))
    for w in range(W):
        check_reduced(Ref(Dx, per[w], S[w], g[w]), Sx[w], gx[w], ("from_schur", D, X, w))
    # device pointers: the same bits, nothing written outside Sx / gx, the inputs left as they were
    ins = {"S": S, "g": g, **dense.arrays()}
    gi = {k: Guarded(ctx, a) for k, a in ins.items()}
    go = {"Sx": Guarded(ctx, np.full((W, Dx, Dx), np.nan)), "gx": Guarded(ctx, np.full((W, Dx), np.nan))}
    dd = dense.struct({k: gi[k].ptr for k in dense.arrays()})
    rd = abi.ReducedOut()
    rd.Sx, rd.gx = go["Sx"].ptr, go["gx"].ptr
    ctx._check(ctx.lib.viml_reduced_from_schur(ctx.h, W, D, gi["S"].ptr, gi["g"].ptr, C.byref(dd), C.byref(rd), pkg.PTRS_DEVICE))
    ctx.sync()
    assert np.array_equal(go["Sx"].check(), Sx) and np.array_equal(go["gx"].check(), gx)
    for k, v in gi.items():
        assert np.array_equal(v.check().view(np.uint8), np.ascontiguousarray(ins[k]).view(np.uint8)), k
    for v in list(gi.values()) + list(go.values()):
        v.free()


# ---- (g) repeatability ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("Dx", [171, 227])
def test_step_repeats_bit_for_bit(pkg, ctx, Dx):
    """Without visual factors every kernel of the step is order-deterministic (no atomics): two calls give the same bits."""
    rng = np.random.default_rng(Dx + 5)
    per = [structured(rng, Dx, 1e6) for _ in range(4)]
    a = run_step(pkg, ctx, 11, Dx - 72, per, 1e-3, seed=9)[2]
    b = run_step(pkg, ctx, 11, Dx - 72, per, 1e-3, seed=9)[2]
    for k in a:
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), k
