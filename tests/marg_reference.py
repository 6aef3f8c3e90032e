"""Extended-precision reference of MarginalizationInfo::marginalize's dense core (marginalization_factor.cpp:264-293).

Given A (pos x pos), b, m and eps in float64, marginalize() computes in np.longdouble (80-bit on x86-64: u_ld = 2^-64):

  Amm_s = (Amm + Amm^T) / 2, its eigenpairs, Amm^+ = V diag(l > eps ? 1 / l : 0) V^T,
  A_s = Arr - Arm Amm^+ Amr,  b_s = brr - Arm Amm^+ bmm,
  the eigenpairs of A_s with its upper triangle mirrored from the lower one (SelfAdjointEigenSolver reads the lower triangle),
  and the outputs that do not depend on the sign of an eigenvector: J^T J = sum_{l > eps} l v v^T, J^T r = P_{>eps} b_s, and per
  eigenpair J_k^T r_k = v_k (v_k . b_s).

Each eigen-decomposition starts from float64 numpy.linalg.eigh and is refined by cyclic Jacobi sweeps in longdouble on V^T A V,
all n / 2 disjoint rotations of a round-robin round applied at once, until off(A)^2 <= (n u_ld)^2 |A|_F^2.  What the bars of the
tests need comes with the result: the eigenvalues, how far the nearest one is from eps, the gap between the kept and the dropped
ones, |Arm Amm^+|, |Amm^+ Amr|, |Arm P_dropped|, |Amm^+| and kappa of the kept part of Amm.

An eigenvalue within `band` of eps (the perturbation a backward-stable float64 eigen-decomposition may make, see `jacobi_eps`)
makes the threshold undecidable: the reference reports it (`undecidable`) and does not pick a side."""
import numpy as np

LD = np.longdouble
U = 2.0 ** -53
U_LD = float(np.finfo(LD).eps) / 2


def jacobi_eps(n, sweeps, unit=U, stop=1e-15):
    """Relative backward error |E|_F / |A|_F of a cyclic Jacobi of `sweeps` sweeps on an n x n matrix: a sweep is n - 1 rounds
    (odd n: n rounds) of disjoint rotations, and a round applied on both sides perturbs A by at most 12 u |A|_F (each side: c and
    s carry 2 u from their formulas, each updated entry two products and a sum; Higham, Accuracy and Stability of Numerical
    Algorithms, 2nd ed., Lemmas 19.8-19.9).  The device's stopping rule adds the off-diagonal it leaves, at most 1e-15 |A|_F when
    the rule is met; when the sweep cap stops it instead, what remains is the floor the rounding of the sweeps leaves, which the
    first term bounds.  The same count bounds the loss of orthogonality |V^T V - I|_2 of the accumulated rotations."""
    rounds = n if n % 2 else n - 1
    return 12.0 * sweeps * max(rounds, 1) * unit + stop


def eigh_ld(A, tol=None, max_sweeps=12):
    """Eigenpairs of the symmetric longdouble matrix A, ascending: (w, V) in longdouble, off(V^T A V) <= tol |A|_F."""
    A = np.asarray(A, LD)
    n = A.shape[0]
    if n == 0:
        return np.zeros(0, LD), np.zeros((0, 0), LD)
    w0, V0 = np.linalg.eigh(A.astype(np.float64))
    V = V0.astype(LD)
    I = np.eye(n, dtype=LD)
    for _ in range(2):   # Newton-Schulz: |V^T V - I| from ~n u to ~(n u)^2, then to the longdouble floor
        V = V @ (3 * I - V.T @ V) / 2
    B = V.T @ A @ V
    B = (B + B.T) / 2
    nrm2 = (A * A).sum()
    tol2 = (n * U_LD) ** 2 if tol is None else tol * tol
    ne = n + (n & 1)
    k = np.arange(ne // 2)
    rounds = []
    for r in range(ne - 1):
        p = np.where(k == 0, ne - 1, (r + k) % (ne - 1))
        q = (r + (ne - 1) - k) % (ne - 1)
        p, q = np.minimum(p, q), np.maximum(p, q)
        ok = q < n
        rounds.append((p[ok], q[ok]))
    offd = ~np.eye(n, dtype=bool)
    for _ in range(max_sweeps):
        off = (B[offd] ** 2).sum()
        if off <= tol2 * nrm2 or off == 0:
            break
        for p, q in rounds:
            if len(p) == 0:
                continue
            apq = B[p, q]
            nz = apq != 0
            if not nz.any():
                continue
            p, q, apq = p[nz], q[nz], apq[nz]
            theta = (B[q, q] - B[p, p]) / (2 * apq)
            t = np.where(theta >= 0, LD(1), LD(-1)) / (np.abs(theta) + np.sqrt(theta * theta + 1))
            c = 1 / np.sqrt(t * t + 1)
            s = t * c
            Bp, Bq = B[:, p].copy(), B[:, q].copy()
            B[:, p], B[:, q] = c * Bp - s * Bq, s * Bp + c * Bq
            Vp, Vq = V[:, p].copy(), V[:, q].copy()
            V[:, p], V[:, q] = c * Vp - s * Vq, s * Vp + c * Vq
            Bp, Bq = B[p, :].copy(), B[q, :].copy()
            B[p, :], B[q, :] = c[:, None] * Bp - s[:, None] * Bq, s[:, None] * Bp + c[:, None] * Bq
    w = np.diag(B).copy()
    order = np.argsort(w.astype(np.float64), kind="stable")
    order = order[np.argsort(w[order], kind="stable")]   # longdouble order, ties kept stable
    return w[order], V[:, order]


def _spectrum_info(w, eps, nrm, band_rel):
    """Distance of the nearest eigenvalue to eps, the gap between the kept (> eps) and the dropped ones, and whether one lies in
    the band band_rel * nrm around eps."""
    wf = w.astype(np.float64)
    kept = wf > eps
    dist = float(np.min(np.abs(wf - eps))) if len(wf) else np.inf
    gap = float(wf[kept].min() - wf[~kept].max()) if kept.any() and (~kept).any() else np.inf
    return {"kept": kept, "dist_eps": dist, "gap": gap, "band": band_rel * nrm, "undecidable": bool(dist <= band_rel * nrm)}


def marginalize(A, b, m, eps=1e-8, band_rel=None, eig=True, eigh=eigh_ld, solve=False):
    """The reference of one problem (see the module docstring); band_rel defaults to jacobi_eps(n, 40) for each decomposition
    (the device's sweep cap).  `eigh` computes the eigenpairs (a 40-digit one checks the reference itself).  solve=True (every
    eigenvalue of Amm kept) takes A_s and b_s from schur_solve and Amm's eigenpairs, which then only size the bars, from float64
    numpy.linalg.eigh: the size sweeps' cheaper route."""
    A = np.asarray(A, np.float64)
    b = np.asarray(b, np.float64)
    pos = A.shape[0]
    n = pos - m
    Al, bl = A.astype(LD), b.astype(LD)
    Amm = (Al[:m, :m] + Al[:m, :m].T) / 2
    Arm, Amr, Arr = Al[m:, :m], Al[:m, m:], Al[m:, m:]
    out = {"m": m, "n": n, "eps": eps, "A_in": A, "b_in": b}
    nmm = float(np.sqrt((Amm * Amm).sum())) if m else 0.0
    if m:
        wm, Vm = (np.linalg.eigh(Amm.astype(np.float64)) if solve else eigh(Amm))
        wm, Vm = wm.astype(LD), Vm.astype(LD)
        im = _spectrum_info(wm, eps, nmm, jacobi_eps(m, 40) if band_rel is None else band_rel)
        inv = np.where(im["kept"], 1 / np.where(im["kept"], wm, LD(1)), LD(0))
        if solve:   # X, T and Tr only size the bars: float64 is enough
            assert im["kept"].all() and not im["undecidable"]
            Vf = Vm.astype(np.float64)
            Ainv = ((Vf * inv.astype(np.float64)) @ Vf.T).astype(LD)
            T, Tr = (A[m:, :m] @ Ainv.astype(np.float64)).astype(LD), (Ainv.astype(np.float64) @ A[:m, m:]).astype(LD)
            As, bs = schur_solve(A, b, m)
        else:
            Ainv = (Vm * inv) @ Vm.T
            T = Arm @ Ainv          # Arm Amm^+
            Tr = Ainv @ Amr         # Amm^+ Amr
            As = Arr - T @ Amr
            bs = bl[m:] - T @ bl[:m]
        Pd = Vm[:, ~im["kept"]]
        wk = wm.astype(np.float64)[im["kept"]]
        out.update(Amm_w=wm, Amm_V=Vm, Amm_inv=Ainv, Amm_info=im,
                   nT=float(np.linalg.norm(T.astype(np.float64), 2)), nTr=float(np.linalg.norm(Tr.astype(np.float64), 2)),
                   nArm_d=float(np.linalg.norm((Arm @ Pd).astype(np.float64), 2)) if Pd.shape[1] else 0.0,
                   nAinv=float(1 / wk.min()) if len(wk) else 0.0,
                   kappa_kept=float(wk.max() / wk.min()) if len(wk) else 1.0)
    else:
        As, bs = Arr.copy(), bl.copy()
        out.update(nT=0.0, nTr=0.0, nArm_d=0.0, nAinv=0.0, kappa_kept=1.0, Amm_inv=np.zeros((0, 0), LD))
    out.update(nAmm=nmm, nArm=float(np.linalg.norm(A[m:, :m], 2)) if m else 0.0, A_s=As, b_s=bs)
    if not eig:
        return out
    Al_s = np.tril(As) + np.tril(As, -1).T
    w, V = eigh(Al_s)
    ns = float(np.sqrt((Al_s * Al_s).sum()))
    info = _spectrum_info(w, eps, ns, jacobi_eps(n, 40) if band_rel is None else band_rel)
    kept = info["kept"]
    Vk = V[:, kept]
    proj = Vk.T @ bs
    out.update(w=w, V=V, As_low=Al_s, info=info, nAs=ns,
               JtJ=(Vk * w[kept]) @ Vk.T, Jtr=Vk @ proj,
               pair_Jtr=(V * np.where(kept, V.T @ bs, LD(0))).T)   # row k: J_k^T r_k (0 for a dropped pair)
    return out


def schur_solve(A, b, m):
    """A_s and b_s (longdouble) of a problem whose Amm_s is positive definite with every eigenvalue far above eps, where
    Amm^+ = Amm^-1: a float64 Cholesky solve of Amm_s [Amr | bmm] and three steps of refinement with the residual in longdouble
    (a cheaper route to the same numbers than `marginalize`, for sweeps over many sizes)."""
    import scipy.linalg
    A = np.asarray(A, np.float64)
    Al, bl = A.astype(LD), np.asarray(b, np.float64).astype(LD)
    Amm = (Al[:m, :m] + Al[:m, :m].T) / 2
    R = np.concatenate([Al[:m, m:], bl[:m, None]], axis=1)
    cf = scipy.linalg.cho_factor(Amm.astype(np.float64))
    X = scipy.linalg.cho_solve(cf, R.astype(np.float64)).astype(LD)
    for _ in range(3):
        X = X + scipy.linalg.cho_solve(cf, (R - Amm @ X).astype(np.float64)).astype(LD)
    return Al[m:, m:] - Al[m:, :m] @ X[:, :-1], bl[m:] - Al[m:, :m] @ X[:, -1]


def _n2(M):
    M = np.asarray(M, np.float64)
    return float(np.linalg.norm(M, 2)) if M.size else 0.0


def schur_bars(ref, sweeps, unit=U, stop=1e-15):
    """Bars (2-norm) on A_s and b_s of a route whose Jacobi of Amm_s runs at most `sweeps` sweeps.  With E the backward error of
    that Jacobi (|E| <= jacobi_eps(m, sweeps) |Amm|_F, plus u |Amm|_F for the rounding of the symmetrisation), the kept
    pseudo-inverse X = sum_{kept} v v^T / l moves to first order by  -X E X + sum_{i kept, j dropped} E_ij / (l_i (l_i - l_j))
    (v_j v_i^T + v_i v_j^T), so Arm dX Amr is at most |E| (|Arm X| |X Amr| + (|Arm P_d| |X Amr| + |Arm X| |P_d Amr|) / gap), gap
    the distance between the kept and the dropped eigenvalues; twice that covers the higher orders while |E| |X| <= 1/2 and
    |E| <= gap / 4 (checked).  The computed V is orthogonal to jacobi_eps, which moves X by V's error on either side:
    eps_J (|Arm| |X Amr| + |Arm X| |Amr|).  The products round entrywise by at most u ((3 m + 4) |Arm| |V| |L^+| |V|^T |Amr|
    + |A_s|) (Higham eq. 3.5 for V L^+ V^T, Arm Inv and T Amr, one subtraction), and the comparison in float64 once more u |A_s|.
    b_s: the same with bmm for Amr."""
    m = ref["m"]
    As, bs = ref["A_s"].astype(np.float64), ref["b_s"].astype(np.float64)
    if m == 0:
        return {"A_s": 0.0, "b_s": 0.0, "valid": True}
    ej = jacobi_eps(m, sweeps, unit, stop)
    E = (ej + unit) * ref["nAmm"]
    info, V, w = ref["Amm_info"], ref["Amm_V"].astype(np.float64), ref["Amm_w"]
    kept = info["kept"]
    X = ref["Amm_inv"]
    Al = ref["A_in"].astype(LD)
    Arm, Amr, bmm = Al[m:, :m], Al[:m, m:], ref["b_in"][:m].astype(LD)
    Pd = ref["Amm_V"][:, ~kept]
    nXr, nXb = ref["nTr"], _n2(X @ bmm)
    nT = ref["nT"]
    nAd, nAmr_d, nbd = ref["nArm_d"], _n2(Pd.T @ Amr), _n2(Pd.T @ bmm)
    gap = info["gap"]
    nX = ref["nAinv"]
    valid = E * nX <= 0.5 and E <= gap / 4 and not info["undecidable"]
    first_A = 2 * E * (nT * nXr + (nAd * nXr + nT * nAmr_d) / gap)
    first_b = 2 * E * (nT * nXb + (nAd * nXb + nT * nbd) / gap)
    nArm, nAmr = ref["nArm"], _n2(Amr)
    orth_A = ej * (nArm * nXr + nT * nAmr)
    orth_b = ej * (nArm * nXb + nT * _n2(bmm))
    Labs = np.where(kept, 1 / np.abs(np.where(kept, w, LD(1))), LD(0)).astype(np.float64)
    VLV = (np.abs(V) * Labs) @ np.abs(V).T
    aArm = np.abs(Arm.astype(np.float64))
    rA = unit * (3 * m + 4) * _n2(aArm @ VLV @ np.abs(Amr.astype(np.float64))) + 2 * unit * _n2(np.abs(As))
    rb = unit * (3 * m + 4) * _n2(aArm @ VLV @ np.abs(bmm.astype(np.float64))) + 2 * unit * _n2(np.abs(bs))
    k = 1.01   # gamma(k) = k u / (1 - k u) over k u
    return {"A_s": k * (first_A + orth_A + rA), "b_s": k * (first_b + orth_b + rb), "valid": bool(valid)}


def check(ref, As, bs, J, r, sweeps, tag, pairs=True, unit=U, stop=1e-15, bounded=True):
    """Holds one problem's outputs (A_s, b_s, J, r; A_s and b_s, or J and r, may be None) to the bars of schur_bars and those
    below; returns the largest error / bar.  Let delta = bar(A_s) + jacobi_eps(n, sweeps) |A_s|_F bound how far the matrix the second Jacobi
    decomposes exactly is from the reference's A_s (lower triangle).  The threshold must be decidable (no eigenvalue within
    delta of eps, gap >= 4 delta) and Amm inside schur_bars' first-order range; with bounded=False (graded rows, where the
    normwise bars are too wide for either) a case outside them has only its finiteness checked.  Then (Davis-Kahan,
    sin theta <= delta / (gap - delta) <= 2 delta / gap):
      J^T J:  2 delta + 4 max|l_dropped| delta / gap + 2 eps_J |A_s P| + u (n + 5) | |J|^T |J| |   (A P moved by the perturbation
              and by the rotation of P; V orthogonal to eps_J; sqrt(S) v rounds twice, numpy's Gram n times);
      J^T r:  2 delta / gap |b_s| + bar(b_s) + 2 eps_J |b_s| + u (n + 4) (| |V_k| |V_k|^T |b_s| | + | |J|^T |r| |) + u |J^T r|;
      per pair k of a simple eigenvalue with gap_k >= 4 delta: 4 delta / gap_k |b_s| + bar(b_s) + 2 eps_J |b_s| + the rounding;
      rows:   the first (dropped) rows of J and r are exactly +-0; the squared norm of kept row i is l_i to
              delta + l_i (2 eps_J + (n + 4) u), and |J_i . J_j| <= sqrt(|J_i|^2 |J_j|^2) (2 eps_J + (n + 4) u)."""
    n = ref["n"]
    bars = schur_bars(ref, sweeps, unit, stop)
    if not bars["valid"]:
        assert not bounded, (tag, "Amm outside the bars' first-order range", ref["Amm_info"])
        for x in [x for x in (As, bs, J, r) if x is not None]:
            assert np.all(np.isfinite(np.asarray(x, np.float64))), tag
        return np.nan
    rb = ref["b_s"].astype(np.float64)
    worst = 0.0
    if As is not None:
        eA = _n2((As.astype(LD) - ref["A_s"]).astype(np.float64))
        eb = float(np.linalg.norm((bs.astype(LD) - ref["b_s"]).astype(np.float64)))
        assert eA <= bars["A_s"], (tag, "A_s", eA, bars["A_s"])
        assert eb <= bars["b_s"], (tag, "b_s", eb, bars["b_s"])
        worst = max(worst, eA / bars["A_s"] if bars["A_s"] else (0.0 if eA == 0 else np.inf),
                    eb / bars["b_s"] if bars["b_s"] else (0.0 if eb == 0 else np.inf))
    if J is None:
        return worst
    ej = jacobi_eps(n, sweeps, unit, stop)
    info, w = ref["info"], ref["w"].astype(np.float64)
    kept = info["kept"]
    delta = bars["A_s"] + ej * ref["nAs"]
    if info["dist_eps"] <= delta or delta > info["gap"] / 4:
        assert not bounded, (tag, "threshold undecidable", info["dist_eps"], delta, info["gap"])
        assert np.all(np.isfinite(J)) and np.all(np.isfinite(r)), tag
        return worst
    d = int((~kept).sum())
    assert np.all(~kept[:d]) and np.all(kept[d:])
    assert np.all(J[:d] == 0.0) and np.all(r[:d] == 0.0), (tag, "dropped rows not zero")
    gap = info["gap"]
    ld = float(np.abs(w[~kept]).max()) if d else 0.0
    JtJ = J.T @ J
    aJ = np.abs(J)
    bJ = (2 * delta + (4 * ld * delta / gap if d and d < n else 0.0) + 2 * ej * _n2(ref["JtJ"])
          + unit * (n + 5) * _n2(aJ.T @ aJ))
    eJ = _n2((JtJ.astype(LD) - ref["JtJ"]).astype(np.float64))
    assert eJ <= bJ, (tag, "J^T J", eJ, bJ)
    nb = float(np.linalg.norm(rb))
    Vk = np.abs(ref["V"].astype(np.float64)[:, kept])
    rnd = unit * (n + 4) * (float(np.linalg.norm(Vk @ (Vk.T @ np.abs(rb)))) + float(np.linalg.norm(aJ.T @ np.abs(r))))
    Jtr = J.T @ r
    br = ((2 * delta / gap * nb if d and d < n else 0.0) + bars["b_s"] + 2 * ej * nb + rnd
          + unit * float(np.linalg.norm(Jtr)))
    er = float(np.linalg.norm((Jtr.astype(LD) - ref["Jtr"]).astype(np.float64)))
    assert er <= br, (tag, "J^T r", er, br)
    worst = max(worst, eJ / bJ if bJ else float(eJ > 0) * np.inf, er / br if br else float(er > 0) * np.inf)
    sq = (J * J).sum(axis=1)
    tol = 2 * ej + (n + 4) * unit
    bl = delta + w * tol
    assert np.all(np.abs(sq[d:] - w[d:]) <= bl[d:]), (tag, "row norms", float(np.max(np.abs(sq[d:] - w[d:]) / bl[d:])))
    G = J @ J.T
    off = np.abs(G - np.diag(np.diag(G)))
    assert np.all(off <= np.sqrt(np.outer(sq, sq)) * tol), (tag, "rows not orthogonal")
    if pairs:
        gaps = np.full(n, np.inf)
        if n > 1:
            dw = np.abs(w[:, None] - w[None, :]) + np.diag(np.full(n, np.inf))
            gaps = dw.min(axis=1)
        for k in np.flatnonzero(kept & (gaps >= 4 * delta)):
            pk = J[k] * r[k]
            bk = 4 * delta / gaps[k] * nb + bars["b_s"] + 2 * ej * nb + rnd
            ek = float(np.linalg.norm((pk.astype(LD) - ref["pair_Jtr"][k]).astype(np.float64)))
            assert ek <= bk, (tag, "pair", k, ek, bk)
    return worst


# ---- problems with a known structure ----------------------------------------------------------------------------------------
def orth(rng, n):
    return np.linalg.qr(rng.standard_normal((n, n)))[0] if n else np.zeros((0, 0))


def sym_with(rng, spec):
    """Q diag(spec) Q^T, Q random orthogonal, symmetrised (float64)."""
    Q = orth(rng, len(spec))
    S = (Q * np.asarray(spec, np.float64)) @ Q.T
    return (S + S.T) / 2


def problem(rng, mm_spec, s_spec, coupling=1.0, skew=0.0, eps=1e-8):
    """A = [[Amm, Amr], [Arm, Arr]] with spec(Amm) = mm_spec and A_s close to a matrix of spectrum s_spec (Arr = that matrix +
    Arm Amm^+ Amr, rounded); skew adds a skew-symmetric part of that relative
    size (the reference symmetrises Amm and reads the lower triangle of A_s).  b random."""
    m, n = len(mm_spec), len(s_spec)
    Amm = sym_with(rng, mm_spec) if m else np.zeros((0, 0))
    S = sym_with(rng, s_spec)
    w, V = np.linalg.eigh(Amm) if m else (np.zeros(0), np.zeros((0, 0)))
    ws, Vs = np.linalg.eigh(S)
    # Arm = |S|^1/2 G |Amm|^1/2 (G random, |G| ~ coupling): Arm Amm^+ Amr stays of the size of S, as in a positive semidefinite A
    Arm = (Vs * np.sqrt(np.abs(ws))) @ Vs.T @ (coupling * rng.standard_normal((n, m)) / np.sqrt(max(m, n, 1))) @ (V * np.sqrt(np.abs(w))) @ V.T
    inv = np.where(w > eps, 1 / np.where(w != 0, w, 1), 0)
    Arr = S + (Arm @ (V * inv) @ V.T) @ Arm.T if m else S
    A = np.block([[Amm, Arm.T], [Arm, (Arr + Arr.T) / 2]])
    if skew:
        K = rng.standard_normal(A.shape)
        A = A + skew * np.abs(A).max() * (K - K.T) / 2
    return A, rng.standard_normal(m + n)


def null_problem(rng, m, n, rank_m, rank, scale_pow=0):
    """A = 2^scale_pow M^T M from an integer M (rank rows, every entry in [-3, 3]) whose first m columns have rank rank_m < m:
    an exact (in float64) positive semidefinite A whose Amm has an exact null space of dimension m - rank_m that Arm does not see
    (Arm v = 0), and whose A_s has one of dimension n - (rank - rank_m) when rank - rank_m < n."""
    X = rng.integers(-1, 2, (rank, rank_m))
    Y = rng.integers(-1, 2, (rank_m, m))
    M = np.concatenate([X @ Y, rng.integers(-3, 4, (rank, n))], axis=1).astype(np.float64)
    A = np.ldexp(M.T @ M, scale_pow)
    return A, np.ldexp(rng.integers(-8, 9, m + n).astype(np.float64), scale_pow)


def graded_problem(rng, rows, kappa_c=1e2):
    """D C D with C a random SPD matrix of condition kappa_c and D the row scales (the realistic inertial window: sqrt_info near
    3e5 on bias rows, FOCAL / 1.5 on visual rows, 1 on the rest): entries over ~11 orders of magnitude."""
    pos = len(rows)
    C = sym_with(rng, np.logspace(0, -np.log10(kappa_c), pos))
    d = np.asarray(rows, np.float64)
    A = d[:, None] * C * d[None, :]
    return (A + A.T) / 2, d * rng.standard_normal(pos)


FOCAL = 460.0
UNBOUNDED = ("graded", "kappa1e+12")   # cases whose eigen outputs the normwise bars cannot decide


def edge_cases(seed=0):
    """(name, A, b, m, eps) of the spectra where an eigen route goes wrong: conditioning, graded rows, exact and near null spaces,
    eigenvalues either side of eps, negative, repeated and clustered eigenvalues, eps = 0 and a large eps, an asymmetric A."""
    rng = np.random.default_rng(seed)
    cs = []
    for kappa in (1e2, 1e6, 1e10, 1e12):   # kappa of the kept Amm, |Amm| = 1e5 (lambda_min >= 1e-7 > eps)
        m = 6 if kappa > 1e10 else 15
        cs.append((f"kappa{kappa:.0e}", *problem(rng, 1e5 * np.logspace(0, -np.log10(kappa), m), np.logspace(2, 0, 20)), m, 1e-8))
    bias, vis = 3e5, FOCAL / 1.5
    rows = [bias] * 3 + [1.0] * 6 + [bias] * 6 + [vis] * 20 + [1.0] * 6 + [bias] * 6
    cs.append(("graded", *graded_problem(rng, rows), 15, 1e-8))
    cs.append(("null", *null_problem(rng, 15, 30, 11, 36), 15, 1e-3))
    cs.append(("null_scaled", *null_problem(rng, 20, 21, 13, 30, scale_pow=-40), 20, np.ldexp(1e-3, -40)))
    gauge = np.concatenate([1e-12 * np.array([1.0, 2.0, 3.0, 4.0]), np.logspace(3, 0, 11)])   # 4-dim near-null gauge space
    cs.append(("gauge", *problem(rng, gauge, np.logspace(2, 0, 18)), 15, 1e-8))
    # eigenvalues at 1e-3 eps and 1e3 eps: in Amm (A_s far from eps), and in A_s (Amm well conditioned)
    cs.append(("eps_sides_mm", *problem(rng, [1e-11, 1e-5, 1e-11, 3.0, 1e-5, 7.0], [1.0, 2.0, 5.0, 3.0]), 6, 1e-8))
    cs.append(("eps_sides_s", *problem(rng, [1.0, 3.0, 7.0, 2.0], [1e-11, 1e-5, 1.0, 2.0, 1e-11, 1e-5, 5.0]), 4, 1e-8))
    cs.append(("negative", *problem(rng, [-5.0, -1e-3, 2.0, 3.0, 1e2, -7.0, 4.0], [-3.0, -1.0, 1e-3, 2.0, 9.0, -2.0]), 7, 1e-8))
    rep = np.repeat([1.0, 2.0, 5.0], 5)
    clu = 3.0 + 1e-12 * np.arange(8)
    cs.append(("repeated", *problem(rng, rep, np.concatenate([np.repeat([4.0, 0.5], 6), clu])), 15, 1e-8))
    cs.append(("cluster", *problem(rng, np.concatenate([clu, [1.0, 9.0]]), np.concatenate([clu, 1 + 1e-9 * np.arange(5)])), 10, 1e-8))
    cs.append(("zero", np.zeros((24, 24)), rng.standard_normal(24), 15, 1e-8))
    cs.append(("eps0", *problem(rng, np.logspace(0, -3, 9), np.logspace(1, -2, 12), eps=0.0), 9, 0.0))
    cs.append(("eps_large", *problem(rng, np.logspace(2, -2, 12), np.logspace(2, -2, 16), eps=0.37), 12, 0.37))
    cs.append(("asymmetric", *problem(rng, np.logspace(1, -1, 15), np.logspace(1, 0, 25), skew=1e-6), 15, 1e-8))
    cs.append(("m_gt_n", *problem(rng, np.logspace(2, 0, 40), np.logspace(1, 0, 3)), 40, 1e-8))
    cs.append(("n1", *problem(rng, np.logspace(1, 0, 15), [2.5]), 15, 1e-8))
    return cs
