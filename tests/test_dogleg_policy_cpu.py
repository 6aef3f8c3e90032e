"""The dogleg restatement of tests/dogleg_policy.py on small dense problems (no GPU): the three cases of the step against the vectors
they stand for, and the radius / mu / reuse transitions of the policy."""
import math

import numpy as np
import pytest

import dogleg_policy as dp


def _problem(seed, n=7, mu=1e-8):
    """A random SPD H and g with Ceres' Jacobi scaling: the vectors and the scalars the device stores."""
    rng = np.random.default_rng(seed)
    J = rng.standard_normal((n + 4, n)) * rng.uniform(0.1, 10.0, n)
    H, g = J.T @ J, J.T @ rng.standard_normal(n + 4)
    s = 1.0 / (1.0 + np.sqrt(np.diag(H)))
    d = np.sqrt(np.minimum(np.maximum(s * s * np.diag(H), 1e-6), 1e32))
    gam = s * g / d
    w = s * gam / d
    dgn = np.linalg.solve(H + np.diag(mu * d * d / (s * s)), -g)
    nv = d * dgn / s
    sc = (float(gam @ gam), float(nv @ nv), float(gam @ nv), float(w @ H @ w), float(w @ H @ dgn), float(dgn @ H @ dgn))
    return H, g, s, d, w, dgn, sc


def _dnorm(d, s, x):
    return float(np.linalg.norm(d * x / s))


@pytest.mark.parametrize("seed", range(8))
def test_three_cases(seed):
    H, g, s, d, w, dgn, sc = _problem(seed)
    gg, nn = sc[0], sc[1]
    alpha = gg / sc[3]
    cauchy, gn_norm = alpha * math.sqrt(gg), math.sqrt(nn)
    assert cauchy < gn_norm   # the Cauchy point lies inside the Gauss-Newton step's sphere
    for radius, want in ((1.01 * gn_norm, 1), (0.5 * cauchy, 2), (0.5 * (cauchy + gn_norm), 3)):
        case, a, b, norm, m = dp.step(*sc, radius)
        assert case == want
        x = a * w + b * dgn
        assert abs(m - (-(g @ x + 0.5 * x @ H @ x))) <= 1e-12 * max(1.0, abs(m))
        assert m > 0.0
        assert abs(norm - _dnorm(d, s, x)) <= 1e-12 * norm
        if case == 1:
            assert np.array_equal(x, dgn) and norm == math.sqrt(nn)
        else:
            assert abs(_dnorm(d, s, x) - radius) <= 1e-12 * radius
        if case == 3:   # on the segment from the Cauchy point -alpha w to dgn
            beta = b
            assert 0.0 < beta < 1.0
            assert np.allclose(x, (1.0 - beta) * (-alpha * w) + beta * dgn, rtol=0, atol=1e-13 * np.abs(x).max())


def test_zero_gradient():
    case, a, b, norm, m = dp.step(0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0)
    assert (case, a, b, norm, m) == (1, 0.0, 1.0, 0.0, -0.0)


def _opt(**kw):
    return dp.Options(**{"max_iterations": 10, **kw})


# (state before, step (f, f+, m, solved, |dx|, |x|, |step|_D), expected radius, mu, reuse, accepted)
TRANSITIONS = [
    # invalid steps: the radius stays, mu rises tenfold, a new step follows
    (dict(radius=4.0, mu=1e-8), (10.0, 9.0, 1.0, 0, 1.0, 1.0, 2.0), 4.0, 1e-7, False, False),
    (dict(radius=4.0, mu=1e-3, reuse=True), (10.0, math.nan, 1.0, 1, 1.0, 1.0, 2.0), 4.0, 1e-2, False, False),
    (dict(radius=4.0, mu=1e-8), (10.0, 9.0, 0.0, 1, 1.0, 1.0, 2.0), 4.0, 1e-7, False, False),
    # rejected: half the radius, reuse the stored step
    (dict(radius=4.0, mu=1e-6), (10.0, 10.5, 1.0, 1, 1.0, 1.0, 2.0), 2.0, 1e-6, True, False),
    # accepted, rho = 0.1 < 1/4: half the radius
    (dict(radius=4.0, mu=1e-6), (10.0, 9.9, 1.0, 1, 1.0, 1.0, 2.0), 2.0, 2e-7, False, True),
    # accepted, 1/4 <= rho = 0.5 <= 3/4: radius unchanged
    (dict(radius=4.0, mu=1e-6), (10.0, 9.5, 1.0, 1, 1.0, 1.0, 2.0), 4.0, 2e-7, False, True),
    # accepted, rho = 0.9 > 3/4: max(radius, 3 |step|_D), capped at max_radius; mu does not fall below 1e-8
    (dict(radius=4.0, mu=1e-8), (10.0, 9.1, 1.0, 1, 1.0, 1.0, 2.0), 6.0, 1e-8, False, True),
    (dict(radius=4.0, mu=1e-8), (10.0, 9.1, 1.0, 1, 1.0, 1.0, 1.0), 4.0, 1e-8, False, True),
    (dict(radius=4.0, mu=1e-8, max_radius=5.0), (10.0, 9.1, 1.0, 1, 1.0, 1.0, 2.0), 5.0, 1e-8, False, True),
]


@pytest.mark.parametrize("before,res,radius,mu,reuse,accepted", TRANSITIONS)
def test_transitions(before, res, radius, mu, reuse, accepted):
    before = dict(before)
    opt = _opt(**({"max_radius": before.pop("max_radius")} if "max_radius" in before else {}))
    st = dp.State(f0=10.0, f=10.0, **before)
    r0 = st.radius
    acc, row = dp.advance(st, opt, *res)
    assert row[3] == r0
    assert (st.radius, st.mu, st.reuse, acc) == (radius, pytest.approx(mu, rel=1e-15), reuse, accepted)
    assert st.iterations == 1 and st.accepted == int(accepted)


def test_stops():
    opt = _opt(max_consecutive_invalid=1, min_radius=1.0)
    st = dp.start(10.0, opt)
    for _ in range(2):
        dp.advance(st, opt, 10.0, math.nan, 1.0, 1, 1.0, 1.0, 1.0)
    assert st.status == dp.FAILURE and st.radius == opt.initial_radius and st.mu == pytest.approx(1e-6)
    st = dp.State(radius=1.5, f0=10.0, f=10.0)
    dp.advance(st, opt, 10.0, 11.0, 1.0, 1, 1.0, 1.0, 1.0)   # rejected: 0.75 < min_radius
    assert st.status == dp.MIN_RADIUS and st.reuse
    st = dp.State(radius=4.0, f0=10.0, f=10.0)
    dp.advance(st, opt, 10.0, 9.0, 1.0, 1, 1e-20, 1.0, 1.0)
    assert st.status == dp.PARAMETER_TOL and st.accepted == 0
    assert dp.start(math.nan, opt).status == dp.FAILURE
