"""Scalar restatement of viml_solve_vi's dogleg strategy (VIML_SOLVE_DOGLEG, include/viml.h): Ceres' traditional dogleg step from the
stored scalars and the trust-region policy with the dogleg's radius / mu / reuse updates, as viml.h states them (not pinned against
Ceres' source).  Plain IEEE doubles in the order the device writes them (no fused multiply-adds), so that dogleg_step_kernel and
policy_kernel agree bit for bit given the same scalars.

A driver calls start() with f(x0); while state.status is None it forms a new Gauss-Newton step when state.reuse is False (with
state.mu), takes step() at state.radius and hands the result to advance()."""
import math
from dataclasses import dataclass

from solve_policy import FAILURE, FUNCTION_TOL, MIN_RADIUS, NO_CONVERGENCE, PARAMETER_TOL, Options  # noqa: F401

MIN_MU, MAX_MU = 1e-8, 1.0


@dataclass
class State:
    radius: float
    mu: float = MIN_MU
    reuse: bool = False
    consecutive_invalid: int = 0
    iterations: int = 0
    accepted: int = 0
    status: object = None
    f0: float = math.nan
    f: float = math.nan


def start(f0, opt):
    st = State(radius=float(opt.initial_radius), f0=float(f0), f=float(f0))
    if not math.isfinite(st.f0):
        st.status = FAILURE
    return st


def step(gg, nn, gn, whw, whd, dhd, radius):
    """The dogleg step at `radius` from |gamma|^2, n.n, gamma.n, w^T H w, w^T H dgn, dgn^T H dgn: (case, a, b, D-space norm,
    model decrease), the step being a w + b dgn."""
    gnorm, nnorm = math.sqrt(gg), math.sqrt(nn)
    alpha = 0.0 if (gg == 0.0 and whw == 0.0) else gg / whw
    if nnorm <= radius:
        case, a, b, norm = 1, 0.0, 1.0, nnorm
    elif alpha * gnorm >= radius:
        case, a, b, norm = 2, -(radius / gnorm), 0.0, radius
    else:
        ag = alpha * gnorm
        a2 = ag * ag
        ba = -(alpha * gn)
        c = ba - a2
        bma = (a2 - 2.0 * ba) + nn
        r2a = radius * radius - a2
        d = math.sqrt(c * c + bma * r2a)
        beta = (d - c) / bma if c <= 0.0 else r2a / (d + c)
        case, a, b = 3, -(alpha * (1.0 - beta)), beta
        norm = math.sqrt((a * a * gg + 2.0 * (a * b) * gn) + b * b * nn)
    lin = a * gg + b * gn
    quad = (a * a * whw + 2.0 * (a * b) * whd) + b * b * dhd
    return case, a, b, norm, -(lin + 0.5 * quad)


def advance(st, opt, f, f_plus, model, solved, step_norm, x_norm, dnorm):
    """One step's result (f(x), f(x+), model decrease, solved, |dx|, |x|, the step's D-space norm) applied to a running window.
    Returns (accepted, trace row [f(x), f(x+), model decrease, radius])."""
    assert st.status is None
    f, f_plus, model = float(f), float(f_plus), float(model)
    row = [f, f_plus, model, st.radius]
    st.f = f
    accepted = False
    if not solved or not math.isfinite(f_plus) or not model > 0.0:
        st.consecutive_invalid += 1
        st.mu = st.mu * 10.0
        st.reuse = False
        if st.consecutive_invalid > opt.max_consecutive_invalid:
            st.status = FAILURE
    else:
        st.consecutive_invalid = 0
        if step_norm <= opt.parameter_tolerance * (x_norm + opt.parameter_tolerance):
            st.status = PARAMETER_TOL
        elif abs(f - f_plus) <= opt.function_tolerance * f:
            st.status = FUNCTION_TOL
        else:
            rho = (f - f_plus) / model
            if rho > opt.min_relative_decrease:
                accepted = True
                st.accepted += 1
                st.f = f_plus
                if rho < 0.25:
                    st.radius = st.radius * 0.5
                elif rho > 0.75:
                    st.radius = min(opt.max_radius, max(st.radius, 3.0 * dnorm))
                st.mu = max(MIN_MU, 2.0 * st.mu / 10.0)
                st.reuse = False
            else:
                st.radius = st.radius * 0.5
                st.reuse = True
    st.iterations += 1
    if st.status is None:
        if st.radius < opt.min_radius:
            st.status = MIN_RADIUS
        elif st.iterations == opt.max_iterations:
            st.status = NO_CONVERGENCE
    return accepted, row
