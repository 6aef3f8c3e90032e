"""Scalar restatement of the trust-region policy of viml_solve_vi (include/viml.h): Ceres' TrustRegionMinimizer with its
LevenbergMarquardtStrategy as viml.h states it (not pinned against Ceres' source).  Plain IEEE doubles, every operation in the
order viml.h writes it, so that the device's policy_kernel (no fused multiply-adds) agrees bit for bit.

A driver calls start() with f(x0), then, while state.status is None, takes the step at x with lambda(state) and hands its result to
advance(), which says whether x+ was accepted."""
import math
from dataclasses import dataclass

NO_CONVERGENCE, FUNCTION_TOL, PARAMETER_TOL, MIN_RADIUS, FAILURE = 0, 1, 2, 3, 4


@dataclass
class Options:
    max_iterations: int = 50
    max_consecutive_invalid: int = 5
    initial_radius: float = 1e4
    max_radius: float = 1e16
    min_radius: float = 1e-32
    min_relative_decrease: float = 1e-3
    function_tolerance: float = 1e-6
    parameter_tolerance: float = 1e-8


@dataclass
class State:
    radius: float
    decrease_factor: float = 2.0
    consecutive_invalid: int = 0
    iterations: int = 0
    accepted: int = 0
    status: object = None      # None while running, else one of the constants above
    f0: float = math.nan
    f: float = math.nan        # f at the current state


def start(f0, opt):
    """The state before the first step; a non-finite f(x0) ends the window at once."""
    st = State(radius=float(opt.initial_radius), f0=float(f0), f=float(f0))
    if not math.isfinite(st.f0):
        st.status = FAILURE
    return st


def lam(st):
    return 1.0 / st.radius


def advance(st, opt, f, f_plus, model, solved, step_norm, x_norm):
    """One step's result (f(x), f(x+), model decrease, solved, |dx|, |x|) applied to a running window's state.  Returns
    (accepted, trace row [f(x), f(x+), model decrease, lambda])."""
    assert st.status is None
    f, f_plus, model = float(f), float(f_plus), float(model)
    row = [f, f_plus, model, lam(st)]
    st.f = f
    accepted = False
    if not solved or not math.isfinite(f_plus) or not model > 0.0:
        st.consecutive_invalid += 1
        st.radius = st.radius / st.decrease_factor
        st.decrease_factor = st.decrease_factor * 2.0
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
                t = 2.0 * rho - 1.0
                st.radius = min(opt.max_radius, st.radius / max(1.0 / 3.0, 1.0 - t * t * t))
                st.decrease_factor = 2.0
            else:
                st.radius = st.radius / st.decrease_factor
                st.decrease_factor = st.decrease_factor * 2.0
    st.iterations += 1
    if st.status is None:
        if st.radius < opt.min_radius:
            st.status = MIN_RADIUS
        elif st.iterations == opt.max_iterations:
            st.status = NO_CONVERGENCE
    return accepted, row
