"""The trust-region policy of viml_solve_vi, restated in tests/solve_policy.py, on hand-computed step sequences; and the ctypes
mirrors of viml_solve_options / viml_solve_out against sizeof / offsetof of the C structs, from a small program that includes
include/viml.h and is compiled with g++.  No GPU."""
import ctypes as C
import json
import math
import os
import subprocess

import pytest

import solve_policy as sp
from conftest import ROOT

X_NORM = 10.0
BIG_STEP = 1.0   # far above parameter_tolerance * (|x| + parameter_tolerance)


def _good(st, opt, rho, f=100.0, model=10.0):
    """A valid step whose quality is rho."""
    return sp.advance(st, opt, f, f - rho * model, model, 1, BIG_STEP, X_NORM)


def _bad(st, opt):
    return sp.advance(st, opt, 100.0, 100.0, 0.0, 0, 0.0, X_NORM)


def test_rho_one_triples_the_radius_and_half_keeps_it():
    opt = sp.Options()
    st = sp.start(100.0, opt)
    acc, row = _good(st, opt, 1.0)
    assert acc and st.radius == 3e4 and st.accepted == 1 and st.f == 90.0
    assert row == [100.0, 90.0, 10.0, 1e-4]
    acc, _ = _good(st, opt, 0.5)    # t = 0: radius / max(1/3, 1) = radius
    assert acc and st.radius == 3e4 and st.decrease_factor == 2.0 and st.status is None


def test_accept_clamps_at_max_radius():
    opt = sp.Options(max_radius=2e4)
    st = sp.start(100.0, opt)
    _good(st, opt, 1.0)
    assert st.radius == 2e4
    _good(st, opt, 1.0)
    assert st.radius == 2e4


def test_rejections_double_the_decrease_factor_and_acceptance_resets_it():
    opt = sp.Options()
    st = sp.start(100.0, opt)
    for k, (radius, factor) in enumerate([(5e3, 4.0), (1.25e3, 8.0), (156.25, 16.0)]):
        acc, _ = _good(st, opt, 1e-4)   # rho below min_relative_decrease: reject
        assert not acc and st.radius == radius and st.decrease_factor == factor and st.consecutive_invalid == 0
    acc, _ = _good(st, opt, 1.0)
    assert acc and st.decrease_factor == 2.0 and st.radius == 468.75
    assert st.accepted == 1 and st.iterations == 4


def test_invalid_steps_end_in_failure():
    opt = sp.Options(max_consecutive_invalid=2)
    st = sp.start(100.0, opt)
    _bad(st, opt)
    assert st.status is None and st.consecutive_invalid == 1 and st.radius == 5e3 and st.decrease_factor == 4.0
    _good(st, opt, 1.0)                 # a valid step resets the count
    assert st.consecutive_invalid == 0
    for _ in range(2):
        _bad(st, opt)
        assert st.status is None
    _bad(st, opt)                       # the third in a row: more than max_consecutive_invalid
    assert st.status == sp.FAILURE and st.iterations == 5
    # every kind of invalid step counts: unsolved, f(x+) not finite, model decrease not positive
    for args in ((100.0, 90.0, 10.0, 0), (100.0, math.inf, 10.0, 1), (100.0, math.nan, 10.0, 1), (100.0, 90.0, 0.0, 1),
                 (100.0, 90.0, -1.0, 1), (100.0, 90.0, math.nan, 1)):
        st = sp.start(100.0, sp.Options(max_consecutive_invalid=0))
        acc, _ = sp.advance(st, sp.Options(max_consecutive_invalid=0), *args, BIG_STEP, X_NORM)
        assert not acc and st.status == sp.FAILURE and st.iterations == 1, args


def test_min_radius():
    opt = sp.Options(initial_radius=1.0, min_radius=0.3)
    st = sp.start(100.0, opt)
    _good(st, opt, 1e-4)                # 1 / 2 = 0.5
    assert st.status is None
    _good(st, opt, 1e-4)                # 0.5 / 4 = 0.125 < 0.3
    assert st.status == sp.MIN_RADIUS and st.radius == 0.125 and st.iterations == 2


def test_function_tolerance_stops_at_x():
    opt = sp.Options(function_tolerance=1e-3)
    st = sp.start(100.0, opt)
    acc, row = sp.advance(st, opt, 100.0, 99.95, 0.06, 1, BIG_STEP, X_NORM)
    assert not acc and st.status == sp.FUNCTION_TOL and st.accepted == 0 and st.f == 100.0 and st.radius == 1e4
    assert row == [100.0, 99.95, 0.06, 1e-4]


def test_parameter_tolerance_stops_at_x():
    opt = sp.Options(parameter_tolerance=1e-3)
    st = sp.start(100.0, opt)
    acc, _ = sp.advance(st, opt, 100.0, 50.0, 60.0, 1, 1e-3 * (X_NORM + 1e-3), X_NORM)   # |dx| == the bound: stop
    assert not acc and st.status == sp.PARAMETER_TOL and st.f == 100.0
    st = sp.start(100.0, opt)
    acc, _ = sp.advance(st, opt, 100.0, 50.0, 60.0, 1, 2e-2, X_NORM)
    assert acc and st.status is None


def test_iteration_cap():
    opt = sp.Options(max_iterations=3)
    st = sp.start(100.0, opt)
    for k in range(3):
        assert st.status is None
        _good(st, opt, 1.0, f=100.0 - 10 * k)
    assert st.status == sp.NO_CONVERGENCE and st.iterations == 3 and st.accepted == 3
    # the cap is checked after the radius: both at once give MIN_RADIUS
    opt = sp.Options(max_iterations=1, initial_radius=1.0, min_radius=0.75)
    st = sp.start(100.0, opt)
    _good(st, opt, 1e-4)
    assert st.status == sp.MIN_RADIUS


@pytest.mark.parametrize("f0", [math.nan, math.inf, -math.inf])
def test_non_finite_initial_cost(f0):
    st = sp.start(f0, sp.Options())
    assert st.status == sp.FAILURE and st.iterations == 0 and st.accepted == 0


def test_radius_update_is_ieee_exact():
    """rho = 0.9: t = 0.8, 1 - t^3 = 0.488 (rounded), radius / 0.488 — the operations in viml.h's order, no fused multiply-add."""
    opt = sp.Options()
    st = sp.start(100.0, opt)
    _good(st, opt, 0.9)
    rho = (100.0 - (100.0 - 0.9 * 10.0)) / 10.0
    t = 2.0 * rho - 1.0
    assert st.radius == 1e4 / (1.0 - t * t * t)


PROGRAM = r"""
#include <cstddef>
#include <cstdio>
#include "viml.h"
#define F(S, m) std::printf("\"%s.%s\": %zu,\n", #S, #m, offsetof(S, m))
int main() {
  std::printf("{\n");
  F(viml_solve_options, max_iterations); F(viml_solve_options, max_consecutive_invalid); F(viml_solve_options, initial_radius);
  F(viml_solve_options, max_radius); F(viml_solve_options, min_radius); F(viml_solve_options, min_relative_decrease);
  F(viml_solve_options, function_tolerance); F(viml_solve_options, parameter_tolerance);
  F(viml_solve_out, poses); F(viml_solve_out, ex_pose); F(viml_solve_out, inv_depth); F(viml_solve_out, extra);
  F(viml_solve_out, status); F(viml_solve_out, iterations); F(viml_solve_out, accepted); F(viml_solve_out, cost);
  F(viml_solve_out, radius); F(viml_solve_out, trace);
  std::printf("\"codes\": [%d, %d, %d, %d, %d],\n", VIML_SOLVE_NO_CONVERGENCE, VIML_SOLVE_FUNCTION_TOL, VIML_SOLVE_PARAMETER_TOL,
              VIML_SOLVE_MIN_RADIUS, VIML_SOLVE_FAILURE);
  std::printf("\"sizeof.viml_solve_options\": %zu,\n\"sizeof.viml_solve_out\": %zu\n}\n", sizeof(viml_solve_options),
              sizeof(viml_solve_out));
}
"""


@pytest.fixture(scope="module")
def c_layout(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("solve_abi")
    cpp = tmp / "layout.cpp"
    cpp.write_text(PROGRAM)
    exe = tmp / "layout"
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(cpp)])
    return json.loads(subprocess.check_output([str(exe)]))


@pytest.mark.parametrize("cname, attr", [("viml_solve_options", "SolveOptions"), ("viml_solve_out", "SolveOut")])
def test_ctypes_layout_matches_c(pkg, c_layout, cname, attr):
    cls = getattr(pkg._abi, attr)
    assert C.sizeof(cls) == c_layout["sizeof." + cname]
    fields = [f[0] for f in cls._fields_]
    assert sorted(fields) == sorted(k.split(".", 1)[1] for k in c_layout if k.startswith(cname + "."))
    for name in fields:
        assert getattr(cls, name).offset == c_layout[f"{cname}.{name}"], name


def test_status_codes_match_c(pkg, c_layout):
    abi = pkg._abi
    codes = [abi.SOLVE_NO_CONVERGENCE, abi.SOLVE_FUNCTION_TOL, abi.SOLVE_PARAMETER_TOL, abi.SOLVE_MIN_RADIUS, abi.SOLVE_FAILURE]
    assert codes == c_layout["codes"]
    assert codes == [sp.NO_CONVERGENCE, sp.FUNCTION_TOL, sp.PARAMETER_TOL, sp.MIN_RADIUS, sp.FAILURE]
    assert tuple(f[0] for f in abi.SolveOut._fields_) == abi.SOLVE_OUT_FIELDS
