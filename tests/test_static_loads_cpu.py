"""CPU tests of the static shape problem under distributed loads, a rotated clamp and a given Gamma: the numpy restatement
(static_loads_ref.py) of its residual Jacobian, Newton solve and implicit adjoint, pinned against central differences with
sagging loads (g = 1, tip loads up to 0.6); and the argument errors of the three entry points that take a sri_static_problem."""
import ctypes

import numpy as np
import pytest

from static_loads_ref import loaded_problem, unit_quaternion

H0 = np.array([1.0, 1.0, 0.77])


def _kw(t):
    return {k: t[k] for k in ("K0", "q0", "Gamma", "fbar", "lbar")}


@pytest.mark.parametrize("N", [5, 9, 16])
def test_residual_jacobian_against_central_differences(make_oracle, N):
    from static_loads_ref import residual, residual_and_jacobian
    o = make_oracle(N)
    rng = np.random.default_rng(500 + N)
    B, ne, h = 3, 3, 1e-6
    t = loaded_problem(rng, B, N)
    qe = rng.uniform(-0.5, 0.5, size=(B, 3 * ne))
    _, J = residual_and_jacobian(o, qe, t["F_tip"], t["M_tip"], H0, ne, **_kw(t))
    for d in range(3 * ne):
        e = np.zeros_like(qe); e[:, d] = h
        fd = (residual(o, qe + e, t["F_tip"], t["M_tip"], H0, ne, **_kw(t)) -
              residual(o, qe - e, t["F_tip"], t["M_tip"], H0, ne, **_kw(t))) / (2 * h)
        assert np.abs(fd - J[:, :, d]).max() <= 1e-7 * np.abs(J).max(), (N, d)


def test_reference_without_loads_is_the_tip_load_reference(make_oracle):
    """With q0, Gamma, fbar, lbar absent the loaded restatement is static_adjoint_ref's (built on oracle/tangent's J_d)."""
    import static_adjoint_ref as tip
    from static_loads_ref import adjoint, newton
    N, B, ne = 9, 2, 3
    o = make_oracle(N)
    rng = np.random.default_rng(8)
    F, Mt = rng.uniform(-0.6, 0.6, size=(B, 3)), rng.uniform(-0.6, 0.6, size=(B, 3))
    qe, gmax = newton(o, F, Mt, H0, ne)
    qt, _ = tip.newton_static_shape(o, F, Mt, H0, ne)
    assert gmax < 1e-13 and np.abs(qe - qt).max() <= 1e-13
    gqe = rng.normal(size=(B, 3 * ne))
    a, b = adjoint(o, qe, F, Mt, H0, ne, gqe), tip.static_shape_vjp(o, qe, F, Mt, H0, ne, gqe)
    for k in ("F_tip", "M_tip", "K0", "H", "lambda"):
        assert np.abs(a[k] - b[k]).max() <= 1e-12 * max(1.0, np.abs(b[k]).max()), k


@pytest.mark.parametrize("N", [5, 9, 16])
def test_equilibrium_gradient_against_central_differences_of_the_newton_solve(make_oracle, N):
    from static_loads_ref import INPUTS, adjoint, newton
    o = make_oracle(N)
    rng = np.random.default_rng(600 + N)
    B, ne, h = 2, 3, 1e-5
    theta = loaded_problem(rng, B, N)
    gqe = rng.normal(size=(B, 3 * ne))

    def solve(t):
        qe, gmax = newton(o, t["F_tip"], t["M_tip"], H0, ne, **_kw(t))
        assert gmax < 1e-13, gmax
        return qe

    qe = solve(theta)
    assert np.abs(qe).max() > 0.3   # the sag is not small
    g = adjoint(o, qe, theta["F_tip"], theta["M_tip"], H0, ne, gqe, **_kw(theta))
    dirs = {k: rng.normal(size=theta[k].shape) for k in INPUTS}
    for keys in [(k,) for k in INPUTS] + [INPUTS]:   # each alone, so that an error in one cannot hide behind another
        tp = dict(theta, **{k: theta[k] + h * dirs[k] for k in keys})
        tm = dict(theta, **{k: theta[k] - h * dirs[k] for k in keys})
        fd = float(np.sum(gqe * (solve(tp) - solve(tm)))) / (2 * h)
        terms = [g[k] * dirs[k] for k in keys]
        ad = sum(float(t.sum()) for t in terms)
        scale = max(abs(ad), sum(float(np.abs(t).sum()) for t in terms))
        assert abs(fd - ad) <= 1e-7 * scale, (N, keys, fd, ad)


def test_analytic_jacobian_still_preconditions_under_loads(make_oracle):
    """J_a of sri_shape_jacobian at an equilibrium under self-weight and a rotated clamp is J_d to the discretisation error
    (DESIGN section 5e's table: 8.5e-6 at N = 9, 1.8e-12 at N = 16)."""
    from static_loads_ref import contraction, newton
    rng = np.random.default_rng(40)
    B, ne = 4, 4
    worst = {}
    for N in (9, 16):
        o = make_oracle(N)
        F, Mt = rng.uniform(-0.6, 0.6, size=(B, 3)), rng.uniform(-0.6, 0.6, size=(B, 3))
        kw = {"q0": unit_quaternion(rng, B), "fbar": np.tile([[0.0], [0.0], [-1.0]], (B, 1, N))}
        qe, gmax = newton(o, F, Mt, H0, ne, **kw)
        assert gmax < 1e-13
        worst[N] = float(contraction(o, qe, F, Mt, H0, ne, **kw).max())
    assert worst[9] < 1e-4 and worst[16] < 1e-10, worst


def test_null_handle_and_argument_errors(sri_lib):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import _lib
    H = (ctypes.c_double * 3)(1.0, 1.0, 0.77)
    prob = _lib.StaticProblem(batch=0, ne=3, H_diag=ctypes.addressof(H))
    rep = _lib.NewtonReport()
    assert sri_lib.sri_newton_static_problem(None, ctypes.byref(prob), None, 1e-10, 30, 0.0, 0, _lib.ALLREDUCE_FN(), None,
                                             ctypes.byref(rep)) == -1
    assert b"handle" in sri_lib.sri_last_error_string().lower()
    grads = _lib.StaticProblemGrad()
    assert sri_lib.sri_static_problem_vjp(None, ctypes.byref(prob), None, None, 3, ctypes.byref(grads)) == -1
    assert b"handle" in sri_lib.sri_last_error_string().lower()
    assert sri_lib.sri_newton_static_problem_sharded(None, ctypes.byref(prob), None, 1e-10, 30, 0.0, ctypes.byref(rep)) == -1
    assert sri_lib.sri_newton_static_problem_sharded(ctypes.c_void_p(1), None, None, 1e-10, 30, 0.0, ctypes.byref(rep)) == -1
    assert b"problem" in sri_lib.sri_last_error_string()
