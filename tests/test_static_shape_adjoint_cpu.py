"""CPU tests of the reverse mode of the static shape problem: the numpy restatement (static_adjoint_ref.py) of the Galerkin
residual's VJP and of the implicit adjoint of the equilibrium, each pinned by a dot-product test against central differences
of the oracle; and the argument errors of the two entry points sri_galerkin_residual_vjp / sri_static_shape_vjp."""
import ctypes

import numpy as np
import pytest

RES_INPUTS = ("K", "K0", "H", "Q", "q0", "m", "M_tip")
H0 = np.array([1.0, 1.0, 0.77])


def _state(rng, B, N):
    M = N - 1
    Q = rng.normal(size=(B, 4, M))
    q0 = rng.normal(size=(B, 4))
    return {"K": rng.uniform(-2, 2, size=(B, 3, N)), "K0": rng.uniform(-1, 1, size=(B, 3, N)),
            "H": H0 + rng.uniform(0, 0.5, size=3), "Q": Q, "q0": q0, "m": rng.normal(size=(B, 3, M)),
            "M_tip": rng.normal(size=(B, 3))}


@pytest.mark.parametrize("N", [2, 5, 16, 33])
def test_residual_vjp_dot_product_against_central_differences(make_oracle, N):
    from static_adjoint_ref import galerkin_residual, galerkin_residual_vjp
    o = make_oracle(N)
    rng = np.random.default_rng(300 + N)
    B, ne, h = 3, 4, 1e-6
    x = _state(rng, B, N)
    gg = rng.normal(size=(B, 3 * ne))
    res = lambda s: galerkin_residual(o, s["K"], s["H"], s["Q"], s["m"], s["M_tip"], ne, K0=s["K0"], q0=s["q0"])
    g = galerkin_residual_vjp(o, x["K"], x["H"], x["Q"], x["m"], x["M_tip"], gg, K0=x["K0"], q0=x["q0"])
    g["H"] = g["H"].sum(0)   # one H for the batch
    dirs = {k: rng.normal(size=v.shape) for k, v in x.items()}

    def directional(keys):
        xp = {k: v + h * dirs[k] if k in keys else v for k, v in x.items()}
        xm = {k: v - h * dirs[k] if k in keys else v for k, v in x.items()}
        fd = float(np.sum(gg * (res(xp) - res(xm)))) / (2 * h)
        return fd, sum(float(np.sum(g[k] * dirs[k])) for k in keys), sum(float(np.abs(g[k] * dirs[k]).sum()) for k in keys)

    fd, ad, scale = directional(RES_INPUTS)
    assert abs(fd - ad) <= 1e-7 * scale, (N, fd, ad)
    for k in RES_INPUTS:   # each input alone, so that an error in one gradient cannot hide behind a larger one
        fd, ad, scale = directional((k,))
        assert abs(fd - ad) <= 1e-7 * scale, (N, k, fd, ad)


def test_residual_vjp_defaults_are_zero_K0_and_identity_q0(make_oracle):
    from static_adjoint_ref import galerkin_residual_vjp
    N, B = 7, 2
    o = make_oracle(N)
    rng = np.random.default_rng(2)
    x = _state(rng, B, N)
    gg = rng.normal(size=(B, 9))
    a = galerkin_residual_vjp(o, x["K"], x["H"], x["Q"], x["m"], x["M_tip"], gg)
    b = galerkin_residual_vjp(o, x["K"], x["H"], x["Q"], x["m"], x["M_tip"], gg, K0=np.zeros((B, 3, N)),
                              q0=np.tile([1.0, 0, 0, 0], (B, 1)))
    for k in RES_INPUTS:
        assert np.array_equal(a[k], b[k]), k


def _loads(rng, B, scale=0.6):
    return rng.uniform(-scale, scale, size=(B, 3)), rng.uniform(-scale, scale, size=(B, 3))


@pytest.mark.parametrize("N", [5, 9, 16])
def test_static_shape_vjp_against_central_differences_of_the_newton_solve(make_oracle, N):
    from static_adjoint_ref import newton_static_shape, static_shape_vjp
    o = make_oracle(N)
    rng = np.random.default_rng(400 + N)
    B, ne, h = 2, 3, 1e-5
    F, Mt = _loads(rng, B)
    K0 = rng.uniform(-0.3, 0.3, size=(B, 3, N))
    theta = {"F_tip": F, "M_tip": Mt, "K0": K0, "H": H0.copy()}
    gqe = rng.normal(size=(B, 3 * ne))

    def solve(t):
        qe, gmax = newton_static_shape(o, t["F_tip"], t["M_tip"], t["H"], ne, K0=t["K0"])
        assert gmax < 1e-13, gmax
        return qe

    qe = solve(theta)
    g = static_shape_vjp(o, qe, F, Mt, H0, ne, gqe, K0=K0)
    g["H"] = g["H"].sum(0)
    for k in ("F_tip", "M_tip", "K0", "H"):
        d = rng.normal(size=theta[k].shape)
        tp = dict(theta, **{k: theta[k] + h * d})
        tm = dict(theta, **{k: theta[k] - h * d})
        fd = float(np.sum(gqe * (solve(tp) - solve(tm)))) / (2 * h)
        ad = float(np.sum(g[k] * d))
        scale = max(abs(ad), float(np.abs(g[k] * d).sum()))
        assert abs(fd - ad) <= 1e-7 * scale, (N, k, fd, ad)


def test_null_handle_and_argument_errors(sri_lib):
    H = (ctypes.c_double * 3)(1.0, 1.0, 0.77)
    assert sri_lib.sri_galerkin_residual_vjp(None, 0, 3, *[None] * 2, H, *[None] * 12) == -1
    assert b"handle" in sri_lib.sri_last_error_string().lower()
    assert sri_lib.sri_static_shape_vjp(None, 0, 3, H, *[None] * 5, 3, *[None] * 7) == -1
    assert b"handle" in sri_lib.sri_last_error_string().lower()
