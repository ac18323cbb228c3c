"""The static shape problem under distributed loads, a rotated clamp and a given Gamma, in numpy: the restatement that
sri_newton_static_problem and sri_static_problem_vjp are checked against (test infrastructure, like oracle/; nothing in the
product imports it).

The problem of include/sri.h (sri_static_problem): theta = (F_tip, M_tip, K0, q0, Gamma, fbar, lbar) and H,
    g(qe; theta) = sum_i w_i P(t_i)^T rho_i,   rho_i = H (K_i - K0_i) - R(q_i)^T m_i,   K = Phi qe,
with (Q, n, m) the oracle's four stages (oracle.integrate_all) under q0, Gamma, fbar, lbar and the tip loads.

J_d, the exact Jacobian of the discrete residual, is assembled row by row from 3 ne reverse-mode products per rod: row j is
J_d^T e_j = Phi^T (gK_dir + gK_int), gK_dir from static_adjoint_ref.galerkin_residual_vjp with cotangent e_j and gK_int from
oracle/adjoint.integrate_all_vjp of that VJP's (gQ, gm) -- the chain(lam) of DESIGN section 5e with lam = e_j.  The
equilibrium gradient is then lam = J_d^-T gqe and theta-grad = -(dg/dtheta)^T lam from one more chain(lam):
    F_tip: -gF_int,  M_tip: -(gM_dir + gM_int),  K0: -gK0_dir,  H: -gH_dir,  q0: -(gq0_dir + gq0_int),
    Gamma: -gGamma_int,  fbar: -gfbar_int,  lbar: -glbar_int.
"""
from __future__ import annotations

import numpy as np

from oracle.adjoint import integrate_all_vjp
from oracle.tangent import cc_weights, jacobian_by_quadrature_from_state
from static_adjoint_ref import galerkin_residual, galerkin_residual_vjp, legendre_table

INPUTS = ("q0", "Gamma", "fbar", "lbar")


def unit_quaternion(rng, B):
    q = rng.normal(size=(B, 4))
    return q / np.linalg.norm(q, axis=1, keepdims=True)


def loaded_problem(rng, B, N, g=1.0):
    """Tip loads U(-0.6, 0.6)^3, K0, a random clamp rotation, Gamma near e1, the weight (0, 0, -g) plus a varying part, lbar."""
    F, Mt = rng.uniform(-0.6, 0.6, size=(B, 3)), rng.uniform(-0.6, 0.6, size=(B, 3))
    Gamma = rng.uniform(-0.1, 0.1, size=(B, 3, N)); Gamma[:, 0] += 1.0
    fbar = rng.uniform(-0.2, 0.2, size=(B, 3, N)); fbar[:, 2] -= g
    return {"F_tip": F, "M_tip": Mt, "K0": rng.uniform(-0.3, 0.3, size=(B, 3, N)), "q0": unit_quaternion(rng, B),
            "Gamma": Gamma, "fbar": fbar, "lbar": rng.uniform(-0.3, 0.3, size=(B, 3, N))}


def forward(oracle, qe, F_tip, M_tip, ne, q0=None, Gamma=None, fbar=None, lbar=None):
    """K = Phi qe and the stages (Q, n, m) of the loaded rods."""
    K = oracle.strain_from_modes(qe, ne)
    out = oracle.integrate_all(K, F_tip, M_tip, q0=q0, Gamma=Gamma, fbar=fbar, lbar=lbar, explicit_inverse=False,
                               want=("Q", "n", "m"))
    return K, out["Q"], out["n"], out["m"]


def residual(oracle, qe, F_tip, M_tip, H, ne, K0=None, q0=None, Gamma=None, fbar=None, lbar=None):
    """g [B][3 ne] of the loaded problem."""
    K, Q, _, m = forward(oracle, qe, F_tip, M_tip, ne, q0, Gamma, fbar, lbar)
    return galerkin_residual(oracle, K, H, Q, m, M_tip, ne, K0=K0, q0=q0)


def _chain(oracle, state, lam, F_tip, M_tip, H, ne, K0, q0, Gamma):
    """The residual VJP with cotangent lam, then the integration VJP of its (gQ, gm): (direct, integration) gradients."""
    K, Q, n, m = state
    d = galerkin_residual_vjp(oracle, K, H, Q, m, M_tip, lam, K0=K0, q0=q0)
    i = integrate_all_vjp(oracle, K, Q, n=n, q0=q0, Gamma=Gamma, gQ=d["Q"], gm=d["m"])
    return d, i


def residual_and_jacobian(oracle, qe, F_tip, M_tip, H, ne, K0=None, q0=None, Gamma=None, fbar=None, lbar=None):
    """g [B][3 ne] and the exact J_d [B][3 ne][3 ne] (J[b][j][d] = dg_j / dqe_d), J_d^T from 3 ne VJPs per rod."""
    n = 3 * ne
    state = forward(oracle, qe, F_tip, M_tip, ne, q0, Gamma, fbar, lbar)
    K, Q, _, m = state
    g = galerkin_residual(oracle, K, H, Q, m, M_tip, ne, K0=K0, q0=q0)
    P = legendre_table(oracle, ne)
    J = np.empty((qe.shape[0], n, n))
    for j in range(n):
        e = np.zeros((qe.shape[0], n)); e[:, j] = 1.0
        d, i = _chain(oracle, state, e, F_tip, M_tip, H, ne, K0, q0, Gamma)
        J[:, j, :] = np.einsum("bci,ki->bck", d["K"] + i["K"], P).reshape(-1, n)     # Phi^T, no weights
    return g, J


def newton(oracle, F_tip, M_tip, H, ne, K0=None, q0=None, Gamma=None, fbar=None, lbar=None, qe0=None, tol=1e-14, max_iter=40):
    """Newton with the exact J_d until max|g| < tol (or no further decrease once below 1e-12).  Returns (qe, max|g|)."""
    B = F_tip.shape[0]
    qe = np.zeros((B, 3 * ne)) if qe0 is None else np.array(qe0, dtype=np.float64)
    best = np.inf
    for _ in range(max_iter):
        g, J = residual_and_jacobian(oracle, qe, F_tip, M_tip, H, ne, K0, q0, Gamma, fbar, lbar)
        gmax = float(np.abs(g).max())
        if gmax < tol or (gmax < 1e-12 and gmax >= best):
            break
        best = min(best, gmax)
        qe = qe - np.stack([np.linalg.solve(J[b], g[b]) for b in range(B)])
    return qe, gmax


def adjoint(oracle, qe, F_tip, M_tip, H, ne, gqe, K0=None, q0=None, Gamma=None, fbar=None, lbar=None):
    """theta-gradients of <gqe, qe*> at the equilibrium qe (formula of the module docstring), exact J_d, direct solve.
    Returns a dict with F_tip, M_tip, K0, H (per rod), q0, Gamma, fbar, lbar and lambda."""
    _, J = residual_and_jacobian(oracle, qe, F_tip, M_tip, H, ne, K0, q0, Gamma, fbar, lbar)
    lam = np.stack([np.linalg.solve(J[b].T, gqe[b]) for b in range(qe.shape[0])])
    state = forward(oracle, qe, F_tip, M_tip, ne, q0, Gamma, fbar, lbar)
    d, i = _chain(oracle, state, lam, F_tip, M_tip, H, ne, K0, q0, Gamma)
    return {"F_tip": -i["F_tip"], "M_tip": -(d["M_tip"] + i["M_tip"]), "K0": -d["K0"], "H": -d["H"],
            "q0": -(d["q0"] + i["q0"]), "Gamma": -i["Gamma"], "fbar": -i["fbar"], "lbar": -i["lbar"], "lambda": lam}


def analytic_jacobian(oracle, qe, F_tip, M_tip, H, ne, q0=None, Gamma=None, fbar=None, lbar=None):
    """J_a of sri_shape_jacobian at the loaded state (oracle/tangent.jacobian_by_quadrature_from_state with the varying n)."""
    _, Q, n, m = forward(oracle, qe, F_tip, M_tip, ne, q0, Gamma, fbar, lbar)
    Dn, M = oracle.dn(), oracle.M
    S, S_T = np.linalg.inv(Dn[:M, :M]), np.linalg.inv(Dn[1:, 1:])
    return jacobian_by_quadrature_from_state(Q, n, m, M_tip, np.asarray(H, dtype=np.float64), ne, legendre_table(oracle, ne),
                                             cc_weights(oracle.N), S, S_T, q0=q0, Gamma=Gamma)


def contraction(oracle, qe, F_tip, M_tip, H, ne, K0=None, q0=None, Gamma=None, fbar=None, lbar=None):
    """||J_a^-1 J_d - I||_2 per rod: the contraction factor of the adjoint's iterative refinement (DESIGN section 5e)."""
    _, Jd = residual_and_jacobian(oracle, qe, F_tip, M_tip, H, ne, K0, q0, Gamma, fbar, lbar)
    Ja = analytic_jacobian(oracle, qe, F_tip, M_tip, H, ne, q0, Gamma, fbar, lbar)
    eye = np.eye(3 * ne)
    return np.array([np.linalg.norm(np.linalg.solve(Ja[b], Jd[b]) - eye, 2) for b in range(qe.shape[0])])
