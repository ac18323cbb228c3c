"""Reverse mode of the static shape problem in numpy: the restatement that sri_galerkin_residual_vjp and
sri_static_shape_vjp are checked against (test infrastructure, like oracle/; nothing in the product imports it).

Notation of include/sri.h and oracle/tangent.py: t_i = 2 x_i - 1, w_i the Clenshaw-Curtis weights, P_k the Legendre modes,
    rho_i = H (K_i - K0_i) - R(q_i)^T m_i      (node 0: m = M_tip; node N-1: q = q0),
    g[c*ne+k] = sum_i w_i P_k(t_i) rho[c][i].

1. VJP of the residual, cotangent gg [3 ne]:  rb[c][i] = w_i sum_k P_k(t_i) gg[c*ne+k], then
    gK = H rb,  gK0 = -H rb,  gH[c] = sum_i rb[c][i] (K - K0)[c][i],
    gm[:, i-1] = -R(q_i) rb_i (i = 1..N-1),  gM_tip = -R(q_0) rb_0,
    gQ[:, i] = -rotation_vjp(q_i, rb_i, m_i) (i = 0..M-1),  gq0 = -rotation_vjp(q0, rb_{N-1}, m_{N-1}).

2. Implicit adjoint of the equilibrium g(qe*; F_tip, M_tip, K0, H) = 0 (q0 = identity, Gamma = e1, no distributed loads):
    J_d^T lam = gqe  (J_d the exact Jacobian of the discrete residual, oracle/tangent.py),   theta-grad = -(dg/dtheta)^T lam,
where (dg/dtheta)^T lam is the residual VJP with cotangent lam followed by the integration's VJP (oracle/adjoint.py) of its
(gQ, gm): F_tip-grad = -gF_tip_int, M_tip-grad = -(gM_tip_dir + gM_tip_int), K0-grad = H rb, H-grad = -gH.
"""
from __future__ import annotations

import numpy as np
from numpy.polynomial import legendre as _L

from oracle.adjoint import integrate_all_vjp, rotation_vjp
from oracle.tangent import cc_weights, galerkin_residual_and_jacobian, rotation


def _nodal(Q, q0, m, M_tip, b):
    """[N][4] rotations (base node = q0 or identity) and [N][3] couples (node 0 = M_tip) of rod b."""
    qb = np.array([1.0, 0.0, 0.0, 0.0]) if q0 is None else q0[b]
    return np.concatenate([Q[b].T, [qb]]), np.concatenate([[M_tip[b]], m[b].T])


def legendre_table(oracle, ne):
    x = oracle.chebyshev_points()
    return np.stack([_L.legval(2 * x - 1, [0] * k + [1]) for k in range(ne)])   # [ne][N]


def galerkin_residual(oracle, K, H, Q, m, M_tip, ne, K0=None, q0=None):
    """g [B][3 ne] (the numpy form of sri_galerkin_residual)."""
    P, w = legendre_table(oracle, ne), cc_weights(oracle.N)
    H = np.asarray(H, dtype=np.float64)
    g = np.empty((K.shape[0], 3 * ne))
    for b in range(K.shape[0]):
        qn, mn = _nodal(Q, q0, m, M_tip, b)
        Kd = K[b] - (0.0 if K0 is None else K0[b])
        rho = H[:, None] * Kd - np.einsum("ikc,ik->ci", rotation(qn), mn)
        g[b] = np.einsum("ci,ki,i->ck", rho, P, w).reshape(-1)
    return g


def galerkin_residual_vjp(oracle, K, H, Q, m, M_tip, gg, K0=None, q0=None):
    """Gradients of <gg, g> with respect to K, K0, H (per rod, [B][3]), Q, q0, m, M_tip (formula 1 above)."""
    B, N, M = K.shape[0], oracle.N, oracle.M
    ne = gg.shape[1] // 3
    P, w = legendre_table(oracle, ne), cc_weights(N)
    H = np.asarray(H, dtype=np.float64)
    out = {"K": np.empty((B, 3, N)), "K0": np.empty((B, 3, N)), "H": np.empty((B, 3)), "Q": np.empty((B, 4, M)),
           "q0": np.empty((B, 4)), "m": np.empty((B, 3, M)), "M_tip": np.empty((B, 3))}
    for b in range(B):
        qn, mn = _nodal(Q, q0, m, M_tip, b)
        rb = w[None, :] * np.einsum("ck,ki->ci", gg[b].reshape(3, ne), P)                 # [3][N]
        Kd = K[b] - (0.0 if K0 is None else K0[b])
        out["K"][b] = H[:, None] * rb
        out["K0"][b] = -H[:, None] * rb
        out["H"][b] = np.sum(rb * Kd, axis=1)
        Rrb = np.einsum("ikc,ci->ik", rotation(qn), rb)                                    # R(q_i) rb_i, [N][3]
        out["M_tip"][b] = -Rrb[0]
        out["m"][b] = -Rrb[1:].T
        gq = np.array([-rotation_vjp(qn[i], rb[:, i], mn[i]) for i in range(N)])            # [N][4]
        out["Q"][b] = gq[:M].T
        out["q0"][b] = gq[M]
    return out


def static_shape_vjp(oracle, qe, F_tip, M_tip, H, ne, gqe, K0=None):
    """theta-gradients of <gqe, qe*> at the equilibrium qe (formula 2 above) with the exact J_d and a direct solve.
    Returns a dict with F_tip, M_tip, K0, H (per rod) and lambda."""
    B, n = qe.shape[0], 3 * ne
    _, J = galerkin_residual_and_jacobian(oracle, qe, F_tip, M_tip, H, ne, K0=K0)
    lam = np.stack([np.linalg.solve(J[b].T, gqe[b]) for b in range(B)])
    K = oracle.strain_from_modes(qe, ne)
    fwd = oracle.integrate_all(K, F_tip, M_tip, explicit_inverse=False, want=("Q", "n", "m"))
    d = galerkin_residual_vjp(oracle, K, H, fwd["Q"], fwd["m"], M_tip, lam, K0=K0)
    i = integrate_all_vjp(oracle, K, fwd["Q"], n=fwd["n"], gQ=d["Q"], gm=d["m"])
    return {"F_tip": -i["F_tip"], "M_tip": -(d["M_tip"] + i["M_tip"]), "K0": -d["K0"], "H": -d["H"], "lambda": lam}


def newton_static_shape(oracle, F_tip, M_tip, H, ne, K0=None, qe0=None, tol=1e-14, max_iter=40):
    """Newton with the exact J_d until max|g| < tol (or no further decrease once below 1e-12).  Returns (qe, max|g|)."""
    B = F_tip.shape[0]
    qe = np.zeros((B, 3 * ne)) if qe0 is None else np.array(qe0, dtype=np.float64)
    best = np.inf
    for _ in range(max_iter):
        g, J = galerkin_residual_and_jacobian(oracle, qe, F_tip, M_tip, H, ne, K0=K0)
        gmax = float(np.abs(g).max())
        if gmax < tol or (gmax < 1e-12 and gmax >= best):
            break
        best = min(best, gmax)
        qe = qe - np.stack([np.linalg.solve(J[b], g[b]) for b in range(B)])
    return qe, gmax
