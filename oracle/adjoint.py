"""Reverse-mode derivatives (vector-Jacobian products) of the DISCRETE four-stage map, in numpy.

TEST INFRASTRUCTURE ONLY (like everything under oracle/): nothing in the product imports this.  It restates, on the
oracle's operators, what sri_integrate_all_vjp computes, and is pinned by a dot-product test against central differences
of Oracle.integrate_all (tests/test_adjoint_cpu.py).

Notation (include/sri.h, oracle/sri_oracle.c): S = Dn_NN^-1, S_T = D_TT^-1, b_i = R(q_i) Gamma_i with R Eigen's
un-normalised toRotationMatrix (node N-1 uses q0), A(k) the 4x4 block of updateA (sri_oracle.c:273).  Given the output
cotangents gQ [4][M], gr, gn, gm [3][M] of one rod, the adjoint runs the stages backwards:

    stage 4   nu = S_T^T gm            lbar-grad[1:] = -nu,  M_tip-grad = -sum_i D_TI[i] nu_i,
                                       g_b[1:] += -n x nu,   gn += b[1:] x nu
    stage 3   xi = S_T^T gn            fbar-grad[1:] = -xi,  F_tip-grad = -sum_i D_TI[i] xi_i
    stage 2   mu = S^T gr              g_b[:M] += mu,        r0-grad = -sum_i Dn_IN[i] mu_i
    b = R Gamma                        Gamma-grad_i = R(q_i)^T g_b_i,  gq_i = d/dq (g_b_i^T R(q_i) Gamma_i)
                                       (nodes 0..M-1 add to gQ, node N-1 to q0-grad)
    stage 1   A_NN(K)^T lam = gQ       K-grad[c][i] = 1/2 lam_i^T A(e_c) Q_i (i < N-1; 0 at the base node),
                                       q0-grad += -sum_i Dn_IN[i] lam_i
"""
from __future__ import annotations

import numpy as np

from .tangent import rotation

E1 = np.array([1.0, 0.0, 0.0])


def block_A(k: np.ndarray) -> np.ndarray:
    """The 4x4 block of updateA for the strain k (sri_oracle.c:273): A(k) q = q (x) (0, k)."""
    k0, k1, k2 = k
    return np.array([[0, -k0, -k1, -k2], [k0, 0, k2, -k1], [k1, -k2, 0, k0], [k2, k1, -k0, 0]], dtype=np.float64)


def rotation_vjp(q: np.ndarray, gamma: np.ndarray, a: np.ndarray) -> np.ndarray:
    """d/dq of a^T R(q) gamma for the un-normalised R: R gamma = gamma + 2w (v x gamma) + 2 v x (v x gamma), v = (x,y,z)."""
    w, v = q[0], q[1:]
    gw = 2.0 * a @ np.cross(v, gamma)
    gv = 2.0 * w * np.cross(gamma, a) + 2.0 * (a @ v) * gamma + 2.0 * (v @ gamma) * a - 4.0 * (a @ gamma) * v
    return np.concatenate([[gw], gv])


def integrate_all_vjp(oracle, K, Q, n=None, q0=None, Gamma=None, gQ=None, gr=None, gn=None, gm=None):
    """Gradients of <gQ, Q> + <gr, r> + <gn, n> + <gm, m> with respect to the eight inputs of oracle.integrate_all.

    K [B][3][N]; Q [B][4][M] and (when gm is given) n [B][3][M]: the forward outputs at these inputs; q0 [B][4], Gamma
    [B][3][N] optional as in the forward (identity, e1).  Cotangents may be None (zero).  The forward's other inputs
    (r0, fbar, lbar, F_tip, M_tip) enter linearly and do not appear.  Returns a dict with K, q0, r0, Gamma, fbar, lbar,
    F_tip, M_tip gradients and `bad`, the number of rods whose transposed stage-1 system was singular."""
    K = np.asarray(K, dtype=np.float64)
    B, N, M = K.shape[0], oracle.N, oracle.M
    S, Dn_IN, D_TI, S_T = (oracle.operator(w) for w in (3, 2, 5, 6))
    z = lambda shape: np.zeros((B,) + shape)
    gQ = z((4, M)) if gQ is None else np.asarray(gQ, dtype=np.float64)
    gr = z((3, M)) if gr is None else np.asarray(gr, dtype=np.float64)
    gn = z((3, M)) if gn is None else np.asarray(gn, dtype=np.float64)
    out = {k: z(s) for k, s in (("K", (3, N)), ("q0", (4,)), ("r0", (3,)), ("Gamma", (3, N)), ("fbar", (3, N)),
                                ("lbar", (3, N)), ("F_tip", (3,)), ("M_tip", (3,)))}
    bad = 0
    for b in range(B):
        qn = np.concatenate([Q[b].T, [np.array([1.0, 0, 0, 0]) if q0 is None else q0[b]]])   # [N][4], base node = q0
        gam = np.tile(E1, (N, 1)) if Gamma is None else Gamma[b].T                            # [N][3]
        Rn = rotation(qn)
        bn = np.einsum("ikc,ic->ik", Rn, gam)                                                 # b_i = R_i Gamma_i
        g_b = np.zeros((N, 3))
        gn_b = gn[b].T.copy()                                                                 # [M][3], nodes 1..N-1
        if gm is not None:
            nu = S_T.T @ gm[b].T
            out["lbar"][b][:, 1:] = -nu.T
            out["M_tip"][b] = -D_TI @ nu
            nj = n[b].T
            g_b[1:] += -np.cross(nj, nu)
            gn_b += np.cross(bn[1:], nu)
        xi = S_T.T @ gn_b
        out["fbar"][b][:, 1:] = -xi.T
        out["F_tip"][b] = -D_TI @ xi
        mu = S.T @ gr[b].T
        g_b[:M] += mu
        out["r0"][b] = -Dn_IN @ mu
        out["Gamma"][b] = np.einsum("ikc,ik->ci", Rn, g_b)                                   # R_i^T g_b_i
        gq = np.array([rotation_vjp(qn[i], gam[i], g_b[i]) for i in range(N)])               # [N][4]
        rhs = (gQ[b] + gq[:M].T).reshape(-1)                                                  # stack [c*M+i]
        A = oracle.assemble_A(K[b])
        try:
            lam = np.linalg.solve(A.T, rhs).reshape(4, M).T                                   # [M][4]
        except np.linalg.LinAlgError:
            bad += 1
            lam = np.full((M, 4), np.nan)
        for c in range(3):
            ec = np.zeros(3); ec[c] = 1.0
            Ae = block_A(ec)
            out["K"][b][c, :M] = 0.5 * np.einsum("ia,ab,ib->i", lam, Ae, qn[:M])
        out["q0"][b] = gq[M] - Dn_IN @ lam
    out["bad"] = bad
    return out
