"""Extended-precision reference for the system every fused-integration kernel actually solves (numpy only).

All six elimination kernels (the tensor-core first pass and the row-pivoting second pass, for N <= 16, <= 32 and <= 64)
solve, per rod, the preconditioned quaternion collocation system

    sum_j Q_j (x) c_ij = g_i q0,     c_ij = (delta_ij, -1/2 S_ij K_j),   S = Dn_NN^-1,   g = -S Dn_IN

(sri_fused16.cuh, stage 1; sri_tiled.cuh, stage 1; tools/dmma_gj_emulator.py).  Here it is built as a real 4M x 4M matrix C
with blocks Rmat(c_ij), where vec(a (x) c) = Rmat(c) vec(a), the unknowns ordered node by node (x[4j + c] = Q[c][j]).
The entries are formed with the kernels' own double operations, fl(fl(-1/2 S_ij) K_j) and fl(g_i q0_c), so C and b are
exactly the float64 system the device eliminates, and a backward error measured against them says how well it was solved
whatever the conditioning.

Stages 2-4 are evaluated from GIVEN quaternions (and internal forces, for the couple) in long double, each with the
componentwise magnitude |T| |x| of its contraction (the right-hand side's own products included), so that a kernel's
stage outputs can be checked entry by entry against (M + 4) u |T| |x| instead of a bound normalised by the rod's largest
entry.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

LD = np.longdouble
U = 2.0 ** -53  # unit roundoff of float64


@dataclass
class Tables:
    """The float64 operator tables of one node count.  g and gT are the long-double products rounded once, as the library's
    host code forms them (sri_host_math.hpp)."""
    S: np.ndarray      # Dn_NN^-1, M x M
    Dn_IN: np.ndarray  # M
    ST: np.ndarray     # D_TT^-1, M x M
    D_TI: np.ndarray   # M

    def __post_init__(self):
        self.M = self.S.shape[0]
        self.N = self.M + 1
        self.g = (-(self.S.astype(LD) @ self.Dn_IN.astype(LD))).astype(np.float64)
        self.gT = (-(self.ST.astype(LD) @ self.D_TI.astype(LD))).astype(np.float64)

    @classmethod
    def from_handle(cls, h) -> "Tables":
        return cls(h.operator("Dn_NN_inv"), h.operator("Dn_IN"), h.operator("D_TT_inv"), h.operator("D_TI"))

    @classmethod
    def from_oracle(cls, o) -> "Tables":
        return cls(o.operator(3), o.operator(2), o.operator(6), o.operator(5))

    def dmma16_stress_delta(self):
        """The N <= 16 tensor-core kernel computes n with J S J in place of -D_TT^-1 and J g in place of gT (J = exchange
        matrix; sri_fused16_dmma.cuh, stages 2-3).  Returns |(-J S J) - ST| and |J g - gT| of the float64 tables."""
        dT = np.abs(-self.S[::-1, ::-1].astype(LD) - self.ST.astype(LD))
        dg = np.abs(self.g[::-1].astype(LD) - self.gT.astype(LD))
        return dT, dg


def q_to_x(Q):
    """Q [B][4][M] -> x [B][4M], node-major."""
    return np.ascontiguousarray(np.swapaxes(Q, 1, 2)).reshape(Q.shape[0], -1)


def x_to_q(x, M):
    return np.ascontiguousarray(np.swapaxes(x.reshape(x.shape[0], M, 4), 1, 2))


def system(tab: Tables, K, q0=None):
    """(C [B][4M][4M], b [B][4M]) in float64, entries rounded exactly as the kernels form them."""
    B, M = K.shape[0], tab.M
    C = quaternion_operator(-0.5 * tab.S, K)                    # the kernels' table entry -1/2 S_ij (exact)
    q0 = np.tile([1.0, 0.0, 0.0, 0.0], (B, 1)) if q0 is None else q0
    b = (tab.g[None, :, None] * q0[:, None, :]).reshape(B, 4 * M)
    return C, b


def quaternion_operator(s, K):
    """The real 4M x 4M matrix [B][4M][4M] of x -> (sum_j x_j (x) c_ij)_i with c_ij = (delta_ij, fl(s_ij K_j)), node-major."""
    B, M = K.shape[0], s.shape[0]
    v = s[None, :, :, None] * np.swapaxes(K[:, :, :M], 1, 2)[:, None, :, :]  # [B][i][j][3] = fl(s_ij K_j)
    w = np.broadcast_to(np.eye(M), (B, M, M))
    C = np.zeros((B, M, 4, M, 4))
    v0, v1, v2 = v[..., 0], v[..., 1], v[..., 2]
    rows = ((w, -v0, -v1, -v2), (v0, w, v2, -v1), (v1, -v2, w, v0), (v2, v1, -v0, w))  # Rmat(c), p (x) c = Rmat(c) p
    for r in range(4):
        for c in range(4):
            C[:, :, r, :, c] = rows[r][c]
    return C.reshape(B, 4 * M, 4 * M)


def residual(C, x, b):
    """b - C x in long double (C and b are float64 and exact; x may be long double)."""
    return b.astype(LD) - np.matmul(C.astype(LD), x.astype(LD)[..., None])[..., 0]


def backward_error(C, x, b):
    """Normwise backward error per rod: ||b - C x||_inf / (||C||_inf ||x||_inf + ||b||_inf), residual in long double."""
    r = np.abs(residual(C, x, b)).max(axis=1)
    nC = np.abs(C).sum(axis=2).max(axis=1)
    return (r / (nC * np.abs(x).max(axis=1) + np.abs(b).max(axis=1))).astype(np.float64)


def cond_inf(C):
    return np.abs(C).sum(axis=2).max(axis=1) * np.abs(np.linalg.inv(C)).sum(axis=2).max(axis=1)


def refine_step(C, x, b):
    """One step of iterative refinement: long-double residual, float64 correction, long-double accumulation.  Returns the
    new x and the relative size of the correction, per rod."""
    d = np.linalg.solve(C, residual(C, x, b).astype(np.float64)[..., None])[..., 0]
    x = x + d.astype(LD)
    return x, (np.abs(d).max(axis=1) / np.abs(x).max(axis=1).astype(np.float64))


def refined_solve(C, b, steps: int = 4, tol=1e-17):
    """float64 LAPACK solve, then `steps` refinement steps.  Raises unless the last correction is below tol relative
    (scalar or one value per rod).  b may be float64 or long double.  Returns x in long double."""
    x = np.linalg.solve(C, b.astype(np.float64)[..., None])[..., 0].astype(LD)
    for _ in range(steps):
        x, rel = refine_step(C, x, b)
    bad = np.nonzero(rel > tol)[0]
    if bad.size:
        raise ArithmeticError(f"refinement did not converge for rods {bad[:8].tolist()}: last correction {rel[bad].max():.2e}")
    return x


# ---- stages 2-4 from given quaternions, long double -----------------------------------------------------------

def _rot(q, g):
    """R(q) g (the un-normalised rotation of sri_device.cuh q_rotate) and its magnitude: every product of the evaluation in
    absolute value.  q [..][4], g [..][3], long double."""
    w, x, y, z = (q[..., k] for k in range(4))
    R = [[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
         [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
         [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]]
    A = [[1 + 2 * (y * y + z * z), 2 * (abs(x * y) + abs(w * z)), 2 * (abs(x * z) + abs(w * y))],
         [2 * (abs(x * y) + abs(w * z)), 1 + 2 * (x * x + z * z), 2 * (abs(y * z) + abs(w * x))],
         [2 * (abs(x * z) + abs(w * y)), 2 * (abs(y * z) + abs(w * x)), 1 + 2 * (x * x + y * y)]]
    out = np.stack([R[c][0] * g[..., 0] + R[c][1] * g[..., 1] + R[c][2] * g[..., 2] for c in range(3)], axis=-1)
    mag = np.stack([A[c][0] * abs(g[..., 0]) + A[c][1] * abs(g[..., 1]) + A[c][2] * abs(g[..., 2]) for c in range(3)], axis=-1)
    return out, mag


def _nodal(a, B, N, default):
    """[B][3][N] -> [B][N][3] long double; None -> the default vector at every node."""
    if a is None:
        return np.broadcast_to(np.asarray(default, dtype=LD), (B, N, 3))
    return np.swapaxes(np.asarray(a), 1, 2).astype(LD)


def _tip(a, B):
    return np.zeros((B, 3), dtype=LD) if a is None else np.asarray(a).astype(LD)


def stage_r(tab: Tables, Q, Gamma=None, r0=None):
    """r = S (R(q) Gamma) + g r0 at the M unknown nodes; returns (r, |S| |R(q) Gamma| + |g| |r0|), [B][3][M] each."""
    B, M = Q.shape[0], tab.M
    q = np.swapaxes(Q, 1, 2).astype(LD)                                   # [B][M][4]
    b, bm = _rot(q, _nodal(Gamma, B, tab.N, (1.0, 0.0, 0.0))[:, :M])       # [B][M][3]
    S, g = tab.S.astype(LD), tab.g.astype(LD)
    r0 = _tip(r0, B)
    r = np.einsum("ij,bjc->bci", S, b) + g[None, None, :] * r0[:, :, None]
    mag = np.einsum("ij,bjc->bci", abs(S), bm) + abs(g)[None, None, :] * abs(r0)[:, :, None]
    return r, mag


def stage_n(tab: Tables, B, F_tip=None, fbar=None):
    """n = D_TT^-1 (-fbar[1:] - D_TI F_tip) at nodes 1..N-1; returns (n, |D_TT^-1| (|fbar| + |D_TI| |F|) + |gT| |F|)."""
    M = tab.M
    f = _nodal(fbar, B, tab.N, (0.0, 0.0, 0.0))[:, 1:]                      # [B][M][3]
    F = _tip(F_tip, B)
    ST, dti, gT = tab.ST.astype(LD), tab.D_TI.astype(LD), tab.gT.astype(LD)
    rhs = -f - dti[None, :, None] * F[:, None, :]
    n = np.einsum("ij,bjc->bci", ST, rhs)
    mag = (np.einsum("ij,bjc->bci", abs(ST), abs(f) + abs(dti)[None, :, None] * abs(F)[:, None, :])
           + abs(gT)[None, None, :] * abs(F)[:, :, None])
    assert n.shape == (B, 3, M)
    return n, mag


def stage_n_dmma16_extra(tab: Tables, B, F_tip=None, fbar=None):
    """The part of the stage-3 bound that the N <= 16 tensor-core kernel's operator adds: |J S J + D_TT^-1| |fbar| +
    |J g - gT| |F|, [B][3][M]."""
    dT, dg = tab.dmma16_stress_delta()
    f = _nodal(fbar, B, tab.N, (0.0, 0.0, 0.0))[:, 1:]
    F = _tip(F_tip, B)
    return np.einsum("ij,bjc->bci", dT, abs(f)) + dg[None, None, :] * abs(F)[:, :, None]


def stage_m(tab: Tables, Q, n, q0=None, Gamma=None, lbar=None, M_tip=None):
    """m = D_TT^-1 (-(r' x n + lbar)[1:] - D_TI M_tip) with r' = R(q) Gamma (node N-1: q0) and the GIVEN n; returns (m, its
    magnitude), [B][3][M]."""
    B, M, N = Q.shape[0], tab.M, tab.N
    q = np.concatenate([np.swapaxes(Q, 1, 2).astype(LD),
                        (np.tile(LD([1, 0, 0, 0]), (B, 1)) if q0 is None else np.asarray(q0).astype(LD))[:, None, :]], axis=1)
    rp, rpm = _rot(q[:, 1:], _nodal(Gamma, B, N, (1.0, 0.0, 0.0))[:, 1:])   # nodes 1..N-1, [B][M][3]
    nn = np.swapaxes(np.asarray(n), 1, 2).astype(LD)
    an = abs(nn)
    cr = np.stack([rp[..., 1] * nn[..., 2] - rp[..., 2] * nn[..., 1], rp[..., 2] * nn[..., 0] - rp[..., 0] * nn[..., 2],
                   rp[..., 0] * nn[..., 1] - rp[..., 1] * nn[..., 0]], axis=-1)
    crm = np.stack([rpm[..., 1] * an[..., 2] + rpm[..., 2] * an[..., 1], rpm[..., 2] * an[..., 0] + rpm[..., 0] * an[..., 2],
                    rpm[..., 0] * an[..., 1] + rpm[..., 1] * an[..., 0]], axis=-1)
    lb = _nodal(lbar, B, N, (0.0, 0.0, 0.0))[:, 1:]
    T = _tip(M_tip, B)
    ST, dti, gT = tab.ST.astype(LD), tab.D_TI.astype(LD), tab.gT.astype(LD)
    m = np.einsum("ij,bjc->bci", ST, -(cr + lb) - dti[None, :, None] * T[:, None, :])
    mag = (np.einsum("ij,bjc->bci", abs(ST), crm + abs(lb) + abs(dti)[None, :, None] * abs(T)[:, None, :])
           + abs(gT)[None, None, :] * abs(T)[:, :, None])
    return m, mag


def stage_bound(tab: Tables, mag):
    """The componentwise bound (M + 4) u |T| |x| of a stage contraction."""
    return (tab.M + 4) * U * mag.astype(np.float64)


def stage_excess(got, ref, bound):
    """max over entries of |got - ref| / bound per rod (<= 1 passes); entries with a zero bound must match exactly."""
    err = np.abs(np.asarray(got).astype(LD) - ref).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
    return ratio.reshape(ratio.shape[0], -1).max(axis=1)
