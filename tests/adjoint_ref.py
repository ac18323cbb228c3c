"""Extended-precision reference for what the reverse-mode kernels compute (numpy only).

The kernels vjp16_kernel<15|0> (sri_vjp16.cuh) and vjp_tiled_kernel (sri_vjp_tiled.cuh) run the four stages backwards from
the forward's float64 Q and n and the output cotangents gQ, gr, gn, gm (oracle/adjoint.py states the derivation):

    stage 4  nu = S_T^T gm   lbar-grad[1:] = -nu, M_tip-grad = -D_TI^T nu, g_b[1:] += -n x nu, gn += b[1:] x nu
    stage 3  xi = S_T^T gn   fbar-grad[1:] = -xi, F_tip-grad = -D_TI^T xi
    stage 2  mu = S^T gr     g_b[:M] += mu,       r0-grad = -Dn_IN^T mu
    rotation b = R(q) Gamma: Gamma-grad = R^T g_b, gq = d/dq (g_b^T R(q) Gamma)
    stage 1  sum_j lam_j (x) c'_ij = b'_i,  c'_ij = delta_ij + (0, fl(fl(1/2 S_ji) K_j)),  b' = S^T (gQ + gq[:M])
             K-grad[c][i] = 1/2 <lam_i, q_i (x) (0, e_c)>,  q0-grad = gq[M] - sum_i Dn_IN[i] lam_i

with S = Dn_NN^-1 and S_T = D_TT^-1 the handle's float64 tables.  Here every stage is evaluated in long double from the
GIVEN float64 Q, n, q0, Gamma and cotangents, with the componentwise magnitude |T| |x| of each result (every product of the
evaluation in absolute value, the rotation and its derivative included), so that the kernels' stage gradients can be
checked entry by entry against (depth M + C_OPS) u |T| |x|, where depth is the number of M-term sums on the longest path
to the output (gF_tip: nu, xi, then the D_TI sum).

Stage 1 is checked by a forward-error bound instead: the transposed system C' is built with the kernels' own double
operations, so C' is exactly the float64 matrix they eliminate; lam' is its refined long-double solution for the exact b',
and a solve with backward error C_ETA u for a right-hand side computed with error db' lies within
    E = ||C'^-1|| (C_ETA u (||C'|| ||lam'|| + ||b'||) + ||db'||),   ||db'|| <= (2M + C_OPS) u |S^T| (|gQ| + mag(gq))
of lam' (infinity norms, per rod), which reaches K-grad through 1/2 |q_i| and q0-grad through |Dn_IN|.  lam itself is no
output (K-grad shows three of its four components per node), so stage 1 has no backward error to check.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from elimination_ref import LD, U, Tables, _nodal, _rot, quaternion_operator, refined_solve

C_ETA = 64   # the stage-1 solve's backward error allowance, in units of u
C_OPS = 16   # roundings outside the M-term sums on any path: rotation, its derivative, cross products, adds of parts
INPUTS = ("K", "q0", "r0", "Gamma", "fbar", "lbar", "F_tip", "M_tip")
DEPTH = {"lbar": 1, "M_tip": 2, "fbar": 2, "F_tip": 3, "r0": 2, "Gamma": 1}


def _cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1], a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1)


def _cross_mag(a, b):
    """The magnitude of a x b from magnitudes a, b >= 0."""
    return np.stack([a[..., 1] * b[..., 2] + a[..., 2] * b[..., 1], a[..., 2] * b[..., 0] + a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] + a[..., 1] * b[..., 0]], axis=-1)


def _tT(T, v):
    """sum_j T[j][i] v[b][j][c] (T^T applied node-wise), long double."""
    return np.einsum("ji,bjc->bic", np.asarray(T).astype(LD), v)


def _rows(a, B, M, k):
    """[B][k][M] cotangent -> [B][M][k] long double; None -> zeros."""
    return np.zeros((B, M, k), dtype=LD) if a is None else np.swapaxes(np.asarray(a), 1, 2).astype(LD)


def _cols(v):
    """[B][nodes][k] -> [B][k][nodes]."""
    return np.ascontiguousarray(np.swapaxes(v, 1, 2))


def rotation_vjp(q, g, a, am):
    """d/dq of a^T R(q) g for the un-normalised R (sri_vjp16.cuh rotation_vjp) and its magnitude; am is the magnitude of a
    (q and g are exact inputs).  [..][4], [..][3], [..][3], [..][3] -> ([..][4], [..][4])."""
    w, v = q[..., 0], q[..., 1:]
    aw, av_, ag_ = abs(w), abs(v), abs(g)
    vg, vgm = _cross(v, g), _cross_mag(av_, ag_)
    av, avm = (a * v).sum(-1), (am * av_).sum(-1)
    vgd, vgdm = (v * g).sum(-1), (av_ * ag_).sum(-1)
    ag, agm = (a * g).sum(-1), (am * ag_).sum(-1)
    gw, gwm = 2 * (a * vg).sum(-1), 2 * (am * vgm).sum(-1)
    gv = 2 * (w[..., None] * _cross(g, a) + av[..., None] * g + vgd[..., None] * a) - 4 * ag[..., None] * v
    gvm = 2 * (aw[..., None] * _cross_mag(ag_, am) + avm[..., None] * ag_ + vgdm[..., None] * am) + 4 * agm[..., None] * av_
    return np.concatenate([gw[..., None], gv], axis=-1), np.concatenate([gwm[..., None], gvm], axis=-1)


def strain_grad(lam, q):
    """1/2 <lam_i, q_i (x) (0, e_c)> for c = 0..2, [..][4] x [..][4] -> [..][3] (sri_vjp16.cuh strain_grad)."""
    lw, lx, ly, lz = (lam[..., k] for k in range(4))
    qw, qx, qy, qz = (q[..., k] for k in range(4))
    return 0.5 * np.stack([(lx * qw - lw * qx) + (ly * qz - lz * qy), (ly * qw - lw * qy) + (lz * qx - lx * qz),
                           (lz * qw - lw * qz) + (lx * qy - ly * qx)], axis=-1)


def reverse_stages(tab: Tables, Q, n=None, q0=None, Gamma=None, gQ=None, gr=None, gn=None, gm=None):
    """Stages 4 -> 2 and the rotation in long double.  Returns a dict with
        out[name] = (gradient in the kernels' output layout, its magnitude) for lbar, M_tip, fbar, F_tip, r0, Gamma;
        nu, xi, mu [B][M][3] and g_b [B][N][3] (values);  qn [B][N][4] (q_i, base node q0);
        gq, gq_mag [B][N][4] (the rotation's share);  r, r_mag [B][M][4] (the stage-1 right-hand side gQ + gq[:M])."""
    B, M, N = Q.shape[0], tab.M, tab.N
    qn = np.concatenate([np.swapaxes(np.asarray(Q), 1, 2).astype(LD),
                         (np.tile(LD([1, 0, 0, 0]), (B, 1)) if q0 is None else np.asarray(q0).astype(LD))[:, None, :]], axis=1)
    gam = _nodal(Gamma, B, N, (1.0, 0.0, 0.0))
    b, bm = _rot(qn, gam)
    S, ST, dti, dnin = tab.S, tab.ST, tab.D_TI.astype(LD), tab.Dn_IN.astype(LD)
    g_b, gbm = np.zeros((B, N, 3), dtype=LD), np.zeros((B, N, 3), dtype=LD)
    gnb = _rows(gn, B, M, 3)
    gnm = abs(gnb)
    gmv = _rows(gm, B, M, 3)
    nu, num = _tT(ST, gmv), _tT(abs(ST), abs(gmv))
    if gm is not None:
        nn = _rows(n, B, M, 3)
        g_b[:, 1:] += -_cross(nn, nu)
        gbm[:, 1:] += _cross_mag(abs(nn), num)
        gnb = gnb + _cross(b[:, 1:], nu)
        gnm = gnm + _cross_mag(bm[:, 1:], num)
    xi, xim = _tT(ST, gnb), _tT(abs(ST), gnm)
    grv = _rows(gr, B, M, 3)
    mu, mum = _tT(S, grv), _tT(abs(S), abs(grv))
    g_b[:, :M] += mu
    gbm[:, :M] += mum

    def nodal_minus(v, vm):  # -v at nodes 1..N-1, an exact zero at node 0
        z = np.zeros((B, 1, 3), dtype=LD)
        return _cols(np.concatenate([z, -v], axis=1)), _cols(np.concatenate([z, vm], axis=1))

    def tip(d, v, vm):  # -sum_i d_i v_i
        return -np.einsum("i,bic->bc", d, v), np.einsum("i,bic->bc", abs(d), vm)

    qT = qn.copy()
    qT[..., 0] = -qT[..., 0]                       # R(-w, x, y, z) = R(w, x, y, z)^T
    out = {"lbar": nodal_minus(nu, num), "M_tip": tip(dti, nu, num), "fbar": nodal_minus(xi, xim),
           "F_tip": tip(dti, xi, xim), "r0": tip(dnin, mu, mum),
           "Gamma": (_cols(_rot(qT, g_b)[0]), _cols(_rot(qn, gbm)[1]))}
    gq, gqm = rotation_vjp(qn, gam, g_b, gbm)
    gQv = _rows(gQ, B, M, 4)
    return {"out": out, "nu": nu, "xi": xi, "mu": mu, "g_b": g_b, "qn": qn, "gq": gq, "gq_mag": gqm,
            "r": gQv + gq[:, :M], "r_mag": abs(gQv) + gqm[:, :M]}


def stage_bounds(tab: Tables, out):
    """(DEPTH[name] M + C_OPS) u |T| |x| for every stage gradient of reverse_stages()['out']."""
    return {k: (DEPTH[k] * tab.M + C_OPS) * U * mag.astype(np.float64) for k, (_, mag) in out.items()}


def transposed_system(tab: Tables, K):
    """C' [B][4M][4M] in float64, node-major as system(): c'_ij = delta_ij + (0, fl(fl(1/2 S_ji) K_j)), the entries
    rounded exactly as the kernels form them."""
    return quaternion_operator(0.5 * tab.S.T, K)


def stage1_grads(qn, lam, gq, Dn_IN):
    """K-grad [B][3][N] (zero at the base node) and q0-grad [B][4] from lam [B][M][4], in long double."""
    B, N = qn.shape[0], qn.shape[1]
    gK = np.zeros((B, N, 3), dtype=LD)
    gK[:, :N - 1] = strain_grad(lam, qn[:, :N - 1])
    gq0 = gq[:, N - 1] - np.einsum("i,bic->bc", np.asarray(Dn_IN).astype(LD), lam)
    return _cols(gK), gq0


def norm_inf(C):
    return np.abs(C).sum(axis=2).max(axis=1)


@dataclass
class Adjoint:
    value: dict      # the eight gradients, long double, the kernels' output layouts
    bound: dict      # float64 bound on |kernel - value| per entry (0: must match exactly)
    lam: np.ndarray  # lam' [B][M][4], long double
    C: np.ndarray    # C' [B][4M][4M]
    b: np.ndarray    # b' [B][4M], long double
    cinv: np.ndarray  # ||C'^-1||_inf per rod
    E: np.ndarray    # the forward-error bound of lam' per rod
    stages: dict     # reverse_stages()


def integrate_all_vjp(tab: Tables, K, Q, n=None, q0=None, Gamma=None, gQ=None, gr=None, gn=None, gm=None, tol=1e-17):
    """Every gradient of sri_integrate_all_vjp with its bound, from the given float64 inputs (see the module docstring)."""
    K = np.asarray(K, dtype=np.float64)
    B, M = K.shape[0], tab.M
    st = reverse_stages(tab, Q, n, q0, Gamma, gQ, gr, gn, gm)
    S = tab.S
    bp = _tT(S, st["r"]).reshape(B, 4 * M)
    bpm = _tT(abs(S), st["r_mag"]).reshape(B, 4 * M).astype(np.float64)
    C = transposed_system(tab, K)
    nC = norm_inf(C)
    cinv = norm_inf(np.linalg.inv(C))
    # the reference must be far more accurate than the bound it checks: correction <= 1e-4 C_ETA u kappa
    lam = refined_solve(C, bp, steps=4, tol=np.maximum(tol, 1e-4 * C_ETA * U * nC * cinv)).reshape(B, M, 4)
    lam_inf = np.abs(lam).max(axis=(1, 2)).astype(np.float64)
    db = (2 * M + C_OPS) * U * bpm.max(axis=1)
    E = cinv * (C_ETA * U * (nC * lam_inf + np.abs(bp).max(axis=1).astype(np.float64)) + db)
    gK, gq0 = stage1_grads(st["qn"], lam, st["gq"], tab.Dn_IN)
    qabs = np.abs(st["qn"][:, :M]).sum(axis=2).astype(np.float64)                  # ||q_i||_1
    lq = (np.abs(lam).sum(axis=2) * np.abs(st["qn"][:, :M]).sum(axis=2)).astype(np.float64)
    bK = np.zeros((B, M + 1))
    bK[:, :M] = 0.5 * E[:, None] * qabs + 8 * U * 0.5 * lq                             # the base node: exactly zero
    dn = np.abs(tab.Dn_IN)
    sum_mag = st["gq_mag"][:, M].astype(np.float64) + np.einsum("i,bic->bc", dn, np.abs(lam).astype(np.float64))
    bq0 = E[:, None] * dn.sum() + (2 * M + C_OPS) * U * sum_mag
    value = {"K": gK, "q0": gq0}
    bound = {"K": np.repeat(bK[:, None, :], 3, axis=1), "q0": bq0}
    sb = stage_bounds(tab, st["out"])
    for k, (v, _) in st["out"].items():
        value[k], bound[k] = v, sb[k]
    return Adjoint(value, bound, lam, C, bp, cinv, E, st)


def excess(got, ref: Adjoint, name):
    """max over entries of |got - value| / bound per rod (<= 1 passes; a zero bound demands an exact match)."""
    err = np.abs(np.asarray(got).astype(LD) - ref.value[name]).astype(np.float64)
    bound = ref.bound[name]
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
    ratio = np.where(np.isnan(err), np.inf, ratio)
    return ratio.reshape(ratio.shape[0], -1).max(axis=1)


def pivot_order(C, quantized=False):
    """The pivot rows, step by step, of the kernels' Gauss-Jordan elimination on C' [B][4M][4M]: arg-max of |c'_ik|^2 over
    the unused rows, first row on ties; quantized=True compares the norms as vjp16_kernel does, by the high word of the
    double with its last four bits cleared (gauss_jordan16, pivot_candidate).  Float64 arithmetic: it may differ from a
    kernel's choice between rows whose norms agree to the last bits.  Returns perm [B][M]."""
    B, M = C.shape[0], C.shape[1] // 4
    c = np.ascontiguousarray(C.reshape(B, M, 4, M, 4)[:, :, :, :, 0].transpose(0, 1, 3, 2))  # c[b][i][j] = c'_ij
    used = np.zeros((B, M), dtype=bool)
    perm = np.empty((B, M), dtype=np.int64)
    rb = np.arange(B)
    for k in range(M):
        nrm = (c[:, :, k] ** 2).sum(axis=-1)
        if quantized:
            nrm = ((nrm.view(np.uint64) >> np.uint64(32)) & np.uint64(0xFFFFFFF0)).astype(np.float64)
        nrm = np.where(used, -1.0, nrm)
        p = nrm.argmax(axis=1)
        perm[:, k] = p
        used[rb, p] = True
        cp = c[rb, p].copy()                                    # [B][M][4] the pivot row
        pk = cp[:, k]
        pinv = pk * np.array([1.0, -1.0, -1.0, -1.0]) / (pk ** 2).sum(axis=-1, keepdims=True)
        m = _qmul(pinv[:, None], c[:, :, k])                     # m_i = c'_pk^-1 (x) c'_ik
        c[:, :, k + 1:] -= _qmul(cp[:, None, k + 1:], m[:, :, None])
        c[rb, p, k + 1:] = _qmul(cp[:, k + 1:], pinv[:, None])   # the pivot row, normalised
    return perm


def _qmul(a, b):
    aw, ax, ay, az = (a[..., k] for k in range(4))
    bw, bx, by, bz = (b[..., k] for k in range(4))
    return np.stack([aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx, aw * bz + ax * by - ay * bx + az * bw], axis=-1)
