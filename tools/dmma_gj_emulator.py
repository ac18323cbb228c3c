"""Lane-exact numpy emulation of the DMMA Gauss-Jordan of csrc/sri_fused16_dmma.cuh (stage 1, one rod per warp).

Purpose: the CUDA kernel's index algebra (which lane holds which entry, every shuffle source, every sign) is
checked HERE, on the CPU, against the oracle, before any GPU time is spent.  Registers are arrays over the 32
lanes; `shfl` and `mma_m8n8k4` follow the PTX fragment layouts
    A (8x4, row):  lane l holds A[l>>2][l&3]
    B (4x8, col):  lane l holds B[l&3][l>>2]
    C (8x8):       lane l holds C[l>>2][2*(l&3) + e], e = 0, 1.

Real layout of the M x M quaternion system  sum_j Q_j (x) c_ij = b_i  (DESIGN.md section 1):
    Cr[4*i + r][j] = component r of c_ij,  j = 0..14;  Cr[4*i + r][15] = component r of b_i
16 tiles of 8 x 8: tile (t, ct) = rows 8t..8t+7 (quaternion rows 2t, 2t+1), columns 8ct..8ct+7.

Step k (static pivot order, growth check instead of a search):
    u'_j  = u_j (x) c_kk^-1                 (pivot row normalised: one DMMA per column tile)
    c_ij -= u'_j (x) c_ik   for all rows i  (vec(a (x) b) = Rmat(b) vec(a): [Rmat(c_ik) stacked] * [-U'] : DMMAs)
    pivot row itself: Rmat(c_kk - 1), which leaves exactly u'_j.
`solve_rod` is that Gauss-Jordan over all rows; `solve_rod_lu` is the schedule the kernel runs: the same steps on the
rows below the pivot only, then a back-substitution on DMMA.
"""
from __future__ import annotations

import numpy as np

LANES = np.arange(32)
RHO, CP = LANES >> 2, LANES & 3
HI, R = RHO >> 2, RHO & 3

# Rmat(b)[r][s] = SG[r][s] * b[r ^ s]   (vec(a (x) b) = Rmat(b) vec(a), components w, x, y, z)
SG = np.array([[1, -1, -1, -1], [1, 1, 1, -1], [1, -1, 1, 1], [1, 1, -1, 1]], dtype=np.float64)


def shfl(v, src):
    return v[src]


def mma_m8n8k4(c0, c1, a, b):
    A = np.zeros((8, 4)); B = np.zeros((4, 8)); C = np.zeros((8, 8))
    A[RHO, CP] = a
    B[CP, RHO] = b
    C[RHO, 2 * CP] = c0
    C[RHO, 2 * CP + 1] = c1
    D = C.copy()
    for q in range(4):  # sequential FMA chain over k, as the hardware accumulates
        D = D + np.outer(A[:, q], B[q, :])
    return D[RHO, 2 * CP], D[RHO, 2 * CP + 1]


def tables(S, g, M):
    """Stx[16][16]: -1/2 S_ij (i, j < M), column 15 = g_i, zero elsewhere."""
    Stx = np.zeros((16, 16))
    Stx[:M, :M] = -0.5 * S
    Stx[:M, 15] = g
    return Stx


def solve_rod(Stx, K, q0, M, growth=8.0):
    """K: [3][N]; returns (Q [M][4], flagged)."""
    kx = np.zeros((4, 16))
    kx[1:, :M] = K[:, :M]
    kx[:, 15] = q0
    # ---- assembly -------------------------------------------------------------------------------------------
    c = np.zeros((8, 2, 2, 32))
    for t in range(8):
        for ct in range(2):
            for e in range(2):
                i = 2 * t + HI
                j = 8 * ct + 2 * CP + e
                diag = ((R == 0) & (i == j) & (j < 15)).astype(np.float64)
                c[t, ct, e] = Stx[i, j] * kx[R, j] + diag
    flagged = False
    # lane constants
    sgL = SG[R, CP]
    srcL_base = 16 * (LANES >> 4) + 4 * (R ^ CP)
    n_even = (RHO & 1) == 0
    sp = RHO >> 1  # s' of the normalisation operand (even output columns only)
    idxN = sp ^ CP
    conj = np.where(idxN == 0, 1.0, -1.0)
    sgN = np.where(n_even, -SG[sp, CP] * conj, 0.0)
    for k in range(M):
        kt, kh, kc, kcp, ke = k >> 1, k & 1, k >> 3, (k & 7) >> 1, k & 1
        cts = [ct for ct in range(2) if 8 * ct + 7 > k]  # column tiles with live columns (j > k), rhs included
        # 1. pivot row -> B fragments
        src = 16 * kh + 4 * CP + (LANES >> 3)
        Ub = {}
        for ct in range(kc, 2):  # the pivot column's tile is needed for c_kk even when it has no live column left
            v0 = shfl(c[kt, ct, 0], src)
            v1 = shfl(c[kt, ct, 1], src)
            Ub[ct] = np.where((RHO & 1) == 1, v1, v0)
        # 2. this lane's entry of -Rmat(conj c_kk), straight from the pivot's tile; un0 = -U (x) conj(c_kk) by DMMA;
        #    its (column k, w) entry is -|c_kk|^2
        pcs = shfl(c[kt, kc, ke], 16 * kh + 4 * idxN + kcp)
        bn0 = sgN * pcs
        un0 = {ct: mma_m8n8k4(np.zeros(32), np.zeros(32), Ub[ct], bn0)[0] for ct in Ub}
        nu = -shfl(un0[kc], np.full(32, 4 * (k & 7)))
        nrm = nu
        inv = 1.0 / nu
        # 3. L fragments (column k of every row tile), before anything is updated
        srcL = srcL_base + kcp
        La = []
        colmax = np.zeros(32)
        for t in range(8):
            v = shfl(c[t, kc, ke], srcL)
            if t > kt:
                colmax = np.maximum(colmax, np.abs(v))
            elif t == kt:
                colmax = np.maximum(colmax, np.where(HI > kh, np.abs(v), 0.0))
            a = sgL * v
            if t == kt:
                a = a - ((HI == kh) & (R == CP)).astype(np.float64)
            La.append(a)
        if not (colmax.max() ** 2 <= growth * growth * nrm[0]) or not (nrm[0] > 1e-300):
            flagged = True
        # 4. normalise the pivot row (negated), 5. update
        for ct in cts:
            d0 = un0[ct] * inv
            for t in range(8):
                c[t, ct, 0], c[t, ct, 1] = mma_m8n8k4(c[t, ct, 0], c[t, ct, 1], La[t], d0)
    Q = np.zeros((16, 4))
    for t in range(8):
        sel = CP == 3
        Q[2 * t + HI[sel], R[sel]] = c[t, 1, 1][sel]
    return Q[:M], flagged


# ---- the shipped schedule: elimination below the pivot only, back-substitution with the solved quaternion as A -------
# Lmat(a)[r][s] = SGL[r][s] * a[r ^ s]   (vec(a (x) b) = Lmat(a) vec(b))
SGL = np.array([[1, -1, -1, -1], [1, 1, -1, 1], [1, 1, 1, -1], [1, -1, 1, 1]], dtype=np.float64)
STAGE_DMMAS = 16  # stages 2-4 of the kernel: two [16 x 16] x [16 x 3] contractions, 2 row tiles x 4 k steps each


def w_col(j):
    """Start of column j of the per-warp store of -U' ([col j][row i][s], doubles).  Column j < 8 is only written by
    steps k <= 6 and read for rows i < j: 7 rows, in the 92-double slot of column j + 8 (16 rows).  The slot stride is
    12 mod 16, so the eight columns of one B fragment start on distinct bank quads (conflict-free stores)."""
    j = np.asarray(j)
    return np.where(j < 8, 92 * j + 64, 92 * (j - 8))


W_DOUBLES = 740


def solve_rod_lu(Stx, K, q0, M, growth=8.0, stats=None):
    """Same system and same pivot order as solve_rod, on the kernel's schedule:
    forward  step k updates only tile rows t >= (k+1)//2 (rows at or above a stored pivot row are dead); the
             last step updates nothing; -U'_k (B-fragment layout: lane holds component CP of column 8ct+RHO) is
             stored to W[w_col(8ct+RHO) + 4k + CP].
    backward with C' = -Q accumulated in one C tile per 8-row block (C'[s][n] = row 8b+n, component s; m >= 4 zero):
             -Q_i = W_i,15 + sum_{j>i} Lmat(-Q_j) W_ij, j = M-1..0; A = Lmat(C'_j) by one shuffle and a sign,
             B = W column j over the block (one contiguous 32-double read).
    Returns (Q [M][4], flagged); `stats` (dict) collects the DMMA count per kind."""
    st = stats if stats is not None else {}
    for key in ("update", "normalise", "backsub"):
        st.setdefault(key, 0)
    kx = np.zeros((4, 16))
    kx[1:, :M] = K[:, :M]
    kx[:, 15] = q0
    c = np.zeros((8, 2, 2, 32))
    for t in range(8):
        for ct in range(2):
            for e in range(2):
                i = 2 * t + HI
                j = 8 * ct + 2 * CP + e
                diag = ((R == 0) & (i == j) & (j < 15)).astype(np.float64)
                c[t, ct, e] = Stx[i, j] * kx[R, j] + diag
    W = np.full(W_DOUBLES, np.nan)  # rows never written must never reach a live result
    flagged = False
    sgL = SG[R, CP]
    srcL_base = 16 * (LANES >> 4) + 4 * (R ^ CP)
    n_even = (RHO & 1) == 0
    sp = RHO >> 1
    idxN = sp ^ CP
    conj = np.where(idxN == 0, 1.0, -1.0)
    sgN = np.where(n_even, -SG[sp, CP] * conj, 0.0)
    for k in range(M):
        kt, kh, kc, kcp, ke = k >> 1, k & 1, k >> 3, (k & 7) >> 1, k & 1
        cts = [ct for ct in range(2) if 8 * ct + 7 > k]
        t0 = (k + 1) >> 1  # first live tile row: kt itself only while the row below the pivot (2kt + 1) shares it
        src = 16 * kh + 4 * CP + (LANES >> 3)
        Ub = {}
        for ct in range(kc, 2):
            v0 = shfl(c[kt, ct, 0], src)
            v1 = shfl(c[kt, ct, 1], src)
            Ub[ct] = np.where((RHO & 1) == 1, v1, v0)
        pcs = shfl(c[kt, kc, ke], 16 * kh + 4 * idxN + kcp)
        bn0 = sgN * pcs
        un0 = {ct: mma_m8n8k4(np.zeros(32), np.zeros(32), Ub[ct], bn0)[0] for ct in Ub}
        st["normalise"] += len(Ub)
        nu = -shfl(un0[kc], np.full(32, 4 * (k & 7)))
        inv = 1.0 / nu
        srcL = srcL_base + kcp
        La = {}
        colmax = np.zeros(32)
        for t in range(t0, 8):
            v = shfl(c[t, kc, ke], srcL)
            if t > kt:
                colmax = np.maximum(colmax, np.abs(v))
            else:  # t == kt, kh == 0: the row below the pivot in the same tile
                colmax = np.maximum(colmax, np.where(HI > kh, np.abs(v), 0.0))
            a = sgL * v
            if t == kt:
                a = a - ((HI == kh) & (R == CP)).astype(np.float64)
            La[t] = a
        if not (colmax.max() ** 2 <= growth * growth * nu[0]) or not (nu[0] > 1e-300):
            flagged = True
        for ct in cts:
            d0 = un0[ct] * inv
            W[w_col(8 * ct + RHO) + 4 * k + CP] = d0
            if k < M - 1:
                for t in range(t0, 8):
                    c[t, ct, 0], c[t, ct, 1] = mma_m8n8k4(c[t, ct, 0], c[t, ct, 1], La[t], d0)
                    st["update"] += 1
    # ---- back-substitution --------------------------------------------------------------------------------------
    sgLm = SGL[RHO & 3, CP]
    y = {}
    for b in range(2):
        y[b] = [np.where(RHO < 4, W[w_col(15) + 4 * (8 * b + 2 * CP + e) + (RHO & 3)], 0.0) for e in range(2)]
    Q = np.zeros((16, 4))
    for j in range(M - 1, -1, -1):
        b, n = j >> 3, j & 7
        v = shfl(y[b][n & 1], 4 * (RHO ^ CP) + (n >> 1))  # lane (rho, cp) gets C'_j[rho ^ cp]; rho >= 4: zero rows
        sel = (CP == 0) & (RHO < 4)
        Q[j, RHO[sel]] = -v[sel]
        a = sgLm * v
        for bb in range(b + 1):
            if 8 * bb < j:  # blocks holding a row i < j
                y[bb][0], y[bb][1] = mma_m8n8k4(y[bb][0], y[bb][1], a, W[w_col(j) + 32 * bb + LANES])
                st["backsub"] += 1
    return Q[:M], flagged


def main():
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
    from oracle.oracle import Oracle

    rng = np.random.default_rng(7)
    for N in (16, 9, 4):
        M = N - 1
        orc = Oracle(N)
        S = orc.operator(3)
        Dn_IN = orc.operator(2)
        g = -S @ Dn_IN
        Stx = tables(S, g, M)
        B = 6
        x = orc.chebyshev_points()
        al, be = rng.uniform(-2, 2, (B, 3, 1)), rng.uniform(-2, 2, (B, 3, 1))
        K = al + be * (2 * x[None, None, :] - 1)
        q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
        ref = orc.integrate_all(K, q0=q0, want=("Q",))["Q"]
        worst = 0.0
        for b in range(B):
            Q, flagged = solve_rod(Stx, K[b], q0[b], M)
            err = np.abs(Q.T - ref[b]).max() / np.abs(ref[b]).max()
            worst = max(worst, err)
            assert not flagged
        print(f"N={N}: max rel err vs oracle {worst:.2e}")
        assert worst < 1e-12
    # large curvature: the growth check must fire for some rods
    orc = Oracle(16); S = orc.operator(3); g = -S @ orc.operator(2); Stx = tables(S, g, 15)
    x = orc.chebyshev_points()
    nflag = 0; worst = 0.0
    for b in range(20):
        K = rng.uniform(-70, 70, (3, 1)) + rng.uniform(-30, 30, (3, 1)) * (2 * x[None, :] - 1)
        q0 = np.array([1.0, 0, 0, 0])
        ref = orc.integrate_all(K[None], q0=q0[None], want=("Q",))["Q"][0]
        Q, flagged = solve_rod(Stx, K, q0, 15)
        nflag += flagged
        if not flagged:
            worst = max(worst, np.abs(Q.T - ref).max() / np.abs(ref).max())
    print(f"|K|<=70: {nflag}/20 rods flagged for the pivoting kernel; worst unflagged rel err {worst:.2e}")


if __name__ == "__main__":
    main()
