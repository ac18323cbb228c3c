// sri_vjp16.cuh -- reverse-mode four-stage kernel (sri_integrate_all_vjp) for N <= 16 Chebyshev nodes.
//
// Given the forward's Q (and n) and the output cotangents gQ, gr, gn, gm of a rod, runs the stages backwards
// (DESIGN.md "Reverse mode"; oracle/adjoint.py restates it in numpy):
//   stage 4  nu = S_T^T gm      lbar-grad = -nu, M_tip-grad = -D_TI^T nu, g_b += -n x nu, gn += b x nu
//   stage 3  xi = S_T^T gn      fbar-grad = -xi, F_tip-grad = -D_TI^T xi
//   stage 2  mu = S^T gr        g_b += mu, r0-grad = -Dn_IN^T mu
//   b = R(q) Gamma              Gamma-grad = R^T g_b, gq = d/dq (g_b^T R(q) Gamma)  (-> gQ; base node -> q0-grad)
//   stage 1  A_NN(K)^T lam = gQ, K-grad[c][i] = 1/2 <lam_i, Q_i (x) (0,e_c)>, q0-grad += -Dn_IN^T lam
// with S = Dn_NN^-1, S_T = D_TT^-1.  Stage 1 preconditioned by S^T is again a quaternion system of the forward's form,
//   sum_j lam_j (x) c'_ij = (S^T gQ)_i,   c'_ij = delta_ij + 1/2 S_ji (0, K_j),
// i.e. the forward elimination with the S table read transposed and the sign of K flipped; it runs through the same
// register-resident Gauss-Jordan with row pivoting (gauss_jordan16, sri_fused16.cuh).
//
// Mapping as in sri_fused16.cuh: TWO rods per warp, lane `row` of a half-warp owns row `row` of its rod (node `row` for
// the nodal quantities, reduced row `row` = node row+1 for the stage 3/4 quantities).
#pragma once
#include "sri_device.cuh"
#include "sri_fused16.cuh"  // MP16, gauss_jordan16, contract16, kFusedThreads, kFusedMinBlocks

namespace sri {

// Arguments of the reverse-mode kernels (device pointers; optional inputs / cotangents NULL = default / zero, gradient
// outputs NULL = not wanted).  Every wanted gradient is written, not accumulated.
struct VjpParams {
    long long batch;
    int N, M;
    const double* S_rm;   // Dn_NN^-1, row-major [M][M]: S_rm[j*M+i] = S(j,i), i.e. row i of S^T read with stride M
    const double* ST_rm;  // D_TT^-1, row-major [M][M]
    const double* DTI;    // D_TI [M]
    const double* DnIN;   // Dn_IN [M]
    const double* K;
    const double* q0;
    const double* Gamma;
    const double* Q;      // forward output [batch][4][M] (required)
    const double* n;      // forward output [batch][3][M] (required when gm is given)
    const double* gQ;
    const double* gr;
    const double* gn;
    const double* gm;
    double* gK;
    double* gq0;
    double* gr0;
    double* gGamma;
    double* gfbar;
    double* glbar;
    double* gF_tip;
    double* gM_tip;
    int* info;
};

// Transposed operator tables of the N <= 16 kernel (doubles, stride MP16, zero padded), filled from S_rm / ST_rm per CTA.
struct VjpTables16 {
    static constexpr int St = 0;                   // [15][16] St[j*16+i]  = S(j,i)    (contract16 -> S^T v)
    static constexpr int STt = St + 15 * MP16;     // [15][16] STt[j*16+i] = S_T(j,i)  (contract16 -> S_T^T v)
    static constexpr int DTI = STt + 15 * MP16;    // [16]
    static constexpr int DnIN = DTI + MP16;        // [16]
    static constexpr int total = DnIN + MP16;      // 512 doubles
};

// Per-rod shared scratch (doubles).
struct VjpScratch16 {
    static constexpr int kbuf = 0;              // [3][16] strain samples
    static constexpr int bvec = kbuf + 48;      // [16][4] b_i = R(q_i) Gamma_i by node; later q_i (kept across the solve)
    static constexpr int vec = bvec + 64;       // [16][4] right-hand side of the current contraction
    static constexpr int lam = vec + 64;        // [16][4] lambda by column
    static constexpr int pbuf = lam + 64;       // [2][16][4] pivot-row publish buffers of gauss_jordan16
    static constexpr int total = pbuf + 128;    // 368 doubles
};

// sum over the 16 lanes of a half-warp
__device__ __forceinline__ double segment_sum16(double v) {
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// d/dq of a^T R(q) g for Eigen's un-normalised toRotationMatrix:
// R g = g + 2w (v x g) + 2 v x (v x g), v = (x,y,z)  =>  d/dw = 2 a.(v x g),
// d/dv = 2w (g x a) + 2 (a.v) g + 2 (v.g) a - 4 (a.g) v.
__device__ __forceinline__ quat rotation_vjp(const quat& q, double g0, double g1, double g2, double a0, double a1, double a2) {
    const double vg0 = q.y * g2 - q.z * g1, vg1 = q.z * g0 - q.x * g2, vg2 = q.x * g1 - q.y * g0;  // v x g
    const double av = a0 * q.x + a1 * q.y + a2 * q.z, vgd = q.x * g0 + q.y * g1 + q.z * g2, ag = a0 * g0 + a1 * g1 + a2 * g2;
    quat r;
    r.w = 2.0 * (a0 * vg0 + a1 * vg1 + a2 * vg2);
    r.x = 2.0 * (q.w * (g1 * a2 - g2 * a1) + av * g0 + vgd * a0) - 4.0 * ag * q.x;
    r.y = 2.0 * (q.w * (g2 * a0 - g0 * a2) + av * g1 + vgd * a1) - 4.0 * ag * q.y;
    r.z = 2.0 * (q.w * (g0 * a1 - g1 * a0) + av * g2 + vgd * a2) - 4.0 * ag * q.z;
    return r;
}

// 1/2 <lam, q (x) (0, e_c)>, c = 0..2: the K-gradient of one node (A(e_c) q = q (x) (0, e_c), updateA main.cpp:72-75)
__device__ __forceinline__ void strain_grad(const quat& l, const quat& q, double& k0, double& k1, double& k2) {
    k0 = 0.5 * ((l.x * q.w - l.w * q.x) + (l.y * q.z - l.z * q.y));
    k1 = 0.5 * ((l.y * q.w - l.w * q.y) + (l.z * q.x - l.x * q.z));
    k2 = 0.5 * ((l.z * q.w - l.w * q.z) + (l.x * q.y - l.y * q.x));
}

// out = sum_j T[j*16+row] v[j] over four components (the quaternion right-hand side of stage 1)
template <int MS>
__device__ __forceinline__ quat contract16_quat(const double* T, const double* v, int M, int row) {
    quat a; a.w = 0.0; a.x = 0.0; a.y = 0.0; a.z = 0.0;
    quat e = a;
#pragma unroll
    for (int j = 0; j < 15; ++j) {
        if (MS == 0 && j >= M) break;
        const double t = T[j * MP16 + row];
        const quat u = ld_quat(v + 4 * j);
        quat& s = (j & 1) ? e : a;
        s.w = fma(t, u.w, s.w); s.x = fma(t, u.x, s.x); s.y = fma(t, u.y, s.y); s.z = fma(t, u.z, s.z);
    }
    a.w += e.w; a.x += e.x; a.y += e.y; a.z += e.z;
    return a;
}

template <int MS>
__global__ void __launch_bounds__(kFusedThreads, kFusedMinBlocks) vjp16_kernel(const VjpParams p) {
    extern __shared__ __align__(16) double smem[];
    double* tab = smem;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sub = lane >> 4, row = lane & 15;
    double* scr = smem + VjpTables16::total + (warp * 2 + sub) * VjpScratch16::total;
    double* kbuf = scr + VjpScratch16::kbuf;
    double* bvec = scr + VjpScratch16::bvec;
    double* vec = scr + VjpScratch16::vec;
    double* lamb = scr + VjpScratch16::lam;
    const int M = MS ? MS : p.M;
    const int N = M + 1;

    const long long pairs = (p.batch + 1) >> 1;
    if ((long long)blockIdx.x * (blockDim.x >> 5) >= pairs) return;
    for (int t = threadIdx.x; t < VjpTables16::total; t += blockDim.x) {
        double v = 0.0;
        if (t < VjpTables16::DTI) {
            const int r = t % (15 * MP16), j = r / MP16, i = r % MP16;
            if (i < M && j < M) v = (t < VjpTables16::STt ? p.S_rm : p.ST_rm)[j * M + i];
        } else {
            const int i = (t - VjpTables16::DTI) % MP16;
            if (i < M) v = (t < VjpTables16::DnIN ? p.DTI : p.DnIN)[i];
        }
        tab[t] = v;
    }
    __syncthreads();
    const bool want_solve = p.gK || p.gq0;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);

    for (long long pair = (long long)blockIdx.x * (blockDim.x >> 5) + warp; pair < pairs; pair += warps_total) {
        const long long rod = 2 * pair + sub;
        const bool live = rod < p.batch;
        const bool rrow = live && row < M;  // a reduced row / stage-1 row of a live rod

        // ---- inputs: q at node `row` (base node: q0), Gamma at node `row`, strain samples -------------------------
        quat q0; q0.w = 1.0; q0.x = 0.0; q0.y = 0.0; q0.z = 0.0;
        if (live && p.q0) { const double* s = p.q0 + rod * 4; q0.w = s[0]; q0.x = s[1]; q0.y = s[2]; q0.z = s[3]; }
        quat q = q0;
        if (rrow) { const double* s = p.Q + rod * 4 * M + row; q.w = s[0]; q.x = s[M]; q.y = s[2 * M]; q.z = s[3 * M]; }
        double G0 = 1.0, G1 = 0.0, G2 = 0.0;
        if (live && p.Gamma && row < N) { const double* s = p.Gamma + rod * 3 * N + row; G0 = s[0]; G1 = s[N]; G2 = s[2 * N]; }
        {
            double k0 = 0.0, k1 = 0.0, k2 = 0.0;
            if (live && row < N) { const double* s = p.K + rod * 3 * N + row; k0 = s[0]; k1 = s[N]; k2 = s[2 * N]; }
            kbuf[row] = k0; kbuf[16 + row] = k1; kbuf[32 + row] = k2;
        }
        double b0, b1, b2;
        q_rotate(q, G0, G1, G2, b0, b1, b2);
        { quat t; t.w = b0; t.x = b1; t.y = b2; t.z = 0.0; st_quat(bvec + 4 * row, t); }

        // cotangent of n at this reduced row, completed by stage 4
        double gn0 = 0.0, gn1 = 0.0, gn2 = 0.0;
        if (rrow && p.gn) { const double* s = p.gn + rod * 3 * M + row; gn0 = s[0]; gn1 = s[M]; gn2 = s[2 * M]; }
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;  // g_b at node `row`

        // ---- stage 4: nu = S_T^T gm ------------------------------------------------------------------------------
        double nu0 = 0.0, nu1 = 0.0, nu2 = 0.0;
        if (p.gm) {
            { quat t; t.w = 0.0; t.x = 0.0; t.y = 0.0; t.z = 0.0;
              if (rrow) { const double* s = p.gm + rod * 3 * M + row; t.w = s[0]; t.x = s[M]; t.y = s[2 * M]; }
              st_quat(vec + 4 * row, t); }
            __syncwarp();
            contract16<MS>(tab + VjpTables16::STt, vec, M, row, nu0, nu1, nu2);
            if (row >= M) { nu0 = 0.0; nu1 = 0.0; nu2 = 0.0; }
            double n0 = 0.0, n1 = 0.0, n2 = 0.0;
            if (rrow) { const double* s = p.n + rod * 3 * M + row; n0 = s[0]; n1 = s[M]; n2 = s[2 * M]; }
            const quat bb = ld_quat(bvec + 4 * (row < M ? row + 1 : row));  // b at node row+1
            // g_b at node row+1 += -(n x nu): computed by reduced row `row`, moved one lane up
            const double c0 = -(n1 * nu2 - n2 * nu1), c1 = -(n2 * nu0 - n0 * nu2), c2 = -(n0 * nu1 - n1 * nu0);
            a0 = __shfl_up_sync(0xffffffffu, c0, 1, 16);
            a1 = __shfl_up_sync(0xffffffffu, c1, 1, 16);
            a2 = __shfl_up_sync(0xffffffffu, c2, 1, 16);
            if (row == 0) { a0 = 0.0; a1 = 0.0; a2 = 0.0; }
            gn0 += bb.x * nu2 - bb.y * nu1; gn1 += bb.y * nu0 - bb.w * nu2; gn2 += bb.w * nu1 - bb.x * nu0;
        }
        if (live && p.glbar) {
            double* d = p.glbar + rod * 3 * N;
            if (row < M) { d[row + 1] = -nu0; d[N + row + 1] = -nu1; d[2 * N + row + 1] = -nu2; }
            if (row == 0) { d[0] = 0.0; d[N] = 0.0; d[2 * N] = 0.0; }
        }
        if (p.gM_tip) {
            const double dti = tab[VjpTables16::DTI + row];
            const double s0 = segment_sum16(-dti * nu0), s1 = segment_sum16(-dti * nu1), s2 = segment_sum16(-dti * nu2);
            if (live && row == 0) { double* d = p.gM_tip + rod * 3; d[0] = s0; d[1] = s1; d[2] = s2; }
        }

        // ---- stage 3: xi = S_T^T gn --------------------------------------------------------------------------------
        if (p.gfbar || p.gF_tip) {
            __syncwarp();  // vec has been read by every lane
            { quat t; t.w = gn0; t.x = gn1; t.y = gn2; t.z = 0.0; st_quat(vec + 4 * row, t); }
            __syncwarp();
            double x0, x1, x2;
            contract16<MS>(tab + VjpTables16::STt, vec, M, row, x0, x1, x2);
            if (row >= M) { x0 = 0.0; x1 = 0.0; x2 = 0.0; }
            if (live && p.gfbar) {
                double* d = p.gfbar + rod * 3 * N;
                if (row < M) { d[row + 1] = -x0; d[N + row + 1] = -x1; d[2 * N + row + 1] = -x2; }
                if (row == 0) { d[0] = 0.0; d[N] = 0.0; d[2 * N] = 0.0; }
            }
            if (p.gF_tip) {
                const double dti = tab[VjpTables16::DTI + row];
                const double s0 = segment_sum16(-dti * x0), s1 = segment_sum16(-dti * x1), s2 = segment_sum16(-dti * x2);
                if (live && row == 0) { double* d = p.gF_tip + rod * 3; d[0] = s0; d[1] = s1; d[2] = s2; }
            }
        }

        // ---- stage 2: mu = S^T gr --------------------------------------------------------------------------------
        {
            double m0 = 0.0, m1 = 0.0, m2 = 0.0;
            if (p.gr) {
                __syncwarp();
                { quat t; t.w = 0.0; t.x = 0.0; t.y = 0.0; t.z = 0.0;
                  if (rrow) { const double* s = p.gr + rod * 3 * M + row; t.w = s[0]; t.x = s[M]; t.y = s[2 * M]; }
                  st_quat(vec + 4 * row, t); }
                __syncwarp();
                contract16<MS>(tab + VjpTables16::St, vec, M, row, m0, m1, m2);
                if (row >= M) { m0 = 0.0; m1 = 0.0; m2 = 0.0; }
                a0 += m0; a1 += m1; a2 += m2;
            }
            if (p.gr0) {
                const double dnin = tab[VjpTables16::DnIN + row];
                const double s0 = segment_sum16(-dnin * m0), s1 = segment_sum16(-dnin * m1), s2 = segment_sum16(-dnin * m2);
                if (live && row == 0) { double* d = p.gr0 + rod * 3; d[0] = s0; d[1] = s1; d[2] = s2; }
            }
        }

        // ---- b = R(q) Gamma: Gamma-gradient and the rotation's share of gQ / q0-grad -----------------------------
        if (live && p.gGamma && row < N) {
            double o0, o1, o2;
            q_rotate_T(q, a0, a1, a2, o0, o1, o2);
            double* d = p.gGamma + rod * 3 * N + row;
            d[0] = o0; d[N] = o1; d[2 * N] = o2;
        }
        if (want_solve) {
            const quat gq = rotation_vjp(q, G0, G1, G2, a0, a1, a2);
            quat rhs; rhs.w = 0.0; rhs.x = 0.0; rhs.y = 0.0; rhs.z = 0.0;
            if (rrow) {
                rhs = gq;
                if (p.gQ) {
                    const double* s = p.gQ + rod * 4 * M + row;
                    rhs.w += s[0]; rhs.x += s[M]; rhs.y += s[2 * M]; rhs.z += s[3 * M];
                }
            }
            // the base node's share goes to q0; lane M keeps it in its lam slot 15 (never a column: mycol < M <= 15)
            __syncwarp();
            st_quat(vec + 4 * row, rhs);
            st_quat(bvec + 4 * row, q);
            if (row == M) st_quat(lamb + 4 * 15, gq);
            __syncwarp();

            // ---- stage 1: sum_j lam_j (x) c'_ij = (S^T gQ)_i, c'_ij = delta_ij + 1/2 S_ji (0,K_j) ------------------
            int sing = 0;
            {
                quat b = contract16_quat<MS>(tab + VjpTables16::St, vec, M, row);
                quat c[15];
#pragma unroll
                for (int j = 0; j < 15; ++j) {
                    const double s = 0.5 * tab[VjpTables16::St + j * MP16 + row];
                    c[j].w = (j == row) ? 1.0 : 0.0;
                    c[j].x = s * kbuf[j]; c[j].y = s * kbuf[16 + j]; c[j].z = s * kbuf[32 + j];
                }
                int mycol;
                gauss_jordan16(c, b, M, row, scr + VjpScratch16::pbuf, mycol, sing);
                __syncwarp();
                if (row < M) st_quat(lamb + 4 * mycol, b);
            }
            __syncwarp();
            if (p.info && live && row == 0) p.info[rod] = sing;
            quat lam; lam.w = 0.0; lam.x = 0.0; lam.y = 0.0; lam.z = 0.0;
            if (row < M) lam = ld_quat(lamb + 4 * row);
            if (live && p.gK && row < N) {
                double k0 = 0.0, k1 = 0.0, k2 = 0.0;  // the base node's strain sample does not enter the forward
                if (row < M) strain_grad(lam, ld_quat(bvec + 4 * row), k0, k1, k2);
                double* d = p.gK + rod * 3 * N + row;
                d[0] = k0; d[N] = k1; d[2 * N] = k2;
            }
            if (p.gq0) {
                const double dnin = tab[VjpTables16::DnIN + row];
                quat v; v.w = -dnin * lam.w; v.x = -dnin * lam.x; v.y = -dnin * lam.y; v.z = -dnin * lam.z;
                if (row == M) v = ld_quat(lamb + 4 * 15);
                v.w = segment_sum16(v.w); v.x = segment_sum16(v.x); v.y = segment_sum16(v.y); v.z = segment_sum16(v.z);
                if (live && row == 0) { double* d = p.gq0 + rod * 4; d[0] = v.w; d[1] = v.x; d[2] = v.y; d[3] = v.z; }
            }
        } else if (p.info && live && row == 0) {
            p.info[rod] = 0;
        }
        __syncwarp();  // scratch is reused by the next iteration
    }
}

}  // namespace sri
