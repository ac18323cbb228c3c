// sri_vjp_tiled.cuh -- reverse-mode four-stage kernel (sri_integrate_all_vjp) for 17 <= N <= 64: one rod per CTA.
//
// The same adjoint as sri_vjp16.cuh (see there and DESIGN.md "Reverse mode"); what changes is the layout.  Thread t owns
// node t (nodal quantities) and reduced row t (node t+1, stage 3/4 quantities); the operator tables are read from global
// memory in row-major order, S_rm[j*M+t] = S(j,t), so that the threads of a warp read consecutive addresses of the same
// row j (L1-resident after the first rod of a CTA).  Stage 1 keeps the M x (M+1) quaternion system [C' | S^T gQ] in
// shared memory and eliminates it Gauss-Jordan style with row pivoting (largest |c'_ik|, first row on ties): per step one
// warp finds the pivot and its inverse, the CTA computes the multipliers m_i = c'_pk^-1 (x) c'_ik (pivot row:
// 1 - c'_pk^-1) and takes c'_ij -= c'_pj (x) m_i over the live columns, as sri_tiled.cuh does with its rows in registers.
#pragma once
#include "sri_device.cuh"
#include "sri_vjp16.cuh"  // VjpParams, rotation_vjp, strain_grad

namespace sri {

constexpr int kVjpTiledThreads = 256;

// shared memory of one CTA (doubles): [M][M+1][4] system, then the per-node vectors (64 slots each) and the int area
struct VjpTiledSmem {
    int M;
    __host__ __device__ int sys() const { return 0; }
    __host__ __device__ int kb() const { return M * (M + 1) * 4; }   // [3][64] strain samples
    __host__ __device__ int bvec() const { return kb() + 192; }      // [64][4] b_i, later q_i
    __host__ __device__ int vec() const { return bvec() + 256; }     // [64][4] contraction right-hand side / row values
    __host__ __device__ int mlt() const { return vec() + 256; }      // [64][4] multipliers of the current step
    __host__ __device__ int urow() const { return mlt() + 256; }     // [64][4] pivot row of the current step
    __host__ __device__ int misc() const { return urow() + 256; }    // [8]: pivot inverse (4), q0 gradient of the base node (4)
    __host__ __device__ int ints() const { return misc() + 8; }      // [64] perm, [64] used, prow, sing
    __host__ __device__ size_t bytes() const { return (size_t)ints() * sizeof(double) + 132 * sizeof(int); }
};

// sum over threads t < M of rowval[t] (component c of the [64][4] vector), by thread 0 in a fixed order
__device__ __forceinline__ double rows_sum(const double* v, int M, int c) {
    double s = 0.0;
    for (int t = 0; t < M; ++t) s += v[4 * t + c];
    return s;
}

__global__ void __launch_bounds__(kVjpTiledThreads) vjp_tiled_kernel(const VjpParams p) {
    extern __shared__ __align__(16) double smem[];
    const int M = p.M, N = p.N, W = M + 1;
    const VjpTiledSmem L{M};
    double* sys = smem + L.sys();
    double* kb = smem + L.kb();
    double* bvec = smem + L.bvec();
    double* vec = smem + L.vec();
    double* mlt = smem + L.mlt();
    double* urow = smem + L.urow();
    double* misc = smem + L.misc();
    int* perm = reinterpret_cast<int*>(smem + L.ints());
    int* used = perm + 64;
    int* prow_s = used + 64;
    int* sing_s = prow_s + 1;
    const int t = threadIdx.x;
    const bool want_solve = p.gK || p.gq0;

    // out = sum_j T(j, t) v[j] (T row-major [M][M]) over 3 components; the caller has synchronised v
    auto contract = [&](const double* T, const double* v, double& o0, double& o1, double& o2) {
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, e0 = 0.0, e1 = 0.0, e2 = 0.0;
        int j = 0;
        for (; j + 1 < M; j += 2) {
            const double s0 = __ldg(T + j * M + t), s1 = __ldg(T + (j + 1) * M + t);
            a0 = fma(s0, v[4 * j], a0); a1 = fma(s0, v[4 * j + 1], a1); a2 = fma(s0, v[4 * j + 2], a2);
            e0 = fma(s1, v[4 * j + 4], e0); e1 = fma(s1, v[4 * j + 5], e1); e2 = fma(s1, v[4 * j + 6], e2);
        }
        if (j < M) {
            const double s0 = __ldg(T + j * M + t);
            a0 = fma(s0, v[4 * j], a0); a1 = fma(s0, v[4 * j + 1], a1); a2 = fma(s0, v[4 * j + 2], a2);
        }
        o0 = a0 + e0; o1 = a1 + e1; o2 = a2 + e2;
    };
    auto put3 = [&](double* v, double x0, double x1, double x2) { quat q; q.w = x0; q.x = x1; q.y = x2; q.z = 0.0; st_quat(v, q); };

    for (long long rod = blockIdx.x; rod < p.batch; rod += gridDim.x) {
        const bool node = t < N, rrow = t < M;
        // ---- inputs ---------------------------------------------------------------------------------------------
        quat q0; q0.w = 1.0; q0.x = 0.0; q0.y = 0.0; q0.z = 0.0;
        if (p.q0) { const double* s = p.q0 + rod * 4; q0.w = s[0]; q0.x = s[1]; q0.y = s[2]; q0.z = s[3]; }
        quat q = q0;
        if (rrow) { const double* s = p.Q + rod * 4 * M + t; q.w = s[0]; q.x = s[M]; q.y = s[2 * M]; q.z = s[3 * M]; }
        double G0 = 1.0, G1 = 0.0, G2 = 0.0;
        if (p.Gamma && node) { const double* s = p.Gamma + rod * 3 * N + t; G0 = s[0]; G1 = s[N]; G2 = s[2 * N]; }
        if (node) {
            const double* s = p.K + rod * 3 * N + t;
            kb[t] = s[0]; kb[64 + t] = s[N]; kb[128 + t] = s[2 * N];
        }
        double b0 = 0.0, b1 = 0.0, b2 = 0.0;
        if (node) { q_rotate(q, G0, G1, G2, b0, b1, b2); put3(bvec + 4 * t, b0, b1, b2); }
        double gn0 = 0.0, gn1 = 0.0, gn2 = 0.0;
        if (rrow && p.gn) { const double* s = p.gn + rod * 3 * M + t; gn0 = s[0]; gn1 = s[M]; gn2 = s[2 * M]; }
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;  // g_b at node t

        // ---- stage 4 ------------------------------------------------------------------------------------------------
        double nu0 = 0.0, nu1 = 0.0, nu2 = 0.0;
        if (p.gm && rrow) { const double* s = p.gm + rod * 3 * M + t; put3(vec + 4 * t, s[0], s[M], s[2 * M]); }
        __syncthreads();
        if (p.gm) {
            double c0 = 0.0, c1 = 0.0, c2 = 0.0;
            if (rrow) {
                contract(p.ST_rm, vec, nu0, nu1, nu2);
                const double* s = p.n + rod * 3 * M + t;
                const double n0 = s[0], n1 = s[M], n2 = s[2 * M];
                const double* bb = bvec + 4 * (t + 1);
                c0 = -(n1 * nu2 - n2 * nu1); c1 = -(n2 * nu0 - n0 * nu2); c2 = -(n0 * nu1 - n1 * nu0);
                gn0 += bb[1] * nu2 - bb[2] * nu1; gn1 += bb[2] * nu0 - bb[0] * nu2; gn2 += bb[0] * nu1 - bb[1] * nu0;
            }
            __syncthreads();  // vec has been read
            if (rrow) put3(vec + 4 * (t + 1), c0, c1, c2);  // g_b of node t+1
            if (t == 0) put3(vec, 0.0, 0.0, 0.0);
            __syncthreads();
            if (node) { const quat v = ld_quat(vec + 4 * t); a0 = v.w; a1 = v.x; a2 = v.y; }
            __syncthreads();
        }
        if (p.glbar && node) {
            double* d = p.glbar + rod * 3 * N;
            if (rrow) { d[t + 1] = -nu0; d[N + t + 1] = -nu1; d[2 * N + t + 1] = -nu2; }
            if (t == 0) { d[0] = 0.0; d[N] = 0.0; d[2 * N] = 0.0; }
        }
        if (p.gM_tip) {
            if (rrow) { const double dt = __ldg(p.DTI + t); put3(mlt + 4 * t, -dt * nu0, -dt * nu1, -dt * nu2); }
            __syncthreads();
            if (t < 3) p.gM_tip[rod * 3 + t] = rows_sum(mlt, M, t);
            __syncthreads();
        }

        // ---- stage 3 ------------------------------------------------------------------------------------------------
        if (p.gfbar || p.gF_tip) {
            if (rrow) put3(vec + 4 * t, gn0, gn1, gn2);
            __syncthreads();
            double x0 = 0.0, x1 = 0.0, x2 = 0.0;
            if (rrow) contract(p.ST_rm, vec, x0, x1, x2);
            if (p.gfbar && node) {
                double* d = p.gfbar + rod * 3 * N;
                if (rrow) { d[t + 1] = -x0; d[N + t + 1] = -x1; d[2 * N + t + 1] = -x2; }
                if (t == 0) { d[0] = 0.0; d[N] = 0.0; d[2 * N] = 0.0; }
            }
            if (rrow) { const double dt = __ldg(p.DTI + t); put3(mlt + 4 * t, -dt * x0, -dt * x1, -dt * x2); }
            __syncthreads();
            if (p.gF_tip && t < 3) p.gF_tip[rod * 3 + t] = rows_sum(mlt, M, t);
            __syncthreads();
        }

        // ---- stage 2 ------------------------------------------------------------------------------------------------
        if (p.gr || p.gr0) {
            double m0 = 0.0, m1 = 0.0, m2 = 0.0;
            if (p.gr) {
                if (rrow) { const double* s = p.gr + rod * 3 * M + t; put3(vec + 4 * t, s[0], s[M], s[2 * M]); }
                __syncthreads();
                if (rrow) contract(p.S_rm, vec, m0, m1, m2);
                a0 += m0; a1 += m1; a2 += m2;
            }
            if (rrow) { const double dn = __ldg(p.DnIN + t); put3(mlt + 4 * t, -dn * m0, -dn * m1, -dn * m2); }
            __syncthreads();
            if (p.gr0 && t < 3) p.gr0[rod * 3 + t] = rows_sum(mlt, M, t);
            __syncthreads();
        }

        // ---- b = R(q) Gamma ------------------------------------------------------------------------------------------
        if (p.gGamma && node) {
            double o0, o1, o2;
            q_rotate_T(q, a0, a1, a2, o0, o1, o2);
            double* d = p.gGamma + rod * 3 * N + t;
            d[0] = o0; d[N] = o1; d[2 * N] = o2;
        }
        if (!want_solve) {
            if (p.info && t == 0) p.info[rod] = 0;
            continue;  // (no shared buffer is written after the last barrier)
        }
        {
            const quat gq = rotation_vjp(q, G0, G1, G2, a0, a1, a2);
            if (rrow) {
                quat rhs = gq;
                if (p.gQ) { const double* s = p.gQ + rod * 4 * M + t; rhs.w += s[0]; rhs.x += s[M]; rhs.y += s[2 * M]; rhs.z += s[3 * M]; }
                st_quat(vec + 4 * t, rhs);
            }
            if (t == M) st_quat(misc + 4, gq);
            if (node) st_quat(bvec + 4 * t, q);
            if (t < 64) used[t] = (t < M) ? 0 : 1;
            if (t == 0) *sing_s = 0;
        }
        __syncthreads();
        // ---- stage 1: assemble [C' | S^T gQ] ------------------------------------------------------------------------------
        for (int idx = t; idx < M * M; idx += blockDim.x) {
            const int i = idx % M, j = idx / M;  // consecutive threads: consecutive rows i of S(j, .)
            const double s = 0.5 * __ldg(p.S_rm + j * M + i);
            quat c; c.w = (i == j) ? 1.0 : 0.0; c.x = s * kb[j]; c.y = s * kb[64 + j]; c.z = s * kb[128 + j];
            st_quat(sys + 4 * (i * W + j), c);
        }
        if (rrow) {
            quat r; r.w = 0.0; r.x = 0.0; r.y = 0.0; r.z = 0.0;
            for (int j = 0; j < M; ++j) {
                const double s = __ldg(p.S_rm + j * M + t);
                const quat u = ld_quat(vec + 4 * j);
                r.w = fma(s, u.w, r.w); r.x = fma(s, u.x, r.x); r.y = fma(s, u.y, r.y); r.z = fma(s, u.z, r.z);
            }
            st_quat(sys + 4 * (t * W + M), r);
        }
        __syncthreads();
        // ---- Gauss-Jordan with row pivoting ---------------------------------------------------------------------------
        for (int k = 0; k < M; ++k) {
            if (t < 32) {
                double best = -1.0;
                int bi = 64;
                for (int i = t; i < M; i += 32) {
                    if (used[i]) continue;
                    const quat c = ld_quat(sys + 4 * (i * W + k));
                    double nrm = q_norm2(c);
                    if (!(nrm <= 1.0e308)) nrm = 1.0e308 * 10.0;  // Inf / NaN: chosen first, then reported below
                    if (nrm > best) { best = nrm; bi = i; }
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, off);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
                    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
                }
                if (t == 0) {
                    const quat c = ld_quat(sys + 4 * (bi * W + k));
                    const double nrm = q_norm2(c);
                    if (!(nrm > 0.0 && nrm <= 1.0e308) && *sing_s == 0) *sing_s = k + 1;  // zero or non-finite pivot
                    const double inv = 1.0 / nrm;
                    quat pinv; pinv.w = c.w * inv; pinv.x = -c.x * inv; pinv.y = -c.y * inv; pinv.z = -c.z * inv;
                    st_quat(misc, pinv);
                    *prow_s = bi;
                    perm[k] = bi;
                    used[bi] = 1;
                }
            }
            __syncthreads();
            const int pr = *prow_s;
            const quat pinv = ld_quat(misc);
            if (t < M) {
                quat mm;
                if (t == pr) { mm.w = 1.0 - pinv.w; mm.x = -pinv.x; mm.y = -pinv.y; mm.z = -pinv.z; }
                else mm = q_mul(pinv, ld_quat(sys + 4 * (t * W + k)));
                st_quat(mlt + 4 * t, mm);
            }
            for (int j = k + 1 + t; j <= M; j += blockDim.x) st_quat(urow + 4 * j, ld_quat(sys + 4 * (pr * W + j)));
            __syncthreads();
            const int live_cols = M - k;  // columns k+1 .. M
            for (int idx = t; idx < M * live_cols; idx += blockDim.x) {
                const int j = k + 1 + idx % live_cols, i = idx / live_cols;
                quat c = ld_quat(sys + 4 * (i * W + j));
                q_sub_mul(c, ld_quat(urow + 4 * j), ld_quat(mlt + 4 * i));
                st_quat(sys + 4 * (i * W + j), c);
            }
            __syncthreads();
        }
        // ---- epilogue: lam_k = rhs of the row that pivoted in step k ----------------------------------------------------
        quat lam; lam.w = 0.0; lam.x = 0.0; lam.y = 0.0; lam.z = 0.0;
        if (rrow) lam = ld_quat(sys + 4 * (perm[t] * W + M));
        if (p.info && t == 0) p.info[rod] = *sing_s;
        if (p.gK && node) {
            double k0 = 0.0, k1 = 0.0, k2 = 0.0;  // the base node's strain sample does not enter the forward
            if (rrow) strain_grad(lam, ld_quat(bvec + 4 * t), k0, k1, k2);
            double* d = p.gK + rod * 3 * N + t;
            d[0] = k0; d[N] = k1; d[2 * N] = k2;
        }
        if (p.gq0) {
            if (rrow) { const double dn = -__ldg(p.DnIN + t); quat v; v.w = dn * lam.w; v.x = dn * lam.x; v.y = dn * lam.y; v.z = dn * lam.z; st_quat(mlt + 4 * t, v); }
            __syncthreads();
            if (t < 4) {
                double s = misc[4 + t];
                for (int i = 0; i < M; ++i) s += mlt[4 * i + t];
                p.gq0[rod * 4 + t] = s;
            }
        }
        __syncthreads();  // shared buffers are reused by the next rod
    }
}

}  // namespace sri
