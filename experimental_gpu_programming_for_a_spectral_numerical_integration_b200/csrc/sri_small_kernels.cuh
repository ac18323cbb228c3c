// sri_small_kernels.cuh -- the kernels around the integration path: modal strain adapter and its cached Legendre table,
// shape residual / Galerkin residual / projection, local-frame wrench (pointwise), Newton driver helpers, the batched
// small solve, the synthetic benchmark rods and the two FP64 peak probes.  All HBM- or latency-bound and small; the
// integration kernels themselves live in sri_fused16*.cuh, sri_tiled*.cuh, sri_stage_*.cuh and sri_wrench_solve.cuh.
// Included by sri_api.cu only (anonymous namespace: one translation unit).
#pragma once
#include <cstdint>

#include "sri_device.cuh"
#include "sri_stage_dmma.cuh"  // dmma_m8n8k4
#include "sri_wrench_solve.cuh"  // quat_to_rot_rm

namespace {

// ---- small kernels ---------------------------------------------------------------------------------------------

// K[b][c][i] = sum_k P_k(t_i) qe[b][c*ne+k]   (Phi<3,ne>(x_i)*qe, main.cpp:69; Legendre recurrence of utilities.h:59)
__global__ void strain_from_modes_kernel(long long batch, int N, int ne, const double* __restrict__ tnodes,
                                         const double* __restrict__ qe, double* __restrict__ K, const int* __restrict__ skip) {
    if (skip && *skip) return;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = batch * 3 * N;
    if (idx >= total) return;
    const int i = (int)(idx % N);
    const long long bc = idx / N;  // b*3 + c
    const double t = tnodes[i];
    const double* q = qe + bc * ne;
    double pm = 1.0, p = t, acc = q[0];
    if (ne > 1) acc = fma(p, q[1], acc);
    for (int k = 1; k + 1 < ne; ++k) {
        const double pn = ((2 * k + 1) * t * p - k * pm) / (k + 1);
        pm = p;
        p = pn;
        acc = fma(p, q[k + 1], acc);
    }
    K[idx] = acc;
}

// P_k(t_i), k < 8, by the recurrence of utilities.h:59 -- once per handle; [k][N]
__global__ void legendre_table_kernel(int N, const double* __restrict__ tnodes, double* __restrict__ ptab) {
    const int i = threadIdx.x;
    if (i >= N) return;
    const double t = tnodes[i];
    double pm = 1.0, p = t;
    ptab[i] = 1.0;
    ptab[N + i] = t;
    for (int k = 1; k + 1 < 8; ++k) {
        const double pn = ((2 * k + 1) * t * p - k * pm) / (k + 1);
        pm = p;
        p = pn;
        ptab[(k + 1) * N + i] = p;
    }
}

// strain_from_modes for ne <= 8 with the cached Legendre table: NL (a power of two >= N) lanes per (rod, component), no
// integer division, no recurrence; same order of the additions as strain_from_modes_kernel.
template <int NL>
__global__ void __launch_bounds__(256) strain_from_modes_table_kernel(long long rows /* batch*3 */, int N, int ne,
                                                                      const double* __restrict__ ptab,
                                                                      const double* __restrict__ qe, double* __restrict__ K,
                                                                      const int* __restrict__ skip) {
    if (skip && *skip) return;
    const int i = threadIdx.x & (NL - 1);
    const long long bc = (long long)blockIdx.x * (256 / NL) + (threadIdx.x / NL);
    if (bc >= rows || i >= N) return;
    const double* q = qe + bc * ne;
    double acc = q[0];
    for (int k = 1; k < ne; ++k) acc = fma(ptab[k * N + i], q[k], acc);
    K[bc * N + i] = acc;
}

// rho = H (K - K0) - R(q)^T m at all N nodes; block-reduced sum(rho^2) and max|rho| via atomics.
__global__ void shape_residual_kernel(long long batch, int N, const double* __restrict__ K,
                                      const double* __restrict__ K0, double h0, double h1, double h2,
                                      const double* __restrict__ Q, const double* __restrict__ q0,
                                      const double* __restrict__ m, const double* __restrict__ M_tip,
                                      double* __restrict__ rho, double* __restrict__ red) {
    const int M = N - 1;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double s2 = 0.0, mx = 0.0;
    if (idx < batch * N) {
        const long long b = idx / N;
        const int i = (int)(idx % N);
        sri::quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
        if (i < M) {
            const double* s = Q + b * 4 * M + i;
            q.w = s[0]; q.x = s[M]; q.y = s[2 * M]; q.z = s[3 * M];
        } else if (q0) {
            const double* s = q0 + b * 4;
            q.w = s[0]; q.x = s[1]; q.y = s[2]; q.z = s[3];
        }
        double m0, m1, m2;
        if (i == 0) { const double* s = M_tip + b * 3; m0 = s[0]; m1 = s[1]; m2 = s[2]; }
        else { const double* s = m + b * 3 * M + (i - 1); m0 = s[0]; m1 = s[M]; m2 = s[2 * M]; }
        double t0, t1, t2;
        sri::q_rotate_T(q, m0, m1, m2, t0, t1, t2);
        const double* k = K + b * 3 * N + i;
        double k0 = k[0], k1 = k[N], k2 = k[2 * N];
        if (K0) { const double* z = K0 + b * 3 * N + i; k0 -= z[0]; k1 -= z[N]; k2 -= z[2 * N]; }
        const double r0 = h0 * k0 - t0, r1 = h1 * k1 - t1, r2 = h2 * k2 - t2;
        if (rho) { double* d = rho + b * 3 * N + i; d[0] = r0; d[N] = r1; d[2 * N] = r2; }
        s2 = r0 * r0 + r1 * r1 + r2 * r2;
        mx = fmax(fabs(r0), fmax(fabs(r1), fabs(r2)));
    }
    if (red) {
        for (int off = 16; off >= 1; off >>= 1) {
            s2 += __shfl_xor_sync(0xffffffffu, s2, off);
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        }
        __shared__ double sh_s[32], sh_m[32];
        const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
        if (l == 0) { sh_s[w] = s2; sh_m[w] = mx; }
        __syncthreads();
        if (w == 0) {
            const int nw = blockDim.x >> 5;
            s2 = l < nw ? sh_s[l] : 0.0;
            mx = l < nw ? sh_m[l] : 0.0;
            for (int off = 16; off >= 1; off >>= 1) {
                s2 += __shfl_xor_sync(0xffffffffu, s2, off);
                mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            }
            if (l == 0) {
                atomicAdd(&red[0], s2);
                // max of non-negative doubles == max of their bit patterns as unsigned integers
                atomicMax(reinterpret_cast<unsigned long long*>(&red[1]), (unsigned long long)__double_as_longlong(mx));
            }
        }
    }
}

// Lambda[b][0..2][i] = R(q_i)^T m_i, Lambda[b][3..5][i] = R(q_i)^T n_i; one thread per (rod, node)
__global__ void wrench_local_kernel(long long batch, int N, const double* __restrict__ Q, const double* __restrict__ q0,
                                    const double* __restrict__ n, const double* __restrict__ m,
                                    const double* __restrict__ F_tip, const double* __restrict__ M_tip,
                                    double* __restrict__ Lambda) {
    const int M = N - 1;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= batch * N) return;
    const long long b = idx / N;
    const int i = (int)(idx % N);
    sri::quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
    if (i < M) {
        const double* s = Q + b * 4 * M + i;
        q.w = s[0]; q.x = s[M]; q.y = s[2 * M]; q.z = s[3 * M];
    } else if (q0) {
        const double* s = q0 + b * 4;
        q.w = s[0]; q.x = s[1]; q.y = s[2]; q.z = s[3];
    }
    double m0, m1, m2, n0, n1, n2;
    if (i == 0) {
        const double* s = M_tip + b * 3; m0 = s[0]; m1 = s[1]; m2 = s[2];
        const double* f = F_tip + b * 3; n0 = f[0]; n1 = f[1]; n2 = f[2];
    } else {
        const double* s = m + b * 3 * M + (i - 1); m0 = s[0]; m1 = s[M]; m2 = s[2 * M];
        const double* f = n + b * 3 * M + (i - 1); n0 = f[0]; n1 = f[M]; n2 = f[2 * M];
    }
    double c0, c1, c2, f0, f1, f2;
    sri::q_rotate_T(q, m0, m1, m2, c0, c1, c2);
    sri::q_rotate_T(q, n0, n1, n2, f0, f1, f2);
    double* d = Lambda + b * 6 * N + i;
    d[0] = c0; d[N] = c1; d[2 * N] = c2; d[3 * N] = f0; d[4 * N] = f1; d[5 * N] = f2;
}

// out[b][c*ne+k] = scale * sum_i w_i P_k(t_i) f[b*rod_stride + c*N + i]: one thread per (rod, component), cached Legendre
// table.  rod_stride = 3 N, scale = 1: projection of a nodal field; rod_stride = 6 N, scale = -1: generalised forces of the
// couple part of a wrench field.  ccw == NULL: w_i = 1, the transpose of the modal strain adapter.
__global__ void project_onto_modes_kernel(long long batch, int N, int ne, long long rod_stride, double scale,
                                          const double* __restrict__ ptab, const double* __restrict__ ccw,
                                          const double* __restrict__ f, double* __restrict__ out) {
    const long long bc = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (bc >= batch * 3) return;
    const long long b = bc / 3;
    const int c = (int)(bc - 3 * b);
    double acc[8];
    for (int k = 0; k < ne; ++k) acc[k] = 0.0;
    const double* fi = f + b * rod_stride + c * N;
    for (int i = 0; i < N; ++i) {
        const double wf = ccw ? ccw[i] * fi[i] : fi[i];
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < ne) acc[k] = fma(wf, ptab[k * N + i], acc[k]);
    }
    for (int k = 0; k < ne; ++k) out[bc * ne + k] = scale * acc[k];
}

// g[b][c*ne+k] = sum_i w_i P_k(t_i) rho[b][c][i],  rho_i = H (K_i - K0_i) - R(q_i)^T m_i: shape_residual_kernel and
// project_onto_modes_kernel in one pass (rho never reaches memory).  G lanes per rod (16 for N <= 16, else 32), node i in
// lane i % G; the sums over the nodes are a shuffle tree.  Optional norms of g over the batch, reduced in a fixed order
// (per block, then the last block to finish adds the block partials by index): bitwise reproducible.
template <int G, int NE>
__global__ void __launch_bounds__(256, 4) galerkin_residual_kernel(long long batch, int N, const double* __restrict__ ptab,
                                                                const double* __restrict__ ccw, const double* __restrict__ K,
                                                                const double* __restrict__ K0, double h0, double h1, double h2,
                                                                const double* __restrict__ Q, const double* __restrict__ q0,
                                                                const double* __restrict__ m, const double* __restrict__ M_tip,
                                                                double* __restrict__ g, double* __restrict__ partial,
                                                                unsigned* __restrict__ counter, double* __restrict__ red,
                                                                const int* __restrict__ skip) {
    if (skip && *skip) return;
    constexpr int ne = NE;
    const int M = N - 1;
    const int lane = threadIdx.x & 31, sub = lane & (G - 1);
    double s2 = 0.0, mx = 0.0;
    // persistent blocks: chunk `blk` of 256 / G rods per pass (one fence + ticket per block at the end instead of one per 16 rods:
    // 42 us instead of 73 us per 10^5 rods; the per-thread, per-block and per-grid summation orders are fixed by the launch
    // geometry, so the norms stay reproducible from run to run)
    const long long nblk = (batch * G + blockDim.x - 1) / blockDim.x;
    for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    const long long b = (blk * blockDim.x + threadIdx.x) / G;
    double acc[3][NE];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int k = 0; k < NE; ++k) acc[c][k] = 0.0;
    if (b < batch) {
        for (int i = sub; i < N; i += G) {
            // every load is issued before the first use: pointers are selected, not branched on (the kernel is bound by the
            // latency of these loads)
            const bool inner = i < M;
            const double* qs = inner ? Q + b * 4 * M + i : (q0 ? q0 + b * 4 : nullptr);
            const int qst = inner ? M : 1;
            const double* ms = i == 0 ? M_tip + b * 3 : m + b * 3 * M + (i - 1);
            const int mst = i == 0 ? 1 : M;
            const double* kp = K + b * 3 * N + i;
            sri::quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
            if (qs) { q.w = qs[0]; q.x = qs[qst]; q.y = qs[2 * qst]; q.z = qs[3 * qst]; }
            const double m0 = ms[0], m1 = ms[mst], m2 = ms[2 * mst];
            double k0 = kp[0], k1 = kp[N], k2 = kp[2 * N];
            if (K0) { const double* z = K0 + b * 3 * N + i; k0 -= z[0]; k1 -= z[N]; k2 -= z[2 * N]; }
            double t0, t1, t2;
            sri::q_rotate_T(q, m0, m1, m2, t0, t1, t2);
            const double w = ccw[i];
            const double wf[3] = {w * (h0 * k0 - t0), w * (h1 * k1 - t1), w * (h2 * k2 - t2)};
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                const double pk = ptab[k * N + i];
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[c][k] = fma(wf[c], pk, acc[c][k]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            {
                double v = acc[c][k];
#pragma unroll
                for (int off = G / 2; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                const int j = c * ne + k;
                if (b < batch && sub == (j & (G - 1))) {
                    g[b * 3 * ne + j] = v;
                    s2 = fma(v, v, s2);
                    mx = fmax(mx, fabs(v));
                }
            }
        }
    }  // chunks of this block
    if (!red) return;
    for (int off = 16; off >= 1; off >>= 1) {
        s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    }
    __shared__ double sh_s[8], sh_m[8];
    __shared__ bool last;
    const int w = threadIdx.x >> 5;
    if (lane == 0) { sh_s[w] = s2; sh_m[w] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, z = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += sh_s[i]; z = fmax(z, sh_m[i]); }
        partial[2 * blockIdx.x] = a; partial[2 * blockIdx.x + 1] = z;
        __threadfence();
        last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && w == 0) {
        __threadfence();
        double a = 0.0, z = 0.0;
        for (unsigned i = lane; i < gridDim.x; i += 32) { a += __ldcg(partial + 2 * i); z = fmax(z, __ldcg(partial + 2 * i + 1)); }
        for (int off = 16; off >= 1; off >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, off);
            z = fmax(z, __shfl_xor_sync(0xffffffffu, z, off));
        }
        if (lane == 0) { red[0] = a; red[1] = z; *counter = 0u; }
    }
}

// Reverse mode of galerkin_residual_kernel (sri_galerkin_residual_vjp), same lane layout: with the cotangent gg of g,
//     rb[c][i] = w_i sum_k P_k(t_i) gg[c*ne+k]                     (the cotangent of rho)
//     gK = H rb,  gK0 = -H rb,  gH[c] = sum_i rb[c][i] (K - K0)[c][i],  gm_i = -R(q_i) rb_i (node 0: gM_tip),
//     gq_i = -d/dq (m_i^T R(q) rb_i) at q_i  (nodes 0..M-1: gQ, node N-1: gq0),
// R the un-normalised rotation of q_rotate.  Every output pointer may be NULL (skipped); all are written, none accumulated.
// gH is a per-rod shuffle tree over the G lanes in a fixed order: bitwise reproducible.
template <int G, int NE>
__global__ void __launch_bounds__(256, 2) galerkin_residual_vjp_kernel(
        long long batch, int N, const double* __restrict__ ptab, const double* __restrict__ ccw, const double* __restrict__ K,
        const double* __restrict__ K0, double h0, double h1, double h2, const double* __restrict__ Q,
        const double* __restrict__ q0, const double* __restrict__ m, const double* __restrict__ M_tip,
        const double* __restrict__ gg, double* __restrict__ gK, double* __restrict__ gK0, double* __restrict__ gH,
        double* __restrict__ gQ, double* __restrict__ gq0, double* __restrict__ gm, double* __restrict__ gM_tip) {
    constexpr int ne = NE;
    const int M = N - 1;
    const int sub = threadIdx.x & (G - 1);
    const double hc[3] = {h0, h1, h2};
    const long long nblk = (batch * G + blockDim.x - 1) / blockDim.x;
    for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    const long long b = (blk * blockDim.x + threadIdx.x) / G;
    double hp[3] = {0.0, 0.0, 0.0};
    if (b < batch) {
        double gb[3][NE];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int k = 0; k < NE; ++k) gb[c][k] = gg[b * 3 * ne + c * ne + k];
        for (int i = sub; i < N; i += G) {
            const bool inner = i < M;
            const double* qs = inner ? Q + b * 4 * M + i : (q0 ? q0 + b * 4 : nullptr);
            const int qst = inner ? M : 1;
            const double* ms = i == 0 ? M_tip + b * 3 : m + b * 3 * M + (i - 1);
            const int mst = i == 0 ? 1 : M;
            const double* kp = K + b * 3 * N + i;
            sri::quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
            if (qs) { q.w = qs[0]; q.x = qs[qst]; q.y = qs[2 * qst]; q.z = qs[3 * qst]; }
            const double a0 = ms[0], a1 = ms[mst], a2 = ms[2 * mst];
            double kd[3] = {kp[0], kp[N], kp[2 * N]};
            if (K0) { const double* z = K0 + b * 3 * N + i; kd[0] -= z[0]; kd[1] -= z[N]; kd[2] -= z[2 * N]; }
            const double w = ccw[i];
            double rb[3] = {0.0, 0.0, 0.0};
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                const double pk = ptab[k * N + i];
#pragma unroll
                for (int c = 0; c < 3; ++c) rb[c] = fma(gb[c][k], pk, rb[c]);
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                rb[c] *= w;
                hp[c] = fma(rb[c], kd[c], hp[c]);
                if (gK) gK[b * 3 * N + c * N + i] = hc[c] * rb[c];
                if (gK0) gK0[b * 3 * N + c * N + i] = -(hc[c] * rb[c]);
            }
            if (i == 0 ? gM_tip != nullptr : gm != nullptr) {
                double r0, r1, r2;
                sri::q_rotate(q, rb[0], rb[1], rb[2], r0, r1, r2);
                double* d = i == 0 ? gM_tip + b * 3 : gm + b * 3 * M + (i - 1);
                d[0] = -r0; d[mst] = -r1; d[2 * mst] = -r2;
            }
            double* dq = inner ? (gQ ? gQ + b * 4 * M + i : nullptr) : (gq0 ? gq0 + b * 4 : nullptr);
            if (dq) {
                // d/dq a^T R(q) g, R g = g + 2w (v x g) + 2 v x (v x g), v = (x, y, z), a = m_i, g = rb_i
                const double g0 = rb[0], g1 = rb[1], g2 = rb[2];
                const double vxg0 = q.y * g2 - q.z * g1, vxg1 = q.z * g0 - q.x * g2, vxg2 = q.x * g1 - q.y * g0;
                const double gxa0 = g1 * a2 - g2 * a1, gxa1 = g2 * a0 - g0 * a2, gxa2 = g0 * a1 - g1 * a0;
                const double av = a0 * q.x + a1 * q.y + a2 * q.z, vg = q.x * g0 + q.y * g1 + q.z * g2;
                const double ag = a0 * g0 + a1 * g1 + a2 * g2;
                dq[0] = -2.0 * (a0 * vxg0 + a1 * vxg1 + a2 * vxg2);
                dq[qst] = -(2.0 * q.w * gxa0 + 2.0 * av * g0 + 2.0 * vg * a0 - 4.0 * ag * q.x);
                dq[2 * qst] = -(2.0 * q.w * gxa1 + 2.0 * av * g1 + 2.0 * vg * a1 - 4.0 * ag * q.y);
                dq[3 * qst] = -(2.0 * q.w * gxa2 + 2.0 * av * g2 + 2.0 * vg * a2 - 4.0 * ag * q.z);
            }
        }
    }
    if (gH) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            double v = hp[c];
#pragma unroll
            for (int off = G / 2; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (b < batch && sub == 0) gH[b * 3 + c] = v;
        }
    }
    }  // chunks of this block
}

// NaN-propagating max (fmax drops a NaN operand; a non-finite residual must show)
__device__ __forceinline__ double max_nan(double a, double b) { return (a > b || a != a) ? a : b; }

// One refinement step of the implicit adjoint of the static shape solve (sri_static_shape_vjp).  jd = Phi^T (gKd + gKi) is
// J_d^T lam, the exact transposed Jacobian of the discrete residual applied to lam (gKd: direct K-gradient of the
// residual's VJP, gKi: K-gradient of the integration's VJP); rhs = jd - gqe (the negated residual r = gqe - jd, so that
// the Newton update kernel lam -= J_a^-T rhs applies the step) and resid = max|r| / max|gqe| (max|r| when gqe = 0).  The
// call after the last chain also writes the parameter gradients F-grad = -gFi, M-grad = -(gMd + gMi), H-grad = -gHw,
// q0-grad = -(gq0d + gq0i) and info = sinfo | vinfo << 8, and negates in place the Gamma, fbar and lbar gradients that the
// last integration VJP wrote into the caller's buffers (no extra launch).  G lanes per rod as in galerkin_residual_kernel;
// NULL outputs are skipped.
struct AdjointRefineParams {
    long long batch;
    int N;
    const double* ptab;
    const double* gqe;   // [B][3 ne] cotangent of qe*
    const double* gKd;   // [B][3][N]
    const double* gKi;   // [B][3][N]
    double* rhs;         // [B][3 ne]
    double* resid;       // [B]
    const double *gFi, *gMd, *gMi, *gHw;   // [B][3] (final call)
    double *gF, *gM, *gH;                  // [B][3] (final call)
    const double *gq0d, *gq0i;             // [B][4] (final call)
    double* gq0;                           // [B][4] (final call)
    double *gGamma, *gfbar, *glbar;        // [B][3][N] (final call, negated in place)
    const int *sinfo, *vinfo;              // [B]
    int* info;                             // [B]
};
template <int G, int NE>
__global__ void __launch_bounds__(256) static_adjoint_refine_kernel(AdjointRefineParams p) {
    constexpr int ne = NE;
    const int N = p.N;
    const int sub = threadIdx.x & (G - 1);
    const long long nblk = (p.batch * G + blockDim.x - 1) / blockDim.x;
    for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    const long long b = (blk * blockDim.x + threadIdx.x) / G;
    double acc[3][NE];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int k = 0; k < NE; ++k) acc[c][k] = 0.0;
    if (b < p.batch) {
        for (int i = sub; i < N; i += G) {
            const double* d = p.gKd + b * 3 * N + i;
            const double* e = p.gKi + b * 3 * N + i;
            const double s[3] = {d[0] + e[0], d[N] + e[N], d[2 * N] + e[2 * N]};
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                const double pk = p.ptab[k * N + i];
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[c][k] = fma(s[c], pk, acc[c][k]);
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const long long o = b * 3 * N + c * N + i;
                if (p.gGamma) p.gGamma[o] = -p.gGamma[o];
                if (p.gfbar) p.gfbar[o] = -p.gfbar[o];
                if (p.glbar) p.glbar[o] = -p.glbar[o];
            }
        }
    }
    double rmax = 0.0, gmax = 0.0;
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            double v = acc[c][k];
#pragma unroll
            for (int off = G / 2; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            const int j = c * ne + k;
            if (b < p.batch && sub == (j & (G - 1))) {
                const double gj = p.gqe[b * 3 * ne + j];
                const double r = gj - v;
                if (p.rhs) p.rhs[b * 3 * ne + j] = v - gj;
                rmax = max_nan(rmax, fabs(r));
                gmax = max_nan(gmax, fabs(gj));
            }
        }
    if (p.resid) {
#pragma unroll
        for (int off = G / 2; off >= 1; off >>= 1) {
            rmax = max_nan(rmax, __shfl_xor_sync(0xffffffffu, rmax, off));
            gmax = max_nan(gmax, __shfl_xor_sync(0xffffffffu, gmax, off));
        }
        if (b < p.batch && sub == 0) p.resid[b] = gmax > 0.0 ? rmax / gmax : rmax;
    }
    if (b < p.batch && sub < 3) {
        const long long o = b * 3 + sub;
        if (p.gF) p.gF[o] = -p.gFi[o];
        if (p.gM) p.gM[o] = -(p.gMd[o] + p.gMi[o]);
        if (p.gH) p.gH[o] = -p.gHw[o];
        if (p.info && sub == 0) p.info[b] = (p.sinfo ? p.sinfo[b] : 0) | ((p.vinfo ? p.vinfo[b] : 0) << 8);
    }
    if (p.gq0 && b < p.batch && sub < 4) p.gq0[b * 4 + sub] = -(p.gq0d[b * 4 + sub] + p.gq0i[b * 4 + sub]);
    }  // chunks of this block
}

// ---- analytic Jacobian of the Galerkin residual (sri_shape_jacobian) ---------------------------------------------------
// J[b][j'][d] = d g_j' / d qe_d without any linear solve: the variation of the rotation is left-trivialised,
// dR = [dtheta]x R with dtheta' = R dK, dtheta(base) = 0, so a direction dK = P_k(t) e_c costs two contractions with the
// cached integration matrices S = Dn_NN^-1 (base condition) and S_T = D_TT^-1 (tip condition):
//     u_i = P_k(t_i) R_i[:, c]                  dtheta = S u                       (nodes 0..M-1; 0 at the base node)
//     v_j = -((dtheta_j x b_j) x n_j)          dm     = S_T v                     (nodes 1..N-1; 0 at the tip node)
//     drho_i = H dK_i - R_i^T (dm_i - dtheta_i x m_i),      dg = sum_i w_i P(t_i)^T drho_i.
// One warp per rod; nodal data and the per-direction vectors in the warp's shared-memory scratch, S and S_T in the CTA's.
struct JacobianScratch {  // doubles per warp, for N nodes
    __host__ __device__ static int total(int N) { return 9 * N + 3 * N + 3 * N + 3 * N + 3 * N + 3 * N + 3 * N + 3 * N + 3 * N; }
};
__global__ void __launch_bounds__(128) shape_jacobian_kernel(long long batch, int N, int ne, const double* __restrict__ S_rm,
                                                             const double* __restrict__ ST_rm, const double* __restrict__ ptab,
                                                             const double* __restrict__ ccw, double h0, double h1, double h2,
                                                             const double* __restrict__ Q, const double* __restrict__ q0,
                                                             const double* __restrict__ Gamma, const double* __restrict__ nin,
                                                             const double* __restrict__ m, const double* __restrict__ M_tip,
                                                             double* __restrict__ J, const int* __restrict__ skip) {
    if (skip && *skip) return;
    extern __shared__ __align__(16) double jsm[];
    const int M = N - 1, n = 3 * ne;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* Ss = jsm;                 // [M][M] row-major
    double* STs = jsm + M * M;        // [M][M] row-major
    double* Ps = jsm + 2 * M * M;     // [8][N] Legendre table
    double* Ws = Ps + 8 * N;          // [N] quadrature weights
    double* scr = Ws + N + warp * JacobianScratch::total(N);
    double* Rn = scr;                 // [N][9] rotation matrices, row-major
    double* bn = Rn + 9 * N;          // [N][3] R Gamma
    double* nn = bn + 3 * N;          // [M][3] internal force at nodes 1..N-1
    double* mn = nn + 3 * N;          // [N][3] internal couple, node 0 = M_tip
    double* u = mn + 3 * N;           // [M][3]
    double* th = u + 3 * N;           // [N][3] dtheta, base node = 0
    double* v = th + 3 * N;           // [M][3]
    double* dm = v + 3 * N;           // [N][3] dm, tip node = 0
    double* wr = dm + 3 * N;          // [3][N] w_i drho_i
    for (int e = threadIdx.x; e < M * M; e += blockDim.x) { Ss[e] = S_rm[e]; STs[e] = ST_rm[e]; }
    for (int e = threadIdx.x; e < 8 * N; e += blockDim.x) Ps[e] = ptab[e];
    for (int e = threadIdx.x; e < N; e += blockDim.x) Ws[e] = ccw[e];
    __syncthreads();
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long b = (long long)blockIdx.x * (blockDim.x >> 5) + warp; b < batch; b += warps_total) {
        for (int i = lane; i < N; i += 32) {
            sri::quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
            if (i < M) { const double* s = Q + b * 4 * M + i; q.w = s[0]; q.x = s[M]; q.y = s[2 * M]; q.z = s[3 * M]; }
            else if (q0) { const double* s = q0 + b * 4; q.w = s[0]; q.x = s[1]; q.y = s[2]; q.z = s[3]; }
            double* R = Rn + 9 * i;
            sri::quat_to_rot_rm(q, R);
            double g0 = 1.0, g1 = 0.0, g2 = 0.0;
            if (Gamma) { const double* gm = Gamma + b * 3 * N + i; g0 = gm[0]; g1 = gm[N]; g2 = gm[2 * N]; }
            bn[3 * i] = R[0] * g0 + R[1] * g1 + R[2] * g2;
            bn[3 * i + 1] = R[3] * g0 + R[4] * g1 + R[5] * g2;
            bn[3 * i + 2] = R[6] * g0 + R[7] * g1 + R[8] * g2;
            if (i == 0) { const double* s = M_tip + b * 3; mn[0] = s[0]; mn[1] = s[1]; mn[2] = s[2]; }
            else { const double* s = m + b * 3 * M + (i - 1); mn[3 * i] = s[0]; mn[3 * i + 1] = s[M]; mn[3 * i + 2] = s[2 * M]; }
            if (i < M) { const double* s = nin + b * 3 * M + i; nn[3 * i] = s[0]; nn[3 * i + 1] = s[M]; nn[3 * i + 2] = s[2 * M]; }
        }
        if (lane < 3) { th[3 * M + lane] = 0.0; dm[lane] = 0.0; }
        __syncwarp();
        for (int d = 0; d < n; ++d) {
            const int c = d / ne, k = d - c * ne;
            const double hc = c == 0 ? h0 : (c == 1 ? h1 : h2);
            for (int e = lane; e < 3 * M; e += 32) { const int i = e / 3, comp = e - 3 * i; u[e] = Ps[k * N + i] * Rn[9 * i + 3 * comp + c]; }
            __syncwarp();
            for (int e = lane; e < 3 * M; e += 32) {
                const int i = e / 3, comp = e - 3 * i;
                const double* srow = Ss + i * M;
                double acc = 0.0;
                for (int j = 0; j < M; ++j) acc = fma(srow[j], u[3 * j + comp], acc);
                th[e] = acc;
            }
            __syncwarp();
            for (int j = lane; j < M; j += 32) {  // node j + 1
                const double* t = th + 3 * (j + 1); const double* bb = bn + 3 * (j + 1); const double* f = nn + 3 * j;
                const double d0 = t[1] * bb[2] - t[2] * bb[1], d1 = t[2] * bb[0] - t[0] * bb[2], d2 = t[0] * bb[1] - t[1] * bb[0];
                v[3 * j] = -(d1 * f[2] - d2 * f[1]);
                v[3 * j + 1] = -(d2 * f[0] - d0 * f[2]);
                v[3 * j + 2] = -(d0 * f[1] - d1 * f[0]);
            }
            __syncwarp();
            for (int e = lane; e < 3 * M; e += 32) {
                const int j = e / 3, comp = e - 3 * j;
                const double* srow = STs + j * M;
                double acc = 0.0;
                for (int l = 0; l < M; ++l) acc = fma(srow[l], v[3 * l + comp], acc);
                dm[3 + e] = acc;  // node j + 1
            }
            __syncwarp();
            for (int i = lane; i < N; i += 32) {
                const double* t = th + 3 * i; const double* mm = mn + 3 * i; const double* dmi = dm + 3 * i; const double* R = Rn + 9 * i;
                const double t0 = dmi[0] - (t[1] * mm[2] - t[2] * mm[1]);
                const double t1 = dmi[1] - (t[2] * mm[0] - t[0] * mm[2]);
                const double t2 = dmi[2] - (t[0] * mm[1] - t[1] * mm[0]);
                const double w = Ws[i], hk = hc * Ps[k * N + i];
                wr[i] = w * ((c == 0 ? hk : 0.0) - (R[0] * t0 + R[3] * t1 + R[6] * t2));
                wr[N + i] = w * ((c == 1 ? hk : 0.0) - (R[1] * t0 + R[4] * t1 + R[7] * t2));
                wr[2 * N + i] = w * ((c == 2 ? hk : 0.0) - (R[2] * t0 + R[5] * t1 + R[8] * t2));
            }
            __syncwarp();
            for (int jp = lane; jp < n; jp += 32) {
                const int cp = jp / ne, kp = jp - cp * ne;
                double acc = 0.0;
                for (int i = 0; i < N; ++i) acc = fma(Ps[kp * N + i], wr[cp * N + i], acc);
                J[(b * n + jp) * n + d] = acc;
            }
            __syncwarp();
        }
    }
}

// ---- Newton driver helpers (sri_newton_static_shape) ---------------------------------------------------------------
// qw[d][b][j] = qe[b][j] + (j == d ? step : 0): the n forward-difference copies of the batch
__global__ void fd_perturb_kernel(long long B, int n, double step, const double* __restrict__ qe, double* __restrict__ qw,
                                  const int* __restrict__ skip) {
    if (skip && *skip) return;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long per = B * n;
    if (idx >= per * n) return;
    const int d = (int)(idx / per);
    const long long bj = idx - d * per;
    const int j = (int)(bj % n);
    const double v = qe[bj];
    qw[idx] = (j == d) ? v + step : v;
}

// J[b][i][d] = (gw[d][b][i] - g0[b][i]) / step
__global__ void fd_jacobian_kernel(long long B, int n, double step, const double* __restrict__ gw,
                                   const double* __restrict__ g0, double* __restrict__ J, const int* __restrict__ skip) {
    if (skip && *skip) return;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * n * n) return;
    const int d = (int)(idx % n);
    const long long bi = idx / n;  // b * n + i
    J[idx] = (gw[(long long)d * B * n + bi] - g0[bi]) / step;
}

using sri::NewtonState;

// qe -= delta for the rods whose Newton system was regular; counts the others.
__global__ void newton_update_kernel(long long B, int n, double* __restrict__ qe, const double* __restrict__ delta,
                                     const int* __restrict__ sinfo, NewtonState* __restrict__ state,
                                     const int* __restrict__ skip) {
    if (skip && *skip) return;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * n) return;
    const long long b = idx / n;
    if (sinfo && sinfo[b] != 0) {
        if (state && idx == b * n) atomicAdd(&state->singular, 1ULL);
        return;
    }
    qe[idx] -= delta[idx];
}

// Convergence test on the device: gathered[r] = (sum g^2, max |g|) of rank r, added in rank order (every rank computes the
// same bits); records the pair and raises the flag when sqrt(sum / dof) < tol.
__global__ void newton_check_kernel(const double* __restrict__ gathered, int nranks, double dof, double tol,
                                    NewtonState* __restrict__ state) {
    if (threadIdx.x != 0 || state->done) return;
    double s = 0.0, m = 0.0;
    for (int r = 0; r < nranks; ++r) { s += gathered[2 * r]; m = fmax(m, gathered[2 * r + 1]); }
    const int t = state->tested;
    if (t < 64) { state->hist[t][0] = s; state->hist[t][1] = m; }
    state->tested = t + 1;
    const double rms = dof > 0.0 ? sqrt(s / dof) : 0.0;
    if (rms < tol) state->done = 1;
}

// in-place (sum, max) over the ranks of an all-gathered norm pair (sri_nccl_allreduce_norms)
__global__ void fold_norms_kernel(const double* __restrict__ gathered, int nranks, double* __restrict__ out) {
    if (threadIdx.x != 0) return;
    double s = 0.0, m = 0.0;
    for (int r = 0; r < nranks; ++r) { s += gathered[2 * r]; m = fmax(m, gathered[2 * r + 1]); }
    out[0] = s; out[1] = m;
}

// A_NN = I4 (x) Dn_NN - 1/2 blockdiag A(K_i), column-major 4M x 4M per rod: updateA main.cpp:55-88 with the index map
// row = r M + i, col = c M + i of main.cpp:80-81 and the 4 x 4 block of main.cpp:72-75.  One CTA per rod.
__global__ void assemble_A_kernel(long long batch, int N, const double* __restrict__ Dnn_cm, const double* __restrict__ K,
                                  double* __restrict__ A) {
    const int M = N - 1, n = 4 * M;
    for (long long b = blockIdx.x; b < batch; b += gridDim.x) {
        const double* k = K + b * 3 * N;
        double* a = A + b * (long long)n * n;
        for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
            const int col = e / n, row = e - col * n;
            const int r = row / M, i = row - r * M, c = col / M, j = col - c * M;
            double v = (r == c) ? Dnn_cm[j * M + i] : 0.0;
            if (i == j) {
                const double k0 = k[i], k1 = k[N + i], k2 = k[2 * N + i];
                // A(K) rows: (0,-k0,-k1,-k2), (k0,0,k2,-k1), (k1,-k2,0,k0), (k2,k1,-k0,0)
                const double blk[4][4] = {{0.0, -k0, -k1, -k2}, {k0, 0.0, k2, -k1}, {k1, -k2, 0.0, k0}, {k2, k1, -k0, 0.0}};
                v = v - 0.5 * blk[r][c];
            }
            a[e] = v;
        }
    }
}

// One thread per system: Gaussian elimination with partial pivoting.  The block's systems (contiguous in global memory)
// are staged in shared memory element-major, a[e * (T + 1) + thread]: coalesced copies, conflict-free in both phases.
// TRANS: solves A^T x = b (element (i, j) of A lands at (j, i) while staged, no copy of A), and a non-finite pivot counts
// as singular too (the implicit adjoint of the static shape solve reports rods with non-finite loads through it).
template <bool TRANS>
__global__ void solve_small_kernel(long long batch, int n, const double* __restrict__ A, const double* __restrict__ b,
                                   double* __restrict__ x, int* __restrict__ info, const int* __restrict__ skip) {
    if (skip && *skip) return;
    extern __shared__ double ssm[];
    const int T = blockDim.x, LD = T + 1, tid = threadIdx.x, nn = n * n;
    const long long s0 = (long long)blockIdx.x * T;
    const int count = (int)((batch - s0) < T ? (batch - s0) : T);
    double* a = ssm + tid;           // a[e * LD]: this thread's matrix, row-major element e
    double* rhs = ssm + nn * LD + tid;
    {
        const double* src = A + s0 * nn;
        for (int e = tid; e < count * nn; e += T) {
            const int sys = e / nn;
            int el = e - sys * nn;
            if constexpr (TRANS) { const int r = el / n; el = (el - r * n) * n + r; }
            ssm[el * LD + sys] = src[e];
        }
        const double* bs = b + s0 * n;
        for (int e = tid; e < count * n; e += T) { const int sys = e / n, el = e - sys * n; ssm[(nn + el) * LD + sys] = bs[e]; }
    }
    __syncthreads();
    int bad = 0;
    if (tid < count) {
        for (int k = 0; k < n; ++k) {
            int p = k;
            double best = fabs(a[(k * n + k) * LD]);
            for (int i = k + 1; i < n; ++i) { const double v = fabs(a[(i * n + k) * LD]); if (v > best) { best = v; p = i; } }
            if (best == 0.0 || (TRANS && !isfinite(best))) { if (!bad) bad = k + 1; continue; }
            if (p != k) {
                for (int j = k; j < n; ++j) { const double t = a[(k * n + j) * LD]; a[(k * n + j) * LD] = a[(p * n + j) * LD]; a[(p * n + j) * LD] = t; }
                const double t = rhs[k * LD]; rhs[k * LD] = rhs[p * LD]; rhs[p * LD] = t;
            }
            const double inv = 1.0 / a[(k * n + k) * LD];
            const double rk = rhs[k * LD];
            for (int i = k + 1; i < n; ++i) {
                const double l = a[(i * n + k) * LD] * inv;
                for (int j = k + 1; j < n; ++j) a[(i * n + j) * LD] = fma(-l, a[(k * n + j) * LD], a[(i * n + j) * LD]);
                rhs[i * LD] = fma(-l, rk, rhs[i * LD]);
            }
        }
        for (int k = n - 1; k >= 0; --k) {
            double v = rhs[k * LD];
            for (int j = k + 1; j < n; ++j) v = fma(-a[(k * n + j) * LD], rhs[j * LD], v);
            rhs[k * LD] = v / a[(k * n + k) * LD];
        }
        if (info) info[s0 + tid] = bad;
    }
    __syncthreads();
    double* xs = x + s0 * n;
    for (int e = tid; e < count * n; e += T) { const int sys = e / n, el = e - sys * n; xs[e] = ssm[(nn + el) * LD + sys]; }
}

// The same solve for the small orders of the shape problem (n = 3 ne, ne <= 3) with the whole system in registers: every
// index is a compile-time constant, the row exchange of the partial pivoting is a chain of predicated swaps, and the
// thread reads its own contiguous 8 n (n + 1) bytes straight from global memory (a warp's systems are one contiguous
// region, so every fetched sector is consumed).  Same arithmetic as solve_small_kernel: identical results.  TRANS as there.
template <int NN, bool TRANS>
__global__ void __launch_bounds__(64) solve_small_reg_kernel(long long batch, const double* __restrict__ A, const double* __restrict__ b,
                                                             double* __restrict__ x, int* __restrict__ info, const int* __restrict__ skip) {
    if (skip && *skip) return;
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= batch) return;
    double a[NN][NN], r[NN];
    {
        const double* src = A + s * NN * NN;
#pragma unroll
        for (int i = 0; i < NN; ++i)
#pragma unroll
            for (int j = 0; j < NN; ++j) a[i][j] = src[TRANS ? j * NN + i : i * NN + j];
        const double* bs = b + s * NN;
#pragma unroll
        for (int e = 0; e < NN; ++e) r[e] = bs[e];
    }
    int bad = 0;
#pragma unroll
    for (int k = 0; k < NN; ++k) {
        int p = k;
        double best = fabs(a[k][k]);
#pragma unroll
        for (int i = k + 1; i < NN; ++i) { const double v = fabs(a[i][k]); if (v > best) { best = v; p = i; } }
        const bool ok = best != 0.0 && (!TRANS || isfinite(best));   // a zero column is skipped (multipliers 0), as in solve_small_kernel
        if (!ok && !bad) bad = k + 1;
#pragma unroll
        for (int i = k + 1; i < NN; ++i) {  // row exchange k <-> p by selects: no branch, every index static
            const bool sw = ok && (p == i);
#pragma unroll
            for (int j = k; j < NN; ++j) { const double t = a[k][j]; a[k][j] = sw ? a[i][j] : t; a[i][j] = sw ? t : a[i][j]; }
            const double t = r[k]; r[k] = sw ? r[i] : t; r[i] = sw ? t : r[i];
        }
        const double inv = ok ? 1.0 / a[k][k] : 0.0;
        const double rk = r[k];
#pragma unroll
        for (int i = k + 1; i < NN; ++i) {
            const double l = a[i][k] * inv;
#pragma unroll
            for (int j = k + 1; j < NN; ++j) a[i][j] = fma(-l, a[k][j], a[i][j]);
            r[i] = fma(-l, rk, r[i]);
        }
    }
#pragma unroll
    for (int k = NN - 1; k >= 0; --k) {
        double v = r[k];
#pragma unroll
        for (int j = k + 1; j < NN; ++j) v = fma(-a[k][j], r[j], v);
        r[k] = v / a[k][k];
    }
    if (info) info[s] = bad;
    double* xs = x + s * NN;
#pragma unroll
    for (int e = 0; e < NN; ++e) xs[e] = r[e];
}

// x[b][...] *= length[b] (or the one length `uniform` when `length` is NULL) for up to four [batch][per_rod] arrays: the
// input scaling that maps a rod of length l onto the unit-interval integrators (rod_modeling.pdf eq. 2.17).
__global__ void scale_for_length_kernel(long long batch, int per_rod, const double* __restrict__ length, double uniform,
                                        double* __restrict__ a0, double* __restrict__ a1, double* __restrict__ a2,
                                        double* __restrict__ a3) {
    const long long total = batch * per_rod;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
        const double l = length ? length[idx / per_rod] : uniform;
        if (a0) a0[idx] *= l;
        if (a1) a1[idx] *= l;
        if (a2) a2[idx] *= l;
        if (a3) a3[idx] *= l;
    }
}

// SURVEY 8(d) synthetic rods.  One thread per rod.
__global__ void generate_rods_kernel(unsigned long long seed, long long first_rod, long long batch, int N,
                                     const double* __restrict__ tnodes, double* __restrict__ K,
                                     double* __restrict__ F_tip, double* __restrict__ M_tip,
                                     double* __restrict__ fbar) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    const unsigned long long rod = (unsigned long long)(first_rod + b);
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t c0 = (uint32_t)rod, c1 = (uint32_t)(rod >> 32);
    uint32_t w[4];
    double u[14];
    for (int s = 0; s < 7; ++s) {
        sri::philox4x32_10(c0, c1, (uint32_t)s, 0u, k0, k1, w);
        u[2 * s] = sri::u01_from_bits(w[0], w[1]);
        u[2 * s + 1] = sri::u01_from_bits(w[2], w[3]);
    }
    if (K) {
        for (int c = 0; c < 3; ++c) {
            const double alpha = 4.0 * u[2 * c] - 2.0, beta = 4.0 * u[2 * c + 1] - 2.0;
            for (int i = 0; i < N; ++i) K[(b * 3 + c) * N + i] = fma(beta, tnodes[i], alpha);
        }
    }
    if (F_tip) for (int c = 0; c < 3; ++c) F_tip[b * 3 + c] = 2.0 * u[6 + c] - 1.0;
    if (M_tip) for (int c = 0; c < 3; ++c) M_tip[b * 3 + c] = 2.0 * u[9 + c] - 1.0;
    if (fbar) {
        const double gload = u[12];
        for (int i = 0; i < N; ++i) {
            fbar[(b * 3 + 0) * N + i] = 0.0;
            fbar[(b * 3 + 1) * N + i] = 0.0;
            fbar[(b * 3 + 2) * N + i] = -gload;
        }
    }
}

// FP64 FMA peak probe: 16 independent dependent-chains per thread.
__global__ void fp64_peak_kernel(double* out, int iters, double s) {
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = threadIdx.x * 1e-9 + i;
    const double b = s, c = 1.0 - s;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = fma(a[i], b, c);
    }
    double r = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) r += a[i];
    if (r == 123.456) out[0] = r;
}

// FP64 tensor-core (DMMA m8n8k4) peak probe: 16 independent accumulator tiles per warp.
__global__ void dmma_peak_kernel(double* out, int iters, double s) {
    double c0[16], c1[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { c0[i] = threadIdx.x * 1e-9 + i; c1[i] = i; }
    const double a = s, b = 1.0 - s;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) sri::dmma_m8n8k4(c0[i], c1[i], a, b);
    }
    double r = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) r += c0[i] + c1[i];
    if (r == 123.456) out[0] = r;
}

}  // namespace
