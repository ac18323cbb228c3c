// sri_tiled.cuh -- fused four-stage kernel for 17 <= N <= 64 Chebyshev nodes, register resident.
//
// Same algebra as sri_fused16.cuh (Gauss-Jordan over the quaternions with implicit row pivoting); what changes is how
// the M x (M+1) quaternion system [C | b] is spread over a CTA:
//   * every lane owns TWO rows of a rod (rows ln and ln + LPR), so a pivot-row quaternion loaded from shared memory
//     feeds two quaternion updates (32 DFMA) instead of one -- the pivot-row traffic through the LSU is what bounds
//     these kernels, not the FP64 pipe;
//   * the columns are dealt cyclically to the H warps of the CTA (column j lives in warp j mod H), 8 column slots per
//     lane, 2 x 8 quaternions = 128 registers per lane;
//   * LPR = 16, H = 4 (N <= 32): two rods per CTA, sixteen lanes per rod, both rods' pivot lanes publish with the same
//     store instruction.  LPR = 32, H = 8 (N <= 64): one rod per CTA.
// Step k: the warp that owns column k finds the pivot row, computes the multipliers m_i of all rows and publishes
// them; one CTA barrier; every warp's pivot lane publishes its own slice of the pivot row (warp-local), every lane
// updates its live slots.  The owner writes its results one slot down (sliding window, as in sri_fused16.cuh), so
// slot 0 of a warp is always its next pivot column and every register index stays a compile-time constant.
#pragma once
#include "sri_device.cuh"
#include "sri_fused16.cuh"  // FusedParams, fast_rcp, q_mul_tree, shfl_quat
#include "sri_generic.cuh"  // OpsLayoutGeneric

#ifndef SRI_TILED_LOOKAHEAD
#define SRI_TILED_LOOKAHEAD 0  // measured on B200: the look-ahead form is not faster (N=32: 15.9 vs 17.6 Mrods/s)
#endif

namespace sri {

template <int LPR, int H>
struct TiledSmem {
    static constexpr int RPW = 32 / LPR;   // rods per CTA
    static constexpr int ROWS = 2 * LPR;   // row capacity per rod = table stride
    static constexpr int SC = 8;           // column slots per lane
    __host__ __device__ static int tab() { return 0; }
    __host__ __device__ static int mbuf() { return OpsLayoutGeneric{ROWS}.total(); }          // [2][RPW][ROWS][4]
    __host__ __device__ static int ubuf() { return mbuf() + 2 * RPW * ROWS * 4; }             // [2][H][RPW][SC][4]
    __host__ __device__ static int qtmp() { return ubuf() + 2 * H * RPW * SC * 4; }           // [RPW][ROWS][4]
    __host__ __device__ static int vec() { return qtmp() + RPW * ROWS * 4; }                  // [RPW][64][4]
    __host__ __device__ static int vec2() { return vec() + RPW * 64 * 4; }                    // [RPW][64][4]
    __host__ __device__ static int Kb() { return vec2() + RPW * 64 * 4; }                     // [RPW][3][64]
    __host__ __device__ static int misc() { return Kb() + RPW * 3 * 64; }                     // [RPW][16]
    __host__ __device__ static int ints() { return misc() + RPW * 16; }                       // int area: 256 ints
    __host__ __device__ static int total() { return ints() + 128; }
};

template <int LPR, int H>
__global__ void __launch_bounds__(32 * H, (LPR == 16 ? 3 : 1)) tiled_kernel(const FusedParams p) {
    using SM = TiledSmem<LPR, H>;
    constexpr int RPW = SM::RPW, ROWS = SM::ROWS, SC = SM::SC;
    if (p.skip && *p.skip) return;  // Newton loop: the solve has already converged (device-side flag), nothing to do
    extern __shared__ __align__(16) double smem[];
    const OpsLayoutGeneric L{ROWS};
    double* tab = smem + SM::tab();
    double* mbuf = smem + SM::mbuf();
    double* ubuf = smem + SM::ubuf();
    double* qtmp = smem + SM::qtmp();
    int* ints = reinterpret_cast<int*>(smem + SM::ints());
    int* pinfo = ints;              // [2][RPW]
    int* sing = ints + 8;           // [RPW]
    int* perm = ints + 16;          // [RPW][64]

    const int M = p.M, N = p.N;
    const int h = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sub = lane / LPR, ln = lane % LPR;
    const int threads_per_rod = (32 * H) / RPW;
    const int tsub = threadIdx.x / threads_per_rod, tn = threadIdx.x % threads_per_rod;  // stage-phase mapping
    double* vec = smem + SM::vec() + tsub * 256;
    double* vec2 = smem + SM::vec2() + tsub * 256;
    double* Kb_t = smem + SM::Kb() + tsub * 192;
    double* misc_t = smem + SM::misc() + tsub * 16;

    // second pass over the rods the DMMA kernel (sri_tiled_dmma.cuh) handed back: rods rod_list[0 .. *rod_count)
    const bool listed = p.rod_list != nullptr;
    const long long batch = listed ? (long long)*p.rod_count : p.batch;
    const long long groups = (batch + RPW - 1) / RPW;
    if ((long long)blockIdx.x >= groups) return;  // whole CTA idle (the usual case of a second pass)
    for (int idx = threadIdx.x; idx < L.total(); idx += blockDim.x) tab[idx] = p.ops[idx];
    __syncthreads();
    for (long long grp = blockIdx.x; grp < groups; grp += gridDim.x) {
        // ---- inputs (stage-phase mapping: thread tn of rod tsub) --------------------------------------------
        const long long tidx = grp * RPW + tsub;
        const bool tlive = tidx < batch;
        const long long trod = (tlive && listed) ? (long long)p.rod_list[tidx] : tidx;
        if (tn < 64) {
            double k0 = 0.0, k1 = 0.0, k2 = 0.0;
            if (tlive && tn < N) { const double* s = p.K + trod * 3 * N + tn; k0 = s[0]; k1 = s[N]; k2 = s[2 * N]; }
            Kb_t[tn] = k0; Kb_t[64 + tn] = k1; Kb_t[128 + tn] = k2;
        }
        if (tn < 3) {
            misc_t[tn] = (tlive && p.F_tip) ? p.F_tip[trod * 3 + tn] : 0.0;
            misc_t[3 + tn] = (tlive && p.M_tip) ? p.M_tip[trod * 3 + tn] : 0.0;
            misc_t[6 + tn] = (tlive && p.r0) ? p.r0[trod * 3 + tn] : 0.0;
        }
        if (tn < 4) misc_t[9 + tn] = (tlive && p.q0) ? p.q0[trod * 4 + tn] : (tn == 0 ? 1.0 : 0.0);
        if (tn == 0) sing[tsub] = 0;
        __syncthreads();
        quat q0t; q0t.w = misc_t[9]; q0t.x = misc_t[10]; q0t.y = misc_t[11]; q0t.z = misc_t[12];

        quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
        {
            // ---- stage 1: assemble this lane's 2 rows x 8 column slots ---------------------------------------
            const double* Kb = smem + SM::Kb() + sub * 192;
            const double* misc = smem + SM::misc() + sub * 16;
            quat c[2][SC];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int i = ln + r * LPR;
#pragma unroll
                for (int s = 0; s < SC; ++s) {
                    const int j = s * H + h;
                    quat v; v.w = 0.0; v.x = 0.0; v.y = 0.0; v.z = 0.0;
                    if (i < M && j < M) {
                        const double sv = -0.5 * tab[L.Sp() + j * ROWS + i];
                        v.w = (j == i) ? 1.0 : 0.0; v.x = sv * Kb[j]; v.y = sv * Kb[64 + j]; v.z = sv * Kb[128 + j];
                    } else if (i < M && j == M) {
                        const double gi = tab[L.g() + i];
                        v.w = gi * misc[9]; v.x = gi * misc[10]; v.y = gi * misc[11]; v.z = gi * misc[12];
                    }
                    c[r][s] = v;
                }
            }
            int cnt = (h <= M) ? (M - h) / H + 1 : 0;  // live column slots of this warp (columns k..M)
            bool used0 = (ln >= M), used1 = (ln + LPR >= M);

            // ---- Gauss-Jordan over the quaternions -------------------------------------------------------------
            // Pivot search, candidate inverse and multipliers of step kk from slot 0 of the warp that owns column kk;
            // results go to the (kk & 1) halves of mbuf / pinfo.  All rows of a rod live in this one warp, so the
            // owner of step k+1 could do this as soon as ITS slot 0 has been updated in step k (SRI_TILED_LOOKAHEAD).
            auto pivot_work = [&](int kk) {
                const int par = kk & 1;
                const double n0 = fma(c[0][0].w, c[0][0].w, c[0][0].x * c[0][0].x) + fma(c[0][0].y, c[0][0].y, c[0][0].z * c[0][0].z);
                const double n1 = fma(c[1][0].w, c[1][0].w, c[1][0].x * c[1][0].x) + fma(c[1][0].y, c[1][0].y, c[1][0].z * c[1][0].z);
                const unsigned k0 = used0 ? 0u : ((((unsigned)__double2hiint(n0)) & 0xFFFFFFC0u) | (unsigned)(63 - ln));
                const unsigned k1 = used1 ? 0u : ((((unsigned)__double2hiint(n1)) & 0xFFFFFFC0u) | (unsigned)(63 - ln - LPR));
                const bool pick1 = k1 > k0;
                unsigned key = pick1 ? k1 : k0;
                const quat cb = pick1 ? c[1][0] : c[0][0];
                const double inv = fast_rcp(pick1 ? n1 : n0);
                quat cand; cand.w = cb.w * inv; cand.x = -cb.x * inv; cand.y = -cb.y * inv; cand.z = -cb.z * inv;
#pragma unroll
                for (int off = LPR / 2; off >= 1; off >>= 1) {
                    const unsigned other = __shfl_xor_sync(0xffffffffu, key, off);
                    key = key > other ? key : other;
                }
                const int prow = 63 - (int)(key & 63u);
                const quat pinv = shfl_quat(cand, (lane & ~(LPR - 1)) | (prow % LPR));
                quat m0 = q_mul_tree(pinv, c[0][0]);
                quat m1 = q_mul_tree(pinv, c[1][0]);
                if (ln == prow) { m0.w = 1.0 - pinv.w; m0.x = -pinv.x; m0.y = -pinv.y; m0.z = -pinv.z; }
                if (ln + LPR == prow) { m1.w = 1.0 - pinv.w; m1.x = -pinv.x; m1.y = -pinv.y; m1.z = -pinv.z; }
                double* mb = mbuf + ((par * RPW + sub) * ROWS) * 4;
                st_quat(mb + 4 * ln, m0);
                st_quat(mb + 4 * (ln + LPR), m1);
                if (ln == 0) {
                    pinfo[par * RPW + sub] = prow;
                    perm[sub * 64 + kk] = prow;
                    if (((key >> 6) == 0u || (key >> 6) >= 0x01ffc000u) && sing[sub] == 0) sing[sub] = kk + 1;  // zero or non-finite pivot
                }
            };
#if SRI_TILED_LOOKAHEAD
            if (h == 0 && M > 0) pivot_work(0);
            __syncthreads();
#endif
            for (int k = 0; k < M; ++k) {
                const int par = k & 1;
                const bool owner = (h == k % H);
#if SRI_TILED_LOOKAHEAD
                const bool next_owner = (k + 1 < M) && (h == (k + 1) % H);
#else
                const bool next_owner = false;
                if (owner) pivot_work(k);
                __syncthreads();
#endif
                const int prow = pinfo[par * RPW + sub];
                const int pl = prow % LPR;
                const bool prhi = prow >= LPR;
                double* ub = ubuf + (((par * H + h) * RPW + sub) * SC) * 4;
                if (ln == pl) {
#pragma unroll
                    for (int s = 0; s < SC; ++s)
                        if (s < cnt && (s > 0 || !owner)) st_quat(ub + 4 * s, prhi ? c[1][s] : c[0][s]);
                }
                if (prow == ln) used0 = true;
                if (prow == ln + LPR) used1 = true;
                __syncwarp();
                const double* mb = mbuf + ((par * RPW + sub) * ROWS) * 4;
                const quat m0 = ld_quat(mb + 4 * ln);
                const quat m1 = ld_quat(mb + 4 * (ln + LPR));
                if (owner) {
                    // sliding window: results go one slot down, slot 0 (the eliminated column) disappears
#pragma unroll
                    for (int s = 1; s < SC; ++s) {
                        if (s < cnt) {
                            const quat u = ld_quat(ub + 4 * s);
                            quat t0 = c[0][s], t1 = c[1][s];
                            q_sub_mul(t0, u, m0);
                            q_sub_mul(t1, u, m1);
                            c[0][s - 1] = t0; c[1][s - 1] = t1;
                        } else {
                            c[0][s - 1].w = 0.0; c[0][s - 1].x = 0.0; c[0][s - 1].y = 0.0; c[0][s - 1].z = 0.0;
                            c[1][s - 1] = c[0][s - 1];
                        }
                    }
                    c[0][SC - 1].w = 0.0; c[0][SC - 1].x = 0.0; c[0][SC - 1].y = 0.0; c[0][SC - 1].z = 0.0;
                    c[1][SC - 1] = c[0][SC - 1];
                    cnt -= 1;
                } else {
                    {   // slot 0 first: for the owner of step k+1 it is the next pivot column
                        const quat u = ld_quat(ub);
                        if (0 < cnt) { q_sub_mul(c[0][0], u, m0); q_sub_mul(c[1][0], u, m1); }
                    }
                    if (next_owner) pivot_work(k + 1);
#pragma unroll
                    for (int s = 1; s < SC; ++s) {
                        if (s < cnt) {
                            const quat u = ld_quat(ub + 4 * s);
                            q_sub_mul(c[0][s], u, m0);
                            q_sub_mul(c[1][s], u, m1);
                        }
                    }
                }
#if SRI_TILED_LOOKAHEAD
                __syncthreads();
#endif
            }
            // ---- the rhs column (j = M) now sits in slot 0 of warp M mod H: rows -> shared ----------------------
            if (h == M % H) {
                st_quat(qtmp + (sub * ROWS + ln) * 4, c[0][0]);
                st_quat(qtmp + (sub * ROWS + ln + LPR) * 4, c[1][0]);
            }
            __syncthreads();
            if (tn < M) q = ld_quat(qtmp + (tsub * ROWS + perm[tsub * 64 + tn]) * 4);
            if (tn == M) q = q0t;
            if (p.info && tlive && tn == 0) p.info[trod] = sing[tsub];
            if (p.Q && tlive && tn < M) {
                double* d = p.Q + trod * 4 * M + tn;
                d[0] = q.w; d[M] = q.x; d[2 * M] = q.y; d[3 * M] = q.z;
            }
        }

        if (p.r || p.n || p.m) {
            // ---- stage 2 (thread tn = node tn of rod tsub) -----------------------------------------------------
            if (tn <= M) {
                double b0, b1, b2;
                if (p.Gamma && tlive) { const double* s = p.Gamma + trod * 3 * N + tn; q_rotate(q, s[0], s[N], s[2 * N], b0, b1, b2); }
                else q_rotate_e1(q, b0, b1, b2);
                quat v; v.w = b0; v.x = b1; v.y = b2; v.z = 0.0;
                st_quat(vec + 4 * tn, v);
            }
            const bool contract3 = (p.n || p.m) && p.fbar;
            const double F0 = misc_t[0], F1 = misc_t[1], F2 = misc_t[2];
            if (contract3 && tn < M) {
                const double dti = tab[L.DTI() + tn];
                double f0 = 0.0, f1 = 0.0, f2 = 0.0;
                if (tlive) { const double* s = p.fbar + trod * 3 * N + tn + 1; f0 = s[0]; f1 = s[N]; f2 = s[2 * N]; }
                quat v; v.w = -f0 - dti * F0; v.x = -f1 - dti * F1; v.y = -f2 - dti * F2; v.z = 0.0;
                st_quat(vec2 + 4 * tn, v);
            }
            __syncthreads();
            if (p.r && tn < M) {
                double a0 = 0.0, a1 = 0.0, a2 = 0.0, e0 = 0.0, e1 = 0.0, e2 = 0.0;
                for (int j = 0; j + 1 < M; j += 2) {
                    const double s0 = tab[L.Sp() + j * ROWS + tn], s1 = tab[L.Sp() + (j + 1) * ROWS + tn];
                    a0 = fma(s0, vec[4 * j], a0); a1 = fma(s0, vec[4 * j + 1], a1); a2 = fma(s0, vec[4 * j + 2], a2);
                    e0 = fma(s1, vec[4 * j + 4], e0); e1 = fma(s1, vec[4 * j + 5], e1); e2 = fma(s1, vec[4 * j + 6], e2);
                }
                if (M & 1) {
                    const int j = M - 1;
                    const double s0 = tab[L.Sp() + j * ROWS + tn];
                    a0 = fma(s0, vec[4 * j], a0); a1 = fma(s0, vec[4 * j + 1], a1); a2 = fma(s0, vec[4 * j + 2], a2);
                }
                const double gi = tab[L.g() + tn];
                a0 = fma(gi, misc_t[6], a0 + e0); a1 = fma(gi, misc_t[7], a1 + e1); a2 = fma(gi, misc_t[8], a2 + e2);
                if (tlive) { double* d = p.r + trod * 3 * M + tn; d[0] = a0; d[M] = a1; d[2 * M] = a2; }
            }
            if (p.n || p.m) {
                // ---- stage 3: thread tn = reduced row (node tn+1) ------------------------------------------------
                double n0 = 0.0, n1 = 0.0, n2 = 0.0;
                if (tn < M) {
                    if (contract3) {
                        double e0 = 0.0, e1 = 0.0, e2 = 0.0;
                        for (int j = 0; j + 1 < M; j += 2) {
                            const double s0 = tab[L.STt() + j * ROWS + tn], s1 = tab[L.STt() + (j + 1) * ROWS + tn];
                            n0 = fma(s0, vec2[4 * j], n0); n1 = fma(s0, vec2[4 * j + 1], n1); n2 = fma(s0, vec2[4 * j + 2], n2);
                            e0 = fma(s1, vec2[4 * j + 4], e0); e1 = fma(s1, vec2[4 * j + 5], e1); e2 = fma(s1, vec2[4 * j + 6], e2);
                        }
                        if (M & 1) {
                            const int j = M - 1;
                            const double s0 = tab[L.STt() + j * ROWS + tn];
                            n0 = fma(s0, vec2[4 * j], n0); n1 = fma(s0, vec2[4 * j + 1], n1); n2 = fma(s0, vec2[4 * j + 2], n2);
                        }
                        n0 += e0; n1 += e1; n2 += e2;
                    } else {
                        const double gi = tab[L.gT() + tn];
                        n0 = gi * F0; n1 = gi * F1; n2 = gi * F2;
                    }
                    if (p.n && tlive) { double* d = p.n + trod * 3 * M + tn; d[0] = n0; d[M] = n1; d[2 * M] = n2; }
                }
                if (p.m) {
                    // ---- stage 4 ---------------------------------------------------------------------------
                    __syncthreads();  // vec2 (stage 3 rhs) has been consumed
                    if (tn < M) {
                        const double* rp = vec + 4 * (tn + 1);
                        double l0 = 0.0, l1 = 0.0, l2 = 0.0;
                        if (p.lbar && tlive) { const double* s = p.lbar + trod * 3 * N + tn + 1; l0 = s[0]; l1 = s[N]; l2 = s[2 * N]; }
                        const double dti = tab[L.DTI() + tn];
                        const double c0 = rp[1] * n2 - rp[2] * n1, c1 = rp[2] * n0 - rp[0] * n2, c2 = rp[0] * n1 - rp[1] * n0;
                        quat v; v.w = -(c0 + l0) - dti * misc_t[3]; v.x = -(c1 + l1) - dti * misc_t[4]; v.y = -(c2 + l2) - dti * misc_t[5]; v.z = 0.0;
                        st_quat(vec2 + 4 * tn, v);
                    }
                    __syncthreads();
                    if (tn < M) {
                        double m0 = 0.0, m1 = 0.0, m2 = 0.0, e0 = 0.0, e1 = 0.0, e2 = 0.0;
                        for (int j = 0; j + 1 < M; j += 2) {
                            const double s0 = tab[L.STt() + j * ROWS + tn], s1 = tab[L.STt() + (j + 1) * ROWS + tn];
                            m0 = fma(s0, vec2[4 * j], m0); m1 = fma(s0, vec2[4 * j + 1], m1); m2 = fma(s0, vec2[4 * j + 2], m2);
                            e0 = fma(s1, vec2[4 * j + 4], e0); e1 = fma(s1, vec2[4 * j + 5], e1); e2 = fma(s1, vec2[4 * j + 6], e2);
                        }
                        if (M & 1) {
                            const int j = M - 1;
                            const double s0 = tab[L.STt() + j * ROWS + tn];
                            m0 = fma(s0, vec2[4 * j], m0); m1 = fma(s0, vec2[4 * j + 1], m1); m2 = fma(s0, vec2[4 * j + 2], m2);
                        }
                        if (tlive) { double* d = p.m + trod * 3 * M + tn; d[0] = m0 + e0; d[M] = m1 + e1; d[2 * M] = m2 + e2; }
                    }
                }
            }
        }
        __syncthreads();  // shared buffers are reused by the next group
    }
}

}  // namespace sri
