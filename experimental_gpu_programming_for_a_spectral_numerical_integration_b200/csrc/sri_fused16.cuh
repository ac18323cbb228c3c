// sri_fused16.cuh -- row-pivoting fused four-stage kernel for N <= 16 Chebyshev nodes (M = N-1 <= 15 unknown nodes).
//
// Role: second pass of the N <= 16 path.  The tensor-core kernel (sri_fused16_dmma.cuh) eliminates in static pivot order
// and hands the rods that fail its growth check back to this kernel through FusedParams::rod_list; with
// SRI_FUSED16_IMPL=scalar it runs the whole batch (1.97e8 rods/s on one B200).  FusedParams and the small PTX helpers
// shared by all fused kernels live here too.
//
// Mapping: TWO rods per warp.  Lanes 0..15 own rod A, lanes 16..31 rod B; lane `row` of a half-warp owns row
// `row` of that rod's M x M quaternion collocation operator (M quaternions + the right-hand side = 64 doubles,
// all in registers, every register index a compile-time constant).  Lane 15 of each half is padding.
//
// Replaces, per rod: updateA (main.cpp:55-88), A_NN.inverse()*(b-ivp) (main.cpp:113), updatePositionb
// (main.cpp:121-140), Dn_NN_inv*(b_NN-ivp) (main.cpp:172) and the two spec'd stages (rod_modeling.pdf 1.17-1.18).
//
// What shapes the code (measured on B200, tools/*microbench*, profiles/):
//   * the FP64 pipe issues one warp-DFMA per 2 cycles per SM sub-partition but a dependent DFMA waits ~36 cycles,
//     so every serial FP64 chain on the elimination's critical path is kept as short as possible (tree-shaped
//     products, branch-free Newton reciprocal) and the pivot search / reciprocal of step k+1 is issued before the
//     bulk update of step k so that it hides behind this warp's own DFMA stream;
//   * a row lives in ONE lane, and getting it out costs LSU time whichever way (8.4 SM-cycles per quaternion for a 2-lane
//     shared-memory store + 4.2 for the loads, 8.2 for eight SHFL.IDX); the shared-memory form ships because the shuffle
//     form (-DSRI_BCAST_SHFL=1) pushes the hot code past the instruction cache;
//   * per-rod inputs that are only needed after the elimination are prefetched with cp.async at the top of the
//     iteration, as are the next pair's strain samples.
#pragma once
#include "sri_device.cuh"

namespace sri {

constexpr int MP16 = 16;  // padded rows per rod in this kernel

constexpr int kFusedThreads = 128;  // threads per CTA of the fused kernel
constexpr int kFusedMinBlocks = 3;

// Packed operator tables (doubles), stride MP16, zero padded.  Built on the host by sri_api.cu.
struct OpsLayout16 {
    static constexpr int St = 0;                   // [15][16]  St[j*16+i]  = -1/2 (Dn_NN^-1)(i,j)   (pre-scaled)
    static constexpr int Sp = St + 15 * MP16;      // [15][16]  Sp[j*16+i]  = (Dn_NN^-1)(i,j)
    static constexpr int STt = Sp + 15 * MP16;     // [15][16]  STt[j*16+i] = (D_TT^-1)(i,j)
    static constexpr int g = STt + 15 * MP16;      // [16]  g  = -(Dn_NN^-1 Dn_IN)
    static constexpr int gT = g + MP16;            // [16]  gT = -(D_TT^-1 D_TI)
    static constexpr int DTI = gT + MP16;          // [16]  D_TI
    static constexpr int DnIN = DTI + MP16;        // [16]  Dn_IN
    static constexpr int total = DnIN + MP16;      // 784 doubles
};

struct FusedParams {
    long long batch;
    int N, M;
    const double* ops;  // OpsLayout16 (device)
    const double* ops2; // N > 16: tables of the DMMA kernel (TiledDmmaCfg: Stx | AS | AT)
    const double* K;
    const double* q0;
    const double* r0;
    const double* Gamma;
    const double* fbar;
    const double* lbar;
    const double* F_tip;
    const double* M_tip;
    const double* Qin;  // stage kernels only: quaternions computed by an earlier call
    const double* nin;  // stage kernels only: internal forces computed by an earlier call
    double* Q;
    double* r;
    double* n;
    double* m;
    int* info;
    // Rods that need row pivoting: written by the DMMA kernel (sri_fused16_dmma.cuh), then read by the scalar kernel,
    // which in that mode integrates rods rod_list[0 .. *rod_count) instead of 0 .. batch.
    int* rod_list;
    int* rod_count;
    int growth_log;  // DMMA kernel: 2^20 log2(G^2), G = accepted sub-diagonal growth max_{i>k} |c_ik| / |c_kk|
    const int* skip; // optional device flag: when set and non-zero the kernel exits at once (sri_newton_static_shape)
};

// Per-rod shared scratch (doubles).
struct RodScratch {
    static constexpr int kbuf = 0;              // [2][4][16] strain samples (double buffered): K0,K1,K2 rows + q0 row
    static constexpr int fbar = kbuf + 128;     // [3][16]
    static constexpr int lbar = fbar + 48;      // [3][16]
    static constexpr int gam = lbar + 48;       // [3][16]
    static constexpr int misc = gam + 48;       // [16]: F_tip 0..2, M_tip 3..5, r0 6..8
    static constexpr int qnode = misc + 16;     // [16][4] quaternions by node (slot M = base node)
    static constexpr int vec = qnode + 64;      // [16][4] nodal 3-vectors (r')
    static constexpr int vec2 = vec + 64;       // [16][4]
    static constexpr int pbuf = vec2 + 64;      // [2][16][4] pivot-row publish buffers (double buffered)
    static constexpr int total = pbuf + 128;    // 608 doubles
};
constexpr int kWarpScratch16 = 2 * RodScratch::total;  // doubles per warp

// ---- small PTX helpers --------------------------------------------------------------------------------------

__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N_) : "memory"); }

// Branch-free reciprocal: MUFU.RCP64H seed (~20 bits) and one cubically convergent correction
// r <- r (1 + e + e^2), e = 1 - x r: three dependent FP64 operations instead of the ~8 of the IEEE division.
// Relative error ~1e-16 (not correctly rounded; the elimination does not need it to be).
__device__ __forceinline__ double fast_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);
    const double t = fma(e, e, e);
    return fma(r, t, r);
}

// Broadcast of one quaternion from lane `src` (per half-warp) to every lane of that half.
__device__ __forceinline__ quat shfl_quat(const quat& q, int src) {
    quat r;
    r.w = __shfl_sync(0xffffffffu, q.w, src);
    r.x = __shfl_sync(0xffffffffu, q.x, src);
    r.y = __shfl_sync(0xffffffffu, q.y, src);
    r.z = __shfl_sync(0xffffffffu, q.z, src);
    return r;
}

// p (x) c with each component evaluated as (t1 + t2) + (t3 + t4): dependent depth 3 instead of 4.
__device__ __forceinline__ quat q_mul_tree(const quat& p, const quat& c) {
    quat r;
    r.w = fma(-p.x, c.x, p.w * c.w) - fma(p.z, c.z, p.y * c.y);
    r.x = fma(p.x, c.w, p.w * c.x) + fma(-p.z, c.y, p.y * c.z);
    r.y = fma(-p.x, c.z, p.w * c.y) + fma(p.z, c.x, p.y * c.w);
    r.z = fma(p.x, c.y, p.w * c.z) + fma(p.z, c.w, -p.y * c.x);
    return r;
}

// Pivot candidate of a row for column value c: key = top 28 bits of |c|^2 (monotone for non-negative doubles) with
// the row index in the low 4 bits, so that the segment-wide maximum also names the winning lane; rows already
// used as pivots get key 0.  cand = c^-1 = conj(c)/|c|^2, computed by EVERY lane for its own row while the
// butterfly runs, so that the winner only has to broadcast it.
__device__ __forceinline__ void pivot_candidate(const quat& c, bool used, int row, unsigned& key, quat& cand) {
    const double nrm = fma(c.w, c.w, c.x * c.x) + fma(c.y, c.y, c.z * c.z);
    key = used ? 0u : ((((unsigned)__double2hiint(nrm)) & 0xFFFFFFF0u) | (unsigned)(15 - row));
    const double inv = fast_rcp(nrm);
    cand.w = c.w * inv; cand.x = -c.x * inv; cand.y = -c.y * inv; cand.z = -c.z * inv;
}

// max over the 16-lane segment (xor offsets 8,4,2,1 never leave the half-warp)
__device__ __forceinline__ unsigned segment_max16(unsigned key) {
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) {
        const unsigned other = __shfl_xor_sync(0xffffffffu, key, off);
        key = key > other ? key : other;
    }
    return key;
}

#ifndef SRI_BCAST_SHFL
#define SRI_BCAST_SHFL 0  // 0: pivot row through shared memory; 1: SHFL.IDX
#endif

// One Gauss-Jordan step over the quaternions with implicit row pivoting, ROLLED form.
//
// B200's instruction supply sustains full FP64 rate only for loops of <= 32 KB of code (tools/icache_microbench:
// 36 TF at 32 KB, 7-20 TF at 64 KB with de-synchronised warps), and a fully unrolled 15-step elimination is ~86 KB.
// So the row is kept in a sliding window instead: slot 0 always holds the pivot column of the current step, every
// update writes its result one slot down (c[j-1] = c[j] - u_j (x) m; the shift costs no instruction), and the same
// body serves several steps.  L = number of window slots the body touches; a body may run while the live width
// 15-k is <= L (the slots beyond it hold zeros and stay zero).  Four bodies (L = 15, 11, 7, 3; two or three bodies
// measured 1-6 % slower) cost 17 % more quaternion updates than the exact triangle and fit the whole kernel in the
// instruction cache.
//
//   equations:  sum_j Q_j (x) c_ij = b_i.   Row i takes  c_ij -= u_j (x) m_i  with u = pivot row and
//   m_i = c_pk^-1 (x) c_ik; the pivot row takes m_p = 1 - c_pk^-1, which normalises it with the same update.
// On entry key/cand describe slot 0 (key already segment-reduced); on exit they describe the new slot 0.
template <int L, int NC>
__device__ __forceinline__ void gj_step_rolled(quat (&c)[15], quat& b, int k, int live, int row, double* pbuf,
                                               bool& used, int& mycol, int& sing, unsigned& key, quat& cand) {
    // live = number of window slots that still hold columns (M - k); a body with window L and NC conditional slots
    // serves live in (L-1-NC, L]: slots 1..L-1-NC are always live, the last NC slots only while slot < live
    // (warp-uniform tests).
    const int prow = 15 - (int)(key & 15u);
    const bool is_pivot = (row == prow) && !used;
    // zero pivot, or a non-finite one (hi word of |c|^2 >= 0x7ff00000: Inf / NaN in the strain samples)
    if (((key >> 4) == 0u || (key >> 4) >= 0x07ff0000u) && sing == 0) sing = k + 1;
#if SRI_BCAST_SHFL
    const int src = ((threadIdx.x & 16) | prow);
#define SRI_PIVOT_ROW(j) shfl_quat(c[j], src)
#define SRI_PIVOT_RHS() shfl_quat(b, src)
    const quat pinv = shfl_quat(cand, src);
#else
    // the pivot lane publishes c_pk^-1 (slot 0), its live window slots and its rhs (slot 15)
    double* buf = pbuf + (k & 1) * (16 * 4);
    if (is_pivot) {
        st_quat(buf, cand);
        st_quat(buf + 4 * 15, b);
#pragma unroll
        for (int j = 1; j < L; ++j)
            if (j <= L - 1 - NC || j < live) st_quat(buf + 4 * j, c[j]);
    }
    __syncwarp();
#define SRI_PIVOT_ROW(j) ld_quat(buf + 4 * (j))
#define SRI_PIVOT_RHS() ld_quat(buf + 4 * 15)
    const quat pinv = ld_quat(buf);
#endif
    quat mlt = q_mul_tree(pinv, c[0]);
    if (is_pivot) { mlt.w = 1.0 - pinv.w; mlt.x = -pinv.x; mlt.y = -pinv.y; mlt.z = -pinv.z; mycol = k; used = true; }
    // slot 1 first: it becomes the next pivot column, and its candidate/key latency hides behind the bulk update
    if (L > 1 && (1 <= L - 1 - NC || 1 < live)) {
        const quat u = SRI_PIVOT_ROW(1);
        quat t = c[L > 1 ? 1 : 0];
        q_sub_mul(t, u, mlt);
        c[0] = t;
    } else {
        c[0].w = 0.0; c[0].x = 0.0; c[0].y = 0.0; c[0].z = 0.0;
    }
    pivot_candidate(c[0], used, row, key, cand);
    {
        const quat u = SRI_PIVOT_RHS();
        q_sub_mul(b, u, mlt);
    }
    unsigned other = 0u;
#pragma unroll
    for (int j = 2; j < L; ++j) {
        const int stage = j - 2;  // butterfly stage interleaved with this slot
        if (stage < 4) other = __shfl_xor_sync(0xffffffffu, key, 8 >> stage);
        if (j <= L - 1 - NC || j < live) {
            const quat u = SRI_PIVOT_ROW(j);
            quat t = c[j];
            q_sub_mul(t, u, mlt);
            c[j - 1] = t;
        }  // a slot >= live is dead: it is never published, loaded or updated again, so it needs no zero fill
        if (stage < 4) key = key > other ? key : other;
    }
#pragma unroll
    for (int stage = (L - 2 > 0 ? L - 2 : 0); stage < 4; ++stage) {
        other = __shfl_xor_sync(0xffffffffu, key, 8 >> stage);
        key = key > other ? key : other;
    }
#undef SRI_PIVOT_ROW
#undef SRI_PIVOT_RHS
}

// Full elimination of an M x M system, M <= 15 at run time (rows and columns >= M are zero padding and never
// pivot).  On return b holds Q_{mycol}.
__device__ __forceinline__ void gauss_jordan16(quat (&c)[15], quat& b, int M, int row, double* pbuf, int& mycol,
                                               int& sing) {
    bool used = (row >= M);
    mycol = row;
    sing = 0;
    unsigned key;
    quat cand;
    pivot_candidate(c[0], used, row, key, cand);
    key = segment_max16(key);
    int k = 0;
    // the body is chosen by the live width M - k, so a short system (N < 16) starts directly with a small window
#pragma unroll 1
    for (; M - k > 11; ++k) gj_step_rolled<15, 3>(c, b, k, M - k, row, pbuf, used, mycol, sing, key, cand);
#pragma unroll 1
    for (; M - k > 7; ++k) gj_step_rolled<11, 3>(c, b, k, M - k, row, pbuf, used, mycol, sing, key, cand);
#pragma unroll 1
    for (; M - k > 3; ++k) gj_step_rolled<7, 3>(c, b, k, M - k, row, pbuf, used, mycol, sing, key, cand);
#pragma unroll 1
    for (; M - k > 0; ++k) gj_step_rolled<3, 3>(c, b, k, M - k, row, pbuf, used, mycol, sing, key, cand);
}

// out_c = sum_j T[j*16+row] * v[j][c], c = 0..2, with three interleaved partial sums per component so that the
// dependent DFMA chains are 5 long instead of 15.
template <int MS>
__device__ __forceinline__ void contract16(const double* T, const double* v, int M, int row, double& o0, double& o1,
                                           double& o2) {
    double a[3][3];
#pragma unroll
    for (int s = 0; s < 3; ++s) { a[s][0] = 0.0; a[s][1] = 0.0; a[s][2] = 0.0; }
#pragma unroll
    for (int j = 0; j < 15; ++j) {
        if (MS == 0 && j >= M) break;
        const double t = T[j * MP16 + row];
        const double2 v01 = *reinterpret_cast<const double2*>(v + 4 * j);
        const double v2 = v[4 * j + 2];
        a[j % 3][0] = fma(t, v01.x, a[j % 3][0]);
        a[j % 3][1] = fma(t, v01.y, a[j % 3][1]);
        a[j % 3][2] = fma(t, v2, a[j % 3][2]);
    }
    o0 = (a[0][0] + a[1][0]) + a[2][0];
    o1 = (a[0][1] + a[1][1]) + a[2][1];
    o2 = (a[0][2] + a[1][2]) + a[2][2];
}

// All four stages starting from the strain samples K.  MS = M when it is fixed at compile time (15), else 0.
template <int MS>
__global__ void __launch_bounds__(kFusedThreads, kFusedMinBlocks) fused16_kernel(const FusedParams p) {
    if (p.skip && *p.skip) return;  // Newton loop: the solve has already converged (device-side flag), nothing to do
    extern __shared__ __align__(16) double smem[];
    double* tab = smem;  // OpsLayout16::total doubles
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sub = lane >> 4, row = lane & 15;
    double* scr = smem + OpsLayout16::total + warp * kWarpScratch16 + sub * RodScratch::total;
    double* qnode = scr + RodScratch::qnode;
    double* vec = scr + RodScratch::vec;
    double* vec2 = scr + RodScratch::vec2;
    double* misc = scr + RodScratch::misc;

    const bool listed = p.rod_list != nullptr;  // second pass over the rods the DMMA kernel handed back
    const long long batch = listed ? (long long)*p.rod_count : p.batch;
    const long long pairs = (batch + 1) >> 1;
    if ((long long)blockIdx.x * (blockDim.x >> 5) >= pairs) return;  // whole CTA idle (the usual case of a second pass)
    for (int i = threadIdx.x; i < OpsLayout16::total; i += blockDim.x) tab[i] = p.ops[i];
    __syncthreads();

    const int M = MS ? MS : p.M;
    const int N = M + 1;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    const long long pair0 = (long long)blockIdx.x * (blockDim.x >> 5) + warp;

    // strain samples (and q0) of the rod at position `idx_` -> kbuf[slot]; lanes outside the rod / batch write zeros
    // (q0: identity)
    auto prefetch_K = [&](long long idx_, int slot) {
        double* kb = scr + RodScratch::kbuf + slot * 64;
        const bool ok = idx_ < batch;
        const long long rod_ = (ok && listed) ? (long long)p.rod_list[idx_] : idx_;
        if (ok && row < N) {
            const double* s = p.K + rod_ * 3 * N + row;
            cp_async8(kb + row, s); cp_async8(kb + 16 + row, s + N); cp_async8(kb + 32 + row, s + 2 * N);
        } else {
            kb[row] = 0.0; kb[16 + row] = 0.0; kb[32 + row] = 0.0;
        }
        if (row < 4) {
            if (ok && p.q0) cp_async8(kb + 48 + row, p.q0 + rod_ * 4 + row);
            else kb[48 + row] = (row == 0) ? 1.0 : 0.0;
        }
    };

    if (pair0 < pairs) prefetch_K(2 * pair0 + sub, 0);
    cp_async_commit();

    int it = 0;
    for (long long pair = pair0; pair < pairs; pair += warps_total, ++it) {
        const long long idx = 2 * pair + sub;
        const bool live = idx < batch;
        const long long rod = (live && listed) ? (long long)p.rod_list[idx] : idx;
        const int cur = it & 1;

        // ---- prefetch: this pair's late inputs and the next pair's strain samples -----------------------
        if (live && row < N) {
            if (p.fbar) { const double* s = p.fbar + rod * 3 * N + row; double* d = scr + RodScratch::fbar + row;
                          cp_async8(d, s); cp_async8(d + 16, s + N); cp_async8(d + 32, s + 2 * N); }
            if (p.lbar) { const double* s = p.lbar + rod * 3 * N + row; double* d = scr + RodScratch::lbar + row;
                          cp_async8(d, s); cp_async8(d + 16, s + N); cp_async8(d + 32, s + 2 * N); }
            if (p.Gamma) { const double* s = p.Gamma + rod * 3 * N + row; double* d = scr + RodScratch::gam + row;
                           cp_async8(d, s); cp_async8(d + 16, s + N); cp_async8(d + 32, s + 2 * N); }
        }
        if (live && row < 3) {
            if (p.F_tip) cp_async8(misc + row, p.F_tip + rod * 3 + row);
            if (p.M_tip) cp_async8(misc + 3 + row, p.M_tip + rod * 3 + row);
            if (p.r0) cp_async8(misc + 6 + row, p.r0 + rod * 3 + row);
        }
        if (pair + warps_total < pairs) prefetch_K(2 * (pair + warps_total) + sub, cur ^ 1);
        cp_async_commit();
        cp_async_wait<1>();  // everything but the group just committed: this pair's K and q0 have landed
        __syncwarp();

        const double* kb = scr + RodScratch::kbuf + cur * 64;
        quat q0;
        {
            const double2 a = *reinterpret_cast<const double2*>(kb + 48);
            const double2 c2 = *reinterpret_cast<const double2*>(kb + 50);
            q0.w = a.x; q0.x = a.y; q0.y = c2.x; q0.z = c2.y;
        }
        quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
        // ---- stage 1: assemble c_ij = delta_ij - 1/2 S_ij (0,K_j) and eliminate -------------------------
        int sing;
        {
            quat c[15], b;
#pragma unroll
            for (int j = 0; j < 15; ++j) {
                const double s = tab[OpsLayout16::St + j * MP16 + row];  // -1/2 S_ij
                c[j].w = (j == row) ? 1.0 : 0.0;
                c[j].x = s * kb[j]; c[j].y = s * kb[16 + j]; c[j].z = s * kb[32 + j];
            }
            {
                const double gi = tab[OpsLayout16::g + row];
                b.w = gi * q0.w; b.x = gi * q0.x; b.y = gi * q0.y; b.z = gi * q0.z;
            }
            int mycol;
            gauss_jordan16(c, b, M, row, scr + RodScratch::pbuf, mycol, sing);
            __syncwarp();
            if (row < M) st_quat(qnode + 4 * mycol, b);
        }
        if (row == M) st_quat(qnode + 4 * M, q0);
        if (p.info && live && row == 0) p.info[rod] = sing;
        cp_async_wait<0>();
        __syncwarp();
        if (row <= M) q = ld_quat(qnode + 4 * row);
        if (p.Q && live && row < M) {
            double* d = p.Q + rod * 4 * M + row;
            d[0] = q.w; d[M] = q.x; d[2 * M] = q.y; d[3 * M] = q.z;
        }

        if (p.r || p.n || p.m) {
            // ---- stage 2: r = S (R(q) Gamma) + g r0 -----------------------------------------------------
            double bv0 = 0.0, bv1 = 0.0, bv2 = 0.0;
            if (row <= M) {
                if (p.Gamma && live) {
                    const double* gm = scr + RodScratch::gam + row;
                    q_rotate(q, gm[0], gm[16], gm[32], bv0, bv1, bv2);
                } else {
                    q_rotate_e1(q, bv0, bv1, bv2);
                }
            }
            {
                quat t; t.w = bv0; t.x = bv1; t.y = bv2; t.z = 0.0;
                st_quat(vec + 4 * row, t);
            }
            // ---- stage 3 right-hand side (independent of stage 2; issued before the barrier) -----------
            double F0 = 0.0, F1 = 0.0, F2 = 0.0;
            if ((p.n || p.m) && live && p.F_tip) { F0 = misc[0]; F1 = misc[1]; F2 = misc[2]; }
            const bool contract3 = (p.n || p.m) && p.fbar;
            if (contract3) {
                const double dti = tab[OpsLayout16::DTI + row];
                double f0 = 0.0, f1 = 0.0, f2 = 0.0;
                if (live && row < M) { const double* s = scr + RodScratch::fbar + row + 1; f0 = s[0]; f1 = s[16]; f2 = s[32]; }
                quat t; t.w = -f0 - dti * F0; t.x = -f1 - dti * F1; t.y = -f2 - dti * F2; t.z = 0.0;
                st_quat(vec2 + 4 * row, t);
            }
            __syncwarp();
            if (p.r) {
                double a0, a1, a2;
                contract16<MS>(tab + OpsLayout16::Sp, vec, M, row, a0, a1, a2);
                if (p.r0 && live) {
                    const double gi = tab[OpsLayout16::g + row];
                    a0 = fma(gi, misc[6], a0); a1 = fma(gi, misc[7], a1); a2 = fma(gi, misc[8], a2);
                }
                if (live && row < M) {
                    double* d = p.r + rod * 3 * M + row;
                    d[0] = a0; d[M] = a1; d[2 * M] = a2;
                }
            }
            if (p.n || p.m) {
                // ---- stage 3: n = D_TT^-1 (-fbar - D_TI F_tip^T); lane `row` = reduced index (node row+1)
                double n0, n1, n2;
                if (contract3) {
                    contract16<MS>(tab + OpsLayout16::STt, vec2, M, row, n0, n1, n2);
                } else {
                    const double gi = tab[OpsLayout16::gT + row];
                    n0 = gi * F0; n1 = gi * F1; n2 = gi * F2;
                }
                if (p.n && live && row < M) {
                    double* d = p.n + rod * 3 * M + row;
                    d[0] = n0; d[M] = n1; d[2 * M] = n2;
                }
                if (p.m) {
                    // ---- stage 4: m = D_TT^-1 (-(r' x n + lbar) - D_TI M_tip^T) ------------------------
                    double T0 = 0.0, T1 = 0.0, T2 = 0.0;
                    if (live) { T0 = misc[3]; T1 = misc[4]; T2 = misc[5]; }
                    const int nb = (row < M) ? row + 1 : row;  // node of this reduced row
                    const double2 rp01 = *reinterpret_cast<const double2*>(vec + 4 * nb);
                    const double rp2 = vec[4 * nb + 2];
                    double l0 = 0.0, l1 = 0.0, l2 = 0.0;
                    if (p.lbar && live && row < M) { const double* s = scr + RodScratch::lbar + row + 1; l0 = s[0]; l1 = s[16]; l2 = s[32]; }
                    const double dti = tab[OpsLayout16::DTI + row];
                    const double c0 = rp01.y * n2 - rp2 * n1, c1 = rp2 * n0 - rp01.x * n2, c2 = rp01.x * n1 - rp01.y * n0;
                    quat t; t.w = -(c0 + l0) - dti * T0; t.x = -(c1 + l1) - dti * T1; t.y = -(c2 + l2) - dti * T2; t.z = 0.0;
                    if (row >= M) { t.w = 0.0; t.x = 0.0; t.y = 0.0; }
                    __syncwarp();  // every lane has read vec2 (stage 3) before it is overwritten
                    st_quat(vec2 + 4 * row, t);
                    __syncwarp();
                    double m0, m1, m2;
                    contract16<MS>(tab + OpsLayout16::STt, vec2, M, row, m0, m1, m2);
                    if (live && row < M) {
                        double* d = p.m + rod * 3 * M + row;
                        d[0] = m0; d[M] = m1; d[2 * M] = m2;
                    }
                }
            }
        }
        __syncwarp();  // scratch is reused by the next iteration
    }
    cp_async_wait<0>();
}

}  // namespace sri
