// sri_fused16_dmma.cuh -- fused four-stage kernel for N <= 16 with the quaternion elimination on the FP64 tensor
// cores (DMMA m8n8k4).  ONE rod per warp.  Lane-exact numpy model of stage 1: tools/dmma_gj_emulator.py (solve_rod_lu).
//
// Replaces, per rod, the same reference code as sri_fused16.cuh (updateA main.cpp:55-88, A_NN.inverse()*(b-ivp)
// main.cpp:113, updatePositionb main.cpp:121-140, Dn_NN_inv*(b_NN-ivp) main.cpp:172) plus rod_modeling.pdf 1.17-1.18.
//
// Why: in the scalar kernel a row lives in one lane and the pivot row has to be broadcast through the LSU, which is
// what bounds it (DESIGN.md 2.1).  The DMMA data path does that broadcast for free.  The M x M quaternion system
//      sum_j Q_j (x) c_ij = b_i
// is stored as the REAL 64 x 16 matrix  Cr[4 i + r][j] = component r of c_ij  (column 15 = b_i), i.e. 8 x 2 DMMA
// accumulator tiles of 8 x 8 = 32 doubles per lane.  With vec(a (x) b) = Rmat(b) vec(a), elimination step k is
//      U'  = Rmat(c_kk^-1) U            U = pivot row as a 4 x 16 matrix (one DMMA per column tile)
//      Cr -= [...; Rmat(c_kk - 1); Rmat(c_k+1,k); ...] U'     (rank-4 update of the tile rows below the pivot, k = 4)
// 4 x 4 real blocks appear only in the A operand (the multipliers); the matrix itself stays in quaternion (4-vector)
// form, so the DMMAs execute exactly the 16 FMAs per quaternion multiply-add of the scalar kernel.
// Per step the LSU only moves the pivot row into B-fragment layout (2 SHFL.64 per column tile), one component of the
// pivot element and its squared norm to every lane (2 SHFL.64) and the pivot column into A-fragment layout (1 SHFL.64
// per live row tile), and stores -U' to shared memory.  The back-substitution then runs with the rows on the n axis:
//      -Q_i = -U'_i,15 + sum_{j>i} Lmat(-Q_j) (-U'_ij),    vec(a (x) b) = Lmat(a) vec(b),
// so one DMMA (A = Lmat(-Q_j), B = column j of -U' over 8 rows) serves 8 rows.  Per rod: 107 updates, 23
// normalisations, 20 back-substitution DMMAs.  Stages 2-4 are [16 x 16] x [16 x 3] DMMA contractions in the same
// warp (16 DMMAs; Q never leaves the SM): 166 DMMAs in all.
//
// Pivoting: the order is static (pivot k = row k).  The left-preconditioned operator I - 1/2 S diag(kappa) has
// |c_kk| >= 1 and measured sub-diagonal growth <= 0.15 for |K| <= 10 and <= 2.4 for |K| <= 300, so a search would
// almost never move a row.  Every step still checks  max_{i>k} |c_ik| <= G |c_kk|  (and c_kk != 0); a rod that
// fails is appended to a list and re-solved by the row-pivoting scalar kernel (sri_fused16.cuh) right after.
#pragma once
#include "sri_fused16.cuh"
#include "sri_stage_dmma.cuh"

namespace sri {

#ifndef SRI_DMMA_MINBLOCKS
#define SRI_DMMA_MINBLOCKS 4
#endif
#ifndef SRI_DMMA_THREADS
#define SRI_DMMA_THREADS 128
#endif
constexpr int kDmmaThreads = SRI_DMMA_THREADS;
constexpr double kDmmaGrowthDefault = 4.0;  // accepted max_{i>k} |c_ik| / |c_kk| (SRI_DMMA_GROWTH overrides)

// Tables appended to the StageTables block (all strain independent, built by sri_api.cu):
//   Stx[i][j] (row-major 16 x 16) = -1/2 (Dn_NN^-1)(i,j) for i, j < M,  Stx[i][15] = g_i = -(Dn_NN^-1 Dn_IN)_i
//   AS, AT: A fragments of the stage operators in DMMA fragment order, X[(mt*4 + kt)*32 + lane] =
//           Xt[8 mt + lane/4][4 kt + lane%4], with the boundary term as k index 15:
//           St[i][j<15] = (Dn_NN^-1)(i,j), St[i][15] = g_i;   Tt[i][j<15] = -(D_TT^-1)(i,j), Tt[i][15] = gT_i
struct DmmaTables {
    static constexpr int Stx = StageTables::total;
    static constexpr int AS = Stx + 256;
    static constexpr int AT = AS + 256;
    static constexpr int total = AT + 256;
};
constexpr int kDmmaTabDoubles = 768;  // Stx | AS | AT in shared memory

// Per-warp shared scratch (doubles).  The [4][20] arrays hold a 3 x 16 right-hand side by (component, k index) with
// the boundary value in k slot 15 and an all-zero fourth row (the unused columns of the B fragments); row stride 20
// keeps the four rows on disjoint banks.
struct DmmaScratch {
    static constexpr int kx = 0;                // [2][4][16] (double buffered): row 0 = (0,..,0,q0w), rows 1..3 = (K_c[0..M-1], 0.., q0_c)
    static constexpr int bs = kx + 128;         // [4][20] r' = R(q) Gamma at nodes 0..14 | r0
    static constexpr int fbs = bs + 80;         // [4][20] fbar at nodes 1..M in REVERSED order (slot j = node M-j) | F_tip
    static constexpr int xs = fbs + 80;         // [4][20] r' x n + lbar at nodes 1..15 | M_tip
    static constexpr int rps = xs + 80;         // [3][16] r' at all 16 nodes
    static constexpr int lbs = rps + 48;        // [3][16] lbar at nodes 1..15 (slot j = node j+1)
    static constexpr int gam = lbs + 48;        // [3][16] Gamma by node
    static constexpr int ns = gam + 48;         // [3][16] n by reduced row
    static constexpr int qnode = ns + 48;       // [16][4] quaternions by node (slot M = base node)
    static constexpr int ust = qnode + 64;      // -U' of every pivot row, [col j][row i][s] from ucol(j) (see below)
    static constexpr int total = ust + 740;     // 1364 doubles
};
// Column j of the stored -U'.  Column j < 8 is written by steps k <= 6 and read for rows i < j only, so it needs 7
// rows and shares a 92-double slot with column j + 8 (16 rows): one store pointer serves both column tiles.  The slot
// stride is 12 mod 16 doubles, so the eight columns one B fragment stores start on distinct bank quads and a step's
// store is conflict free.  A back-substitution read is 32 consecutive doubles (8 rows, those at or below j unused).
__host__ __device__ constexpr int ucol(int j) { return j < 8 ? 92 * j + 64 : 92 * (j - 8); }
static_assert(ucol(7) + 32 <= 740, "DmmaScratch::ust size");
constexpr size_t kDmmaSmem = (kDmmaTabDoubles + (kDmmaThreads / 32) * DmmaScratch::total) * sizeof(double);

#ifndef SRI_DMMA_VOLATILE
#define SRI_DMMA_VOLATILE
#endif
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm SRI_DMMA_VOLATILE("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ double dmma_zero(double a, double b) {  // column 0/2/4/6 of A*B (C fragment register 0)
    double d0, d1;
    const double z = 0.0;
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%4,%4};" : "=d"(d0), "=d"(d1) : "d"(a), "d"(b), "d"(z));
    (void)d1;
    return d0;
}
__device__ __forceinline__ double flip_sign(double v, unsigned mask) {
    return __hiloint2double(__double2hiint(v) ^ (int)mask, __double2loint(v));
}

// One cached-operator stage on the tensor cores: out[16 x 3] = At[16 x 16] * rhs[16 x 3], A fragments from the
// fragment-ordered table `at`, B fragments from a [4][20] right-hand side (lane reads component min(rho,3), k = 4kt+cp).
template <int KT0>
__device__ __forceinline__ void stage_dmma16(const double* at, const double* rhs_lane, int lane, double (&acc)[2][2]) {
    acc[0][0] = 0.0; acc[0][1] = 0.0; acc[1][0] = 0.0; acc[1][1] = 0.0;
#pragma unroll
    for (int kt = KT0; kt < 4; ++kt) {
        const double b = rhs_lane[4 * kt];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) dmma(acc[mt][0], acc[mt][1], at[(mt * 4 + kt) * 32 + lane], b);
    }
}
// C fragment -> [3][M] stack in global memory: lane (rho, cp) holds reduced row 8 mt + rho, components 2cp, 2cp+1
__device__ __forceinline__ void store_stage(double* out, int M, int rho, int cp, const double (&acc)[2][2]) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int i = 8 * mt + rho;
        if (i < M) {
            if (cp == 0) { out[i] = acc[mt][0]; out[M + i] = acc[mt][1]; }
            else if (cp == 1) out[2 * M + i] = acc[mt][0];
        }
    }
}

template <int MS>
#ifdef SRI_DMMA_MAXNREG
__global__ void __maxnreg__(SRI_DMMA_MAXNREG) fused16_dmma_kernel(const FusedParams p) {
#else
__global__ void __launch_bounds__(kDmmaThreads, SRI_DMMA_MINBLOCKS) fused16_dmma_kernel(const FusedParams p) {
#endif
    if (p.skip && *p.skip) return;  // Newton loop: the solve has already converged (device-side flag), nothing to do
    extern __shared__ __align__(16) double smem[];
    double* stx = smem;             // 256 doubles
    double* tabAS = smem + 256;     // 256
    double* tabAT = smem + 512;     // 256
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* scr = smem + kDmmaTabDoubles + warp * DmmaScratch::total;
    double* qnode = scr + DmmaScratch::qnode;

    constexpr int kWarps = kDmmaThreads / 32;
    if ((long long)blockIdx.x * kWarps >= p.batch) return;  // whole CTA idle
    for (int i = threadIdx.x; i < kDmmaTabDoubles; i += kDmmaThreads) smem[i] = p.ops[DmmaTables::Stx + i];
    for (int i = lane; i < DmmaScratch::total; i += 32) scr[i] = 0.0;
    __syncthreads();

    const int M = MS ? MS : p.M;
    const int N = M + 1;
    // fragment coordinates of this lane
    const int rho = lane >> 2, cp = lane & 3;  // C fragment: row rho, columns 2cp, 2cp+1
    const int hi = rho >> 2, rr = rho & 3;     // quaternion row within the tile, component
    // node coordinates of the pointwise stage work
    const int row = lane & 15, half = lane >> 4;

    // lane constants of the elimination (see tools/dmma_gj_emulator.py)
    const int srcU_base = 4 * cp + (lane >> 3);
    const bool odd_col = (rho & 1) != 0;
    const int srcL_base = 16 * hi + 4 * (rr ^ cp);
    // Rmat(b)[r][s] = sg(r,s) b[r^s]: rows (+,-,-,-), (+,+,+,-), (+,-,+,+), (+,+,-,+)
    const unsigned neg_tab = 0x428Eu;  // bit (4r+s) set where sg(r,s) = -1: r0: s1,s2,s3; r1: s3; r2: s1; r3: s2
    const unsigned sgL_mask = ((neg_tab >> (4 * rr + cp)) & 1u) << 31;
    const double dpiv0 = (hi == 0 && rr == cp) ? 1.0 : 0.0;  // the pivot's tile row is live only for even k
    const unsigned hi_mask = hi ? 0x7fffffffu : 0u;
    // normalisation operand: B[q = cp][n = rho]; even n = 2 s' carries Rmat(conj c)[s'][q] = sg(s',q) conj(c)[s'^q]
    // (odd columns feed C-fragment register 1, which is discarded: don't-care)
    const int sp = rho >> 1;
    const int idxN = sp ^ cp;
    const unsigned sgN_mask = ((((neg_tab >> (4 * sp + cp)) & 1u) != 0) != (idxN != 0)) ? 0x80000000u : 0u;
    // identity entries of the assembly: tile (t, ct), register e holds delta_ij iff rr == 0, hi == e, cp == t - 4 ct
    const int diag_code = (rr == 0) ? (4 * hi + cp) : -1;
    // -U' store of step k: lane (rho, cp) holds component cp of column 8 ct + rho
    double* const ustl = scr + DmmaScratch::ust + 92 * rho + cp;
    // B-fragment read offset into a [4][20] right-hand side
    const int offb = (rho < 3 ? rho : 3) * 20 + cp;
    // stages 2+3 in one contraction: columns 0..2 = r' (bs), columns 3..5 = reversed fbar (fbs), the rest the zero row of bs
    const int offb23 = (rho < 3 ? DmmaScratch::bs + rho * 20 : (rho < 6 ? DmmaScratch::fbs + (rho - 3) * 20 : DmmaScratch::bs + 60)) + cp;

    const long long stride = (long long)gridDim.x * kWarps;
    const long long rod0 = (long long)blockIdx.x * kWarps + warp;

    // strain samples and q0 of rod `rod_` -> kx[slot]
    auto prefetch_K = [&](long long rod_, int slot) {
        double* kb = scr + DmmaScratch::kx + slot * 64;
        if (row < M) {
            const double* s = p.K + rod_ * 3 * N + row;
            if (half == 0) { cp_async8(kb + 16 + row, s); cp_async8(kb + 32 + row, s + N); }
            else cp_async8(kb + 48 + row, s + 2 * N);
        }
        if (lane < 4) {
            if (p.q0) cp_async8(kb + 16 * lane + 15, p.q0 + rod_ * 4 + lane);
            else kb[16 * lane + 15] = (lane == 0) ? 1.0 : 0.0;
        }
    };

    if (rod0 < p.batch) prefetch_K(rod0, 0);
    cp_async_commit();

    int it = 0;
    for (long long rod = rod0; rod < p.batch; rod += stride, ++it) {
        const int cur = it & 1;
        // ---- prefetch: this rod's late inputs (nodal loads shifted to reduced rows, boundary values into k slot 15)
        //      and the next rod's strain samples -------------------------------------------------------------------
        if (row < N) {
            const int c0 = half ? 2 : 0, c1 = half ? 3 : 2;  // half 0: components 0, 1; half 1: component 2
            for (int c = c0; c < c1; ++c) {
                if (p.fbar && row >= 1) cp_async8(scr + DmmaScratch::fbs + 20 * c + (M - row), p.fbar + (rod * 3 + c) * N + row);  // flipped, see stages 2+3
                if (p.lbar && row >= 1) cp_async8(scr + DmmaScratch::lbs + 16 * c + row - 1, p.lbar + (rod * 3 + c) * N + row);
                if (p.Gamma) cp_async8(scr + DmmaScratch::gam + 16 * c + row, p.Gamma + (rod * 3 + c) * N + row);
            }
        }
        if (lane < 3) { if (p.F_tip) cp_async8(scr + DmmaScratch::fbs + 20 * lane + 15, p.F_tip + rod * 3 + lane); }
        else if (lane >= 4 && lane < 7) { if (p.M_tip) cp_async8(scr + DmmaScratch::xs + 20 * (lane - 4) + 15, p.M_tip + rod * 3 + lane - 4); }
        else if (lane >= 8 && lane < 11) { if (p.r0) cp_async8(scr + DmmaScratch::bs + 20 * (lane - 8) + 15, p.r0 + rod * 3 + lane - 8); }
        if (rod + stride < p.batch) prefetch_K(rod + stride, cur ^ 1);
        cp_async_commit();
        cp_async_wait<1>();  // everything but the group just committed: this rod's K and q0 have landed
        __syncwarp();

        const double* kb = scr + DmmaScratch::kx + cur * 64;
        // ---- stage 1: assemble Cr = delta - 1/2 S_ij (0,K_j) | g_i q0 in C-fragment layout -------------------------
        double c[8][2][2];
        {
            double kq[2][2];
#pragma unroll
            for (int ct = 0; ct < 2; ++ct) {
                const double2 v = *reinterpret_cast<const double2*>(kb + 16 * rr + 8 * ct + 2 * cp);
                kq[ct][0] = v.x; kq[ct][1] = v.y;
            }
#pragma unroll
            for (int t = 0; t < 8; ++t)
#pragma unroll
                for (int ct = 0; ct < 2; ++ct) {
                    const double2 s = *reinterpret_cast<const double2*>(stx + (2 * t + hi) * 16 + 8 * ct + 2 * cp);
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int dcode = 4 * e + (t - 4 * ct);  // compile-time
                        const bool candidate = (t - 4 * ct >= 0) && (t - 4 * ct < 4) && !(ct == 1 && t == 7 && e == 1);
                        const double d = (candidate && diag_code == dcode) ? 1.0 : 0.0;
                        c[t][ct][e] = fma(e ? s.y : s.x, kq[ct][e], d);
                    }
                }
        }
        // ---- forward elimination over the quaternions on DMMA, static pivot order, software pipelined ----------
        // Step k normalises pivot row k, stores it (-U'_k) to shared memory and eliminates column k from the rows
        // below it.  A stored pivot row is never read from the tiles again, so step k updates only tile rows
        // t >= (k+1)/2 (the pivot's own tile row only while row k+1 shares it), and the last step updates nothing.
        // Iteration k issues the rank-4 update of step k and, behind it, everything step k+1 needs: its tile row, the
        // first live one, is updated first, then the next pivot row is gathered and normalised; each la[t] is
        // re-gathered for step k+1 as soon as tile row t has been updated.  k = -1 is the prologue (no update).
        // Scalar FP64 instructions share the pipe with the DMMAs and queue behind them, so the serial scalar chain is
        // kept to three operations per step: U (x) conj(c_kk) is itself a DMMA, whose (column k, w) entry is |c_kk|^2,
        // and its reciprocal (MUFU seed, e = 1 - nu r0, t2 = e + e^2) is folded into the scaling of that product.
        bool bad = false;
        const int growth_log = p.growth_log;
        double la[8], un[2];
#pragma unroll
        for (int k = -1; k < 15; ++k) {
            const int kn = k + 1;  // the step being prepared
            const bool upd = (k >= 0) && (k < 14) && (MS != 0 || k < M - 1);
            const bool prep = (kn < 15) && (MS != 0 || kn < M);
            const int nt = (kn >> 1) & 7, nh = kn & 1, nc = (kn >> 3) & 1, ncp = (kn & 7) >> 1, ne = kn & 1;
            // 1. step k on the tile row of the next pivot (= its first live tile row)
            if (upd) {
#pragma unroll
                for (int ct = 0; ct < 2; ++ct)
                    if (8 * ct + 7 > k) dmma(c[nt][ct][0], c[nt][ct][1], la[nt], un[ct]);
            }
            double un0[2] = {0.0, 0.0}, r0n = 0.0, t2 = 0.0;
            unsigned mx = 0u;
            int thr = 0;
            if (prep) {
                // next pivot row -> B fragments: lane wants U[s = cp][col = 8 ct + rho]
                const int srcU = 16 * nh + srcU_base;
                // this lane's entry of Rmat(conj c_kk), straight from the pivot's tile
                const double pcs = __shfl_sync(0xffffffffu, c[nt][nc][ne], 16 * nh + 4 * idxN + ncp);
                const double bn0 = flip_sign(pcs, sgN_mask);
#pragma unroll
                for (int ct = nc; ct < 2; ++ct) {
                    const double v0 = __shfl_sync(0xffffffffu, c[nt][ct][0], srcU);
                    const double v1 = __shfl_sync(0xffffffffu, c[nt][ct][1], srcU);
                    un0[ct] = dmma_zero(odd_col ? v1 : v0, bn0);  // U (x) conj(c_kk), B-fragment layout
                }
                const double nu = __shfl_sync(0xffffffffu, un0[nc], 4 * (kn & 7));  // |c_kk|^2
                double r0;
                asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(nu));
                const double e = fma(-nu, r0, 1.0);
                t2 = fma(e, e, e);  // 1/nu = r0 (1 + e + e^2) to ~1e-16
                r0n = flip_sign(r0, 0x80000000u);
                // growth bound in the log domain (hi word of a positive double ~ 2^20 (log2 + 1023)):
                //   |c_ik| <= G |c_kk|  <=>  2 H(|c_ik|) <= H(nu) + (1023 << 20) + 2^20 log2(G^2)
                const int hn = __double2hiint(nu);
                thr = (int)(((long long)hn + 0x3ff00000LL + (long long)growth_log) >> 1);
                if (hn < 0x05000000 || hn >= 0x7ff00000) thr = -1;  // zero / tiny / negative / inf / NaN pivot norm
            }
            // 2. step k on the other live tile rows; la[t] is re-gathered for step k+1 once tile row t is done (step
            //    k+1 needs tile rows t >= (kn+1)/2: the next pivot's own tile row only when kn is even)
            const int srcL = srcL_base + ncp;
#pragma unroll
            for (int t = nt; t < 8; ++t) {
                if (upd && t != nt) {
#pragma unroll
                    for (int ct = 0; ct < 2; ++ct)
                        if (8 * ct + 7 > k) dmma(c[t][ct][0], c[t][ct][1], la[t], un[ct]);
                }
                if (prep && (t != nt || nh == 0)) {
                    const double v = __shfl_sync(0xffffffffu, c[t][nc][ne], srcL);
                    const unsigned h = (unsigned)__double2hiint(v) & 0x7fffffffu;
                    mx = max(mx, t != nt ? h : (h & hi_mask));
                    la[t] = flip_sign(v, sgL_mask);
                    if (t == nt) la[t] -= dpiv0;  // pivot row: Rmat(c_kk - 1) leaves the normalised row
                }
            }
            // 3. -U' = -(U (x) conj c_kk) / nu for the next step, and into the store for the back-substitution
            if (prep) {
                bad = bad || ((int)mx > thr);
#pragma unroll
                for (int ct = 0; ct < 2; ++ct)
                    if (8 * ct + 7 > kn) {
#ifdef SRI_DMMA_RFOLD
                        un[ct] = un0[ct] * fma(r0n, t2, r0n);
#else
                        const double a = un0[ct] * r0n; un[ct] = fma(a, t2, a);
#endif
                        ustl[(ct ? ucol(8) : ucol(0)) + 4 * kn] = un[ct];
                    }
            }
        }
        const bool flagged = __any_sync(0xffffffffu, bad);
        __syncwarp();  // the -U' stores above are read across lanes below
        // ---- back-substitution on DMMA: with W = -U' (stored) and C' = -Q,  C'_i = W_i,15 + sum_{j>i} Lmat(C'_j) W_ij
        //      (vec(a (x) b) = Lmat(a) vec(b)).  C' lives in one C tile per 8-row block, component s on the m axis
        //      (m >= 4 stays zero) and row 8b + n on the n axis, so one DMMA subtracts Q_j (x) U'_ij from 8 rows: the
        //      A operand is Lmat(C'_j), one shuffle and a sign; the B operand is column j of W over the block.
        //      C'_j is final once every j' > j has been applied, and is written to qnode as Q_j.
        {
            // the lane is re-read here so that its constants below are not held (and spilled) across the elimination
            int ln;
            asm volatile("mov.u32 %0, %%laneid;" : "=r"(ln));
            const int qm = ln >> 2, qs = ln & 3;  // A: row m, k index s;  B: k index s, n = row within the block
            const double* ust = scr + DmmaScratch::ust;
            double y[2][2];
#pragma unroll
            for (int b = 0; b < 2; ++b)
#pragma unroll
                for (int e = 0; e < 2; ++e) y[b][e] = qm < 4 ? ust[ucol(15) + 4 * (8 * b + 2 * qs + e) + (qm & 3)] : 0.0;
            // Lmat(a)[r][s] = sg(r,s) a[r^s]: rows (+,-,-,-), (+,+,-,+), (+,+,+,-), (+,-,+,+)
            const unsigned sgQ_mask = ((0x284Eu >> (4 * (qm & 3) + qs)) & 1u) << 31;
            const int srcQ_base = 4 * (qm ^ qs);  // m >= 4 reads the zero rows 4..7: the padded A rows stay zero
#pragma unroll
            for (int j = 14; j >= 0; --j) {
                if (MS != 0 || j < M) {
                    const int b = j >> 3, n = j & 7;
                    const double v = __shfl_sync(0xffffffffu, y[b][n & 1], srcQ_base + (n >> 1));  // C'_j[qm ^ qs]
                    if (qm < 4 && qs == 0) qnode[4 * j + qm] = flip_sign(v, 0x80000000u);
                    const double a = flip_sign(v, sgQ_mask);
#pragma unroll
                    for (int bb = 0; bb <= b; ++bb)
                        if (8 * bb < j) dmma(y[bb][0], y[bb][1], a, ust[ucol(j) + 32 * bb + ln]);
                }
            }
        }
        cp_async_wait<0>();
        // a flagged rod needs row pivoting: it is handed to the scalar kernel; its stores below are suppressed (no
        // divergent `continue`, which would wrap every later shuffle in WARPSYNC/ENDCOLLECTIVE pairs)
        const bool keep = !(flagged && p.rod_list);
        if (!keep && lane == 0) p.rod_list[atomicAdd(p.rod_count, 1)] = (int)rod;
        __syncwarp();
        if (lane < 4) qnode[4 * M + lane] = kb[16 * lane + 15];  // base node: q0
        if (p.info && keep && lane == 0) p.info[rod] = flagged ? -1 : 0;
        __syncwarp();
        quat q; q.w = 1.0; q.x = 0.0; q.y = 0.0; q.z = 0.0;
        if (row <= M) q = ld_quat(qnode + 4 * row);
        if (p.Q && keep && row < M) {
            double* d = p.Q + rod * 4 * M + (2 * half) * M + row;
            d[0] = half ? q.y : q.w;
            d[M] = half ? q.z : q.x;
        }

        if (p.r || p.n || p.m) {
            // ---- stages 2-4 as [16 x 16] x [16 x 3] DMMA contractions against the cached operators; the boundary terms
            //      (g r0, gT F_tip, gT M_tip) ride along as k index 15, so the only scalar FP64 work left is pointwise:
            //      R(q) Gamma and the cross product r' x n.
            double bv0 = 0.0, bv1 = 0.0, bv2 = 0.0;
            if (row <= M) {
                if (p.Gamma) {
                    const double* gm = scr + DmmaScratch::gam + row;
                    q_rotate(q, gm[0], gm[16], gm[32], bv0, bv1, bv2);
                } else {
                    q_rotate_e1(q, bv0, bv1, bv2);
                }
            }
            if (half == 0) {
                double* rp = scr + DmmaScratch::rps + row;
                rp[0] = bv0; rp[16] = bv1; rp[32] = bv2;
                if (row < 15) { double* b = scr + DmmaScratch::bs + row; b[0] = bv0; b[20] = bv1; b[40] = bv2; }
            }
            __syncwarp();
            double acc[2][2];
            // stages 2 and 3 in ONE contraction against Dn_NN^-1: the Chebyshev matrix is centro-antisymmetric, so
            // -D_TT^-1 = J Dn_NN^-1 J (J = exchange matrix; 4e-16 on the as-built inverses, SURVEY T11) and gT = J g, hence
            //   r      = S (R(q) Gamma)    + g r0^T        -> columns 0..2 of the B operand, rows in natural order
            //   J n    = S (J fbar[1:])    + g F_tip^T     -> columns 3..5, right-hand side and result in reversed order
            // C fragment: lane (rho, cp) holds row 8 mt + rho of columns 2cp, 2cp+1.
            stage_dmma16<0>(tabAS, scr + offb23, lane, acc);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                const int i = 8 * mt + rho;
                if (i < M && keep) {
                    if (p.r) {
                        double* d = p.r + rod * 3 * M + i;
                        if (cp == 0) { d[0] = acc[mt][0]; d[M] = acc[mt][1]; }
                        else if (cp == 1) d[2 * M] = acc[mt][0];
                    }
                    if (p.n) {
                        double* d = p.n + rod * 3 * M + (M - 1 - i);
                        if (cp == 1) d[0] = acc[mt][1];
                        else if (cp == 2) { d[M] = acc[mt][0]; d[2 * M] = acc[mt][1]; }
                    }
                }
            }
            if (p.n || p.m) {
                if (p.m) {
                    // stage 4: m = (-D_TT^-1) (r' x n + lbar)[1:] + gT M_tip^T
                    double* nsv = scr + DmmaScratch::ns;
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        const int i = 8 * mt + rho;
                        if (i < M) {
                            if (cp == 1) nsv[M - 1 - i] = acc[mt][1];
                            else if (cp == 2) { nsv[16 + M - 1 - i] = acc[mt][0]; nsv[32 + M - 1 - i] = acc[mt][1]; }
                        }
                    }
                    __syncwarp();
                    if (half == 0 && row < 15) {
                        const double n0 = nsv[row], n1 = nsv[16 + row], n2 = nsv[32 + row];
                        const double* rp = scr + DmmaScratch::rps + row + 1;  // node of reduced row `row`
                        const double rp0 = rp[0], rp1 = rp[16], rp2 = rp[32];
                        double l0 = 0.0, l1 = 0.0, l2 = 0.0;
                        if (p.lbar) { const double* lb = scr + DmmaScratch::lbs + row; l0 = lb[0]; l1 = lb[16]; l2 = lb[32]; }
                        double* x = scr + DmmaScratch::xs + row;
                        x[0] = fma(rp1, n2, fma(-rp2, n1, l0));
                        x[20] = fma(rp2, n0, fma(-rp0, n2, l1));
                        x[40] = fma(rp0, n1, fma(-rp1, n0, l2));
                    }
                    __syncwarp();
                    stage_dmma16<0>(tabAT, scr + DmmaScratch::xs + offb, lane, acc);
                    if (keep) store_stage(p.m + rod * 3 * M, M, rho, cp, acc);
                }
            }
        }
        __syncwarp();  // scratch is reused by the next iteration
    }
    cp_async_wait<0>();
}

}  // namespace sri
