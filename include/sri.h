/*
 * sri.h -- C ABI of libsri_cuda.so: batched Chebyshev-collocation spectral integration of Cosserat-rod
 * kinematics and statics on NVIDIA B200 (sm_100a), FP64.
 *
 * This is the drop-in boundary for the one hot path of
 * aGotelli/experimental_gpu_programming_for_a_spectral_numerical_integration.  The reference has no FFI layer:
 * its "API" is the set of free functions compiled into main.cpp.  Each entry point below names the reference
 * function (file:line under /root/reference) it replaces.  include/sri_reference_api.hpp keeps the reference's
 * C++ function names on top of these symbols; INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions (identical to the reference so that a single-rod call is byte-compatible with Q_stack/r_stack):
 *   - N Chebyshev nodes, M = N-1.  Node 0 is the rod tip (X=1), node N-1 the base (X=0)
 *     (include/chebyshev_differentiation.h:26).
 *   - per-rod stacks are component-major, node-minor: Q[c*M+i] (main.cpp:80-81,130-133), r[c*M+i] (Eigen
 *     column-major (N-1)x3, main.cpp:172).  Batches are rod-major and contiguous: rod b's Q starts at Q + b*4*M.
 *   - stage 1/2 outputs cover nodes 0..N-2 (the base node carries the boundary condition, main.cpp:94-95);
 *     stage 3/4 outputs cover nodes 1..N-1 (the tip node carries the boundary condition).
 *   - nodal inputs K, Gamma, fbar, lbar are [batch][3][N] (component-major, node-minor, all N nodes).
 *   - every data pointer may be a host pointer or a device pointer on the handle's device (detected with
 *     cudaPointerGetAttributes); host buffers are staged through the handle's device workspace.
 *   - all functions return SRI_OK (0) or a negative sri_status; nothing throws across this boundary.
 *     There is no CPU fallback: without a usable CUDA device sri_create fails with SRI_ERR_CUDA.
 */
#ifndef SRI_H
#define SRI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRI_VERSION_MAJOR 0
#define SRI_VERSION_MINOR 5

typedef enum sri_status {
    SRI_OK = 0,
    SRI_ERR_INVALID_ARGUMENT = -1,
    SRI_ERR_UNSUPPORTED_N = -2,
    SRI_ERR_CUDA = -3,
    SRI_ERR_ALLOC = -4,
    SRI_ERR_SINGULAR = -5 /* at least one rod hit a zero / non-finite pivot: returned by calls with HOST buffers and a non-NULL
                             info array, after every output (the info array included) has been written; calls with device
                             buffers are asynchronous and report through info[] only */
} sri_status;

typedef struct sri_context* sri_handle;

/* ---- strain-independent spectral operator (host side, FP64, reference formula order) ------------------- */

/* ComputeChebyshevPoints<N,L>()  include/chebyshev_differentiation.h:19-30.  x[N], descending from L to 0. */
int sri_chebyshev_points(int N, double L, double* x);
/* GetCoefficients_c<N>()         include/chebyshev_differentiation.h:37-52.  c[N]. */
int sri_chebyshev_coefficients(int N, double* c);
/* getDn<N>()                     include/chebyshev_differentiation.h:59-108. Dn[N*N], column-major. */
int sri_chebyshev_dn(int N, double* Dn_colmajor);
/* Phi<na,ne>(X, begin, end)      include/utilities.h:49-67.  out[na * na*ne], column-major na x (na*ne). */
int sri_phi(int na, int ne, double X, double begin, double end, double* out_colmajor);

/* ---- handle ------------------------------------------------------------------------------------------- */

/* Builds the operator set for N nodes once (replaces the getDn/Kronecker/inverse rebuilds at main.cpp:93-100,
 * 157-160) and uploads it to `device`.  2 <= N <= 64. */
int sri_create(int N, int device, sri_handle* out);
int sri_destroy(sri_handle h);
/* Work is enqueued on this CUDA stream (a cudaStream_t passed as void*; NULL = the legacy default stream).
 * A new handle uses a non-blocking stream it owns; sri_reset_stream returns to it.
 * Calls with host buffers synchronise the stream before returning; calls with device buffers do not. */
int sri_set_stream(sri_handle h, void* cuda_stream);
int sri_reset_stream(sri_handle h);
int sri_synchronize(sri_handle h);
int sri_get_N(sri_handle h, int* N);
/* Copies one cached operator to a host buffer.  which: 0 Dn (N*N), 1 Dn_NN (M*M), 2 Dn_IN (M),
 * 3 Dn_NN^-1 (M*M), 4 D_TT (M*M), 5 D_TI (M), 6 D_TT^-1 (M*M); matrices column-major. */
int sri_get_operator(sri_handle h, int which, double* out);

/* ---- modal strain adapter ----------------------------------------------------------------------------- */

/* K = Phi<3,ne>(x_i) * qe at every node (main.cpp:69).  qe [batch][3*ne] -> K [batch][3][N]. */
int sri_strain_from_modes(sri_handle h, int64_t batch, int ne, const double* qe, double* K);
/* Its transpose (no quadrature weights, unlike sri_project_onto_modes): gqe[b][c*ne+k] = sum_i P_k(2 x_i - 1) gK[b][c][i],
 * the gradient with respect to qe of a function of K = Phi qe whose K-gradient is gK.  gK [batch][3][N] -> gqe [batch][3*ne],
 * 1 <= ne <= 8. */
int sri_strain_from_modes_transpose(sri_handle h, int64_t batch, int ne, const double* gK, double* gqe);

/* Rod length (SURVEY 8 f3).  The reference integrates on X in [0,1] with an implicit length of 1 (ComputeChebyshevPoints<N, 1>,
 * main.cpp:15).  For a rod of length l every ODE is multiplied by l (rod_modeling.pdf eq. 2.17): Q' = l/2 Q (x) (0,K),
 * r' = l R Gamma, n' = -l fbar, m' = -(r' x n + l lbar) -- i.e. the integrators are called with (l K, l Gamma, l fbar, l lbar),
 * tip loads and outputs unchanged.  This scales the given [batch][3][N] arrays IN PLACE (any of them may be NULL; host or
 * device pointers) by length[b] ([batch], host or device) or, when length == NULL, by uniform_length.  A rod with the
 * default Gamma = (1,0,0) needs an explicit Gamma array holding (1,0,0) at every node before the call. */
int sri_scale_for_length(sri_handle h, int64_t batch, const double* length, double uniform_length, double* K, double* Gamma,
                         double* fbar, double* lbar);

/* updateA()  main.cpp:55-88 on D_NN = I4 (x) Dn_NN (main.cpp:98,102): the assembled collocation operator of stage 1,
 * A_NN = D_NN - 1/2 blockdiag A(K_i), as the reference holds it before A_NN.inverse() (main.cpp:113).  The integration
 * kernels never form it (they eliminate the left-preconditioned quaternion system in registers); this entry point exists so
 * that the operator itself can be inspected and checked.  K [batch][3][N] -> A_NN [batch][4M*4M], column-major per rod. */
int sri_assemble_A(sri_handle h, int64_t batch, const double* K, double* A_NN);

/* ---- the four integration stages ---------------------------------------------------------------------- */

/* integrateQuaternions()  main.cpp:91-118 with updateA main.cpp:55-88.
 * Solves ((I4 (x) Dn_NN) - 1/2 blockdiag A(K_i)) Q = -D_IN q0 per rod.
 * K [batch][3][N]; q0 [batch][4] (w,x,y,z) or NULL => (1,0,0,0) (main.cpp:106-107); Q [batch][4][M];
 * info [batch] or NULL: 0 ok, k>0 = zero or non-finite pivot met at elimination step k (the reference would return inf/NaN). */
int sri_integrate_quaternions(sri_handle h, int64_t batch, const double* K, const double* q0, double* Q,
                              int* info);

/* integratePosition()  main.cpp:145-176 with updatePositionb main.cpp:121-140, minus the redundant second
 * quaternion solve (main.cpp:147): r = Dn_NN^-1 (R(q) Gamma - Dn_IN r0^T).
 * Q [batch][4][M]; Gamma [batch][3][N] or NULL => (1,0,0) (main.cpp:136); r0 [batch][3] or NULL => 0
 * (main.cpp:151-154); r [batch][3][M]. */
int sri_integrate_position(sri_handle h, int64_t batch, const double* Q, const double* Gamma, const double* r0,
                           double* r);

/* Internal force n' = -fbar, n(1) = F_tip.  Not implemented by the reference; spec: materials/rod_modeling.pdf
 * eq. 1.17 with the BC elimination of main.cpp:94-113 mirrored to the tip node.
 * fbar [batch][3][N] or NULL => 0; F_tip [batch][3]; n [batch][3][M] (nodes 1..N-1). */
int sri_integrate_stress(sri_handle h, int64_t batch, const double* fbar, const double* F_tip, double* n);

/* Internal couple m' = -(r' x n + lbar), m(1) = M_tip, r' = R(q) Gamma.  Spec: rod_modeling.pdf eq. 1.18;
 * cross-product convention of skew() include/utilities.h:16-24.
 * Q [batch][4][M]; q0 as above (rotation of the base node); n [batch][3][M] from sri_integrate_stress;
 * lbar [batch][3][N] or NULL => 0; M_tip [batch][3]; m [batch][3][M] (nodes 1..N-1). */
int sri_integrate_couple(sri_handle h, int64_t batch, const double* Q, const double* q0, const double* Gamma,
                         const double* n, const double* lbar, const double* M_tip, double* m);

/* All four stages in one fused launch (what main() does at main.cpp:197-201, plus stages 3-4).  Q never
 * leaves the SM between stages.  Any of the outputs Q, r, n, m may be NULL to skip storing it; F_tip and
 * M_tip may be NULL only when both n and m are NULL. */
typedef struct sri_rod_batch {
    int64_t batch;
    const double* K;     /* [batch][3][N]  required */
    const double* q0;    /* [batch][4]     or NULL  */
    const double* r0;    /* [batch][3]     or NULL  */
    const double* Gamma; /* [batch][3][N]  or NULL  */
    const double* fbar;  /* [batch][3][N]  or NULL  */
    const double* lbar;  /* [batch][3][N]  or NULL  */
    const double* F_tip; /* [batch][3] */
    const double* M_tip; /* [batch][3] */
    double* Q;           /* [batch][4][M] */
    double* r;           /* [batch][3][M] */
    double* n;           /* [batch][3][M] */
    double* m;           /* [batch][3][M] */
    int* info;           /* [batch] or NULL */
} sri_rod_batch;
int sri_integrate_all(sri_handle h, const sri_rod_batch* rods);

/* Reverse mode of sri_integrate_all (vector-Jacobian product of the discrete four-stage map): given cotangents of the
 * outputs, the gradients of  <gQ,Q> + <gr,r> + <gn,n> + <gm,m>  with respect to the eight inputs, in one launch.
 * rods: the struct of the forward call.  Its inputs are read as in sri_integrate_all (NULL defaults q0 = identity,
 * Gamma = e1; r0, fbar, lbar, F_tip, M_tip enter linearly and are not read); rods->Q, the forward's output, is required;
 * rods->n is required when gm is given; rods->r and rods->m are not read.  rods->info (or NULL) receives the zero /
 * non-finite pivot step of the transposed stage-1 solve A_NN(K)^T lam = gQ (0 when no K / q0 gradient is wanted).
 * Cotangents have the shapes of the outputs (NULL = zero); every non-NULL gradient has the shape of its input and is
 * written, not accumulated (K and fbar/lbar gradients are 0 at the node whose sample the forward does not use).  Host or
 * device pointers, errors and SRI_ERR_SINGULAR as for sri_integrate_all.  N <= 16: two rods per warp, register-resident
 * Gauss-Jordan with row pivoting; 17 <= N <= 64: one rod per CTA. */
typedef struct sri_rod_batch_grad {
    const double* gQ;  /* [batch][4][M] or NULL */
    const double* gr;  /* [batch][3][M] or NULL */
    const double* gn;  /* [batch][3][M] or NULL */
    const double* gm;  /* [batch][3][M] or NULL */
    double* gK;        /* [batch][3][N] or NULL */
    double* gq0;       /* [batch][4]    or NULL */
    double* gr0;       /* [batch][3]    or NULL */
    double* gGamma;    /* [batch][3][N] or NULL */
    double* gfbar;     /* [batch][3][N] or NULL */
    double* glbar;     /* [batch][3][N] or NULL */
    double* gF_tip;    /* [batch][3]    or NULL */
    double* gM_tip;    /* [batch][3]    or NULL */
} sri_rod_batch_grad;
int sri_integrate_all_vjp(sri_handle h, const sri_rod_batch* rods, const sri_rod_batch_grad* grads);

/* ---- several devices in one process (SURVEY 8b/8e: one host thread and one stream per GPU, contiguous rod ranges) -------- */

typedef struct sri_multi_context* sri_multi_handle;
/* Number of CUDA devices visible to this process (so that a host without the CUDA headers can size its shard list). */
int sri_device_count(int* ndev);
/* One sri_handle per listed device (devices == NULL => devices 0..ndev-1).  Rods are independent: no collective. */
int sri_create_multi(int N, const int* devices, int ndev, sri_multi_handle* out);
int sri_destroy_multi(sri_multi_handle mh);
int sri_multi_device_count(sri_multi_handle mh, int* ndev);
/* The handle of the index-th device (owned by mh), e.g. to generate or keep rods resident per device. */
int sri_multi_get_handle(sri_multi_handle mh, int index, sri_handle* h);
/* Rod-index block of shard `rank` of `world`: [floor(rank*total/world), floor((rank+1)*total/world)). */
int sri_shard_range(int64_t total, int rank, int world, int64_t* first, int64_t* last);
/* sri_integrate_all over all devices of mh.  HOST pointers: shard g integrates its contiguous block of rods->batch rods,
 * streamed through its device by its own host thread (pinned memory recommended); returns when every result has landed. */
int sri_integrate_all_sharded(sri_multi_handle mh, const sri_rod_batch* rods);
/* The same with data already resident: per_device[g] describes the rods of device g (device pointers on that device; batch
 * may differ per device or be 0).  Launches on every device, then synchronises all of them. */
int sri_integrate_all_per_device(sri_multi_handle mh, const sri_rod_batch* per_device);

/* ---- static shape problem (SURVEY 8f1; rod_modeling.pdf eq. 1.25) ------------------------------------- */

/* rho_i = H (K_i - K0_i) - R(q_i)^T m_i at all N nodes (m_0 = M_tip, q_{N-1} = q0); H = diag(H_diag[3]).
 * K, K0 (or NULL => 0), rho: [batch][3][N].  Also accumulates sum(rho^2) and max|rho| over the batch into
 * norm2_and_max[2] (device or host pointer, may be NULL). */
int sri_shape_residual(sri_handle h, int64_t batch, const double* K, const double* K0, const double* H_diag,
                       const double* Q, const double* q0, const double* m, const double* M_tip, double* rho,
                       double* norm2_and_max);

/* Local-frame wrench Lambda = [C; N] = [R(q)^T m; R(q)^T n] at all N nodes: the state of the local-frame statics
 * Lambda' = ad^T_xi Lambda - Fbar (rod_modeling.pdf eqs. 1.29, 2.18), couple first as in ad()'s [k; gamma] ordering
 * (include/utilities.h:27-37).  Evaluated pointwise from the global-frame stages (n = R N, m = R C), not by a second
 * collocation solve.  Node 0 carries (M_tip, F_tip), node N-1 the base rotation q0 (NULL => identity).
 * Q [batch][4][M]; n, m [batch][3][M]; F_tip, M_tip [batch][3]; Lambda [batch][6][N]. */
int sri_wrench_local(sri_handle h, int64_t batch, const double* Q, const double* q0, const double* n, const double* m,
                     const double* F_tip, const double* M_tip, double* Lambda);

/* The same wrench obtained by SOLVING the local-frame statics (SURVEY 8 f4; rod_modeling.pdf eqs. 1.29, 2.18):
 *   N' = -K^ N - R^T fbar,  C' = -K^ C - Gamma^ N - R^T lbar,  N(1) = R(1)^T F_tip,  C(1) = R(1)^T M_tip,
 * collocated with the tip node eliminated: the strain-dependent operator D_TT (x) I3 + blockdiag(K^_i) (3M x 3M), one
 * partial-pivot LU per rod and two solves.  Agrees with sri_wrench_local on the global-frame stages to the
 * discretisation error (1e-8 at N = 16, round-off from N = 32).  One rod per warp for N <= 16 (register-resident
 * Gauss-Jordan elimination with partial pivoting), one rod per CTA for 17 <= N <= 64 (the same elimination over 2-3 warps up to
 * N = 33, a CTA-wide LU beyond).  K [batch][3][N]; Q [batch][4][M] from stage 1; optional inputs as
 * in sri_integrate_all; Lambda [batch][6][N], couple first; info [batch] or NULL (zero-pivot step of the LU). */
int sri_integrate_wrench_local(sri_handle h, int64_t batch, const double* K, const double* Q, const double* q0,
                               const double* Gamma, const double* fbar, const double* lbar, const double* F_tip,
                               const double* M_tip, double* Lambda, int* info);

/* Galerkin projection of a nodal field onto the Legendre strain modes (rod_modeling.pdf eqs. 2.14, 2.16; the
 * transpose of Phi, include/utilities.h:49-67): out[b][c*ne+k] = sum_i w_i P_k(2 x_i - 1) f[b][c][i], with w the
 * Clenshaw-Curtis weights of the N Chebyshev nodes on [0,1].  f [batch][3][N] -> out [batch][3*ne]. */
int sri_project_onto_modes(sri_handle h, int64_t batch, int ne, const double* f, double* out);

/* Generalised internal forces of the angular strain modes (rod_modeling.pdf eqs. 2.16, 2.20: Q_ad = -int Phi^T B^T Lambda dX
 * with B^T Lambda = the couple part of the local-frame wrench): Qad[b][c*ne+k] = -sum_i w_i P_k(2 x_i - 1) Lambda[b][c][i],
 * c = 0..2.  Lambda [batch][6][N] as written by sri_wrench_local / sri_integrate_wrench_local -> Qad [batch][3*ne].  The
 * static balance 2.20 reads  int Phi^T H (K - K0) dX + Qad = 0. */
int sri_generalised_forces(sri_handle h, int64_t batch, int ne, const double* Lambda, double* Qad);

/* Galerkin residual of the static shape problem in one pass (rod_modeling.pdf eq. 1.25 projected as in 2.14/2.20):
 *   g[b][c*ne+k] = sum_i w_i P_k(2 x_i - 1) rho[b][c][i],   rho_i = H (K_i - K0_i) - R(q_i)^T m_i,
 * i.e. sri_shape_residual followed by sri_project_onto_modes without storing rho.  Arguments as in those two;
 * g [batch][3*ne]; norm2_and_max (2 doubles or NULL): sum g^2 and max |g| over the batch, reduced in a fixed order
 * (bitwise reproducible from run to run). */
int sri_galerkin_residual(sri_handle h, int64_t batch, int ne, const double* K, const double* K0, const double* H_diag,
                          const double* Q, const double* q0, const double* m, const double* M_tip, double* g,
                          double* norm2_and_max);

/* Reverse mode of sri_galerkin_residual: given the cotangent gg [batch][3*ne] of g, with rb[c][i] = w_i sum_k P_k(2 x_i - 1)
 * gg[c*ne+k] (the cotangent of rho), the gradients of <gg, g>:
 *   gK = H rb,  gK0 = -H rb  ([batch][3][N]);  gH[b][c] = sum_i rb[c][i] (K - K0)[c][i]  ([batch][3], per rod: a caller with
 *   one H for the batch sums over b);  gm[:, i-1] = -R(q_i) rb_i for i = 1..N-1  ([batch][3][M]),  gM_tip = -R(q_0) rb_0;
 *   gQ[:, i] = -d/dq (m_i^T R(q) rb_i) at q_i for i = 0..M-1  ([batch][4][M]),  gq0 likewise at node N-1  ([batch][4]),
 * R the un-normalised rotation of the forward.  Inputs as in sri_galerkin_residual (K0, q0 may be NULL); every output may be
 * NULL (skipped) and is written, not accumulated.  One pass, the lane layout of sri_galerkin_residual; gH is reduced in a fixed
 * order (bitwise reproducible). */
int sri_galerkin_residual_vjp(sri_handle h, int64_t batch, int ne, const double* K, const double* K0, const double* H_diag,
                              const double* Q, const double* q0, const double* m, const double* M_tip, const double* gg,
                              double* gK, double* gK0, double* gH, double* gQ, double* gq0, double* gm, double* gM_tip);

/* Jacobian of sri_galerkin_residual with respect to the modal strain coordinates, J[b][j][d] = d g_j / d qe_d, without
 * any linear solve: the variation of the rotation is left-trivialised (dR = [dtheta]x R, dtheta' = R dK, dtheta(0) = 0), so
 * every direction is two contractions with the cached integration matrices Dn_NN^-1 and D_TT^-1,
 *   dtheta = Dn_NN^-1 (R dK),   dm = D_TT^-1 (-((dtheta x R Gamma) x n)),   drho = H dK - R^T (dm - dtheta x m).
 * It is the tangent of the continuous problem collocated; it agrees with the exact tangent of the discrete stages to the
 * discretisation error (1e-10 at N = 16, round-off at N = 32).  Q, n, m: the stage outputs at the current qe
 * ([batch][4][M], [batch][3][M], [batch][3][M]); q0, Gamma optional as in sri_integrate_all; J [batch][3*ne][3*ne]
 * row-major (the layout sri_solve_small_batched takes). */
int sri_shape_jacobian(sri_handle h, int64_t batch, int ne, const double* H_diag, const double* Q, const double* q0,
                       const double* Gamma, const double* n, const double* m, const double* M_tip, double* J);

/* Newton iteration of the static shape problem (BASELINE configs[4]; rod_modeling.pdf section 2.2), the loop inside the
 * library: unknowns qe [batch][3*ne] (modal strain coordinates, in: initial guess, out: solution; device or host pointer),
 * residual g = sri_galerkin_residual of the four-stage integration of K = Phi qe under (F_tip, M_tip), forward-difference
 * Jacobian (the 3*ne perturbed copies of the batch go through ONE sri_integrate_all) or, with fd_step == 0, the
 * analytic Jacobian of sri_shape_jacobian (one integration per iteration); per-rod solve, update; stops when
 * sqrt(sum g^2 / total_dof) < tol or after max_iter iterations (<= 62).  total_dof: number of unknowns over all ranks
 * (0 => batch*3*ne).  reduce (or NULL): called once per iteration with the 2 host doubles [sum g^2, max |g|] of this
 * rank's rods, must replace them by the sum / max over the ranks (e.g. MPI_Allreduce) and return 0 -- the only collective
 * of the method; every rank must call with the same max_iter, also ranks with batch == 0.
 * With reduce == NULL the norms are reduced ON THE DEVICE: over the communicator attached by sri_nccl_init (one
 * ncclAllGather of 16 bytes per iteration on the handle's stream) or, without one, over this handle's rods only.  In that
 * mode the convergence test is a kernel that sets a device-side flag, the host enqueues iteration k+1 before it reads the
 * norms of iteration k (SURVEY section 5: the test lags by one iteration, so the GPU never waits for the host), and every
 * kernel of an iteration enqueued after convergence exits at once: iterates and counts are those of the unlagged loop.
 * On a single rank one iteration + its test is replayed as ONE CUDA graph launch from the second iteration on (captured
 * once per problem shape / H / tol; environment SRI_NEWTON_GRAPH=0 keeps eager launches, a communicator of more than one
 * rank does too).  A handle whose stream is the legacy default stream (which cannot be captured) runs this call on its own
 * stream, ordered after the work already queued on the caller's; the call returns after qe has been copied back either way. */
typedef int (*sri_allreduce_fn)(double* norm2_and_max, void* ctx);
typedef struct sri_newton_report {
    int iterations;        /* Newton updates taken */
    int converged;         /* 1 when the tolerance was met */
    int64_t integrations;  /* four-stage integrations of the batch: 1 + iterations * (3*ne + 1), or 1 + iterations (analytic) */
    double rms, max_abs;   /* of the last residual, over all ranks */
    double rms_history[64];
    int history_len;
    int64_t singular_solves; /* per-rod Newton systems found singular (zero pivot), summed over the iterations; those rods
                                kept their qe in that iteration */
} sri_newton_report;
/* Tip-loaded rods with an identity clamp: sri_newton_static_problem with q0, Gamma, fbar and lbar NULL (the same kernels,
 * results and launches). */
int sri_newton_static_shape(sri_handle h, int64_t batch, int ne, const double* H_diag, const double* F_tip,
                            const double* M_tip, const double* K0, double* qe, double tol, int max_iter, double fd_step,
                            int64_t total_dof, sri_allreduce_fn reduce, void* reduce_ctx, sri_newton_report* report);

/* A static shape problem with every input of the four-stage integration that the residual depends on (r0 moves the rod,
 * not its shape, and is not part of it).  Distributed loads are dead loads: per unit length, in the global frame, independent
 * of the shape (a follower load would make n depend on K).  Per-rod and per-node arrays are host or device pointers as
 * everywhere. */
typedef struct sri_static_problem {
    int64_t batch;
    int ne;                /* Legendre modes per strain component, 1..8: qe [batch][3*ne] */
    const double* H_diag;  /* [3], host or device */
    const double* F_tip;   /* [batch][3] */
    const double* M_tip;   /* [batch][3] */
    const double* K0;      /* [batch][3][N] or NULL (0) */
    const double* q0;      /* [batch][4]    or NULL (identity): rotation of the clamped base */
    const double* Gamma;   /* [batch][3][N] or NULL (e1) */
    const double* fbar;    /* [batch][3][N] or NULL (0), global frame (e.g. the weight (0, 0, -g)) */
    const double* lbar;    /* [batch][3][N] or NULL (0), global frame */
} sri_static_problem;
/* The Newton loop of sri_newton_static_shape (every argument, the report, both Jacobians, the lagged device-side test, the
 * NCCL and callback reductions and the graph replay as documented there) for a sri_static_problem: q0, Gamma, fbar and lbar
 * reach the integration, the residual and the analytic Jacobian, and the forward-difference copies carry them too.  The
 * analytic Jacobian stays exact under dead loads: n does not depend on K, it only varies along the rod. */
int sri_newton_static_problem(sri_handle h, const sri_static_problem* problem, double* qe, double tol, int max_iter,
                              double fd_step, int64_t total_dof, sri_allreduce_fn reduce, void* reduce_ctx,
                              sri_newton_report* report);
/* Tip-loaded rods with an identity clamp: sri_static_problem_vjp with q0, Gamma, fbar and lbar NULL.
 * Gradients of the static shape solution (implicit-function theorem): at an equilibrium qe* of sri_newton_static_shape
 * (g(qe*; F_tip, M_tip, K0, H) = 0, q0 = identity, Gamma = e1, no distributed loads) and a cotangent gqe of qe*, solves
 * J_d^T lam = gqe per rod, J_d the exact Jacobian of the discrete residual, and returns theta-grad = -(dg/dtheta)^T lam:
 *   gF_tip, gM_tip [batch][3];  gK0 [batch][3][N];  gH [batch][3] (per rod: a caller with one H sums over the batch).
 * qe [batch][3*ne] is the caller's converged solution: the call recomputes the four stages and the analytic Jacobian J_a of
 * sri_shape_jacobian there, but does not check that g(qe) ~ 0; the result is the gradient of the equilibrium only when it is.
 * J_d is never formed: lam_0 = J_a^-T gqe, then refine_steps steps lam += J_a^-T (gqe - J_d^T lam), each J_d^T lam being one
 * residual VJP and one sri_integrate_all_vjp.  ||J_a^-1 J_d - I|| (ne = 4, tip loads up to 0.6) is 3e-2 at N = 5, 2e-6 at
 * N = 9, 6e-14 at N = 16 and grows with the load: refine_steps = 3 reaches round-off for N >= 7, N = 5 needs about 12, 0 is
 * enough for N >= 16 (DESIGN section 5e).
 * K0 may be NULL (0); every output may be NULL.  lambda [batch][3*ne]: the adjoint solution; resid [batch]:
 * max|gqe - J_d^T lam| / max|gqe| at the returned lam.  info [batch]: 0, or (s | v << 8) with s the zero / non-finite pivot
 * step of the J_a^T solve (1..3*ne) and v that of the transposed stage-1 solve (as in sri_integrate_all_vjp); such a rod's
 * outputs are not valid.  Host or device pointers, SRI_ERR_SINGULAR with host buffers as in sri_integrate_all_vjp.  The
 * workspace is kept by the handle for the next call of the same shape. */
int sri_static_shape_vjp(sri_handle h, int64_t batch, int ne, const double* H_diag, const double* F_tip, const double* M_tip,
                         const double* K0, const double* qe, const double* gqe, int refine_steps, double* gF_tip,
                         double* gM_tip, double* gK0, double* gH, double* lambda, double* resid, int* info);
/* Outputs of sri_static_problem_vjp.  Every pointer may be NULL (skipped); each is written, not accumulated. */
typedef struct sri_static_problem_grad {
    double* gF_tip;  /* [batch][3] */
    double* gM_tip;  /* [batch][3] */
    double* gK0;     /* [batch][3][N] */
    double* gH;      /* [batch][3], per rod: a caller with one H sums over the batch */
    double* gq0;     /* [batch][4]    (at q0 = identity when problem->q0 is NULL) */
    double* gGamma;  /* [batch][3][N] (at Gamma = e1 when problem->Gamma is NULL) */
    double* gfbar;   /* [batch][3][N] (0 at node 0, whose sample the integration does not use) */
    double* glbar;   /* [batch][3][N] (0 at node 0) */
    double* lambda;  /* [batch][3*ne] the adjoint solution */
    double* resid;   /* [batch] max|gqe - J_d^T lam| / max|gqe| */
    int* info;       /* [batch] 0, or s | v << 8 as in sri_static_shape_vjp */
} sri_static_problem_grad;
/* sri_static_shape_vjp for a sri_static_problem: the forward state and J_a are those of the problem's inputs, J_d^T lam is the
 * residual VJP and sri_integrate_all_vjp with q0 and Gamma, and theta-grad = -(dg/dtheta)^T lam also for theta = q0, Gamma,
 * fbar, lbar (gq0 sums the residual's direct dependence on the base rotation and the integration's).  The refinement, its
 * accuracy per N, the workspace, host / device buffers and SRI_ERR_SINGULAR are those of sri_static_shape_vjp; a rod with a
 * non-finite load is flagged in its own info[b] and leaves the other rods' results unchanged. */
int sri_static_problem_vjp(sri_handle h, const sri_static_problem* problem, const double* qe, const double* gqe, int refine_steps,
                           const sri_static_problem_grad* grads);
/* The same solve over all devices of mh from one host process: HOST pointers, rods sharded by index as in
 * sri_integrate_all_sharded, one host thread per device, the norms reduced between the threads (no NCCL, no MPI).
 * Tip-loaded rods with an identity clamp: sri_newton_static_problem_sharded with q0, Gamma, fbar and lbar NULL. */
int sri_newton_static_shape_sharded(sri_multi_handle mh, int64_t batch, int ne, const double* H_diag, const double* F_tip,
                                    const double* M_tip, const double* K0, double* qe, double tol, int max_iter,
                                    double fd_step, sri_newton_report* report);
/* sri_newton_static_problem over all devices of mh: every per-rod and per-node array of the problem and qe are HOST pointers,
 * sharded by rod index as in sri_integrate_all_sharded; each rod's qe is bit for bit that of a one-device solve taking the same
 * iterations (the norms are added in shard order, so the rms history agrees to round-off). */
int sri_newton_static_problem_sharded(sri_multi_handle mh, const sri_static_problem* problem, double* qe, double tol,
                                      int max_iter, double fd_step, sri_newton_report* report);

/* ---- NCCL residual-norm reduction (BASELINE configs[4]; SURVEY 8e: the only collective, Newton driver only) -----------
 * libnccl.so.2 is opened at run time (dlopen), the library does not link against it.  One process per GPU:
 *   rank 0: sri_nccl_unique_id(id)  ->  broadcast the 128 bytes by any means (MPI, torch.distributed, a file)
 *   all   : sri_nccl_init(h, nranks, rank, id)          (collective: ncclCommInitRank on the handle's device)
 * after which sri_newton_static_shape(h, ..., reduce = NULL, ...) reduces its norms over that communicator on the
 * handle's stream.  sri_nccl_allreduce_norms is that reduction alone (norm2_and_max: 2 doubles on the device, in place:
 * sum over ranks, max over ranks; asynchronous on the handle's stream). */
int sri_nccl_unique_id(void* id128);
int sri_nccl_init(sri_handle h, int nranks, int rank, const void* id128);
int sri_nccl_finalize(sri_handle h);
int sri_nccl_allreduce_norms(sri_handle h, double* norm2_and_max);

/* Batched dense solve A x = b for small systems (n <= 24), partial pivoting, one rod per thread: the Newton step
 * of the static shape problem.  A [batch][n][n] row-major (may be overwritten), b [batch][n] -> x [batch][n].
 * info [batch] or NULL as in sri_integrate_quaternions.  Device pointers only. */
int sri_solve_small_batched(sri_handle h, int64_t batch, int n, double* A, const double* b, double* x, int* info);

/* ---- synthetic inputs of SURVEY 8(d): counter-based, identical for any sharding ------------------------ */

/* Fills K, F_tip, M_tip, fbar for rods [first_rod, first_rod+batch): K_c(X) = alpha + beta (2X-1) with
 * alpha,beta ~ U(-2,2); F_tip,M_tip ~ U(-1,1)^3; fbar = (0,0,-g), g ~ U(0,1).  Philox4x32-10 keyed by seed,
 * counter = rod index.  Any output pointer may be NULL.  Device pointers only. */
int sri_generate_rods(sri_handle h, uint64_t seed, int64_t first_rod, int64_t batch, double* K, double* F_tip,
                      double* M_tip, double* fbar);

/* ---- diagnostics -------------------------------------------------------------------------------------- */

const char* sri_last_error_string(void);
/* Tracing (SURVEY section 5).  Every entry point that takes a handle is an NVTX range named after itself (nvtx3, header only:
 * free unless a profiler is attached).  sri_set_timing(h, 1) additionally brackets the work of every following call on this
 * handle with a CUDA-event pair on the handle's stream; sri_get_last_timing returns the device time of the most recent
 * such call in milliseconds and the name of its entry point (waits for that call to finish).  The separate-stage entry
 * points (sri_integrate_position / _stress / _couple, ...) are thereby timed stage by stage; the fused sri_integrate_all
 * is one launch and one number. */
int sri_set_timing(sri_handle h, int enabled);
int sri_get_last_timing(sri_handle h, float* ms, const char** entry_point);
/* Number of CUDA kernels this library has launched in the calling process (bench.py's gpu_launches). */
int64_t sri_kernel_launch_count(void);
/* N <= 16: the elimination runs on the FP64 tensor cores in static pivot order; a rod whose sub-diagonal growth
 * max_{i>k} |c_ik| / |c_kk| exceeds the accepted bound (4; environment SRI_DMMA_GROWTH at sri_create) is handed
 * back to the row-pivoting kernel inside the same call; 17 <= N <= 64 works the same way with the multi-warp DMMA
 * kernel.  sri_integrate_wrench_local (N <= 33) has the same two passes with scalar kernels.  Returns how many rods of the
 * most recent such device-buffer call on this handle took the second pass (synchronises the handle's stream); 0 when the
 * handle runs the row-pivoting kernels only (SRI_FUSED16_IMPL=scalar; SRI_WRENCH_IMPL set). */
int sri_get_handback_count(sri_handle h, int64_t* count);
/* Runs the library's FP64 FMA peak probe on the handle's device and returns TFLOP/s (roofline denominator). */
int sri_measure_fp64_peak(sri_handle h, double* tflops);
/* The same for the FP64 tensor cores (stream of independent DMMA m8n8k4): the roofline denominator of the N <= 16
 * fused kernel, whose elimination and stage contractions run there. */
int sri_measure_dmma_peak(sri_handle h, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* SRI_H */
