/*
 * psd_b200.h — C ABI of the B200 (sm_100a) dense periodic Schur library.
 *
 * This is the drop-in boundary for the dense pschur! hot path of
 * RalphAS/PeriodicSchurDecompositions.jl (v0.1.6).  The reference has no FFI of its own
 * (pure Julia, multiple dispatch); the Julia glue in
 * periodicschurdecompositions.jl_b200/julia/PeriodicSchurB200.jl overloads the reference's
 * methods for Float64/ComplexF64 matrices and forwards to these entry points via ccall
 * (see INTEGRATION.md).  Each entry point cites the reference method it replaces
 * (file:line relative to the reference repository).
 *
 * Conventions
 *  - Matrices are column-major, order n, leading dimension n, one factor after another:
 *    A[batch][p][n*n].  Complex data are interleaved (re,im) double pairs (Julia ComplexF64).
 *  - Factors are always in the USER's order A_1..A_p.  orientation 0 = :R (product
 *    A_1 A_2 ... A_p, Schur factor is A_1 / schurindex 1), 1 = :L (product A_p ... A_1,
 *    Schur factor is A_p / schurindex p)   [PeriodicSchurDecompositions.jl:40-48,127-131,
 *    1078-1093].
 *  - On return (wantT != 0) A holds the T factors in place, with exact zeros below the
 *    (quasi-)triangle; Z (wantZ != 0) holds the orthogonal/unitary factors indexed as in the
 *    reference result structs (:R  Z_j' A_j Z_{j+1} = T_j ;  :L  Z_{j+1}' A_j Z_j = T_j).
 *  - info[b] = 0 on success, k > 0 = "convergence failed at level k"
 *    (PeriodicSchurDecompositions.jl:891-893, generalized.jl:856-858,
 *    rgeneralized.jl:1057-1059).  One failing problem never aborts the batch.
 *  - All functions return 0 on success and a negative code on error; the message is
 *    available from psd_last_error_string().  No C++ exception crosses this boundary and
 *    nothing calls exit()/abort().
 *  - There is no CPU fallback: without a usable CUDA device every compute entry point
 *    returns PSD_ERR_NO_DEVICE.
 *  - Host entry points are synchronous and thread-safe (per-handle mutex); buffers belong to
 *    the caller and are only touched during the call.
 */
#ifndef PSD_B200_H
#define PSD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSD_VERSION 100 /* 0.1.0 */

#define PSD_OK 0
#define PSD_ERR_BAD_ARG (-1)      /* invalid n/p/batch/flags/pointer                       */
#define PSD_ERR_NO_DEVICE (-2)    /* no CUDA device / extension unusable                    */
#define PSD_ERR_CUDA (-3)         /* CUDA runtime error (see psd_last_error_string)        */
#define PSD_ERR_SIGNATURE (-4)    /* "The leftmost entry in S must be true"                */
                                  /*   (generalized.jl:140, rgeneralized.jl:37)            */
#define PSD_ERR_UNSUPPORTED (-5)  /* shape outside what this build implements              */

typedef struct psd_handle_s* psd_handle_t;

int psd_version(void);
/* Number of visible CUDA devices (0 if none / driver missing). */
int psd_device_count(void);
/* Thread-local description of the last error returned on this thread. */
const char* psd_last_error_string(void);

/* Create a handle owning streams, device workspaces and pinned staging on `ndev` devices
 * (devices[i] = CUDA ordinal); ndev == 0 selects every visible device.  Batched host entry
 * points shard the batch into ndev contiguous ranges, one host thread + stream per device,
 * with no inter-device communication (SURVEY.md §8(e)). */
int psd_create(psd_handle_t* handle, int ndev, const int* devices);
int psd_destroy(psd_handle_t handle);
int psd_handle_device_count(psd_handle_t handle);

/* ---------------------------------------------------------------------------------------
 * Real standard periodic Schur decomposition, batched.
 * Replaces pschur!(A::Vector{Matrix{Float64}}, lr; wantZ, wantT, maxitfac)
 *   driver                      PeriodicSchurDecompositions.jl:120-152
 *   periodic Hessenberg         PeriodicSchurDecompositions.jl:213-259  (+ householder.jl)
 *   explicit Q                  PeriodicSchurDecompositions.jl:136-140,180 (orghr/orgqr)
 *   periodic QR iteration       PeriodicSchurDecompositions.jl:322-1096 (+ rschur2x2.jl)
 * for `batch` independent problems of identical shape.
 *   A    in/out  [batch][p][n][n]   (wantT == 0: contents unspecified on return, as the
 *                                    reference leaves "mangled" matrices, runtests.jl:118)
 *   Z    out     [batch][p][n][n]   or NULL when wantZ == 0
 *   eig  out     [batch][n] complex128 (re,im); complex pairs adjacent, positive imaginary
 *                                    part first (rschur2x2.jl:89-91)
 *   info out     [batch]
 * maxitfac <= 0 selects the reference default 30.
 * n >= 192: blocked reduction + small-bulge multishift iteration with FP64 tensor-core updates,
 * one problem at a time on the whole GPU (DESIGN.md section 9); results of this path are not
 * bit-for-bit reproducible from run to run (floating-point atomics in the blocked reduction,
 * timing-dependent choice between equally valid shift sets), all acceptance predicates hold.
 * maxitfac bounds this iteration too: its rounds are capped at (256 + 100 n / D) maxitfac / 30
 * (D = 32..16 rows per round, by period); a problem that reaches the cap is finished by the
 * single-bulge team iteration with the same maxitfac.
 * ------------------------------------------------------------------------------------- */
int psd_rpschur_batched(psd_handle_t handle, int n, int p, int64_t batch, int orientation,
                        int wantT, int wantZ, int maxitfac, double* A, double* Z, double* eig,
                        int32_t* info);

/* Same computation on buffers already resident on device `dev_index` (index into the
 * handle's device list), enqueued on `stream` (a cudaStream_t passed as void*; NULL = the
 * handle's own stream for that device).  Asynchronous: the caller synchronises the stream.
 * All *_dev calls on one device of a handle share one set of scratch buffers; the library orders
 * them with an event (a call waits for the previous one, whatever stream that was enqueued on), so
 * calls on different streams are safe but do not overlap.  For n >= 192 (large-N path) the call
 * synchronises the stream internally (the iteration is driven from the host).
 * Used by bench.py for the HBM-resident throughput figure and by host code that keeps
 * matrices on the GPU. */
int psd_rpschur_batched_dev(psd_handle_t handle, int dev_index, void* stream, int n, int p,
                            int64_t batch, int orientation, int wantT, int wantZ,
                            int maxitfac, double* dA, double* dZ, double* deig,
                            int32_t* dinfo);

/* Periodic QR iteration on input that is already in Hessenberg-triangular form (rightwards
 * order: A_1 upper Hessenberg, A_2..A_p upper triangular; anything below is ignored and
 * zeroed), Z initialised to the identity.
 * Replaces the inner method pschur!(H1, Hs; wantT, wantZ, maxitfac) with Q === nothing
 * (PeriodicSchurDecompositions.jl:322-1096), which the reference's tests use to keep exact
 * zeros in the input (test/runtests.jl:53-66). */
int psd_rpschur_hessut_batched(psd_handle_t handle, int n, int p, int64_t batch, int wantT,
                               int wantZ, int maxitfac, double* A, double* Z, double* eig,
                               int32_t* info);

/* Same, with the Schur vectors accumulated onto orthogonal matrices of the caller: on entry Q
 * holds Q_1..Q_p of an earlier reduction (storage layout of A), on exit Q_j Z_j.
 * Replaces pschur!(H1, Hs; Q = Q, wantZ = true, ...) (the `Q` keyword of the inner method,
 * PeriodicSchurDecompositions.jl:326, 432-437, as used by the Krylov-Schur driver,
 * krylov.jl:583-591). */
int psd_rpschur_hessut_q_batched(psd_handle_t handle, int n, int p, int64_t batch, int wantT,
                                 int maxitfac, double* A, double* Q, double* eig, int32_t* info);

/* Periodic Hessenberg-triangular reduction only, batched (device or host buffers).
 * Replaces phessenberg!(A) (PeriodicSchurDecompositions.jl:213-259) followed by the explicit
 * Q materialisation of the driver (:136-140): on return A holds H_1 (upper Hessenberg) and
 * H_2..H_p (upper triangular) with exact zeros below, Q (or NULL) the explicit Q_j with
 * Q_j' A_j Q_{j+1} = H_j.  Rightwards order only (the :L driver reverses before calling). */
int psd_rphess_batched(psd_handle_t handle, int n, int p, int64_t batch, int wantQ, double* A,
                       double* Q);

/* Same reduction with the result in the reference's own packed form: on return A_j holds H_j in
 * its upper (Hessenberg for j = 1) part and, below it, the Householder vectors (implicit leading
 * 1, LAPACK convention), and tau[b][j-1][i] their scalars (n per factor; tau[.][0] uses n-1, the
 * trailing entries are 0) - exactly the (A[j], tau[j]) from which phessenberg! builds
 * Hessenberg(A[1], tau[1]) and QR(A[j], tau[j]) (PeriodicSchurDecompositions.jl:229-253).
 * Host buffers, first device of the handle; one CTA per problem at every order (the blocked
 * large-N reduction keeps its reflectors in compact-WY form and is not used here). */
int psd_rphess_packed_batched(psd_handle_t handle, int n, int p, int64_t batch, double* A,
                              double* tau);

/* ---------------------------------------------------------------------------------------
 * Complex (generalized) periodic Schur decomposition, batched.
 * Replaces pschur!(A::Vector{Matrix{ComplexF64}}, S, lr; wantZ, wantT)
 *   driver, :L reversal of A and S      generalized.jl:108-148
 *   generalized Hessenberg-triangular   generalized.jl:988-1082   (_phessenberg!(A, S))
 *   complex periodic QZ (MB03BZ-style)  generalized.jl:166-931
 *   scaled eigenvalue representation    generalized.jl:939-976    (_safeprod)
 * and, with S all true, the complex standard method pschur!(A, lr)
 * (PeriodicSchurDecompositions.jl:1106-1111), whose glue repackages the result as PeriodicSchur
 * with values = alpha ./ beta .* 2^alphascale.
 *   S          in   [p] user order, 1 = factor enters as A_j, 0 = as inv(A_j); the leftmost
 *                   factor after orientation (S[0] for :R, S[p-1] for :L) must be 1, otherwise
 *                   PSD_ERR_SIGNATURE ("The leftmost entry in S must be true", generalized.jl:140)
 *   A          in/out [batch][p][n][n] complex128 (re,im interleaved), user order
 *   Z          out  [batch][p][n][n] complex128 or NULL when wantZ == 0; indexed as in the
 *                   reference result (T_l = Z_l' A_l Z_{l+1} for S_l xor :L, else
 *                   T_l = Z_{l+1}' A_l Z_l; test/testfuncs.jl:175-186)
 *   alpha,beta out  [batch][n] complex128; alphascale out [batch][n] int64:
 *                   lambda_k = alpha_k / beta_k * 2^alphascale_k, |alpha| in [1,2) or 0,
 *                   beta in {0,1} (0 = infinite eigenvalue)
 *   info       out  [batch]
 * On return with wantT != 0 the diagonals of all factors except the Schur factor are real and
 * non-negative (generalized.jl:860-908).  maxitfac <= 0 selects the reference default 30.
 * ------------------------------------------------------------------------------------- */
int psd_cpschur_batched(psd_handle_t handle, int n, int p, int64_t batch, int orientation,
                        const uint8_t* S, int wantT, int wantZ, int maxitfac, double* A,
                        double* Z, double* alpha, double* beta, int64_t* alphascale,
                        int32_t* info);

/* Complex periodic QZ iteration on input already in Hessenberg-triangular form, rightwards
 * order, Z starting from the identity.  Replaces the inner method
 * pschur!(H1, Hs, S; wantT, wantZ) with Q === nothing (generalized.jl:166-931), which the
 * reference's tests call directly to keep planted exact zeros (test/testfuncs.jl:384-409,
 * test/generalized.jl:68-173). */
int psd_cpschur_hessut_batched(psd_handle_t handle, int n, int p, int64_t batch, const uint8_t* S,
                               int wantT, int wantZ, int maxitfac, double* A, double* Z,
                               double* alpha, double* beta, int64_t* alphascale, int32_t* info);

/* ---------------------------------------------------------------------------------------
 * Real generalized periodic Schur decomposition (periodic QZ), batched.
 * Replaces pschur!(A::Vector{Matrix{Float64}}, S, lr; wantZ, wantT)
 *   driver, :L reversal of A and S      rgeneralized.jl:3-45
 *   generalized Hessenberg-triangular   generalized.jl:988-1082   (_phessenberg!(A, S))
 *   real periodic QZ (MB03BD-style)     rgeneralized.jl:49-1083
 *   2x2 periodic eigen-kernels          rpschur2x2.jl:9-317, rgeneralized.jl:1140-1509
 * Arguments as psd_cpschur_batched with real A, Z (float64) and real beta:
 *   alpha out [batch][n] complex128, beta out [batch][n] float64, alphascale [batch][n] int64.
 * On return (wantT != 0) the Schur factor is upper quasi-triangular with exact zeros below the
 * subdiagonal and T1[i+1,i] == 0 wherever eigenvalue i is real; 2x2 diagonal blocks are exactly
 * the complex-conjugate pairs and are left unstandardised as in the reference
 * (rgeneralized.jl:748-790); conjugate pairs are adjacent, positive imaginary part first
 * (rpschur2x2.jl:228-232).  maxitfac <= 0 selects the reference default 120.
 * The reference keyword `aggressive` (rgeneralized.jl:7, off by default) is not offered.
 * ------------------------------------------------------------------------------------- */
int psd_rgpschur_batched(psd_handle_t handle, int n, int p, int64_t batch, int orientation,
                         const uint8_t* S, int wantT, int wantZ, int maxitfac, double* A,
                         double* Z, double* alpha, double* beta, int64_t* alphascale,
                         int32_t* info);

/* Real periodic QZ iteration on Hessenberg-triangular input (rightwards order, Z from the
 * identity): the inner method pschur!(H1, Hs, S; ...) of rgeneralized.jl:49-1083, which the
 * reference's tests call directly for the planted-zero cases (test/generalized.jl:68-153). */
int psd_rgpschur_hessut_batched(psd_handle_t handle, int n, int p, int64_t batch, const uint8_t* S,
                                int wantT, int wantZ, int maxitfac, double* A, double* Z,
                                double* alpha, double* beta, int64_t* alphascale, int32_t* info);

/* Generalized periodic Hessenberg-triangular reduction only, batched (cplx != 0: complex128).
 * Replaces _phessenberg!(A, S; wantQ) (generalized.jl:988-1082, exercised directly by
 * test/generalized.jl:2-40): on return A_1 is upper Hessenberg, A_2..A_p upper triangular (exact
 * zeros below), Q (or NULL) the explicit Q_l with  A_l = Q_l H_l Q_{l+1}'  for S_l = true and
 * A_l = Q_{l+1} H_l Q_l'  for S_l = false.  Rightwards order; S[0] must be 1. */
int psd_gphess_batched(psd_handle_t handle, int cplx, int n, int p, int64_t batch, const uint8_t* S,
                       int wantQ, double* A, double* Q);

/* Row-wise periodic Hessenberg reduction for the left orientation, batched.
 * Replaces _rphessenberg!(Ap, A, Q) (rhessx.jl:53-109; RHouseholder rhessx.jl:7-50), whose only
 * caller is the Krylov-Schur restart (krylov.jl:800-832).  For the product Ap A_{p-1} ... A_1:
 *   Ap  in/out [batch][m][n] column-major, m = n + (extra_row != 0): on return upper Hessenberg
 *               (the extra Arnoldi foot row, if present, is reduced to its last entry)
 *   A   in/out [batch][p-1][n][n]: on return upper triangular (NULL when p == 1)
 *   Q   in/out [batch][p][qrows][n] or NULL: Q_l <- Q_l H' for every reflector applied to the
 *               columns of factor l (l = p is Ap) */
int psd_rphess_rowwise_batched(psd_handle_t handle, int n, int extra_row, int p, int qrows,
                               int64_t batch, double* Ap, double* A, double* Q);

/* Test / measurement hook for the FP64 tensor-core (DMMA) GEMM that carries the large-N blocked
 * updates (csrc/psd_dgemm.cuh): C <- alpha*op(A)*op(B) + beta*C on host buffers, column-major,
 * BLAS dgemm argument meaning (transA/transB: 0 = 'N', 1 = 'T').  With reps > 0 the kernel alone
 * is additionally timed on resident operands (CUDA events, 3 warm-up launches) and the average
 * milliseconds per launch are returned in *ms.  Replaces the BLAS calls the reference reaches
 * through householder.jl:199-218,252 once they are blocked (SURVEY.md section 2.3). */
int psd_dgemm_host(psd_handle_t handle, int transA, int transB, int M, int N, int K, double alpha,
                   const double* A, int lda, const double* B, int ldb, double beta, double* C,
                   int ldc, int reps, double* ms);

/* Synthetic inputs (measurement only, SURVEY.md §8(d)): uniform [0,1) entries from a
 * counter-based generator keyed by (seed, problem, factor, row, col), problems
 * first_b .. first_b+batch-1, written to a host buffer or (asynchronously, on the current
 * device and `stream`) to a device buffer.  cplx != 0 fills interleaved complex128.
 * Mirrors rand(T,n,n) under a fixed seed in the reference's tests (test/testfuncs.jl:12). */
int psd_fill_uniform_host(uint64_t seed, int n, int p, int64_t batch, int64_t first_b, int cplx,
                          double* A);
int psd_fill_uniform_dev(void* stream, uint64_t seed, int n, int p, int64_t batch,
                         int64_t first_b, int cplx, double* dA);

/* Counters of the most recent batched call on this handle (diagnostics; mirrors the
 * reference's niter/maxits reporting, PeriodicSchurDecompositions.jl:458-459,1077):
 * stats[0] = kernel launches, stats[1] = problems solved in shared memory,
 * stats[2] = problems solved in global-memory workspaces, stats[3] = H2D bytes,
 * stats[4] = D2H bytes, stats[5] = kernel time in microseconds summed over devices. */
int psd_last_stats(psd_handle_t handle, int64_t stats[8]);

/* Measurement support (SURVEY.md §8(d)): with profiling on, every kernel the library launches
 * is bracketed by CUDA events on its own stream.  psd_kernel_times waits for the recorded
 * events and returns, accumulated since the previous call, ms[0] = reduction kernels,
 * ms[1] = QR/QZ iteration kernels (milliseconds of device time), ms[2], ms[3] = how many
 * launches of each kind were timed; for the large-N blocked reduction ms[4] = panel kernels,
 * ms[5] = FP64 tensor-core GEMM updates (milliseconds), ms[6] = GEMM flops issued; ms[7] = kernel
 * launches not counted in ms[2..3] because one timer brackets several (the occupancy phases of the
 * eigenvalue-only iteration). */
int psd_set_profiling(psd_handle_t handle, int on);
int psd_kernel_times(psd_handle_t handle, double ms[8]);

/* Counters of the most recent large-N (N >= 192) iteration on this handle: the small-bulge
 * multishift periodic QR sweeps that replace the single double-shift bulge of
 * PeriodicSchurDecompositions.jl:806-886 (mirrors the reference's niter report, :458-459, 1077).
 * out[0] = status (0 finished, 1 fell back to the single-bulge team kernel), out[1] = sweeps,
 * out[2] = rounds (chase + update launches), out[3] = window-rounds, out[4] = shift pairs used,
 * out[5] = exceptional-shift sweeps, out[6] = diagonal blocks finished by the small kernel,
 * out[7] = kernel launches, out[8] = flops of the FP64 tensor-core window updates;
 * with profiling on additionally device milliseconds: out[9] = bulge chase, out[10] = tensor-core
 * updates, out[11] = shift computation, out[12] = deflation scans, out[13] = final blocks. */
int psd_large_stats(psd_handle_t handle, double out[16]);

/* Iteration counts of the real standard paths.  After this call every psd_rpschur_batched /
 * psd_rpschur_hessut(_q)_batched call on `handle` stores in iters[b] the number of periodic QR
 * iterations problem b took (the `niter` the reference reports with @debug,
 * PeriodicSchurDecompositions.jl:458-459, 1077); iters is host memory with room for the batch of
 * those calls, NULL switches the report off.  Problems that take the large-N path (N >= 192)
 * report 0 here and their counters through psd_large_stats. */
int psd_set_iters_output(psd_handle_t handle, int32_t* iters);

/* Page-locked host memory for the callers of the batched entry points (a Julia Array is pageable;
 * buffers from here are copied from / to by DMA directly, without the staging copy).
 * write_combined != 0: for INPUT buffers the host only writes (the device reads them faster over
 * PCIe; host reads of such memory are very slow). */
int psd_host_alloc(size_t bytes, int write_combined, void** out);
int psd_host_free(void* ptr);

/* Integrity check of real periodic Schur decompositions on the device, batched.
 * Replaces checkpsd(P, Hs) (diagnostics.jl:190-263) for PeriodicSchur results (S all true): for
 * problem b and factor l (user order, host arrays in the storage layout of psd_rpschur_batched)
 *   err[b*p + l]  = || Z_l T_l Z_l1' - A_l ||_F / (eps ||A_l||_1)   (:R; Z_l1 T_l Z_l' for :L),
 *                   the "normalized factorization error" the reference returns (O(1) expected,
 *                   its threshold is 100),
 *   tri[b*p + l]  = Frobenius norm of T_l below its (quasi-)triangle (tril(T, -2) for the Schur
 *                   factor, tril(T, -1) for the others; the strict check wants exactly 0),
 *   orth[b*p + l] = || Z_l Z_l' - I ||_F (the reference's limit is 10 eps n).
 * tri and orth may be NULL.  The comparison with the thresholds stays with the caller.  Host
 * buffers; a diagnostic, run on the first device of the handle in plain synchronous chunks. */
int psd_rcheckpsd_batched(psd_handle_t handle, int n, int p, int64_t batch, int orientation,
                          const double* A, const double* T, const double* Z, double* err,
                          double* tri, double* orth);

#ifdef __cplusplus
}
#endif
#endif /* PSD_B200_H */
