/*
 * splpak_b200.h -- C ABI of the B200-native fit-and-evaluate path of splpak.
 *
 * This is the drop-in boundary: every entry point below is what the reference's Fortran
 * module would bind through iso_c_binding (see INTEGRATION.md and fortran/splpak_module.F90).
 * All arrays are laid out exactly as Fortran passes them (column-major, contiguous):
 *   xdata(l1xdat, ndata)  -> coordinates of one point are contiguous, stride l1xdat per point
 *   coef(nodes(1),...,nodes(ndim)) -> dimension 1 fastest
 * No C++ or torch types cross this boundary: plain pointers, sizes and integer codes.
 *
 * Precision: splpak_real is double, or float when the library is built with -DSPLPAK_REAL32
 * (libsplpak_b200_r32.so), mirroring the reference's -DREAL32 switch (src/splpak.F90:33-41).
 * REAL128 has no GPU equivalent and is refused at compile time.
 *
 * There is NO CPU fallback: every compute entry point needs a CUDA device and returns
 * SPLPAK_ERR_CUDA (201) when none is usable.
 *
 * Error convention (src/splpak.F90:674-686 for the fit, :1155-1161 for evaluation):
 *   0    no error
 *   101  ndim < 1 (this library also returns 101 for ndim > 4, which the reference documents
 *        at :1158 but never checks)
 *   102  nodes(idim) < 4 for some idim
 *   103  xmin(idim) == xmax(idim) for some idim
 *   104  fit: ncf < nodes(1)*...*nodes(ndim);   evaluation: nderiv(idim) outside 0..2
 *   105  ndata < 1
 *   106  nwrk too small (nwrk - nwrk1 + 1 < 1, :775-781)
 *   107  solver failure (too few rows, non-positive pivot, or scratch smaller than
 *        ((n+5)n+2)/2 as suprls checks at :1443-1454)
 *   201+ failures that cannot occur in the reference (CUDA, NCCL, bad handle, allocation)
 * The C ABI returns codes silently; printing ' IERR=nnnnn' + message (cfaerr, :399-407) is
 * done by the host-side mirror (splpak_type.hpp / the Fortran shim).
 * Every function returns the same code it stores in *ierror (when it has an ierror argument).
 */
#ifndef SPLPAK_B200_H
#define SPLPAK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifdef REAL128
#error "splpak_b200: REAL128 has no GPU equivalent (src/splpak.F90:37-38); build REAL64 or REAL32"
#endif
#ifdef SPLPAK_REAL32
typedef float splpak_real;
#else
typedef double splpak_real;
#endif

#define SPLPAK_OK              0
#define SPLPAK_ERR_NDIM        101
#define SPLPAK_ERR_NODES       102
#define SPLPAK_ERR_RANGE       103
#define SPLPAK_ERR_NCF         104   /* fit */
#define SPLPAK_ERR_NDERIV      104   /* evaluation */
#define SPLPAK_ERR_NDATA       105
#define SPLPAK_ERR_NWRK        106
#define SPLPAK_ERR_SOLVER      107
#define SPLPAK_ERR_CUDA        201
#define SPLPAK_ERR_NCCL        202
#define SPLPAK_ERR_HANDLE      203
#define SPLPAK_ERR_ALLOC       204

typedef struct splpak_b200_fit_s *splpak_b200_fit_t;   /* opaque streaming-fit handle */

/* sizeof(splpak_real) of this build (8, or 4 for the REAL32 library). */
int splpak_b200_sizeof_real(void);
/* Static string for a code above (the reference's cfaerr message text for 101..107). */
const char *splpak_b200_strerror(int code, int evaluation);

/* ------------------------------------------------------------------------------------------
 * One-shot entry points with HOST arrays: exact replacements for the reference procedures.
 * ---------------------------------------------------------------------------------------- */

/* Replaces splcw (src/splpak.F90:512-513).  wdata: ndata weights, or wdata[0] < 0 meaning
 * "all weights 1, other elements not referenced" (:581-588).  work is accepted for signature
 * compatibility and never touched (the GPU needs no host scratch); nwrk is still checked the way
 * the reference checks it (106, and the suprls scratch test that maps to 107). */
int splpak_b200_splcw(int ndim, const splpak_real *xdata, int l1xdat, const splpak_real *ydata,
                      const splpak_real *wdata, int64_t ndata, const splpak_real *xmin,
                      const splpak_real *xmax, const int *nodes, splpak_real xtrap,
                      splpak_real *coef, int64_t ncf, splpak_real *work, int64_t nwrk, int *ierror);

/* Replaces splcc (src/splpak.F90:421-422): splcw with all weights 1. */
int splpak_b200_splcc(int ndim, const splpak_real *xdata, int l1xdat, const splpak_real *ydata,
                      int64_t ndata, const splpak_real *xmin, const splpak_real *xmax,
                      const int *nodes, splpak_real xtrap, splpak_real *coef, int64_t ncf,
                      splpak_real *work, int64_t nwrk, int *ierror);

/* Replaces splde (src/splpak.F90:1089): one value or partial derivative at one point. */
splpak_real splpak_b200_splde(int ndim, const splpak_real *x, const int *nderiv,
                              const splpak_real *coef, const splpak_real *xmin,
                              const splpak_real *xmax, const int *nodes, int *ierror);

/* Replaces splfe (src/splpak.F90:1258): splde with nderiv = 0. */
splpak_real splpak_b200_splfe(int ndim, const splpak_real *x, const splpak_real *coef,
                              const splpak_real *xmin, const splpak_real *xmax, const int *nodes,
                              int *ierror);

/* Batched splfe/splde: nq points x(l1x, nq), out(nq).  nderiv == NULL means splfe.
 * (New entry point: the reference evaluates one point per call, :1089/:1258.)  HOST arrays. */
int splpak_b200_eval(int ndim, const splpak_real *x, int l1x, int64_t nq, const int *nderiv,
                     const splpak_real *coef, const splpak_real *xmin, const splpak_real *xmax,
                     const int *nodes, splpak_real *out, int *ierror);

/* Same with x, coef and out already in DEVICE memory (xmin/xmax/nodes/nderiv stay on the host).
 * stream is a cudaStream_t passed as void* (NULL = default stream); the call is asynchronous. */
int splpak_b200_eval_device(int ndim, const splpak_real *d_x, int l1x, int64_t nq, const int *nderiv,
                            const splpak_real *d_coef, const splpak_real *xmin,
                            const splpak_real *xmax, const int *nodes, splpak_real *d_out,
                            void *stream, int *ierror);

/* Derivative sets: for every point, all partial derivatives up to total order `order` in one pass (one gather of
 * the point's 4^ndim coefficients for all of them).  out(ncomp, nq): the ncomp results of one point are contiguous.
 *   order 1: ncomp = ndim + 1                 the value, d/dx1 .. d/dxn
 *   order 2: ncomp = (ndim + 1)(ndim + 2) / 2 the order-1 set, then d2/dxi dxj for i <= j in row order
 *            (1,1), (1,2), .., (1,n), (2,2), .., (n,n)
 * Component k is bit-identical to splpak_b200_eval on the same batch with the nderiv it names.  Errors 101..103
 * as splpak_b200_eval; an order other than 1 or 2 returns 104 and writes nothing.  HOST arrays (same staging as
 * splpak_b200_eval) / DEVICE arrays (asynchronous on stream).  The REAL32 library keeps float I/O with float64
 * arithmetic here, as splde does. */
int splpak_b200_eval_derivs(int ndim, const splpak_real *x, int l1x, int64_t nq, int order,
                            const splpak_real *coef, const splpak_real *xmin, const splpak_real *xmax,
                            const int *nodes, splpak_real *out, int *ierror);
int splpak_b200_eval_derivs_device(int ndim, const splpak_real *d_x, int l1x, int64_t nq, int order,
                                   const splpak_real *d_coef, const splpak_real *xmin, const splpak_real *xmax,
                                   const int *nodes, splpak_real *d_out, void *stream, int *ierror);

/* Evaluation on a REGULAR OUTPUT GRID (new; the upstream fit-then-grid use, README.md:60): the value (nderiv NULL)
 * or partial derivative of the spline at every point (a1[i1], .., aN[iN]) of the tensor grid spanned by ndim axes.
 * axes = the axes concatenated (axis d has naxis[d] points, any order, inside or outside [xmin, xmax]);
 * out(naxis(1), .., naxis(ndim)), dimension 1 fastest.  Same basis values as splfe/splde point by point; the
 * contraction runs one dimension at a time, so the cost is 4 FMAs and 8 bytes per output point instead of a
 * 4^ndim gather.  HOST arrays (the output is produced in slabs along the last axis) / DEVICE arrays. */
int splpak_b200_eval_grid(int ndim, const splpak_real *axes, const int64_t *naxis, const int *nderiv,
                          const splpak_real *coef, const splpak_real *xmin, const splpak_real *xmax,
                          const int *nodes, splpak_real *out, int *ierror);
int splpak_b200_eval_grid_device(int ndim, const splpak_real *d_axes, const int64_t *naxis, const int *nderiv,
                                 const splpak_real *d_coef, const splpak_real *xmin, const splpak_real *xmax,
                                 const int *nodes, splpak_real *d_out, void *stream, int *ierror);

/* ------------------------------------------------------------------------------------------
 * Streaming fit handle: create -> add_points (any number of calls, host or device arrays)
 * -> [all-reduce the partial buffer across ranks] -> compute.  This is the assembly / solve
 * split the north star names add_points / compute; splcw above is create+add_points+compute.
 * A handle owns its device buffers and one CUDA stream; use it from one host thread at a time.
 * ---------------------------------------------------------------------------------------- */

/* Validates ndim/nodes/xmin/xmax in the reference's order (101, 102, 103; :718-750). */
int splpak_b200_fit_create(int ndim, const splpak_real *xmin, const splpak_real *xmax,
                           const int *nodes, splpak_real xtrap, splpak_b200_fit_t *handle,
                           int *ierror);

/* Accumulate n more data points into the normal equations (and the sparse-area histogram when
 * xtrap != 0).  weighted = 0 ignores w (splcc, or wdata(1) < 0); zero-weight points are skipped
 * as in :796-800.  HOST arrays; the copy is chunked and overlapped with the kernels. */
int splpak_b200_fit_add_points(splpak_b200_fit_t h, const splpak_real *x, int l1x,
                               const splpak_real *y, const splpak_real *w, int weighted, int64_t n);
/* Same with DEVICE arrays; asynchronous on the handle's stream (splpak_b200_fit_stream), which does NOT
 * synchronise with other streams: the arrays must be complete before the call (synchronise the producing
 * stream or make the handle's stream wait on its event). */
int splpak_b200_fit_add_points_device(splpak_b200_fit_t h, const splpak_real *d_x, int l1x,
                                      const splpak_real *d_y, const splpak_real *d_w, int weighted,
                                      int64_t n);

/* The partial sums a multi-GPU fit must add across ranks before compute: one contiguous DEVICE
 * buffer of *count float64 values [G in stencil storage | g | node histogram | totlwt | nrows].
 * Sum it in place with one all-reduce (NCCL via torch.distributed, or splpak_b200_fit_allreduce). */
int splpak_b200_fit_partial_buffer(splpak_b200_fit_t h, void **d_ptr, int64_t *count);
/* In-place ncclAllReduce(sum, float64) of that buffer on the handle's stream; comm is an
 * ncclComm_t passed as void*.  libnccl.so.2 is loaded lazily; 202 if that or the call fails. */
int splpak_b200_fit_allreduce(splpak_b200_fit_t h, void *nccl_comm);
/* Same for the ncol-long right-hand side of a refinement step (between refine_add_points and refine_compute). */
int splpak_b200_fit_allreduce_rhs(splpak_b200_fit_t h, void *nccl_comm);
/* NCCL communicators for hosts without torch.distributed (a Fortran or C program) -- (new), thin re-exports of
 * ncclCommInitAll / ncclGetUniqueId / ncclCommInitRank / ncclCommDestroy / ncclGroupStart / ncclGroupEnd through the
 * lazily loaded libnccl.so.2; communicators are passed as void*, the ncclUniqueId as its 128 raw bytes.
 *   one process, ndev GPUs : comm_init_all; wrap the per-device fit_allreduce calls in comm_group_start/end
 *   one process per GPU    : rank 0 calls comm_unique_id and distributes the bytes; every rank calls comm_init_rank */
int splpak_b200_comm_init_all(int ndev, const int *devs, void **comms);
int splpak_b200_comm_unique_id(char id[128]);
int splpak_b200_comm_init_rank(int nranks, int rank, const char id[128], void **comm);
int splpak_b200_comm_destroy(void *comm);
int splpak_b200_comm_group_start(void);
int splpak_b200_comm_group_end(void);

/* Add the data-sparse derivative-constraint rows (xtrap != 0), factor and solve.
 * coef/ncf as in splcw (104 if ncf < ncol); nwrk < 0 skips the reference's workspace checks.
 * coef is a HOST array. */
int splpak_b200_fit_compute(splpak_b200_fit_t h, splpak_real *coef, int64_t ncf, int64_t nwrk,
                            int *ierror);
/* Same, leaving the coefficients in DEVICE memory (d_coef, ncol values). */
int splpak_b200_fit_compute_device(splpak_b200_fit_t h, splpak_real *d_coef, int64_t ncf,
                                   int64_t nwrk, int *ierror);

/* Solver selection -- (new).  SPLPAK_SOLVER_CHOLESKY (default): band Cholesky of the normal equations (+ refinement).
 * SPLPAK_SOLVER_ORTHOGONAL: the rows are reduced by Householder reflections only, like the reference's suprls
 * (src/splpak.F90:1375-1695): per-window QR of the data and constraint rows, band QR of the stacked triangles,
 * back-substitution -- accurate at cond(A) instead of cond(A)^2, slower; 1-D..3-D, single GPU.  Must be called before
 * the first add_points (203 otherwise, or when the variant is not available for this grid).  The one-shot splcw /
 * splcc switch to it by themselves when the Cholesky factor reports a non-positive pivot or a pivot-ratio bound of
 * eps*cond(G) above 1e-3 (SPLPAK_B200_FIT=cholesky|orthogonal in the environment forces one). */
#define SPLPAK_SOLVER_CHOLESKY   0
#define SPLPAK_SOLVER_ORTHOGONAL 1
int splpak_b200_fit_set_solver(splpak_b200_fit_t h, int solver);
int splpak_b200_fit_get_solver(splpak_b200_fit_t h);
/* Smoothing -- (new) no counterpart in the reference.  The Cholesky fit then minimises
 *     sum_i (w_i (y_i - s(x_i)))^2  [+ the constraint rows when xtrap != 0]  +  lambda * integral over [xmin, xmax] of P(s)
 * with P(s) = sum_d (d2s/dx_d^2)^2 (SPLPAK_PENALTY_CURVATURE; multilinear functions are not penalised) or that plus
 * 2 sum_{i<j} (d2s/dx_i dx_j)^2 (SPLPAK_PENALTY_THIN_PLATE; affine functions are not penalised), in the caller's
 * coordinates.  fit_compute solves (G + lambda R) c = g; fit_get_normal_equations then returns S + lambda R, and the
 * refinement steps keep the penalty.  With lambda > 0, fewer points than columns is not an error (the penalty makes the
 * system well posed); a non-positive pivot still returns 107.  lambda = 0 (the default) is exactly the unsmoothed fit.
 * The setting persists across fit_reset.  Any time before fit_compute.  Returns 203 for an invalid or finalized handle, for
 * lambda < 0, NaN or inf, for an unknown penalty, and for lambda > 0 on the orthogonal solver (set_solver(ORTHOGONAL) on a
 * handle with lambda > 0 returns 203 too). */
#define SPLPAK_PENALTY_CURVATURE  0
#define SPLPAK_PENALTY_THIN_PLATE 1
int splpak_b200_fit_set_smoothing(splpak_b200_fit_t h, double lambda, int penalty);
/* Choosing lambda by generalized cross-validation -- (new).  With M = G0 + C + lambda R (G0 the assembled data rows, C the
 * constraint rows, R the penalty) and c = M^-1 g:
 *     RSS = sum_i (w_i (y_i - s(x_i)))^2 = ywy - 2 c.g + c^T G0 c,   edf = tr(M^-1 G0),   V = N RSS / (N - edf)^2
 * (N: the data rows counted, V = +inf when N <= edf).  edf is exact: Sigma = M^-1 is formed on the band of the Cholesky
 * factor (selected inverse).  RSS carries a cancellation: its relative error is about eps * ywy / RSS.
 *   enable_gcv          before the first add_points (203 otherwise): every add_points chunk also sums ywy = sum (w y)^2
 *                       into one more slot at the END of the partial buffer, [S | g | cnt | totlwt | nrows | ywy]
 *                       (fit_partial_buffer reports one more double, and the multi-GPU all-reduce sums it too).  Persists
 *                       across fit_reset, which zeroes ywy.  Not with the orthogonal solver (203, in either order).
 *   smoothing_score     after the (all-reduced) assembly, before fit_compute: out[0..4] = {V, RSS, edf, N, ywy}, nout >= 5.
 *                       Changes neither S, g, the counts nor the totals: a later compute is unaffected.  lambda = 0 is
 *                       allowed; a non-positive pivot returns 107.
 *   select_smoothing    V minimised over log10 lambda: a grid at 2 points per decade over [lambda_lo, lambda_hi], then
 *                       golden-section refinement around the best grid point down to 0.02 decades; ties go to the larger
 *                       lambda.  lambda_lo <= 0 or lambda_hi <= 0: rho * [1e-10, 1e4], rho = sum G0_ii / sum R_ii.  Points
 *                       with a non-positive pivot count as V = +inf (107 when all do).  On success it calls
 *                       set_smoothing(best, penalty), writes *lambda, the best point's out, and the evaluated
 *                       [lambda, V, RSS, edf] rows in evaluation order into trace (up to trace_cap rows; *ntrace = count).
 *   get_selected_inverse  parity hook, valid after a score call: out[ncol][b + 1], row i = Sigma(i, i..i+b) of the last
 *                       lambda scored (after select_smoothing: the selected lambda); out may be NULL to query *count.
 * All in FP64 (the REAL32 library too).  Given the same summed partial buffer, every output is bit-identical across calls,
 * handles and ranks, so every rank of a multi-GPU fit selects the same lambda.  203: invalid or finalized handle, GCV
 * not enabled, unknown penalty, lambda < 0 / NaN / inf, lambda_lo > lambda_hi. */
int splpak_b200_fit_enable_gcv(splpak_b200_fit_t h);
int splpak_b200_fit_smoothing_score(splpak_b200_fit_t h, double lambda, int penalty, double *out, int nout, int *ierror);
int splpak_b200_fit_select_smoothing(splpak_b200_fit_t h, int penalty, double lambda_lo, double lambda_hi, double *lambda,
                                     double *out, int nout, double *trace, int64_t trace_cap, int64_t *ntrace,
                                     int *ierror);
int splpak_b200_fit_get_selected_inverse(splpak_b200_fit_t h, double *out, int64_t capacity, int64_t *count);
/* Choosing lambda by REML (restricted maximum likelihood) -- (new).  M = G0 + C + lambda R and c = M^-1 g as above,
 * p = ncol, Mp the dimension of the penalty's null space (2^ndim for CURVATURE, ndim + 1 for THIN_PLATE, 2 for both in
 * 1-D), n the rows of the system COUNTING THE CONSTRAINT ROWS: they enter the likelihood as observations with a zero
 * response (GCV counts them as part of the regulariser instead; as data the score stays exact and needs only the factor).
 *     D_p   = ywy - 2 c.g + c^T M c          (= weighted RSS + constraint-row residuals + lambda c^T R c)
 *     phi   = D_p / (n - Mp)                 (the REML estimate of the noise variance)
 *     V_R   = (n - Mp) log(D_p / (n - Mp)) + log|M| - (p - Mp) log lambda
 * V_R is -2 x the restricted log-likelihood with the noise variance profiled out, WITHOUT its two lambda-independent
 * terms + (n - Mp)(1 + log 2 pi) and - log|R|+ (|R|+ the product of the non-zero eigenvalues of R): compare V_R only
 * across lambda for one grid and penalty.  log|M| = 2 sum log L_jj from the Cholesky factor; no selected inverse.
 * V_R = +inf when n <= Mp.
 *   reml_score          preconditions as smoothing_score (enable_gcv, Cholesky solver, after the all-reduced assembly,
 *                       before fit_compute; S, g, the counts and the totals stay untouched).  lambda > 0 (V_R -> +inf as
 *                       lambda -> 0).  out[0..5] = {V_R, D_p, log|M|, n, ywy, phi}, nout >= 6.  A non-positive pivot
 *                       returns 107.  It overwrites the band storage with a factor: get_selected_inverse returns 203 after
 *                       it, and a following prepare_variance scores by GCV once.
 *   select_smoothing_reml  V_R minimised with the search, default range and tie rule of select_smoothing; points with a
 *                       non-positive pivot count as +inf.  On success set_smoothing(best, penalty), the best point's six
 *                       values in out, trace rows [lambda, V_R, D_p, log|M|].  prepare_variance after it returns GCV's
 *                       sigma2 = RSS / (N - edf), not phi.
 * FP64, fixed-order reductions: bit-identical across calls, handles and ranks given the same summed partial buffer.
 * 203: as smoothing_score, and lambda <= 0. */
int splpak_b200_fit_reml_score(splpak_b200_fit_t h, double lambda, int penalty, double *out, int nout, int *ierror);
int splpak_b200_fit_select_smoothing_reml(splpak_b200_fit_t h, int penalty, double lambda_lo, double lambda_hi,
                                          double *lambda, double *out, int nout, double *trace, int64_t trace_cap,
                                          int64_t *ntrace, int *ierror);
/* Pointwise posterior variances of a smoothing fit -- (new).  With Sigma = M^-1 as above and b_k(x) the row of basis
 * values (nderiv = k: of their partial derivatives) at x,
 *     q_k(x) = b_k(x)^T Sigma b_k(x),     Var[d^k s(x)] = sigma2 q_k(x)     (the Bayesian posterior variance)
 * and w_i^2 q_0(x_i) is the leverage of data point i (the leverages sum to edf).
 *   prepare_variance    after the (all-reduced) assembly, before fit_compute; GCV enabled, Cholesky solver.  Uses the
 *                       handle's current (lambda, penalty): when the selected inverse of exactly that system is held
 *                       (after select_smoothing) it does not score again, otherwise it runs one smoothing_score.  Then it
 *                       builds one table of 10^ndim doubles per window (8 KB per window in 3-D, 80 KB in 4-D) into a
 *                       buffer the handle owns, so the tables survive fit_compute and the refinement steps.
 *                       out[0..5] = {V, RSS, edf, N, ywy, sigma2}, sigma2 = RSS / (N - edf) (+inf when N <= edf); nout >= 6.
 *   variance            HOST arrays x(l1x, nq) -> out(nq) = q(x), unscaled: multiply by sigma2 (or a known noise
 *                       variance).  nderiv: ndim entries in 0..2, NULL = values.
 *   variance_device     the same with device arrays, asynchronous on `stream` (NULL: the handle's stream).
 * Sequence: [select_smoothing ->] prepare_variance -> fit_compute -> variance*.  The tables become invalid with
 * add_points, fit_partial_buffer / fit_allreduce, fit_reset, and set_smoothing to another (lambda, penalty).  Exterior
 * queries use the clamped window and the linearly continued basis, as splde; a NaN coordinate gives NaN.  FP64 arithmetic
 * (the REAL32 library: float I/O).  Bit-identical across calls, and across handles and ranks given the same summed
 * partial buffer.  203: invalid handle, GCV not enabled, orthogonal solver, prepare_variance on a finalized handle or
 * with nout < 6, variance* without valid tables or with l1x < ndim; 104: nderiv outside 0..2 (nothing is computed);
 * 204: the tables cannot be allocated; 107: a non-positive pivot in the score.  nq <= 0 is a no-op.  A variance_device
 * call on another stream must complete before the next prepare_variance of the handle. */
int splpak_b200_fit_prepare_variance(splpak_b200_fit_t h, double *out, int nout, int *ierror);
int splpak_b200_fit_variance(splpak_b200_fit_t h, const splpak_real *x, int l1x, int64_t nq, const int *nderiv,
                             splpak_real *out, int *ierror);
int splpak_b200_fit_variance_device(splpak_b200_fit_t h, const splpak_real *d_x, int l1x, int64_t nq, const int *nderiv,
                                    splpak_real *d_out, void *stream, int *ierror);
/* Robust fit by iteratively reweighted least squares -- (new).  Data row i has coordinate x_i, value y_i and caller weight
 * w_i (1 when weighted = 0); only points with w_i > 0 take part.
 *   residual   r_i = w_i (y_i - s(x_i)), s evaluated as the refinement pass evaluates it
 *   scale      sigma = MAD / 0.6744897501960817, MAD = the k-th smallest |r_i| over the m points with w_i > 0, k = ceil(m/2)
 *              (the lower median, about 0; exact: MAD is one of the |r_i|, bit for bit)
 *   weights    t = r_i / (c sigma);  Huber (c = 1.345 by default): u_i = min(1, 1/|t|);  bisquare (c = 4.685 by default):
 *              u_i = (1 - t^2)^2 for |t| < 1, else 0;  u_i = 0 where w_i <= 0.  The next assembly uses row weights w_i sqrt(u_i).
 *   iteration  c^0 is the fit fit_compute would return for the points (the handle's lambda and penalty, constraint rows
 *              included); iteration k takes the residuals of c^(k-1) to get sigma_k and u^k, re-assembles S and g with the
 *              new row weights, adds the constraint rows and lambda R, factors and solves for c^k.
 *   stopping   max_j |c^k_j - c^(k-1)_j| <= tol max_j |c^k_j|, or k = max_iter.  MAD = 0 (the fit interpolates at least half
 *              the points): stop with the current coefficients, converged.
 *   constraint rows  the node histogram and [totlwt, nrows] come from the first assembly with the caller's weights and stay
 *              fixed for the call: the data-sparse nodes, and so the constraint rows, are the same in every iteration.
 *   refinement when constraint rows fired, two corrected-semi-normal-equation steps after the last solve, with the final row
 *              weights (as splcw for an ordinary fit; none in the REAL32 library).
 * out[0..5] = {iterations completed, the last sigma computed (0 when the MAD = 0 stop fired), the last relative change
 * (0 before the first), sum of u_i, points with w_i > 0 and u_i = 0, converged (0/1)}, nout >= 6.  u (optional, NULL
 * allowed): the u_i of the final solve.  tuning <= 0 selects the default c.
 * Preconditions: a fresh or reset handle (no add_points yet), the Cholesky solver; the call does its own assembly.  After it
 * the handle is finalized as after fit_compute, refine_begin returns 203 (it would re-feed the caller's weights) and the
 * score and variance calls are refused as after fit_compute.
 * Errors: 203 invalid or used handle, orthogonal solver, unknown psi, tuning NaN or inf, max_iter < 1, tol < 0 or NaN,
 * nout < 6, l1x < ndim; 104 ncf < ncol; 105 n < 1; 107 a non-positive pivot in any iteration (coef then holds the last
 * successful iterate, out[0] counts the completed iterations, u the weights of the failed solve); 204 the host entry
 * cannot allocate device copies of the points (it copies them once for the whole call).
 * Multi-GPU: nccl_comm NULL means one GPU; otherwise every rank passes its shard and its communicator (splpak_b200_comm_*)
 * and the call all-reduces, on the handle's stream, the partial buffer after each assembly, the integer histograms of the
 * median selection, the convergence numbers and the right-hand side of the refinement steps: every input of the replicated
 * solve is the same on every rank, so the replicas stay bit-identical.  A process that drives several devices calls the
 * function from one host thread per device.
 * FP64 keys, scale and weights (the REAL32 library: float I/O, the residual from its working-precision splfe).
 * Repeated calls with the same input return bit-identical coef, u and out in SPLPAK_B200_DETERMINISTIC=1 mode, and with
 * the default assembly up to the order of its FP64 atomic sums. */
#define SPLPAK_ROBUST_HUBER    0
#define SPLPAK_ROBUST_BISQUARE 1
int splpak_b200_fit_robust_device(splpak_b200_fit_t h, const splpak_real *d_x, int l1x, const splpak_real *d_y,
                                  const splpak_real *d_w, int weighted, int64_t n, int psi, double tuning, int max_iter,
                                  double tol, void *nccl_comm, splpak_real *d_coef, int64_t ncf, splpak_real *d_u,
                                  double *out, int nout, int *ierror);
/* Same with HOST x, y, w, coef and u. */
int splpak_b200_fit_robust(splpak_b200_fit_t h, const splpak_real *x, int l1x, const splpak_real *y,
                           const splpak_real *w, int weighted, int64_t n, int psi, double tuning, int max_iter,
                           double tol, void *nccl_comm, splpak_real *coef, int64_t ncf, splpak_real *u, double *out,
                           int nout, int *ierror);
/* Generalized smoothing fit by penalized iteratively reweighted least squares (PIRLS) -- (new).  Data row i has
 * coordinate x_i, response y_i, caller weight w_i (1 when weighted = 0) and offset o_i (0 when offset is NULL); only
 * points with w_i > 0 take part.
 *   prior weight      a_i = w_i^2 (row i of a least-squares fit contributes (w_i (y_i - s))^2).  Binomial: y_i is a
 *                     proportion and a_i the number of trials, so pass w_i = sqrt(trials).
 *   linear predictor  eta_i = s(x_i) + o_i, s evaluated as the refinement pass evaluates it.
 *   family            link   mu(eta) and dmu/deta                              V(mu)        valid y     start mu0
 *     POISSON  (0)    log    max(exp(eta), eps), same                          mu           y >= 0      y + 0.1
 *     BINOMIAL (1)    logit  R's logit_linkinv / logit_mu_eta (+-30, eps, 1/eps) mu (1 - mu)  0 <= y <= 1 (a y + 0.5)/(a + 1)
 *     GAMMA    (2)    log    max(exp(eta), eps), same                          mu^2         y > 0       y
 *                     eps = 2^-52: the clamps of R's make.link, the starts of glm.fit.  eta itself is not clamped.
 *   working values    z_i = eta_i - o_i + (y_i - mu_i) / mu'_i, W_i = a_i mu'_i^2 / V(mu_i); the assembly takes the
 *                     response z_i with row weight sqrt(W_i) = w_i mu'_i / sqrt(V); z_i = 0 and row weight 0 where
 *                     w_i <= 0 (y_i is not read there).
 *   deviance          D = sum over w_i > 0 of R's unit deviances (y log y = 0 at y = 0): Poisson 2 a (y log(y/mu) -
 *                     (y - mu)), binomial 2 a (y log(y/mu) + (1-y) log((1-y)/(1-mu))), Gamma -2 a (log(y/mu) -
 *                     (y - mu)/mu);  Pearson X^2 = sum a (y - mu)^2 / V(mu).
 *   iteration k = 1, 2, ...  z and W from the current mu (k = 1: mu0, eta0 = g(mu0), the offset ignored as glm.fit
 *                     does); assemble (k = 1: the ordinary first assembly, whose node histogram and [totlwt, nrows]
 *                     stay fixed for the call; later: S and g only); the constraint rows and lambda R (the handle's
 *                     lambda and penalty); factor and solve for c^k; evaluate eta^k, mu^k and D_k.
 *   step halving      while D_k is not finite: c^k = (c^k + c^(k-1)) / 2 and evaluate again, at most 10 times (glm.fit).
 *                     Still not finite, or not finite at k = 1: 107, coef = the last iterate with a finite deviance
 *                     (c^1 at k = 1).
 *   stopping          |D_k - D_(k-1)| / (|D_k| + 0.1) < tol (D_0: the deviance of mu0), or k = max_iter.  glm.control's
 *                     defaults are tol = 1e-8, max_iter = 25.
 *   refinement        when constraint rows fired and the last iteration took its full step, two corrected-semi-normal-
 *                     equation steps of splcw follow the last solve, with that solve's z and row weights (none in the
 *                     REAL32 library), then one more evaluation: out and mu describe the returned coefficients.
 * out[0..6] = {iterations (solves completed), D, X^2, the last relative deviance change, step halvings in all,
 * converged (0/1), m = points with w_i > 0}, nout >= 7.  mu (optional, NULL allowed): the fitted means at the points.
 * Preconditions: a fresh or reset handle (no add_points yet), the Cholesky solver; the call does its own assembly.  After
 * it the handle is finalized as after fit_compute, refine_begin returns 203 and the score and variance calls are refused
 * as after fit_compute.
 * Errors: 203 invalid or used handle, orthogonal solver, unknown family, max_iter < 1, tol < 0 or NaN, nout < 7,
 * l1x < ndim, or any y_i outside its family's domain (or not finite) where w_i > 0 -- checked on the device before the
 * first assembly, after which the handle is still fresh; 104 ncf < ncol; 105 n < 1 or m = 0; 107 as above, or a
 * non-positive pivot (coef then holds the last successful iterate); 204 the host entry cannot allocate its device
 * copies (it copies the points once for the whole call).
 * Multi-GPU: nccl_comm NULL means one GPU; otherwise every rank passes its shard and the call all-reduces, on the
 * handle's stream, the domain-check counts, the partial buffer after the first assembly, [S | g] after each
 * re-assembly, {D, X^2, ywy} of each evaluation and the right-hand side of the refinement steps: every rank makes the same
 * halving and stopping decisions and the replicas stay bit-identical.
 * All reductions are fixed-order per-CTA partial sums (no FP64 atomics): with SPLPAK_B200_DETERMINISTIC=1 repeated calls
 * and the host and device entries return bit-identical coef, mu and out.  REAL32: float I/O (and float z and row
 * weights for its assembly), FP64 everything else. */
#define SPLPAK_GLM_POISSON  0
#define SPLPAK_GLM_BINOMIAL 1
#define SPLPAK_GLM_GAMMA    2
int splpak_b200_fit_glm_device(splpak_b200_fit_t h, const splpak_real *d_x, int l1x, const splpak_real *d_y,
                               const splpak_real *d_w, int weighted, const splpak_real *d_offset, int64_t n, int family,
                               int max_iter, double tol, void *nccl_comm, splpak_real *d_coef, int64_t ncf,
                               splpak_real *d_mu, double *out, int nout, int *ierror);
/* Same with HOST x, y, w, offset, coef and mu. */
int splpak_b200_fit_glm(splpak_b200_fit_t h, const splpak_real *x, int l1x, const splpak_real *y, const splpak_real *w,
                        int weighted, const splpak_real *offset, int64_t n, int family, int max_iter, double tol,
                        void *nccl_comm, splpak_real *coef, int64_t ncf, splpak_real *mu, double *out, int nout,
                        int *ierror);
/* GLM fit with the smoothing parameter chosen on each PIRLS working system ("performance iteration") -- (new).
 * Everything fit_glm_device says holds (data, families, working values, deviance, halving, stopping, the fixed node
 * histogram and totals, refinement, multi-GPU, determinism), except that lambda is chosen inside the loop.
 *   working system    iteration k assembles S_k, g_k from z and sqrt(W), and ywy_k = sum (sqrt(W_i) z_i)^2;
 *                     M(lambda) = G0_k + C + lambda R with the given penalty.
 *   criterion         the scores of smoothing_score / reml_score on that system (same quantities and counting: REML
 *                     counts the constraint rows as observations, GCV / UBRE count them as part of the regulariser),
 *                     the family deciding whether the scale is known:
 *                                     Poisson, binomial (phi = 1)              Gamma (phi unknown)
 *                       REML          V = D_p + log|M| - (p - Mp) log lambda   the profiled V_R of reml_score
 *                       PREDICTION    UBRE U = RSS / N - 1 + 2 edf / N          GCV V = N RSS / (N - edf)^2
 *   phase 1 (selecting)  k = 1: the search of select_smoothing over [lambda_lo, lambda_hi] (either <= 0: rho [1e-10,
 *                     1e4] with rho from the first working system): a grid at 2 points per decade, golden section to
 *                     0.02 decades, ties to the larger lambda.  k >= 2: the same search over log10 lambda_(k-1) +- 1
 *                     decade clipped to the range, repeated over the whole range when its best grid point is an end of
 *                     the window but not of the range.  Points with a non-positive pivot count as +inf (107 when all
 *                     of a search do).  lambda_k then goes on the handle and the iteration solves with it.
 *   phase 2           phase 1 ends at the first k >= 2 with |log10 lambda_k - log10 lambda_(k-1)| <= 0.05 (settled), or
 *                     after max_select selecting iterations (not settled).  lambda-hat = lambda_k is then frozen and the
 *                     loop continues as fit_glm's fixed-lambda PIRLS; `converged` needs a fixed-lambda iteration to
 *                     meet the stopping rule.  max_iter counts all solves (tol = 0, max_iter = k: iterate k).  A
 *                     converged, settled result is the fixed-lambda GLM fit at lambda-hat.
 *   after the loop    the refinement steps (when constraint rows fired); then the system of the last solve is rebuilt
 *                     (z and sqrt(W) from c^(k-1), or mu0) and one GCV score at lambda-hat gives edf = tr(M^-1 G0) and
 *                     leaves Sigma = M^-1 in the band storage; with variance = 1 the tables of prepare_variance are
 *                     built from it, so fit_variance[_device] return q(x) = b(x)^T M^-1 b(x) of the final working
 *                     system and phi-hat q(x) is the Bayesian variance of eta(x) (mgcv's Vp).  The final evaluation of
 *                     the returned coefficients fills out and mu.
 * out[0..6] as fit_glm; out[7..12] = {lambda-hat, the criterion at lambda-hat in the last selecting iteration, edf,
 * phi-hat, selecting iterations, settled (0/1)}, nout >= 13; phi-hat = 1 (Poisson, binomial) or X^2 / (m - edf) (Gamma;
 * +inf when m <= edf).  trace (may be NULL): one row per iteration, [lambda_k, the criterion at lambda_k (NaN when
 * frozen), scores evaluated, D_k, halvings_k], at most trace_cap rows; *ntrace = rows written.
 * On return the handle's lambda is lambda-hat with the given penalty, GCV is enabled on it (the call enables it on the
 * fresh handle), and get_cholesky_factor returns 203 (Sigma has overwritten the factor).
 * Errors: those of fit_glm_device, and 203 for an unknown criterion or penalty, NaN or inf bounds, lambda_lo > lambda_hi
 * with both > 0, max_select < 1, trace_cap < 0, nout < 13 (a refused call leaves the handle fresh; the domain check
 * still runs before anything touches it); 204 when the score scratch or the variance tables cannot be allocated (before
 * the first assembly: the handle stays fresh).
 * Multi-GPU: every score is computed from the all-reduced system with fixed-order reductions, so every rank takes the
 * same search path and the replicas stay bit-identical.  With SPLPAK_B200_DETERMINISTIC=1 repeated calls and the host
 * and device entries return bit-identical coef, mu, out and trace. */
#define SPLPAK_GLM_SELECT_REML       0
#define SPLPAK_GLM_SELECT_PREDICTION 1   /* UBRE for Poisson / binomial, GCV for Gamma */
int splpak_b200_fit_glm_select_device(splpak_b200_fit_t h, const splpak_real *d_x, int l1x, const splpak_real *d_y,
                                      const splpak_real *d_w, int weighted, const splpak_real *d_offset, int64_t n,
                                      int family, int criterion, int penalty, double lambda_lo, double lambda_hi,
                                      int max_select, int variance, int max_iter, double tol, void *nccl_comm,
                                      splpak_real *d_coef, int64_t ncf, splpak_real *d_mu, double *out, int nout,
                                      double *trace, int64_t trace_cap, int64_t *ntrace, int *ierror);
/* Same with HOST x, y, w, offset, coef and mu. */
int splpak_b200_fit_glm_select(splpak_b200_fit_t h, const splpak_real *x, int l1x, const splpak_real *y,
                               const splpak_real *w, int weighted, const splpak_real *offset, int64_t n, int family,
                               int criterion, int penalty, double lambda_lo, double lambda_hi, int max_select,
                               int variance, int max_iter, double tol, void *nccl_comm, splpak_real *coef, int64_t ncf,
                               splpak_real *mu, double *out, int nout, double *trace, int64_t trace_cap,
                               int64_t *ntrace, int *ierror);
/* Parity-test hook of the orthogonal path: which = 0 -> per-window triangles [nwindows][4^ndim][4^ndim + 1] (R_w | z_w),
 * which = 1 -> band factor [ncol][b + 2] (row i: R[i][i..i+b], then (Q^T r)_i).  out may be NULL to query *count. */
int splpak_b200_fit_get_orthogonal_factor(splpak_b200_fit_t h, int which, double *out, int64_t capacity, int64_t *count);
/* Parity-test hook of the Cholesky path, valid after fit_compute and the refinement steps (203 otherwise, e.g. after a
 * score call, which leaves Sigma or the factor of another M in the band storage).  G = L L^T in lower band storage with
 * lda = (b + 65) rounded up to even, panels of 64 columns.  Columns first_col .. first_col + ncols - 1:
 *   which = 0 -> out[ncols][lda], row j - first_col = the band column j, rows j .. j + lda - 1 (entry r: L(j + r, j)).
 *                Outside the 64 x 64 diagonal blocks these are L, and exactly 0 where j + r >= ncol or r > b.  The
 *                diagonal blocks are scratch and hold no part of L on any route: the panel kernels factor them in shared
 *                memory and keep only L11^-1; what is left there (an updated A11) depends on the route.
 *   which = 1 -> out[nblk][64][64], the block inverses L11^-1 (row-major) of the panels first_col / 64 .. (first_col +
 *                ncols - 1) / 64; a last panel of nb < 64 columns is padded with the identity.
 * out may be NULL to query *count.  203 also for which outside 0..1 or a column range outside 0..ncol-1. */
int splpak_b200_fit_get_cholesky_factor(splpak_b200_fit_t h, int which, int64_t first_col, int64_t ncols, double *out,
                                        int64_t capacity, int64_t *count);
/* (max L_jj / min L_jj)^2 of the last Cholesky factor: a cheap LOWER bound of cond(G); 0 when unknown. */
int splpak_b200_fit_condition_estimate(splpak_b200_fit_t h, double *cond_lower_bound);

/* Refinement by corrected semi-normal equations -- (new) no counterpart in the reference, whose orthogonal
 * solver (suprls, src/splpak.F90:1375-1695) does not need it.  The Cholesky solve works at cond(G) =
 * cond(A)^2; when derivative-constraint rows fire (xtrap != 0 and data holes) that is what separates its
 * coefficients from suprls's.  One step = a second pass over THE SAME points (any chunking), residuals formed row by
 * row, one more solve with the same G:
 *     fit_compute -> [fit_refine_begin -> fit_refine_add_points* -> (all-reduce fit_rhs_buffer across ranks)
 *                     -> fit_refine_compute] x k
 * splpak_b200_splcw / splcc run two steps automatically when constraint rows fired.  A no-op in the REAL32 library. */
int splpak_b200_fit_refine_begin(splpak_b200_fit_t h);
int splpak_b200_fit_refine_add_points(splpak_b200_fit_t h, const splpak_real *x, int l1x,
                                      const splpak_real *y, const splpak_real *w, int weighted, int64_t n);
int splpak_b200_fit_refine_add_points_device(splpak_b200_fit_t h, const splpak_real *d_x, int l1x,
                                             const splpak_real *d_y, const splpak_real *d_w, int weighted,
                                             int64_t n);
int splpak_b200_fit_refine_compute(splpak_b200_fit_t h, splpak_real *coef, int64_t ncf, int *ierror);
int splpak_b200_fit_refine_compute_device(splpak_b200_fit_t h, splpak_real *d_coef, int64_t ncf, int *ierror);
/* 1 if the last fit_compute added derivative-constraint rows (the regime where refinement pays). */
int splpak_b200_fit_constraints_fired(splpak_b200_fit_t h);
/* The right-hand-side slice (ncol float64) of the partial buffer: what a multi-GPU refinement step sums. */
int splpak_b200_fit_rhs_buffer(splpak_b200_fit_t h, void **d_ptr, int64_t *count);

/* Start a new fit on the same grid (zeroes the partial sums). */
int splpak_b200_fit_reset(splpak_b200_fit_t h);
/* cudaStream_t (as void*) the handle launches on. */
void *splpak_b200_fit_stream(splpak_b200_fit_t h);
/* Device-time split of everything since create/reset, milliseconds:
 * ms[0] classify+histogram, ms[1] scan+scatter (binning), ms[2] accumulate, ms[3] constraints (and, with smoothing,
 * the penalty tables and S += lambda R), ms[4] band expand, ms[5] factor, ms[6] back-substitution.  Synchronises the stream. */
int splpak_b200_fit_timings(splpak_b200_fit_t h, double *ms, int n);
/* Kernels this handle has launched since create/reset (for bench.py's gpu_launches). */
int64_t splpak_b200_fit_launch_count(splpak_b200_fit_t h);
/* Debug/parity access: copy the assembled G (stencil storage, ncol*4^ndim float64), g (ncol),
 * node histogram (ncol) and [totlwt, nrows] to HOST arrays (any may be NULL).  After a compute with smoothing
 * (lambda > 0), S holds G + lambda R. */
int splpak_b200_fit_get_normal_equations(splpak_b200_fit_t h, double *S, double *g, double *cnt,
                                         double *totals);
int splpak_b200_fit_destroy(splpak_b200_fit_t h);

/* ------------------------------------------------------------------------------------------
 * Measurement helpers (used by bench.py for the FP64 roofline denominator; MEASURED_PEAKS.json
 * has no FP64 entry).
 * ---------------------------------------------------------------------------------------- */
/* out[0] = DFMA TFLOP/s, out[1] = DMMA.8x8x4 TFLOP/s, out[2] = device copy GB/s (read+write). */
int splpak_b200_measure_peaks(double *out, int n);
/* Total kernels launched by this library in this process. */
int64_t splpak_b200_total_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* SPLPAK_B200_H */
