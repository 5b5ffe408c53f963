/* dnsb.h -- C ABI of libdnsb200.so, the sm_100a CUDA library behind
 * dolfin_navier_scipy_b200.
 *
 * The reference (highlando/dolfin_navier_scipy) is pure Python and has no FFI;
 * its seams are Python call sites (SURVEY.md section 8b).  Every entry point
 * below names the reference code whose arithmetic it replaces.  All pointers
 * are HOST pointers unless the name ends in `_dev`; host arrays are borrowed
 * for the duration of the call.  Indices are int32, values are fp64.
 *
 * Batched ("ensemble") layout: a vector of n entries for nb members is stored
 * member-fastest, x[i*nb + m].  nb = 1 is a plain vector.
 *
 * Return value: 0 = ok, < 0 = error (message via dnsb_last_error);
 * DNSB_E_NOT_CONVERGED: an iterative solve stopped at `maxit` above `tol` --
 * the outputs / the state are valid and can be read, the caller decides (the
 * reference's sparse-LU solve cannot fail this way).  Nothing throws across
 * the ABI.  One context = one device + one stream; a context is
 * not thread-safe.
 *
 * Handles: a dnsb_*_create sets *out only on success; on failure *out is NULL
 * and nothing it allocated stays allocated.  The exception is
 * dnsb_ctx_create, which returns its context on failure as well so that the
 * message can be read with dnsb_last_error; the caller then destroys it.
 * dnsb_*_destroy waits for the work queued on the handle's streams, then
 * frees everything the handle owns (matrices and solvers passed in are
 * borrowed and stay the caller's).
 */
#ifndef DNSB_H
#define DNSB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DNSB_E_NOT_CONVERGED (-3)

typedef struct dnsb_ctx dnsb_ctx;
typedef struct dnsb_csr dnsb_csr;       /* CSR pattern + 1..2 value arrays on the device */
typedef struct dnsb_solver dnsb_solver; /* saddle-point FGMRES solver */
typedef struct dnsb_imex dnsb_imex;     /* device-resident IMEX time stepper */
typedef struct dnsb_cnsweep dnsb_cnsweep; /* device-resident Picard/Newton + Crank-Nicolson sweep */

/* ---- context ------------------------------------------------------------ */
int dnsb_ctx_create(int device, dnsb_ctx **out);
void dnsb_ctx_destroy(dnsb_ctx *ctx);
const char *dnsb_last_error(dnsb_ctx *ctx);
int dnsb_version(void);
/* sm count, total device memory, compute capability major*10+minor */
int dnsb_device_info(dnsb_ctx *ctx, int *sm_count, size_t *mem_bytes, int *cc);
int dnsb_sync(dnsb_ctx *ctx);
/* counters of kernels launched by this context since creation / last reset */
long long dnsb_launch_count(dnsb_ctx *ctx);
void dnsb_launch_count_reset(dnsb_ctx *ctx);

/* per-kernel device timing with CUDA events on the context's stream: begin
 * records up to `max_records` launches, end writes "kernel count total_ms work"
 * lines (sorted by time) into buf and returns the bytes needed; `work` is the
 * sum of a per-launch size some kernels report (Gram-Schmidt: basis vectors
 * read), so that their average algorithmic bytes can be computed. */
int dnsb_profile_begin(dnsb_ctx *ctx, int max_records);
int dnsb_profile_end(dnsb_ctx *ctx, char *buf, int buflen);
/* bytes of device memory and of pinned host memory held by the library in
 * this process, over all contexts (either pointer may be NULL): a leak shows
 * here exactly, unlike in the device's free memory, which other processes
 * share */
void dnsb_live_bytes(long long *device, long long *pinned);

/* ---- mesh + convection assembly (K1a / K1b) ------------------------------
 * dnsb_set_mesh: P2 scalar cell dofmap (ncell*6, local order 3 vertices then
 * the edge opposite to vertex i), affine geometry per cell (ncell*5:
 * grad(lambda_1).x, .y, grad(lambda_2).x, .y, detJ) and a colouring of the
 * cell conflict graph (cells sharing a vertex get different colours), so that
 * the scatter needs no atomics and is deterministic.
 * Replaces the dolfin cell loop behind `dolfin.assemble` in
 * dolfin_to_sparrays.py:462-470 and :358-364. */
int dnsb_set_mesh(dnsb_ctx *ctx, int ncell, int nnodes,
                  const int32_t *cell_nodes, const double *geom,
                  int ncolours, const int32_t *cell_colour);
/* fixed CSR pattern of the P2 vector space (2*nnodes rows) and, per cell, the
 * 144 CSR slots of its 12x12 element matrix (row-major, dof = 2*local+comp) */
int dnsb_set_conv_pattern(dnsb_ctx *ctx, const int32_t *indptr,
                          const int32_t *indices, const int32_t *cell_slots);
/* c = int (grad(u1) u2).phi dx on all 2*nnodes dofs (u2 == NULL: u2 = u1).
 * dolfin_to_sparrays.py:427-472 (get_convvec).  nb members, batched layout. */
int dnsb_convvec(dnsb_ctx *ctx, const double *u1, const double *u2,
                 double *out, int nb);
/* Constant operators of the Taylor-Hood discretisation assembled on the device
 * with the per-cell machinery of K1b (SURVEY.md 8f-1; replaces the dolfin
 * assembles of dolfin_to_sparrays.py:243-275, get_stokessysmats): values of
 * the mass matrix M and of A = nu*int 2 eps(u):grad(v) (symgrad != 0) or
 * 2 nu int grad(u):grad(v) on the pattern of dnsb_set_conv_pattern (zeros
 * kept); optionally J = int q div(u) (P1 x P2-vector) and the pressure mass
 * MP on patterns of the caller: jslots[c*36 + k*12 + 2m+b] / mpslots[c*9 + k*3 + l]
 * give the CSR slot of the element entries of (host) cell c.  j_vals / mp_vals
 * may be NULL.  Boundary terms (outflow correction, Robin) stay on the host. */
int dnsb_assemble_stokes(dnsb_ctx *ctx, double nu, int symgrad, int jnnz,
                         const int32_t *jslots, int mpnnz, const int32_t *mpslots,
                         double *m_vals, double *a_vals, double *j_vals,
                         double *mp_vals);
/* N1, N2 values in the fixed pattern and f3 = N(u0)u0;
 * dolfin_to_sparrays.py:325-376 (get_convmats).  Any output may be NULL. */
int dnsb_convmats(dnsb_ctx *ctx, const double *u0, double *n1_data,
                  double *n2_data, double *f3);

/* ---- CSR matrices and SpMV/SpMM (K2) -------------------------------------
 * value(k, m) = vals1[k] + coef[m]*vals2[k]   (vals2/coef optional).
 * Replaces scipy.sparse `M*v`, `A*v` of time_int_utils.py:125-128 etc. */
int dnsb_csr_create(dnsb_ctx *ctx, int nrows, int ncols, const int32_t *indptr,
                    const int32_t *indices, const double *vals1,
                    const double *vals2, dnsb_csr **out);
void dnsb_csr_destroy(dnsb_csr *mat);
/* y = alpha*A*x + beta*y on host vectors (nb members, coef may be NULL) */
int dnsb_spmm(dnsb_csr *mat, const double *coef, const double *x, double *y,
              int nb, double alpha, double beta);
/* device-resident variant for benchmarking: x_dev/y_dev are device pointers */
int dnsb_spmm_dev(dnsb_csr *mat, const double *coef_dev, const double *x_dev,
                  double *y_dev, int nb, double alpha, double beta);

/* ---- saddle-point solver (K3) --------------------------------------------
 *   [ F_m  JT ] [v]   [rhsv]        F_m = vals1 + coef[m]*vals2 of `fmat`
 *   [ J    0  ] [q] = [rhsp]
 * by right-preconditioned FGMRES(restart) with the block-triangular
 * preconditioner  P = [Fh  JT; 0  -Sh]:  Fh^-1 = `cheb_steps` steps of
 * Jacobi-Chebyshev on F (spectrum of D^-1 F in [lmin, lmax]), Sh^-1 = the
 * pressure hierarchy set with dnsb_solver_set_schur_* (dense inverse and/or
 * AMG V-cycle levels).  Replaces sadptprj_riclyap_adi.lin_alg_utils.
 * solve_sadpnt_smw (SuperLU) at stokes_navier_utils.py:401,458,497,903,1505,
 * 1629 and time_int_utils.py:89-91,134,402,466. */
int dnsb_solver_create(dnsb_ctx *ctx, dnsb_csr *fmat, dnsb_csr *jmat,
                       dnsb_csr *jtmat, const double *coef, int nb,
                       int restart, int cheb_steps, double lmin, double lmax,
                       dnsb_solver **out);
void dnsb_solver_destroy(dnsb_solver *s);
/* Schur approximation level l of the pressure hierarchy (0 = finest).
 * `amat`: the SPD pressure operator on this level, `pmat`: prolongation from
 * level l+1 (NULL on the coarsest), smoother = `nsmooth` Jacobi-Chebyshev steps
 * with bounds [lmin,lmax].  The coarsest level is solved with a dense inverse
 * (row-major n*n) given in `dense_inv`; a sparse level without `pmat`/`rmat`
 * is terminal too and "solved" by its smoother alone. */
int dnsb_solver_add_schur_level(dnsb_solver *s, dnsb_csr *amat, dnsb_csr *pmat,
                                dnsb_csr *rmat, int nsmooth, double lmin,
                                double lmax, const double *dense_inv);
/* coarse levels of the velocity block (level 0 is F itself with `cheb_steps`
 * Chebyshev smoothing): transfer operators between level 0 and level 1, then
 * the levels 1.. like the Schur levels.  Without them Fh^-1 is the plain
 * Chebyshev iteration (enough for the mass-dominated time-stepping matrices;
 * the V-cycle is needed for Stokes/Oseen systems). */
int dnsb_solver_set_velocity_transfer(dnsb_solver *s, dnsb_csr *pmat, dnsb_csr *rmat);
int dnsb_solver_add_velocity_level(dnsb_solver *s, dnsb_csr *amat, dnsb_csr *pmat,
                                   dnsb_csr *rmat, int nsmooth, double lmin,
                                   double lmax, const double *dense_inv);
/* additive term  + mp_scale[m] * diag(mp_dinv) of the Schur approximation
 * (Cahouet-Chabard); with no Schur level set it is the whole approximation
 * (scaled pressure mass matrix, the Stokes/Oseen choice) */
int dnsb_solver_set_schur_mass(dnsb_solver *s, const double *mp_dinv,
                               const double *mp_scale);
/* least-squares-commutator Schur approximation for stiffness dominated blocks
 * (Stokes, Oseen/Picard, Newton; stokes_navier_utils.py:401,458,497):
 *   Sh^-1 = L^-1 (J Du^-1 F Du^-1 JT) L^-1,   L = J Du^-1 JT,
 * `du_inv` = 1/diag(velocity mass matrix) (nv); the Schur levels added before
 * must be the hierarchy of L. */
int dnsb_solver_set_schur_lsc(dnsb_solver *s, const double *du_inv);
/* solve for nb members; x0 may be NULL (zero initial guess); vp has
 * (nv+np)*nb entries.  iters/relres: per-member outputs (may be NULL). */
int dnsb_solver_solve(dnsb_solver *s, const double *rhsv, const double *rhsp,
                      const double *x0, double *vp, double tol, int maxit,
                      int *iters, double *relres);

/* new values of the velocity block `fmat` (single value array, nnz entries in
 * the order of the pattern given at creation): the per-step matrices
 * M + dt/2 (A + N(v)) of the Picard/Newton + Crank-Nicolson sweeps
 * (stokes_navier_utils.py:1484-1512) and of the steady Picard/Newton iteration
 * (:438-525) change values, not pattern; the preconditioner set-up is kept. */
int dnsb_solver_update_fvalues(dnsb_solver *s, const double *vals1);
/* z = P^-1 r: one application of the block-triangular preconditioner to host
 * vectors ((nv+np)*nb); used by the tests to check the multigrid / Schur
 * pieces against a numpy restatement */
int dnsb_solver_apply_prec(dnsb_solver *s, const double *r, double *z);
/* block_diagonal = 1: the preconditioner is applied as diag(Fh^-1, +Sh^-1) (symmetric positive definite, what
 * MINRES needs; Chebyshev velocity block + dense Schur block only); 0 (default): block triangular (FGMRES).
 * Replaces nothing in the reference: its MINRES experiment (`stokes_navier_utils.py:879-890`) is unpreconditioned. */
int dnsb_solver_set_prec_mode(dnsb_solver *s, int block_diagonal);
/* y = K x with K = [[F, JT], [J, 0]] of the solver, host vectors of (nv + np) x nb doubles (operator for host-driven
 * Krylov methods: `lin_alg_utils.solve_sadpnt_smw(krylov='minres')`) */
int dnsb_solver_apply_k(dnsb_solver *s, const double *x, double *y);

/* ---- device-resident IMEX time stepping ----------------------------------
 * CNAB (time_int_utils.py:23-145), SBDF2 (:260-355) incl. the Heun start
 * (:366-477), IMEX Euler (:566-635), the blow-up guard (:94-103) and the
 * convection re-evaluation of stokes_navier_utils.py:1136-1140 per step.
 *   A_m = nu[m]*a0 + arob,   F_m(tau) = M + tau*A_m.
 * `mmat` holds (vals1 = M), `amat` holds (vals1 = arob or zeros, vals2 = a0)
 * on the same pattern; `jmat`/`jtmat` the divergence/gradient blocks.
 * scheme: 0 = CNAB, 1 = SBDF2, 2 = IMEX Euler. */
int dnsb_imex_create(dnsb_ctx *ctx, int scheme, int nb, double dt,
                     dnsb_csr *mmat, dnsb_csr *amat, dnsb_csr *jmat,
                     dnsb_csr *jtmat, const double *nu,
                     const int32_t *invinds, int nv, int nbc,
                     const int32_t *bcinds, const double *bcvals,
                     const double *fv, const double *fp, dnsb_imex **out);
void dnsb_imex_destroy(dnsb_imex *e);
/* the three solvers (loop matrix tau=theta*dt; Heun predictor tau=dt; Heun
 * corrector tau=0), created by the caller with dnsb_solver_create */
int dnsb_imex_set_solvers(dnsb_imex *e, dnsb_solver *loop, dnsb_solver *pred,
                          dnsb_solver *corr);
/* time-dependent forcing  f(t_n) = sum_k useries[(n*nk + k)*nb + m] * b[i*nk + k]
 * (nk input shapes b (nv x nk, row-major), ntimes = nsteps+1 samples);
 * useries[0] belongs to the time level at which this function is called, so a
 * running integration can be fed chunk by chunk */
int dnsb_imex_set_forcing(dnsb_imex *e, int nk, const double *bvecs,
                          int ntimes, const double *useries);
/* initial state (inner velocity nv*nb, pressure np*nb) */
int dnsb_imex_set_state(dnsb_imex *e, const double *v0, const double *p0);
/* run `nsteps` steps from the current state.  Snapshots [v (nv*nb); p (np*nb)]
 * are stored on the device every `snap_stride` steps (0 = none), including the
 * initial state.  tol/maxit: FGMRES controls; guess: 0 = previous solution,
 * 1 = linear extrapolation, k>=2 = projection onto the last k solutions.
 * ffflag (out): 1 if the blow-up guard tripped (time_int_utils.py:99-103);
 * with the per-member guard: 1 if at least one member was retired in this run. */
int dnsb_imex_run(dnsb_imex *e, int nsteps, int snap_stride, double tol,
                  int maxit, int guess, double check_ff_maxv, int ntimeslices,
                  int *ffflag);
/* Per-member blow-up guard.  on = 0 (default): the reference's guard applied
 * to the ensemble as a whole -- the first member with |v_m| > check_ff_maxv
 * (or NaN) ends the run for all.  on = 1: the same test, at the same points
 * (start of each of the ntimeslices slices and of the remainder slice; v_n for
 * CNAB / IMEX Euler, v_c for SBDF2), is applied to every live member, and a
 * member that fails is RETIRED: its state (v_n, p_n) is frozen at that time
 * level (its trip level; what the reference's cnab / sbdftwo returns after
 * its break) and the others integrate on.  A retired member stays retired
 * across runs until dnsb_imex_set_state; the run ends at a check that leaves
 * no member live.  For a retired member:
 *   dnsb_imex_get_state        returns the frozen trip state;
 *   dnsb_imex_get_outputs      gives NaN at every level after the trip level;
 *   snapshots                  hold NaN in its lanes from the trip on (device
 *                              store and pinned mirror alike);
 *   dnsb_imex_gram(_dev)       sums over the members live when called only,
 *                              sum_{m live} X_m^T M X_m, so no NaN of a member
 *                              retired inside the snapshot window enters G.
 * Run verdict in this mode: DNSB_E_NOT_CONVERGED only if a member live at the
 * end of the run has a final relative residual above tol or a non-finite one;
 * the solves of members retired in the same run are forgiven, no others.
 * Allowed between runs; switching it off while members are retired is
 * refused (dnsb_imex_set_state first). */
int dnsb_imex_set_member_guard(dnsb_imex *e, int on);
/* trip_level (nb entries): -1 for a live member, else its trip level */
int dnsb_imex_member_status(dnsb_imex *e, int32_t *trip_level);
/* Field statistics of every member accumulated inside the loop, one
 * elementwise Welford update per time level that only reads the state.
 * on = 1 switches them on (or, when on already, restarts the window); on = 0
 * (default) frees them, and with them off the loop is unchanged.
 * Window: it starts at the current time level at dnsb_imex_set_statistics(1)
 * and dnsb_imex_reset_statistics, and at level 0 at dnsb_imex_set_state.  After
 * a run it holds every level from its first level through the run's final
 * level, inclusive (first, last); a run that continues the trajectory
 * continues the window without gap or double count.  When the stop-all guard
 * trips, the run's final level is the state the run returns.  The Heun levels 0
 * and 1 of CNAB / SBDF2 are ordinary levels.
 * Per member m with count[m] levels (divisors are the count, population
 * statistics):
 *   v_mean (nvf*nb)        mean of the full velocity V (Dirichlet values
 *                          included, full numbering 2*node + comp);
 *   uvcov (3, nnodes, nb)  per P2 node, the covariances uu, vv, uv of its two
 *                          components;
 *   p_mean, p_var (np*nb)  mean and variance of the pressure p = -q/dt;
 *   c_mean (nv*nb)         mean of the convection c(V)[inv] on the inner dofs
 *                          (the sign of dts.get_convvec).
 * p and c are in the device numbering.  A member retired by the per-member
 * guard counts the levels up to its trip level only (0 if it was retired
 * before the window); a member with count 0 has NaN fields.  Any output may be
 * NULL; reset and get are refused while the statistics are off. */
int dnsb_imex_set_statistics(dnsb_imex *e, int on);
int dnsb_imex_reset_statistics(dnsb_imex *e);
int dnsb_imex_get_statistics(dnsb_imex *e, long long *first, long long *last, long long *count,
                             double *v_mean, double *uvcov, double *p_mean, double *p_var,
                             double *c_mean);
/* device time of the last dnsb_imex_run, measured with CUDA events on the
 * context's stream (milliseconds) */
double dnsb_imex_last_run_ms(dnsb_imex *e);
int dnsb_imex_get_state(dnsb_imex *e, double *v, double *p);
int dnsb_imex_num_snapshots(dnsb_imex *e);
/* forget the stored snapshots (the next run records from the current state) */
int dnsb_imex_reset_snapshots(dnsb_imex *e);
/* snapshots as (nsnap, nv+np, nb), rows in output order */
int dnsb_imex_get_snapshots(dnsb_imex *e, double *out);
/* Output row order of the snapshots: output row of device row i is vmap[i]
 * (velocity, nv entries) / pmap[i] (pressure, np entries); NULL = identity.
 * The host-side mirror of the reference API numbers the unknowns along a
 * space-filling curve on the device (locality of the SpMM gathers) and uses
 * this map to hand trajectories back in the caller's numbering
 * (the `savevp(appndbcs(v_n, bcs_n), p_n, time)` hook of
 * time_int_utils.py:143). */
int dnsb_imex_set_output_order(dnsb_imex *e, const int32_t *vmap, const int32_t *pmap);
/* Snapshots are mirrored into pinned host memory by asynchronous D2H copies on
 * a second stream while the integration runs.  `reserve` allocates the mirror
 * ahead of time (nsnap snapshots); `snapshots_host` waits for the copies and
 * returns the mirror itself (valid until the next reserve/run/destroy): a
 * zero-copy view for the ctypes caller. */
int dnsb_imex_reserve_snapshots(dnsb_imex *e, int nsnap);
int dnsb_imex_snapshots_host(dnsb_imex *e, const double **ptr, int *nsnap);
/* Output functionals recorded inside the loop at every time level (the
 * initial state and the Heun level included), for all members, by one kernel
 * per step that only reads the state; the values stay on the device until
 * dnsb_imex_get_outputs.  A record holds (levels, ny + 2, nb) values: ny
 * linear outputs and the x / y force.  It starts empty at dnsb_imex_set_state,
 * dnsb_imex_reset_outputs and whenever the rows change, and a run appends to
 * it (a run on an empty record first records the current state).
 * Linear outputs  y_n = Cv v_n + Cp p_n  (the reference's `cv_mat.dot(v)`,
 * stokes_navier_utils.py:1144-1150): `cv` ny x nv on the inner velocity, `cp`
 * ny x np, columns in the device numbering; either may be NULL, both NULL = no
 * linear outputs. */
int dnsb_imex_set_outputs(dnsb_imex *e, dnsb_csr *cv, dnsb_csr *cp);
/* Force (CNAB only): the CNAB weak residual of residual_checks.get_imex_res
 * (crni/abtw, nu = nu[m]) tested with the indicator Phi of the x / y
 * components of the `ndofs` full-numbering velocity dofs `dofs`:
 *   F_n = Phi^T [ M (V_n - V_{n-1})/dt + nu_m A0 (V_n + V_{n-1})/2
 *                 + 3/2 c(V_{n-1}) - 1/2 c(V_{n-2}) - JT p_n ]
 * with the uncondensed nu = 1 operators reduced to rows: fm = Phi^T M[:, inv]
 * and fa = Phi^T A0[:, inv] (2 x nv), fj = Phi^T JT (2 x np), fa_bc[2] =
 * Phi^T A0[:, bc] u_bc (scaled by nu_m).  Defined for n >= 2 (NaN at levels 0
 * and 1 and at the first level after the rows were set mid-run).  ndofs = 0
 * switches the force off; scheme != 0 is refused. */
int dnsb_imex_set_force(dnsb_imex *e, int ndofs, const int32_t *dofs, dnsb_csr *fm,
                        dnsb_csr *fa, dnsb_csr *fj, const double *fa_bc);
int dnsb_imex_num_output_levels(dnsb_imex *e);
/* y: (levels, ny, nb), force: (levels, 2, nb); either may be NULL */
int dnsb_imex_get_outputs(dnsb_imex *e, double *y, double *force);
int dnsb_imex_reset_outputs(dnsb_imex *e);
/* solver statistics of the last run: total FGMRES iterations (max over
 * members per solve, summed over the loop solves), number of loop solves, and
 * the LARGEST final relative residual over all solves of the run (every
 * member, start-up solves included; NaN if a solve produced one).
 * dnsb_imex_run returns DNSB_E_NOT_CONVERGED when a solve of the run stopped
 * at maxit above tol (unless the blow-up guard fired, which is reported through
 * ffflag like time_int_utils.py:94-103); dnsb_imex_unconverged = how many.
 * With the per-member guard, max_relres is the largest over the members live
 * at the end of the run, and dnsb_imex_unconverged still counts every solve
 * that stopped at maxit with any member above tol. */
int dnsb_imex_stats(dnsb_imex *e, long long *total_iters, long long *nsolves,
                    double *max_relres);
long long dnsb_imex_unconverged(dnsb_imex *e);
/* local POD Gram matrix  G = sum_m X_m^T M X_m  (nsnap x nsnap, row-major;
 * with retired members the sum runs over the live ones only)
 * written to DEVICE memory g_dev (so that torch.distributed / NCCL can
 * all-reduce it in place) -- stokes_navier_utils.py:136-143 is the only
 * Gram-like op of the reference. */
int dnsb_imex_gram_dev(dnsb_imex *e, double *g_dev);
/* the same into HOST memory g (nsnap*nsnap doubles) */
int dnsb_imex_gram(dnsb_imex *e, double *g);

/* ---- device-resident Picard/Newton + Crank-Nicolson sweep -------------------
 * One sweep of stokes_navier_utils.py:1402-1566 over the whole time grid:
 *   (M + dt/2 (A + N_n)) v+ + JT q = M v + dt/2 (f_n + f_c - (A + N_c) v),
 *   J v+ = fp,  p = -q/dt,
 * N_n = condensed Picard (N1) or Newton (N1+N2) matrix about the PREVIOUS
 * sweep's state at t_n (`linpoint`), N_c about the sweep's own state
 * (:1529-1538); f = fv - (N u_bc)[inv] (+ N(v)v[inv] for Newton, :1365,1459).
 * `solver`: single-system solver whose velocity block lives on the union
 * pattern of M, A and the condensed convection pattern; `mvals`/`avals`: M and
 * A on that pattern; (src, pos): slot k of the condensed convection matrix is
 * entry src[k] of the full pattern (dnsb_set_conv_pattern) and entry pos[k] of
 * the solver's pattern.  The reference re-assembles with dolfin and
 * re-factorises with SuperLU every step and passes the trajectory through
 * .npy files (:1424-1431, :1505-1512, :1540-1541); here the step never leaves
 * the device. */
int dnsb_cnsweep_create(dnsb_solver *solver, dnsb_csr *mmat, const double *mvals,
                        const double *avals, int nconv, const int32_t *src,
                        const int32_t *pos, const int32_t *invinds, int nbc,
                        const int32_t *bcinds, const double *bcvals, const double *fv,
                        const double *fp, dnsb_cnsweep **out);
void dnsb_cnsweep_destroy(dnsb_cnsweep *w);
/* dts: nsteps step sizes; linpoint: (nsteps+1) full velocities (V.dim() each);
 * v0 (nv), p0 (np): initial state; vtraj ((nsteps+1)*V.dim()), ptraj
 * ((nsteps+1)*np): the sweep's trajectory; upd_norm = sum_n dt_n |v_n -
 * lin_n|_M^2 (:1557-1560); iters_total: FGMRES iterations of the sweep. */
int dnsb_cnsweep_run(dnsb_cnsweep *w, int nsteps, const double *dts, int picard,
                     const double *linpoint, const double *v0, const double *p0,
                     double tol, int maxit, double *vtraj, double *ptraj,
                     double *upd_norm, long long *iters_total);
/* initial guess of the step solves: 0 = the previous step's solution
 * (`krylovini='old'`, stokes_navier_utils.py:1493-1495), 1 = linear
 * extrapolation of the last two (`'upd'`, :1496-1501; the default) */
int dnsb_cnsweep_set_guess(dnsb_cnsweep *w, int mode);
/* largest final relative residual over the step solves of the last sweep and
 * the number of them that stopped at maxit above tol (then dnsb_cnsweep_run
 * returned DNSB_E_NOT_CONVERGED; the trajectories were still written) */
int dnsb_cnsweep_stats(dnsb_cnsweep *w, double *max_relres, long long *unconverged);

#ifdef __cplusplus
}
#endif
#endif /* DNSB_H */
