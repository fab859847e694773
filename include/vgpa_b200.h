/*
 * vgpa_b200.h -- C ABI of libvgpa_b200.so: the B200 (sm_100a) implementation of
 * VGPA's variational free-energy + gradient evaluation for a BATCH of
 * independent inference problems.
 *
 * The reference (vrettasm/VGPA) is pure Python and has no FFI; its boundary is
 * the pair of callables handed to the SCG optimiser.  Each entry point below
 * names the reference interface it stands in for (paths relative to the
 * reference root).  Plain pointers and sizes only; all arrays are C-contiguous
 * float64 in the reference's own layouts:
 *
 *     x    = [ A (N,D,D) | b (N,D) ]          (variational.py:153-162)
 *     grad = [ dL/dA (N,D,D) | dL/db (N,D) ]  (variational.py:284-288)
 *
 * D = 1 (DW, OU) uses the same layout with 1x1 matrices.
 *
 * Scope: diagonal system noise Sigma, diagonal observation noise R, and an
 * observation operator H that selects components: the identity, or per problem
 * any non-empty subset of the state components (vgpa_create_observed; the
 * sim_params JSON's Observations.operator, simulation.py:107-176).  That is
 * everything the sim_params JSON schema can express (vgpa_main.py:38-40).  A
 * general H and a non-diagonal R are out of scope.  L96 takes any 10 <= D <= 64
 * (lorenz_96.py:104-140 accepts dim_d >= 10): D = 40, the only size simulation.py:20,134
 * constructs, runs hand-tuned kernels, every other D a run-time-D kernel family.
 *
 * Return codes (mapped to the exceptions the reference raises):
 *     VGPA_OK            0
 *     VGPA_EINVAL        1   -> ValueError
 *     VGPA_ENOTPD        2   -> numpy.linalg.LinAlgError   (utilities.py:211,275:
 *                               a covariance S(t) is not positive definite)
 *     VGPA_ECUDA         3   -> RuntimeError
 *
 * Threading: one handle is driven by one host thread at a time (the
 * reference's VarGP.output cache is equally non re-entrant); different
 * handles / devices may run concurrently.  There is NO CPU fallback.
 */
#ifndef VGPA_B200_H
#define VGPA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { VGPA_OK = 0, VGPA_EINVAL = 1, VGPA_ENOTPD = 2, VGPA_ECUDA = 3 };

/* simulation.py:20  dynamical_systems = {"DW","OU","L63","L96"} */
enum { VGPA_MODEL_DW = 0, VGPA_MODEL_OU = 1, VGPA_MODEL_L63 = 2, VGPA_MODEL_L96 = 3 };
/* utilities.py:12   num_integration = {"euler","heun","rk2","rk4"} */
enum { VGPA_ODE_EULER = 0, VGPA_ODE_HEUN = 1, VGPA_ODE_RK2 = 2, VGPA_ODE_RK4 = 3 };

typedef struct vgpa_handle vgpa_handle;

/*
 * Problem-batch descriptor.  Replaces the constructor arguments of
 * VarGP(model, m0, s0, fwd_ode, bwd_ode, likelihood, kl0, obs_y, obs_t)
 * (variational.py:15-71) together with the fields it reads from them:
 * model.sigma / theta / time_step, likelihood.values / times / noise,
 * fwd_ode.method / dt.  Host pointers; copied to the device by vgpa_create.
 *
 * Every per-problem array carries a stride in ELEMENTS between consecutive
 * problems; stride 0 means "shared by all B problems".
 */
typedef struct {
    int32_t model;   /* VGPA_MODEL_*                                              */
    int32_t method;  /* VGPA_ODE_*                                                */
    int32_t D;       /* state dimension (DW, OU: 1; L63: 3; L96: 10 <= D <= 64)   */
    int32_t N;       /* number of time-grid points = len(np.arange(t0,tf+dt,dt))  */
    int32_t M;       /* number of observations                                    */
    int32_t B;       /* number of independent problems in the batch               */
    int32_t device;  /* CUDA device ordinal                                        */
    int32_t reserved;
    double dt;       /* step of the ODE sweeps (fwd_ode.py:14, JSON Time-window.dt) */
    double dt_model; /* model.time_step (stochastic_process.py:117): trapezoid
                        spacing (utilities.py:144) and gradient scale
                        (variational.py:284-285)                                  */
    const double *theta;  int64_t theta_stride;  /* DW/OU/L96: 1 value; L63: 3    */
    const double *sigma;  int64_t sigma_stride;  /* D: diag of the system noise   */
    const double *R;      int64_t R_stride;      /* D: diag of the obs. noise     */
    const int64_t *obs_t;                        /* M sorted unique indices,
                                                    shared by the batch
                                                    (stochastic_process.py:166-175);
                                                    vgpa_create_obs_rows: NULL   */
    const double *obs_y;  int64_t obs_y_stride;  /* M x D observation values      */
    const double *m0;     int64_t m0_stride;     /* D                             */
    const double *s0;     int64_t s0_stride;     /* D x D                         */
    const double *E0;     int64_t E0_stride;     /* 1: prior KL at t=0, constant
                                                    per problem (prior_kl0.py:30-92,
                                                    variational.py:183-185)       */
    int64_t scratch_bytes; /* device scratch budget for trajectories; 0 = default */
} vgpa_desc;

/* VarGP.__init__ (variational.py:15-71): validate, upload, allocate scratch. */
int vgpa_create(const vgpa_desc *desc, vgpa_handle **out);
/* Per-problem observation schedules.  Problem p has M[p] observations, at the time indices
 * obs_t + p * obs_t_stride (sorted, unique, in [0, N)).  Its values are the M[p] x D entries at
 * desc->obs_y + p * desc->obs_y_stride.  desc->M is the row capacity: M[p] <= desc->M, and each
 * obs_y row holds desc->M x D entries (obs_y_stride >= desc->M * D, or 0 = one row shared by all).
 * desc->obs_t must be NULL.  obs_t_stride == 0: one row shared by every problem (the first M[p]
 * entries are problem p's), else obs_t_stride >= desc->M.  M == NULL: every problem has desc->M
 * observations.  With both, this is vgpa_create.  Every entry point of the handle uses each
 * problem's own schedule; vgpa_initialization fails (VGPA_EINVAL, naming the problem) when a
 * problem has no observation or one at the first or last grid index.  The handle keeps a (B, N)
 * int32 table of observation ordinals on the device (B * N * 4 bytes). */
int vgpa_create_obs_rows(const vgpa_desc *desc, const int64_t *obs_t, int64_t obs_t_stride,
                         const int32_t *M, vgpa_handle **out);
/* Partially observed problems.  Bit i of observed[p * observed_stride] set: component i of problem p
 * is observed (D <= 64, so one word holds a mask).  observed_stride == 0: one mask shared by the batch.
 * observed == NULL: exactly vgpa_create_obs_rows; the first four arguments follow its rules.
 * Problem p observes the set O_p: H is the rows of the identity at O_p and R is diagonal over O_p, so
 *   Eobs = 1/2 [ sum_n sum_{i in O} ((y_ni - m_i(t_n))^2 / R_i + S_ii[n] / R_i) + M (D_o log 2pi + sum_{i in O} log R_i) ]
 * (S indexed by the observation ordinal n, as for H = I), the jumps at t_n are -(y_ni - m_i) / R_i and
 * 1/2 / R_i for i in O and 0 otherwise, and vgpa_initialization gives an unobserved component the
 * constant mean path m0[p][i] (b0(t)_i = a_ii m0_i) in place of the spline.  obs_y keeps its M x D rows and
 * R its D values: the entries of unobserved components are never read (NaN allowed).  Every entry point
 * of the handle follows the masks.  With every bit below D set, a handle computes what
 * vgpa_create_obs_rows's does, bit for bit.  VGPA_EINVAL, naming the problem, before any CUDA call: a
 * mask with no bit set, a bit at or above D, a negative observed_stride. */
int vgpa_create_observed(const vgpa_desc *desc, const int64_t *obs_t, int64_t obs_t_stride, const int32_t *M,
                         const uint64_t *observed, int64_t observed_stride, vgpa_handle **out);
void vgpa_destroy(vgpa_handle *h);
/* Text of the last error on this handle (or of the last failed vgpa_create
 * when h is NULL).  Valid until the next call on the handle. */
const char *vgpa_last_error(const vgpa_handle *h);

/*
 * VarGP.free_energy(x) followed by VarGP.gradient(x) on the same x
 * (variational.py:141-200 and :202-289), for all B problems.
 *
 * HOST buffers: x (B rows, x_stride elements apart; 0 = one x shared by all
 * problems), F (B values), grad (B rows, grad_stride apart; may be NULL when
 * want_grad == 0).  Host<->device copies are inside the call; pass memory from
 * vgpa_host_alloc for full PCIe speed.
 */
int vgpa_eval(vgpa_handle *h, const double *x, int64_t x_stride, int want_grad,
              double *F, double *grad, int64_t grad_stride);

/* Optional active set for the following vgpa_eval_device calls: d_active = B int32 flags in DEVICE
 * memory (read when the kernels run), NULL = every problem.  Problems whose flag is 0 are skipped by
 * every kernel: their F, gradient rows and status are left untouched and they cost no sweep time.
 * This is what lets a batched optimiser (SCG runs per problem, optim_scg.py:75-285) stop paying for
 * problems that have converged. */
int vgpa_set_active(vgpa_handle *h, const int32_t *d_active);

/* Compacted launches for thinned-out ensembles (Lorenz-96 handles only): `list` = n problem indices in
 * HOST memory (copied), or NULL / n < 0 to switch the mode off.  The following vgpa_eval_device calls
 * evaluate exactly the listed problems, chunked by list position, so that every pass still fills whole
 * waves of the GPU when most problems of a batch have converged (an active-flag mask alone leaves the
 * chunk of a few survivors under-occupied).  F and gradient rows are still addressed by problem index;
 * the rows of unlisted problems are left untouched.  Host-buffer entry points ignore the list. */
int vgpa_set_active_list(vgpa_handle *h, const int32_t *list, int32_t n);

/*
 * Same evaluation with DEVICE buffers on `stream` (a cudaStream_t passed as
 * void*; NULL = default stream).  Asynchronous: returns after enqueueing.
 * Call vgpa_sync to wait and to collect the positive-definiteness status.
 * A handle owns one scratch: an evaluation enqueued on another stream than the
 * previous one is ordered after it (an event wait on the device, no host
 * synchronisation); for evaluations that should overlap use one handle each.
 */
int vgpa_eval_device(vgpa_handle *h, const double *d_x, int64_t x_stride, int want_grad,
                     double *d_F, double *d_grad, int64_t grad_stride, void *stream);
int vgpa_sync(vgpa_handle *h);

/* model.energy's hyper-parameter gradients for EVERY problem of the handle, each at its own x row
 * (d_x + p * x_stride; 0 = one x shared by all).  DEVICE buffers, asynchronous on `stream`; vgpa_sync
 * waits and reports a non-positive-definite S(t) exactly as after vgpa_eval_device.  Any output may be NULL.
 *   F[p]                           free energy (bitwise what vgpa_eval_device returns for the same x)
 *   Esde[p]                        Esde as energy() returns it (= parts[1] of vgpa_eval_full)
 *   dtheta + p * dtheta_stride     dEsde_dtheta: 1 (DW, OU), 3 (L63), D (L96) values
 *   dsigma + p * dsigma_stride     dEsde_dsigma: 1 value (D = 1) or D x D (diagonal; off-diagonals written as 0)
 * x is 16-byte aligned with an even stride; an output stride is at least the length of its row (0 only when
 * B = 1).  dEsde_dtheta and dEsde_dsigma are the partial derivatives at the problem's m(t), S(t): for DW, OU
 * and L63, dEsde_dtheta is dF/dtheta at fixed x.  Ordering against other calls on the handle is that of
 * vgpa_eval_device.  The active set and the compacted list are suspended for the call (every problem is
 * served) and stay installed for later vgpa_eval_device calls. */
int vgpa_hyper_device(vgpa_handle *h, const double *d_x, int64_t x_stride, double *d_F, double *d_Esde,
                      double *d_dtheta, int64_t dtheta_stride, double *d_dsigma, int64_t dsigma_stride,
                      void *stream);

/*
 * One problem, everything: F, its three parts, the gradient and every
 * intermediate the reference caches in VarGP.output (variational.py:189-196,
 * arg_out :292) or passes between its stages (:169-181).  HOST pointers; any
 * output may be NULL.  x is that problem's own row (N*D*(D+1) values).
 *   parts[3] = {E0, Esde, Eobs};  mt (N,D) st (N,D,D) lamt (N,D) psit (N,D,D)
 *   Efx (N,D) Edf (N,D,D) dEsde_dm (N,D) dEsde_ds (N,D,D)
 */
typedef struct {
    double *F, *parts, *grad;
    double *mt, *st, *lamt, *psit, *Efx, *Edf, *dEsde_dm, *dEsde_ds;
} vgpa_full_out;
int vgpa_eval_full(vgpa_handle *h, int64_t problem, const double *x, const vgpa_full_out *out);

/* The two sweeps on their own, as FwdOde.__call__ (fwd_ode.py:45) and
 * BwdOde.__call__ (bwd_ode.py:45) expose them: one problem, HOST buffers.
 *   fwd: A (N,D,D), b (N,D), m0 (D), s0 (D,D), sigma (D diag) -> mt, st
 *   bwd: A, dEsde_dm (N,D), dEsde_ds (N,D,D), dEobs_dm (N,D), dEobs_ds (N,D,D)
 *        -> lam (N,D), psi (N,D,D)
 * (dense jump tables exactly as GaussianLikelihood.gradients returns them,
 * gaussian_like.py:155-243; the jump added at each step is the one at t-1.) */
int vgpa_solve_fwd(int device, int method, int D, int N, double dt, const double *A,
                   const double *b, const double *m0, const double *s0, const double *sigma,
                   double *mt, double *st);
int vgpa_solve_bwd(int device, int method, int D, int N, double dt, const double *A,
                   const double *dEsde_dm, const double *dEsde_ds, const double *dEobs_dm,
                   const double *dEobs_ds, double *lam, double *psi);

/* model.energy(A, b, m, S, obs_t) of a StochasticProcess subclass
 * (double_well.py:169, ornstein_uhlenbeck.py:165, lorenz_63.py:237,
 * lorenz_96.py:316): the time-parallel stage on its own, one problem, HOST
 * buffers.  Outputs: Esde (1 value), Ef (N,D), Edf (N,D,D), dEsde_dm (N,D),
 * dEsde_ds (N,D,D).  The hyper-parameter gradients dEsde_dtheta / dEsde_dsigma
 * that the reference also returns are discarded by VarGP (variational.py:175)
 * and are not computed. */
int vgpa_model_energy(int device, int model, int D, int N, double dt_model, const double *theta,
                      const double *sigma, const double *A, const double *b, const double *m,
                      const double *S, double *Esde, double *Ef, double *Edf, double *dEsde_dm,
                      double *dEsde_ds, double *dEsde_dtheta, double *dEsde_dsigma);
/* dEsde_dtheta / dEsde_dsigma: the hyper-parameter gradients that energy() returns last
 * (double_well.py:251-257, ornstein_uhlenbeck.py:223-229, lorenz_63.py:327-343 + :572-633,
 * lorenz_96.py:420-434) and VarGP discards.  Both may be NULL (not computed).  Sizes:
 * dEsde_dtheta 1 (DW, OU), 3 (L63), D (L96); dEsde_dsigma 1 (D = 1) or D x D.  The kernels are those of
 * vgpa_hyper_device with one problem. */

/* GaussianLikelihood.__call__ and .gradients (gaussian_like.py:39-243) on their
 * own: one problem, HOST buffers, identity operator, diagonal R (D values).
 * Outputs: Eobs (1 value) and the dense jump tables dEobs_dm (N,D),
 * dEobs_ds (N,D,D), zero except at obs_t. */
int vgpa_obs_energy(int device, int D, int N, int M, const int64_t *obs_t, const double *obs_y,
                    const double *R, const double *mt, const double *st, double *Eobs,
                    double *dEobs_dm, double *dEobs_ds, double *dEobs_dr);
/* dEobs_dr (may be NULL): third output of GaussianLikelihood.gradients -- N values for D = 1
 * (gaussian_like.py:194), N x M x M zeros for D > 1 (the reference never fills it, :226). */
/* The same likelihood for a component-selecting operator: `observed` holds the observed components (bit i =
 * component i; vgpa_create_observed gives the formulas).  obs_y is M x D and R has D values; the entries of
 * unobserved components are not read.  jm (N,D) and js (N,D,D) are the jump tables dEobs_dm, dEobs_ds,
 * zero except at obs_t and at observed components.  With every
 * bit below D set, the outputs are those of vgpa_obs_energy, bit for bit.  VGPA_EINVAL for a mask with no
 * bit set or a bit at or above D. */
int vgpa_obs_energy_observed(int device, int D, int N, int M, const int64_t *obs_t, const double *obs_y,
                             const double *R, uint64_t observed, const double *mt, const double *st,
                             double *Eobs, double *jm, double *js);

/* VarGP.initialization (variational.py:73-139) for every problem of the handle: the starting
 * point x0 = [A0 | b0] from cubic splines (scipy CubicSpline, not-a-knot) through each problem's
 * observations, written to DEVICE rows d_x + p * x_stride on `stream` (asynchronous), or to HOST
 * rows (vgpa_initialization_host, synchronous).  t0 = first point of the time window; the grid
 * is t0 + k * dt_model.  VGPA_EINVAL when an observation sits at the first or last grid index
 * (the reference's CubicSpline raises: knots must be strictly increasing) or M < 1. */
int vgpa_initialization(vgpa_handle *h, double t0, double *d_x, int64_t x_stride, void *stream);
int vgpa_initialization_host(vgpa_handle *h, double t0, double *x, int64_t x_stride);

/* Batched sample paths for ensembles: the Euler-Maruyama loops of DoubleWell / OrnsteinUhlenbeck /
 * Lorenz63 / Lorenz96 .make_trajectory (double_well.py:122-166, ornstein_uhlenbeck.py:128-161,
 * lorenz_63.py:181-233, lorenz_96.py:249-314) for B paths at once.  The standard-normal draws are an
 * INPUT in the layout the reference draws them -- z: (D, N) per path, row 0 of the time axis unused --
 * so a host generator seeded like the reference gives the reference's path bit for bit (every
 * operation is one correctly rounded IEEE operation in the reference's order, no FMA contraction).
 *   theta : DW [theta], OU [theta, mu], L63 [sigma, rho, beta], L96 [F]      (per path, stride 0 = shared)
 *   sigma : (D) diagonal of the system noise;  x_init: (D) state at t0 -- required for DW / OU
 *           (their start consumes the generator, double_well.py:145-151), NULL for L63 / L96 = the
 *           reference's 5000-step burn-in from its fixed starting point
 *   path  : (N, D) per path, row stride path_stride
 * vgpa_make_trajectory: HOST buffers, synchronous.  _device: DEVICE buffers, asynchronous on `stream`.
 * Both take D from the model (L96: 40); the _dim variants take it as an argument (L96: 10 <= D <= 64,
 * the burn-in perturbs component int(D / 2); the other models: their fixed D). */
int vgpa_make_trajectory(int device, int model, int N, int B, double dt, const double *theta,
                         int64_t theta_stride, const double *sigma, int64_t sigma_stride,
                         const double *x_init, int64_t x_init_stride, const double *z, int64_t z_stride,
                         double *path, int64_t path_stride);
int vgpa_make_trajectory_device(int device, int model, int N, int B, double dt, const double *d_theta,
                                int64_t theta_stride, const double *d_sigma, int64_t sigma_stride,
                                const double *d_x_init, int64_t x_init_stride, const double *d_z,
                                int64_t z_stride, double *d_path, int64_t path_stride, void *stream);
int vgpa_make_trajectory_dim(int device, int model, int D, int N, int B, double dt, const double *theta,
                             int64_t theta_stride, const double *sigma, int64_t sigma_stride,
                             const double *x_init, int64_t x_init_stride, const double *z, int64_t z_stride,
                             double *path, int64_t path_stride);
int vgpa_make_trajectory_device_dim(int device, int model, int D, int N, int B, double dt, const double *d_theta,
                                    int64_t theta_stride, const double *d_sigma, int64_t sigma_stride,
                                    const double *d_x_init, int64_t x_init_stride, const double *d_z,
                                    int64_t z_stride, double *d_path, int64_t path_stride, void *stream);

/* StochasticProcess.collect_obs (stochastic_process.py:130-230) for B observation sets:
 * obs_y[p][j][i] = path[p][obs_t[j]][i] + sqrt(R[p][i]) * xi[p][i][j]   (xi: (D, M) draws, the
 * reference's layout; R: (D) diagonal; obs_y: (M, D)).  The observation indices themselves
 * (np.linspace, :172-175) are host-side integers and stay with the caller. */
int vgpa_collect_obs(int device, int D, int N, int M, int B, const int64_t *obs_t, const double *R,
                     int64_t R_stride, const double *path, int64_t path_stride, const double *xi,
                     int64_t xi_stride, double *obs_y, int64_t obs_y_stride);
int vgpa_collect_obs_device(int device, int D, int N, int M, int B, const int64_t *d_obs_t,
                            const double *d_R, int64_t R_stride, const double *d_path,
                            int64_t path_stride, const double *d_xi, int64_t xi_stride,
                            double *d_obs_y, int64_t obs_y_stride, void *stream);

/* Pinned host memory for x / grad staging (cudaHostAlloc / cudaFreeHost). */
void *vgpa_host_alloc(int64_t bytes);
void vgpa_host_free(void *p);
/* memcpy on up to `threads` host threads (filling a pinned staging buffer from pageable memory). */
void vgpa_host_copy(void *dst, const void *src, int64_t bytes, int threads);
/* 1 when the two host ranges hold the same bytes (memcmp on up to `threads` host threads), else 0:
 * the "is this the x of the last evaluation" test of VarGP.free_energy / gradient, whose reference
 * counterpart recomputes unconditionally (variational.py:141-226). */
int vgpa_host_equal(const void *a, const void *b, int64_t bytes, int threads);

/* Introspection for bench.py: kernels launched by the handle so far, the
 * chunk size (problems resident per pass) and the scratch bytes in use. */
int64_t vgpa_launch_count(const vgpa_handle *h);
int64_t vgpa_chunk_size(const vgpa_handle *h);
int64_t vgpa_scratch_in_use(const vgpa_handle *h);
/* Batched vector kernels for the device-resident SCG driver (vgpa_b200/batched_scg.py):
 * the optimiser's own arithmetic (optim_scg.py:137-274) over rows of (B, n) DEVICE arrays
 * with a common row stride; rows are cut into slices so that small batches fill the GPU, and
 * reductions add the slice partials in a fixed order.  `active` (B int32 flags in device memory,
 * or NULL): rows whose flag is 0 are skipped and their outputs left untouched.
 *   vgpa_bdot  : out[p] = x.y, out[B+p] = x.z (z may be NULL), out[2B+p] = x.x
 *   vgpa_baxpy : out = y + a[p] x
 *   vgpa_bdir  : mode[p] 0 keep | 1: d = gamma[p] d - g | 2: d = -g
 *   vgpa_bcopy : dst[p] = src[p] where mask[p] != 0
 *   vgpa_bstats: out[p] = max|x|, out[B+p] = sum|x|                                   */
int vgpa_bdot(int B, int64_t n, const double *x, const double *y, const double *z, int64_t stride,
              double *out3B, const int32_t *active, void *stream);
int vgpa_baxpy(int B, int64_t n, const double *a, const double *x, const double *y, double *out,
               int64_t stride, const int32_t *active, void *stream);
int vgpa_bdir(int B, int64_t n, const int32_t *mode, const double *gamma, double *d, const double *g,
              int64_t stride, void *stream);
int vgpa_bcopy(int B, int64_t n, const int32_t *mask, const double *src, double *dst, int64_t stride,
               void *stream);
int vgpa_bstats(int B, int64_t n, const double *x, int64_t stride, double *out2B, const int32_t *active,
                void *stream);

/* Hand-over of the trajectory scratch between handles.  enable != 0: from now on the large device blocks of a
 * destroyed handle are kept and given to the next vgpa_create that needs exactly the same sizes on the same
 * device (an ensemble processed in sub-batches of one shape: no cudaFree / cudaMalloc of tens of GB per
 * sub-batch; cudaFree was measured at up to 2 s when several processes free at once).  enable == 0: switch it
 * off and free what is kept; returns the bytes released.  Kept blocks are also released when an allocation of
 * this library would otherwise fail.  Off by default.  Thread-safe. */
long long vgpa_scratch_cache(int enable);

/* Per-kernel device timing for bench.py's roofline: when enabled, every kernel
 * launch of vgpa_eval / vgpa_eval_device is bracketed by CUDA events on the
 * launching stream.  vgpa_get_timing synchronises, then returns the accumulated
 * milliseconds and launch counts per kernel kind and clears the accumulators:
 *   kind 0 forward sweep, 1 time-parallel energy, 2 finalize (F), 3 backward+gradient.
 * (D = 1 evaluations with a gradient are ONE launch doing all four: accounted to kind 0.) */
int vgpa_set_timing(vgpa_handle *h, int enable);
int vgpa_get_timing(vgpa_handle *h, double ms[4], int64_t launches[4]);
const char *vgpa_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VGPA_B200_H */
