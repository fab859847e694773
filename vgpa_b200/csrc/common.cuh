// common.cuh -- shared declarations of the sm_100a VGPA kernels.
#pragma once
#include <cstddef>
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

namespace vgpa {

enum Model { MODEL_DW = 0, MODEL_OU = 1, MODEL_L63 = 2, MODEL_L96 = 3 };
enum Method { ODE_EULER = 0, ODE_HEUN = 1, ODE_RK2 = 2, ODE_RK4 = 3 };

// Solver dispatch of the launchers: f(std::integral_constant<int, METHOD>{}) for the run-time method, so that
// f instantiates its kernel for that method.  Values out of range take RK4.
template <typename F>
void with_method(int method, F&& f)
{
    switch (method) {
    case ODE_EULER: f(std::integral_constant<int, ODE_EULER>{}); break;
    case ODE_HEUN:  f(std::integral_constant<int, ODE_HEUN>{}); break;
    case ODE_RK2:   f(std::integral_constant<int, ODE_RK2>{}); break;
    default:        f(std::integral_constant<int, ODE_RK4>{}); break;
    }
}

template <typename K>
void set_smem(K kernel, size_t bytes)
{
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// Device-resident description of a problem batch (all pointers are device
// pointers; *_stride in elements, 0 = shared by every problem).
struct Batch {
    int model, method, D, N, M, B;
    double dt, dt_model;
    const double* theta;  long long theta_stride;
    const double* sigma;  long long sigma_stride;
    const double* R;      long long R_stride;
    const long long* obs_t;   // M
    const int* obs_index;     // N : ordinal of the observation at grid index t, or -1
    const double* obs_y;  long long obs_y_stride;
    const double* m0;     long long m0_stride;
    const double* s0;     long long s0_stride;
    const double* E0;     long long E0_stride;
    const int* active;        // B flags or null: problems whose flag is 0 are skipped by every kernel
                              // (their F, gradient and scratch rows are left untouched)
    const int* plist;         // or null.  Compacted launches of the Lorenz-96 kernels (vgpa_set_active_list): the
                              // pass covers list positions [p0, p0 + count) and the problem at position k is
                              // plist[k], so that a thinned-out ensemble still fills whole waves
    // Per-problem observation schedules (vgpa_create_obs_rows).  Problem p observes at obs_t + p * obs_t_stride, its
    // grid table is obs_index + p * obs_index_stride (a (B, N) table), and it has obs_count[p] observations.  A handle
    // of vgpa_create has both strides 0 and a null count: one schedule of M observations for the batch.
    long long obs_t_stride;
    long long obs_index_stride;
    const int* obs_count;     // B counts <= M, or null = M each
    // Partially observed problems (vgpa_create_observed): B words, bit i of word p set = component i of problem p is
    // observed; null = every component of every problem.  Only the observation energy (free_energy_of) and the
    // initialisation read it.  The sweeps' jumps need no mask: the handle's device copy of R holds +inf and its copy
    // of obs_y holds 0 at every unobserved (problem, component), so the jump -(y - m) / R is a zero and 0.5 / R is 0.
    // (The pointer keeps the fields added with the schedules at 32 bytes: the kernel parameters that follow a Batch
    // keep their 16-byte alignment, and the D = 40 kernels their code and speed.)
    const unsigned long long* observed;
};

// The observed components of problem p (bit i = component i).
__device__ __forceinline__ unsigned long long observed_of(const Batch& b, int p)
{
    return b.observed != nullptr ? b.observed[p] : ~0ull;
}

// problem served by launch position `pos` (= p0 + local index)
__device__ __forceinline__ int problem_at(const Batch& b, int pos) { return b.plist != nullptr ? b.plist[pos] : pos; }

// The observation schedule of problem p: sorted time indices, the ordinal of the observation at each grid index (or
// -1), and the number of observations.
__device__ __forceinline__ const long long* obs_t_of(const Batch& b, int p) { return b.obs_t + p * b.obs_t_stride; }
__device__ __forceinline__ const int* obs_index_of(const Batch& b, int p) { return b.obs_index + p * b.obs_index_stride; }
__device__ __forceinline__ int obs_count_of(const Batch& b, int p) { return b.obs_count != nullptr ? b.obs_count[p] : b.M; }
// Launchers of the kernels that sit at the edge of the instruction cache (the D = 40 backward sweep) instantiate them
// twice: ROWS = false reads the one shared schedule exactly as before per-problem schedules existed.
inline bool obs_rows(const Batch& b) { return b.obs_index_stride != 0; }

// Sum over the CTA in a fixed order (every thread gets it); sh: blockDim.x doubles, blockDim.x a power of two.
__device__ __forceinline__ double block_sum(double v, double* sh)
{
    const int tid = threadIdx.x;
    sh[tid] = v;
    __syncthreads();
    for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
        if (tid < o) sh[tid] += sh[tid + o];
        __syncthreads();
    }
    const double r = sh[0];
    __syncthreads();
    return r;
}

// Esde of problem p from its integrand f(t) (utilities.py:144-201: composite trapezoid, sum(dx * (f[i+1] + f[i]) / 2)).
// Every thread of the CTA calls it.  The partial sums are taken by the first ESDE_THREADS threads whatever the CTA
// size (the rest add zeros to the reduction tree), so that Esde and F are the same bits from finalize_kernel, from
// the fused D = 1 evaluation (SCAN_THREADS) and from the hyper-parameter reduction.
constexpr int ESDE_THREADS = 128;
__device__ __forceinline__ double esde_of(const Batch& b, int p, const double* f, double* sh)
{
    const int tid = threadIdx.x, N = b.N;
    double acc = 0.0;
    if (tid < ESDE_THREADS)
        for (int i = tid; i < N - 1; i += ESDE_THREADS) acc += b.dt_model * (f[i + 1] + f[i]) / 2.0;
    double Esde = block_sum(acc, sh);
    if (b.model == MODEL_DW || b.model == MODEL_OU)  // double_well.py:217, ornstein_uhlenbeck.py:208
        Esde = 0.5 * Esde / b.sigma[p * b.sigma_stride];
    return Esde;
}

// Per-pass (chunk) scratch: trajectories of the marginal moments, the SDE-energy
// gradients and the per-time-step energy.  Problem-major: [p][t][...].
struct Scratch {
    double* mt;      // (C, N, D)
    double* st;      // (C, N, D, D)
    double* dEm;     // (C, N, D)
    double* dEs;     // (C, N, D, D)
    double* esde_t;  // (C, N)
    int* status;     // (C) : 0 ok, else 1 + time index of the first non-PD S(t)
};

// Optional per-problem trajectory outputs (vgpa_eval_full); null = not stored.
struct Extra {
    double* lamt;  // (N, D)
    double* psit;  // (N, D, D)
    double* Efx;   // (N, D)
    double* Edf;   // (N, D, D)
    double* parts; // (3) E0, Esde, Eobs
};

// Batched sample paths / observations (datagen.cu); device pointers, strides in elements (0 = shared).
struct TrajArgs {
    int model, D, N, B;
    double dt;
    const double* theta;  long long theta_stride;    // DW [theta], OU [theta, mu], L63 [sigma, rho, beta], L96 [F]
    const double* sigma;  long long sigma_stride;    // (D) diagonal of the system noise
    const double* x_init; long long x_init_stride;   // (D) state at t0; null (L63, L96) = the reference's burn-in
    const double* z;      long long z_stride;        // (D, N) standard-normal draws, the reference's layout
    double* path;         long long path_stride;     // (N, D)
};
struct ObsArgs {
    int D, N, M, B;
    const long long* obs_t;                          // (M)
    const double* R;      long long R_stride;        // (D) diagonal of the observation noise
    const double* path;   long long path_stride;     // (N, D)
    const double* xi;     long long xi_stride;       // (D, M) standard-normal draws
    double* obs_y;        long long obs_y_stride;    // (M, D)
};

// ---- shared-memory layout of a 40 x 40 matrix in the D = 40 kernels -----------------------
// Rows are contiguous (one bulk / cp.async copy per row); row PAIRS are 84 doubles apart:
//   address(row, col) = 84 * (row >> 1) + 40 * (row & 1) + col      (1680 doubles per matrix)
// i.e. pitch 40 plus a cumulative shift of 4 doubles per row pair.  Modulo the 16 8-byte banks a
// half-warp sees, row r starts at 8 (r & 1) + 4 ((r >> 1) & 3), which makes ALL access shapes of
// the kernels bank-conflict free (64-bit accesses go out per half-warp, 128-bit per quarter-warp):
//   DMMA A fragments  (lane (g,q): row R+g,    col C+q)       rows g = 0..3 start at 0, 8, 4, 12
//   DMMA B fragments  (lane (g,q): row R+q,    col C+g)       same with q and g swapped
//   accumulator pairs (lane (g,q): row R+g,    cols C+2q, +1 as one 16-byte access)
//   transposed reads  (lane (g,q): row R+2q+e, col C+g)       rows 2q+e start at 8e + 4q
// (pitch 44 / 42, used before, made the 16-byte accumulator accesses 2-way conflicted: 22 % of the
// forward sweep's shared-memory wavefronts, profiles/README.md.)
constexpr int SM_MAT = 84 * 20;          // doubles per matrix
constexpr int SM_R8 = 84 * 4;            // offset of 8 rows
__host__ __device__ constexpr int sm_idx(int row, int col) { return 84 * (row >> 1) + 40 * (row & 1) + col; }
// B-fragment addressing: element (8 B + 4 h + q, C + g) is at  B * SM_R8 + C + sm_boff(q, g) + h * SM_BH
__host__ __device__ constexpr int sm_boff(int q, int g) { return 84 * (q >> 1) + 40 * (q & 1) + g; }
constexpr int SM_BH = 84 * 2;

// ---- launchers (one translation unit each) --------------------------------
// p0: first problem of the chunk; count: problems in the chunk.
void launch_small_fwd(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                      int p0, int count, cudaStream_t st);
// D = 1 batches, F and gradient wanted, nothing else kept: the whole evaluation in one launch (small_dim.cu,
// scan1_eval_kernel).  Returns false when it does not apply; the caller then runs the four phases.
bool launch_small_fused(const Batch& b, const double* x, long long x_stride, double* F, double* grad,
                        long long grad_stride, int p0, int count, const Extra& ex, cudaStream_t st);
void launch_small_energy(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                         int p0, int count, const Extra& ex, cudaStream_t st);
void launch_small_bwd(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                      double* grad, long long grad_stride, int p0, int count, const Extra& ex,
                      cudaStream_t st);

// Lorenz-63 batches of up to a few thousand problems: several lanes per problem (l63_lanes.cu)
bool l63_lanes_applies(const Batch& b, int count);
void launch_l63_fwd_lanes(const Batch& b, const Scratch& s, const double* x, long long x_stride, int p0, int count,
                          cudaStream_t st);
void launch_l63_bwd_lanes(const Batch& b, const Scratch& s, const double* x, long long x_stride, double* grad,
                          long long grad_stride, int p0, int count, cudaStream_t st);

void launch_l96_fwd(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                    int p0, int count, cudaStream_t st);
void launch_l96_energy(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                       int p0, int count, const Extra& ex, cudaStream_t st);
void launch_l96_bwd(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                    double* grad, long long grad_stride, int p0, int count, const Extra& ex,
                    cudaStream_t st);

// Lorenz 96 at a run-time 10 <= D <= 64 other than 40 (l96_dyn.cu); the same contracts as the D = 40 launchers.
// D = 40 always runs the tuned kernels above.
__host__ __device__ inline bool l96_tuned(int D) { return D == 40; }
void launch_l96d_fwd(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                     int p0, int count, cudaStream_t st);
void launch_l96d_energy(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                        int p0, int count, const Extra& ex, cudaStream_t st);
void launch_l96d_hyper(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                       cudaStream_t st);
void launch_l96d_bwd(const Batch& b, const Scratch& s, const double* x, long long x_stride,
                     double* grad, long long grad_stride, int p0, int count, const Extra& ex,
                     cudaStream_t st);
void launch_bwd_dense_l96d(int method, int D, int N, double dt, const double* A, const double* dEm,
                           const double* dEs, const double* jm, const double* js, double* lam, double* psi,
                           cudaStream_t st);

// F[p] = E0 + trapz(esde_t) (/sigma for DW, OU) + Eobs.
void launch_finalize(const Batch& b, const Scratch& s, double* F, int p0, int count,
                     const Extra& ex, cudaStream_t st);

// Stand-alone backward sweep with dense jump tables (BwdOde.__call__).
void launch_bwd_dense(int method, int D, int N, double dt, const double* A, const double* dEm,
                      const double* dEs, const double* jm, const double* js, double* lam,
                      double* psi, cudaStream_t st);

// VarGP.initialization for problems p0 .. p0 + count - 1 (init.cu); scratch: count * D * 2 (M + 2) doubles, M the
// handle's row capacity (problem p uses obs_count_of(b, p) + 2 knots of its slot).
void launch_initialization(const Batch& b, int p0, int count, double t0, double* scratch, double* x,
                           long long x_stride, int* err, cudaStream_t st);

// Hyper-parameter gradients of model.energy (hyper.cu).  dEsde/dtheta has one entry per theta value, and for
// Lorenz-96 one per state dimension (lorenz_96.py:431).
__host__ __device__ inline int hyper_ntheta(int model, int D) { return model == MODEL_L63 ? 3 : (model == MODEL_L96 ? D : 1); }
// Per-problem outputs of the reduction: device rows p * stride, any pointer may be null.
struct HyperOut {
    double* Esde;                          // (B)
    double* dth;  long long dth_stride;    // hyper_ntheta values
    double* dsig; long long dsig_stride;   // 1 (D = 1) or D x D (diagonal; off-diagonals written as 0)
};
// The integrands of problems p0 .. p0 + count - 1 at their moments in s.mt, s.st into s.dEs (nth + D values per
// (problem, t); ft only for D = 1).  D = 1 and 3 read s.esde_t later and need the energy stage first; D = 40 runs the
// energy kernel's HYPER instantiation, which writes s.esde_t and the status words itself.
void launch_hyper_terms(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                        cudaStream_t st);
void launch_l96_hyper(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                      cudaStream_t st);
// Esde, dEsde/dtheta, dEsde/dSigma of those problems from s.esde_t and the integrands: one CTA per problem.
void launch_hyper_reduce(const Batch& b, const Scratch& s, int p0, int count, const HyperOut& o, cudaStream_t st);
// dEobs_dr of the 1-D likelihood (N values, zero except at obs_t).
void launch_obs_dr(int N, int M, const long long* obs_t, const double* obs_y, const double* R,
                   const double* mt, const double* st, double* dr, cudaStream_t stream);

// Euler-Maruyama sample paths and noisy observations for ensembles (make_trajectory / collect_obs).
void launch_trajectories(const TrajArgs& a, cudaStream_t st);
void launch_collect_obs(const ObsArgs& a, cudaStream_t st);

// Dense jump tables dEobs_dm (N,D), dEobs_ds (N,D,D) (GaussianLikelihood.gradients); entries of the components
// whose bit of `observed` is clear stay zero.
void launch_jump_tables(int D, int N, int M, const long long* obs_t, const double* obs_y, const double* R,
                        unsigned long long observed, const double* mt, double* jm, double* js, cudaStream_t st);

}  // namespace vgpa
