// l96_dyn.cu -- Lorenz-96 at a run-time state dimension 10 <= D <= 64 other than 40 (D = 40 keeps the
// hand-fitted kernels of l96_sweeps.cu and l96_energy.cu).  The reference's Lorenz96(sigma, theta, r_seed,
// dim_d) takes any dim_d >= 10 (lorenz_96.py:104-140); this family serves every such D up to 64, the size at
// which each per-item working set still sits in shared memory.
//
//   forward sweep  : one CTA per problem, m(t), S(t) into the pass scratch     (ode_solver.py:31-61)
//   energy stage   : one CTA per (problem, t): Esde(t), dEsde/dm, dEsde/dS, or the hyper-parameter
//                    integrands (HYPER)                                       (lorenz_96.py:389-434)
//   backward sweep : one CTA per problem, fused with the gradient assembly    (ode_solver.py:63-95,
//                    variational.py:202-334), observation jumps or dense jump tables
// Plain FP64 arithmetic on D x D row-major matrices (pitch D) in shared memory: thread e of the CTA forms
// the entries e, e + NTH, ... of each product.  The solver tableaux are those of l96_sweeps.cu, quirks included
// (runge_kutta2.py:96: the inner covariance stage is fun_st(S, S, Sigma)); S and Psi stay EXACTLY symmetric
// because each right-hand side is formed as P + P^T from one product P.
#include "common.cuh"

namespace vgpa {
namespace {

constexpr int DMAX = 64;
constexpr int NTH = 256;
constexpr int EPT = DMAX * DMAX / NTH;   // matrix entries per thread at D = 64

enum { K_CUR = 0, K_MID = 1, K_NEXT = 2 };

__host__ __device__ constexpr int n_stages(int m) { return m == ODE_EULER ? 1 : (m == ODE_RK4 ? 4 : 2); }
__host__ __device__ constexpr int stage_kind(int m, int s)
{
    return m == ODE_EULER ? K_CUR
         : m == ODE_HEUN  ? (s == 0 ? K_CUR : K_NEXT)
         : m == ODE_RK2   ? (s == 0 ? K_CUR : K_MID)
                          : (s == 0 ? K_CUR : (s == 3 ? K_NEXT : K_MID));
}
__host__ __device__ constexpr double next_coef(int m, int s) { return m == ODE_HEUN ? 1.0 : m == ODE_RK2 ? 0.5 : (s < 2 ? 0.5 : 1.0); }
__host__ __device__ constexpr double ksum_w(int m, int s)
{
    return m == ODE_RK2 ? (s == 0 ? 0.0 : 1.0) : m == ODE_RK4 ? ((s == 1 || s == 2) ? 2.0 : 1.0) : 1.0;
}
template <int METHOD>
__device__ __forceinline__ double final_step(double dt, double ksum)
{
    if (METHOD == ODE_HEUN) return (0.5 * dt) * ksum;
    if (METHOD == ODE_RK4) return dt * ksum / 6.0;
    return dt * ksum;
}

// operand of kind K from the current and the neighbouring matrix (midpoint: runge_kutta2.py:74-75)
__device__ __forceinline__ double pick(int kind, const double* c, const double* n, int o)
{
    return kind == K_CUR ? c[o] : (kind == K_NEXT ? n[o] : 0.5 * (c[o] + n[o]));
}

// T = L R with L of kind lk from (L0, L1), R of kind rk from (R0, R1); all D x D, pitch D
__device__ void mat_mul(double* __restrict__ T, int lk, const double* L0, const double* L1, int rk, const double* R0,
                        const double* R1, int D)
{
    for (int e = threadIdx.x; e < D * D; e += NTH) {
        const int i = e / D, j = e - i * D;
        double s = 0.0;
        for (int k = 0; k < D; ++k) s = fma(pick(lk, L0, L1, i * D + k), pick(rk, R0, R1, k * D + j), s);
        T[e] = s;
    }
}

// (M v)[i] for i < D, M of kind mk from (M0, M1)
__device__ __forceinline__ double mat_vec_row(int mk, const double* M0, const double* M1, const double* v, int i, int D)
{
    double s = 0.0;
    for (int k = 0; k < D; ++k) s = fma(pick(mk, M0, M1, i * D + k), v[k], s);
    return s;
}

// ===========================================================================
// forward sweep
// ===========================================================================
template <int METHOD>
__global__ void __launch_bounds__(NTH, 1)
l96d_fwd_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0)
{
    extern __shared__ __align__(16) double smd[];
    constexpr int NS = n_stages(METHOD);
    const int D = b.D, DD = D * D, N = b.N, tid = threadIdx.x;
    const int lp = blockIdx.x, p = problem_at(b, p0 + lp);
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    double *Sb = smd, *Hb = Sb + DD, *Tb = Hb + DD, *Ac = Tb + DD, *An = Ac + DD;
    double *mv = An + DD, *vt0 = mv + DMAX, *vt1 = vt0 + DMAX, *sig = vt1 + DMAX, *bc = sig + DMAX, *bn = bc + DMAX;
    const double* A = x + (long long)p * xs;
    const double* bo = A + (long long)N * DD;
    double* mt = s.mt + (long long)lp * N * D;
    double* st = s.st + (long long)lp * N * DD;
    const double dt = b.dt;
    for (int e = tid; e < DD; e += NTH) {
        const double v = b.s0[p * b.s0_stride + e];
        Sb[e] = v;
        st[e] = v;
        Ac[e] = A[e];
    }
    if (tid < D) {
        const double v = b.m0[p * b.m0_stride + tid];
        mv[tid] = v;
        mt[tid] = v;
        sig[tid] = b.sigma[p * b.sigma_stride + tid];
        bc[tid] = bo[tid];
    }
    for (int k = 0; k < N - 1; ++k) {
        for (int e = tid; e < DD; e += NTH) An[e] = A[(long long)(k + 1) * DD + e];
        if (tid < D) bn[tid] = bo[(long long)(k + 1) * D + tid];
        __syncthreads();   // A(k+1), b(k+1) in place; the previous step's S, m visible
        double ksum[EPT];
        double kv = 0.0;
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            const int kind = stage_kind(METHOD, sidx);
            const double* X = (sidx == 0) ? Sb : Hb;
            const double* vX = (sidx == 0) ? mv : ((sidx - 1) & 1 ? vt1 : vt0);
            // T = Aop X  (fun_st: -A S - S A^T + Sigma = Sigma - (T + T^T));  RK2's inner stage: Aop = S
            if (METHOD == ODE_RK2 && sidx == 0) mat_mul(Tb, K_CUR, Sb, Sb, K_CUR, Sb, Sb, D);
            else mat_mul(Tb, kind, Ac, An, K_CUR, X, X, D);
            double ks = 0.0;
            if (tid < D) ks = -mat_vec_row(kind, Ac, An, vX, tid, D) + pick(kind, bc, bn, tid);   // fun_mt: -A m + b
            __syncthreads();   // T complete
            const double wt = ksum_w(METHOD, sidx), cdt = next_coef(METHOD, sidx) * dt;
#pragma unroll
            for (int r = 0; r < EPT; ++r) {
                const int e = tid + r * NTH;
                if (e >= DD) break;
                const int i = e / D, j = e - i * D;
                const double kk = (i == j ? sig[i] : 0.0) - (Tb[e] + Tb[j * D + i]);
                if (wt != 0.0) ksum[r] = (sidx == 0 || METHOD == ODE_RK2) ? wt * kk : ksum[r] + wt * kk;
                if (sidx < NS - 1) {
                    Hb[e] = Sb[e] + cdt * kk;
                } else {
                    const double v = Sb[e] + final_step<METHOD>(dt, ksum[r]);
                    Sb[e] = v;
                    st[(long long)(k + 1) * DD + e] = v;
                }
            }
            if (tid < D) {
                if (wt != 0.0) kv = (sidx == 0 || METHOD == ODE_RK2) ? wt * ks : kv + wt * ks;
                if (sidx < NS - 1) {
                    (sidx & 1 ? vt1 : vt0)[tid] = mv[tid] + cdt * ks;
                } else {
                    const double mn = mv[tid] + final_step<METHOD>(dt, kv);
                    mv[tid] = mn;
                    mt[(long long)(k + 1) * D + tid] = mn;
                }
            }
            __syncthreads();   // next operand visible, T reusable
        }
        double* tmp = Ac; Ac = An; An = tmp;
        tmp = bc; bc = bn; bn = tmp;
    }
}

// ===========================================================================
// energy stage: one CTA per (problem, t)
// ===========================================================================
// With L = chol(S) (lower) and V = L^-1, c = D + kappa, the sigma points are m +- sqrt(c) L[:, j]
// (utilities.py:283-288; chol(c S) = sqrt(c) chol(S)), and as in l96_energy.cu
//   dEsde/dm = (sqrt(c) / 2) V^T q,            q_j = w_i (var_{+j} - var_{-j})
//   dEsde/dS = (c / 2) V^T diag(d) V,          d_j = w_i (var_{+j} + var_{-j}) / 2 - Esde / c
// which is the reference's  dmS[:D] - Esde S^-1 m  and  0.5 (dmS[D:] - Esde S^-1)  (lorenz_96.py:414-418).
// l96() on the (2D+1) x D sigma-point matrix uses numba's FLATTENED np.roll (lorenz_96.py:27-32): the
// neighbours of a sigma point's first and last rows are rows of the adjacent sigma points.
// A non-positive-definite S(t) sets the status word to 1 + t.  (The reference's chol(diag(S)) fallback for
// a failed chol((D + kappa) S), utilities.py:276-279, only serves S that chol(S) then rejects in the gradient,
// variational.py:380: the status word reports that S(t) either way.)
// HYPER: instead of dEsde/dm, dEsde/dS the integrands of hyper.cu, 2D values per (problem, t) in s.dEs:
//   ft_i = <f>_i + (A m)_i - b_i,  fs_i = sum_k w_k r_{k,i}^2  (lorenz_96.py:420-423);  Esde(t) on the same bits.
struct EnView {
    double *Lb, *Vb, *ALb, *mv, *bv, *isg, *am, *ef, *dg, *qv, *dv, *var, *misc;
    int* bad;
};
__device__ __forceinline__ EnView en_view(double* smd, int D)
{
    EnView v;
    const int DD = D * D;
    v.Lb = smd; v.Vb = v.Lb + DD; v.ALb = v.Vb + DD;
    v.mv = v.ALb + DD; v.bv = v.mv + DMAX; v.isg = v.bv + DMAX; v.am = v.isg + DMAX; v.ef = v.am + DMAX;
    v.dg = v.ef + DMAX; v.qv = v.dg + DMAX; v.dv = v.qv + DMAX; v.var = v.dv + DMAX; v.misc = v.var + 2 * DMAX + 2;
    v.bad = reinterpret_cast<int*>(v.misc + 2);
    return v;
}
__host__ __device__ constexpr size_t en_smem(int D) { return sizeof(double) * (3 * (size_t)D * D + 10 * DMAX + 2 + 2 + 2); }

// entry `f` of the flattened sigma-point matrix chi (sigma point f / D, component f % D)
__device__ __forceinline__ double chi_at(const EnView& v, int f, int D, double sc)
{
    const int T = (2 * D + 1) * D;
    f = (f + T) % T;
    const int k = f / D, i = f - k * D;
    if (k == 0) return v.mv[i];
    if (k <= D) return v.mv[i] + sc * v.Lb[i * D + (k - 1)];
    return v.mv[i] - sc * v.Lb[i * D + (k - 1 - D)];
}

// residual r_{k,i} = l96(chi)_k,i + (A chi_k)_i - b_i  (lorenz_96.py:380-381)
__device__ __forceinline__ double residual(const EnView& v, int k, int i, int D, double sc, double theta)
{
    const int f = k * D + i;
    const double fi = (chi_at(v, f + 1, D, sc) - chi_at(v, f - 2, D, sc)) * chi_at(v, f - 1, D, sc) - chi_at(v, f, D, sc) + theta;
    const double al = (k == 0) ? 0.0 : (k <= D ? sc * v.ALb[i * D + (k - 1)] : -(sc * v.ALb[i * D + (k - 1 - D)]));
    return fi + (v.am[i] + al) - v.bv[i];
}

template <bool HYPER>
__global__ void __launch_bounds__(NTH, 2)
l96d_energy_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0, Extra ex)
{
    extern __shared__ __align__(16) double smd[];
    const int D = b.D, DD = D * D, N = b.N, K = 2 * D + 1, tid = threadIdx.x;
    const int lp = blockIdx.x / N, t = blockIdx.x - lp * N, p = problem_at(b, p0 + lp);
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    const EnView v = en_view(smd, D);
    const double* At = x + (long long)p * xs + (long long)t * DD;
    const double* bt = x + (long long)p * xs + (long long)N * DD + (long long)t * D;
    const double* mt = s.mt + ((long long)lp * N + t) * D;
    const double* St = s.st + ((long long)lp * N + t) * DD;
    const double theta = b.theta[p * b.theta_stride];
    const double kap = 1.05 * D, c = D + kap;                 // utilities.py:271
    const double w0 = kap / c, wi = 1.0 / (2.0 * c);          // :290-291
    const double sc = sqrt(c);
    if (tid == 0) *v.bad = 0;
    for (int e = tid; e < DD; e += NTH) {
        v.Lb[e] = St[e];
        v.Vb[e] = At[e];
    }
    if (tid < D) {
        v.mv[tid] = mt[tid];
        v.bv[tid] = bt[tid];
        v.isg[tid] = 1.0 / b.sigma[p * b.sigma_stride + tid];
    }
    __syncthreads();
    // <f> (lorenz_96.py:440-462) from S(t) before it is factored, A m; <df/dx> for vgpa_eval_full
    if (tid < D) {
        const int i = tid, f1 = (i + 1) % D, b1 = (i + D - 1) % D, b2 = (i + D - 2) % D;
        v.ef[i] = (v.Lb[f1 * D + b1] - v.Lb[b2 * D + b1]) + (v.mv[f1] - v.mv[b2]) * v.mv[b1] - v.mv[i] + theta;
        v.am[i] = mat_vec_row(K_CUR, v.Vb, v.Vb, v.mv, i, D);
        if (!HYPER && ex.Efx != nullptr && lp == 0) {
            ex.Efx[(long long)t * D + i] = v.ef[i];
            double* row = ex.Edf + (long long)t * DD + (long long)i * D;
            for (int j = 0; j < D; ++j) row[j] = 0.0;
            row[i] = -1.0;
            row[f1] = v.mv[b1];
            row[b2] = -v.mv[b1];
            row[b1] = v.mv[f1] - v.mv[b2];
        }
    }
    // ---- Cholesky S = L L^T in place (lower triangle; numpy.linalg.cholesky reads the lower triangle) ----
    for (int j = 0; j < D; ++j) {
        __syncthreads();
        const double d = v.Lb[j * D + j];
        const double dj = sqrt(d);
        if (tid == 0) {
            if (!(d > 0.0)) *v.bad = 1;
            v.dg[j] = dj;
        }
        for (int i = j + 1 + tid; i < D; i += NTH) v.Lb[i * D + j] = v.Lb[i * D + j] / dj;
        __syncthreads();
        const int m = D - 1 - j;
        for (int e = tid; e < m * m; e += NTH) {
            const int r = e / m, cc = e - r * m;
            if (cc > r) continue;
            const int i = j + 1 + r, k = j + 1 + cc;
            v.Lb[i * D + k] -= v.Lb[i * D + j] * v.Lb[k * D + j];
        }
    }
    __syncthreads();
    for (int e = tid; e < DD; e += NTH) {
        const int i = e / D, j = e - i * D;
        if (j > i) v.Lb[e] = 0.0;
        else if (j == i) v.Lb[e] = v.dg[i];
    }
    __syncthreads();
    // ---- A L (L lower: k >= j) ----
    for (int e = tid; e < DD; e += NTH) {
        const int i = e / D, j = e - i * D;
        double acc = 0.0;
        for (int k = j; k < D; ++k) acc = fma(v.Vb[i * D + k], v.Lb[k * D + j], acc);
        v.ALb[e] = acc;
    }
    __syncthreads();
    // ---- V = L^-1 over A's buffer (not needed by HYPER) ----
    if (!HYPER) {
        for (int e = tid; e < DD; e += NTH) {
            const int i = e / D, j = e - i * D;
            v.Vb[e] = (i == j) ? 1.0 : 0.0;
        }
        for (int k = 0; k < D; ++k) {
            __syncthreads();
            for (int j = tid; j <= k; j += NTH) v.Vb[k * D + j] = v.Vb[k * D + j] / v.Lb[k * D + k];
            __syncthreads();
            const int m = D - 1 - k;
            for (int e = tid; e < m * (k + 1); e += NTH) {
                const int r = e / (k + 1), j = e - r * (k + 1), i = k + 1 + r;
                v.Vb[i * D + j] -= v.Lb[i * D + k] * v.Vb[k * D + j];
            }
        }
    }
    // ---- residual energies var_k = sum_i r_{k,i}^2 / sigma_i of the 2D + 1 sigma points ----
    for (int k = tid; k < K; k += NTH) {
        double vk = 0.0;
        for (int i = 0; i < D; ++i) {
            const double rr = residual(v, k, i, D, sc, theta);
            vk += v.isg[i] * (rr * rr);
        }
        v.var[k] = vk;
    }
    __syncthreads();
    // Esde(t) = 1/2 sum_k w_k var_k (lorenz_96.py:401), fixed order: lanes stride the points, then a xor tree
    if (tid < 32) {
        double e = 0.0;
        for (int k = tid; k < K; k += 32) e += (k == 0 ? w0 : wi) * v.var[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
        if (tid == 0) v.misc[0] = 0.5 * e;
    }
    __syncthreads();
    const double esde = v.misc[0];
    if (HYPER) {
        if (tid < D) {
            const int i = tid;
            double fs = 0.0;
            for (int k = 0; k < K; ++k) {
                const double rr = residual(v, k, i, D, sc, theta);
                fs += (k == 0 ? w0 : wi) * (rr * rr);
            }
            double* o = s.dEs + ((long long)lp * N + t) * (2 * D);
            o[i] = (v.ef[i] + v.am[i]) - v.bv[i];
            o[D + i] = fs;
        }
    } else {
        if (tid < D) {
            const double vp = v.var[1 + tid], vm = v.var[1 + D + tid];
            v.qv[tid] = wi * (vp - vm);
            v.dv[tid] = 0.5 * (wi * (vp + vm)) - esde * (1.0 / c);
        }
        __syncthreads();
        double* oEm = s.dEm + ((long long)lp * N + t) * D;
        double* oEs = s.dEs + ((long long)lp * N + t) * DD;
        if (tid < D) {
            double acc = 0.0;
            for (int j = tid; j < D; ++j) acc = fma(v.Vb[j * D + tid], v.qv[j], acc);
            oEm[tid] = (0.5 * sc) * acc;
        }
        // lower entries, mirrored: exactly symmetric
        for (int e = tid; e < DD; e += NTH) {
            const int i = e / D, j = e - i * D;
            if (j > i) continue;
            double acc = 0.0;
            for (int k = i; k < D; ++k) acc = fma(v.Vb[k * D + i] * v.dv[k], v.Vb[k * D + j], acc);
            const double val = (0.5 * c) * acc;
            oEs[i * D + j] = val;
            oEs[j * D + i] = val;
        }
    }
    if (tid == 0) {
        s.esde_t[(long long)lp * N + t] = esde;
        if (*v.bad) atomicCAS(&s.status[lp], 0, 1 + t);
    }
}

// ===========================================================================
// backward sweep + gradient assembly
// ===========================================================================
struct DynBwdArgs {
    const double* A;     // (N,D,D) of this launch's first problem (stride xs between problems)
    const double* bo;    // (N,D) offsets (null without gradient)
    long long xs;
    const double* mt; const double* st;       // scratch (problem-major), null without gradient
    const double* dEm; const double* dEs;
    long long traj_v, traj_m;
    double* gA; double* gb; long long gs;     // gradient out (null: none)
    const double* jm_dense; const double* js_dense;
    double* lam_out; double* psi_out;         // first problem only, or null
};

template <int METHOD>
__global__ void __launch_bounds__(NTH, 1)
l96d_bwd_kernel(Batch b, DynBwdArgs a, int p0)
{
    extern __shared__ __align__(16) double smd[];
    constexpr int NS = n_stages(METHOD);
    const int D = b.D, DD = D * D, N = b.N, tid = threadIdx.x;
    const int lp = blockIdx.x, p = problem_at(b, p0 + lp);
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    double *Pb = smd, *Hb = Pb + DD, *Tb = Hb + DD, *Ac = Tb + DD, *An = Ac + DD, *Sb = An + DD;
    double *lam = Sb + DD, *lt0 = lam + DMAX, *lt1 = lt0 + DMAX, *mv = lt1 + DMAX, *bv = mv + DMAX;
    double *isg = bv + DMAX, *Rv = isg + DMAX, *uv = Rv + DMAX;
    // x and the gradient are addressed by PROBLEM (a.A, a.gA point at problem p0), the scratch by launch position
    const long long xrow = (long long)(p - p0);
    const double* A = a.A + xrow * a.xs;
    const double* bo = a.bo ? a.bo + xrow * a.xs : nullptr;
    const double* mt = a.mt ? a.mt + (long long)lp * a.traj_v : nullptr;
    const double* st = a.st ? a.st + (long long)lp * a.traj_m : nullptr;
    const double* dEm = a.dEm + (long long)lp * a.traj_v;
    const double* dEs = a.dEs + (long long)lp * a.traj_m;
    const bool with_grad = a.gA != nullptr;
    double* gA = with_grad ? a.gA + xrow * a.gs : nullptr;
    double* gb = with_grad ? a.gb + xrow * a.gs : nullptr;
    const bool dense = a.jm_dense != nullptr;
    const bool keep = a.lam_out != nullptr && lp == 0;
    const double* oy = dense ? nullptr : b.obs_y + p * b.obs_y_stride;
    const int* oidx = dense ? nullptr : obs_index_of(b, p);
    const double dt = b.dt, dtm = b.dt_model;
    const double theta = (b.theta != nullptr) ? b.theta[p * b.theta_stride] : 0.0;

    for (int e = tid; e < DD; e += NTH) {
        Pb[e] = 0.0;                                          // Psi[N-1] = 0
        Ac[e] = A[(long long)(N - 1) * DD + e];
    }
    if (tid < D) {
        lam[tid] = 0.0;                                       // lam[N-1] = 0
        isg[tid] = (b.sigma != nullptr) ? 1.0 / b.sigma[p * b.sigma_stride + tid] : 0.0;
        Rv[tid] = (b.R != nullptr) ? b.R[p * b.R_stride + tid] : 1.0;
    }
    for (int t = N - 1; t >= 0; --t) {
        if (with_grad) {
            for (int e = tid; e < DD; e += NTH) Sb[e] = st[(long long)t * DD + e];
            if (tid < D) {
                mv[tid] = mt[(long long)t * D + tid];
                bv[tid] = bo[(long long)t * D + tid];
            }
        }
        if (t >= 1)
            for (int e = tid; e < DD; e += NTH) An[e] = A[(long long)(t - 1) * DD + e];
        __syncthreads();   // Psi[t], lam[t], S(t), m(t), b(t), A(t-1) in place
        if (keep) {   // lam[t], Psi[t] for vgpa_eval_full / the stand-alone sweep
            for (int e = tid; e < DD; e += NTH) a.psi_out[(long long)t * DD + e] = Pb[e];
            if (tid < D) a.lam_out[(long long)t * D + tid] = lam[tid];
        }
        // ---- gradient at index t (variational.py:263-334) ----
        if (with_grad) {
            if (tid < D) {
                const int i = tid, f1 = (i + 1) % D, b1 = (i + D - 1) % D, b2 = (i + D - 2) % D;
                const double am = mat_vec_row(K_CUR, Ac, Ac, mv, i, D);
                const double Ef = (Sb[f1 * D + b1] - Sb[b2 * D + b1]) + (mv[f1] - mv[b2]) * mv[b1] - mv[i] + theta;
                const double db = isg[i] * (-Ef - am + bv[i]);
                const double ui = db + lam[i];
                uv[i] = ui;
                gb[(long long)t * D + i] = dtm * ui;
            }
            __syncthreads();
            // (Sigma^-1 (A_t + <df/dx>) - 2 Psi_t) S_t - u m^T, <df/dx> the sparse Lorenz-96 Jacobian at m
            for (int e = tid; e < DD; e += NTH) {
                const int i = e / D, j = e - i * D;
                const int f1 = (i + 1) % D, b1 = (i + D - 1) % D, b2 = (i + D - 2) % D;
                const double cf = mv[b1], cb1 = mv[f1] - mv[b2], si = isg[i];
                double acc = 0.0;
                for (int k = 0; k < D; ++k) {
                    const double edf = (k == i) ? -1.0 : (k == f1) ? cf : (k == b2) ? -cf : (k == b1) ? cb1 : 0.0;
                    acc = fma(fma(si, edf + Ac[i * D + k], -2.0 * Pb[i * D + k]), Sb[k * D + j], acc);
                }
                gA[(long long)t * DD + e] = dtm * (acc - uv[i] * mv[j]);
            }
        }
        if (t == 0) break;
        // ---- one backward step t -> t-1 ----
        double ksum[EPT];
        double kv = 0.0;
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            const int kind = stage_kind(METHOD, sidx);
            const double* X = (sidx == 0) ? Pb : Hb;
            const double* vX = (sidx == 0) ? lam : ((sidx - 1) & 1 ? lt1 : lt0);
            // Q = X Aop (fun_psi: -dE/dS + Psi A + A^T Psi = -G + (Q + Q^T))
            mat_mul(Tb, K_CUR, X, X, kind, Ac, An, D);
            double ks = 0.0;
            if (tid < D) {
                const double gk = pick(kind, dEm + (long long)t * D, dEm + (long long)(t - 1) * D, tid);
                ks = -gk + mat_vec_row(kind, Ac, An, vX, tid, D);   // fun_lam: -dE/dm + A lam
            }
            __syncthreads();   // Q complete
            const double wt = ksum_w(METHOD, sidx), cdt = next_coef(METHOD, sidx) * dt;
            const int n_obs = dense ? -1 : oidx[t - 1];
#pragma unroll
            for (int r = 0; r < EPT; ++r) {
                const int e = tid + r * NTH;
                if (e >= DD) break;
                const int i = e / D, j = e - i * D;
                const double gg = pick(kind, dEs + (long long)t * DD, dEs + (long long)(t - 1) * DD, e);
                const double kk = -gg + (Tb[e] + Tb[j * D + i]);
                if (wt != 0.0) ksum[r] = (sidx == 0 || METHOD == ODE_RK2) ? wt * kk : ksum[r] + wt * kk;
                if (sidx < NS - 1) {
                    Hb[e] = Pb[e] - cdt * kk;
                } else {   // final combination + jump at index t-1
                    double pn = Pb[e] - final_step<METHOD>(dt, ksum[r]);
                    if (dense) pn += a.js_dense[(long long)(t - 1) * DD + e];
                    else if (n_obs >= 0 && i == j) pn += 0.5 / Rv[i];   // gaussian_like.py:238
                    Pb[e] = pn;
                }
            }
            if (tid < D) {
                const int i = tid;
                if (wt != 0.0) kv = (sidx == 0 || METHOD == ODE_RK2) ? wt * ks : kv + wt * ks;
                if (sidx < NS - 1) {
                    (sidx & 1 ? lt1 : lt0)[i] = lam[i] - cdt * ks;
                } else {
                    double ln = lam[i] - final_step<METHOD>(dt, kv);
                    if (dense) ln += a.jm_dense[(long long)(t - 1) * D + i];
                    else if (n_obs >= 0) ln += -(oy[(long long)n_obs * D + i] - mt[(long long)(t - 1) * D + i]) / Rv[i];   // :235
                    lam[i] = ln;
                }
            }
            __syncthreads();   // next operand visible, Q reusable
        }
        double* tmp = Ac; Ac = An; An = tmp;
    }
}

size_t fwd_smem(int D) { return sizeof(double) * (5 * (size_t)D * D + 6 * DMAX); }
size_t bwd_smem(int D) { return sizeof(double) * (6 * (size_t)D * D + 8 * DMAX); }

void bwd_launch(const Batch& b, const DynBwdArgs& a, int p0, int count, cudaStream_t st)
{
    const size_t sh = bwd_smem(b.D);
    with_method(b.method, [&](auto m) {
        set_smem(l96d_bwd_kernel<m>, sh);
        l96d_bwd_kernel<m><<<count, NTH, sh, st>>>(b, a, p0);
    });
}

}  // namespace

void launch_l96d_fwd(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                     cudaStream_t st)
{
    const size_t sh = fwd_smem(b.D);
    with_method(b.method, [&](auto m) {
        set_smem(l96d_fwd_kernel<m>, sh);
        l96d_fwd_kernel<m><<<count, NTH, sh, st>>>(b, s, x, xs, p0);
    });
}

void launch_l96d_energy(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                        const Extra& ex, cudaStream_t st)
{
    const size_t sh = en_smem(b.D);
    set_smem(l96d_energy_kernel<false>, sh);
    l96d_energy_kernel<false><<<(unsigned)((long long)count * b.N), NTH, sh, st>>>(b, s, x, xs, p0, ex);
}

void launch_l96d_hyper(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                       cudaStream_t st)
{
    const size_t sh = en_smem(b.D);
    set_smem(l96d_energy_kernel<true>, sh);
    l96d_energy_kernel<true><<<(unsigned)((long long)count * b.N), NTH, sh, st>>>(b, s, x, xs, p0, Extra{});
}

void launch_l96d_bwd(const Batch& b, const Scratch& s, const double* x, long long xs, double* grad, long long gs,
                     int p0, int count, const Extra& ex, cudaStream_t st)
{
    const long long N = b.N, D = b.D;
    DynBwdArgs a{};
    a.A = x + (long long)p0 * xs;
    a.bo = a.A + N * D * D;
    a.xs = xs;
    a.mt = s.mt; a.st = s.st; a.dEm = s.dEm; a.dEs = s.dEs;
    a.traj_v = N * D; a.traj_m = N * D * D;
    if (grad != nullptr) {
        a.gA = grad + (long long)p0 * gs;
        a.gb = a.gA + N * D * D;
        a.gs = gs;
    }
    a.lam_out = ex.lamt; a.psi_out = ex.psit;
    bwd_launch(b, a, p0, count, st);
}

void launch_bwd_dense_l96d(int method, int D, int N, double dt, const double* A, const double* dEm,
                           const double* dEs, const double* jm, const double* js, double* lam, double* psi,
                           cudaStream_t st)
{
    Batch b{};
    b.model = MODEL_L96; b.method = method; b.D = D; b.N = N; b.B = 1; b.dt = dt; b.dt_model = dt;
    DynBwdArgs a{};
    a.A = A; a.xs = 0; a.dEm = dEm; a.dEs = dEs;
    a.traj_v = (long long)N * D; a.traj_m = (long long)N * D * D;
    a.jm_dense = jm; a.js_dense = js; a.lam_out = lam; a.psi_out = psi;
    bwd_launch(b, a, 0, 1, st);
}

}  // namespace vgpa
