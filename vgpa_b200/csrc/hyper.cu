// hyper.cu -- hyper-parameter gradients of model.energy: dEsde/dtheta and dEsde/dSigma, the last two
// entries of the third return value of StochasticProcess.energy.  The reference's hot path computes
// them on every evaluation and discards them (variational.py:175); here they are produced on request,
// for one problem (vgpa_model_energy) or for every problem of a handle (vgpa_hyper_device):
//   DW   double_well.py:251-257        OU   ornstein_uhlenbeck.py:223-229
//   L63  lorenz_63.py:327-343, Efg_drift_theta :572-633, Efg :414-432
//   L96  lorenz_96.py:420-434 (m_bar of ut_approx, utilities.py:239-310; flattened roll :27-32)
// Per (problem, time index) the integrands go to the pass's dEs scratch, nth + D values each (ft: theta
// integrand, nth values; fs: Sigma integrand, D values; for D = 1 ft only, dEsde/dSigma = -Esde / sigma): one thread per (problem, t)
// for D = 1 and D = 3 (below), the HYPER instantiation of the energy kernel for Lorenz 96 (l96_energy.cu for
// D = 40, l96_dyn.cu for the other D).
// Then one CTA per problem integrates every component with the composite trapezoid
// (utilities.py:144-201) in an order fixed by N alone and applies the final scalings.
#include "common.cuh"

namespace vgpa {
namespace {

// ---- D = 1 (DW, OU) and D = 3 (L63): one thread per (problem, time index) -------------------
template <int MODEL>
__global__ void __launch_bounds__(128)
hyper_small_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0, int count)
{
    constexpr int D = (MODEL == MODEL_L63) ? 3 : 1, DD = D * D, W = (MODEL == MODEL_L63) ? 6 : 1;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int N = b.N;
    if (idx >= (long long)count * N) return;
    const int lp = (int)(idx / N), t = (int)(idx % N), p = p0 + lp;
    const double* xp = x + (long long)p * xs;
    const double* theta = b.theta + p * b.theta_stride;
    const double* m = s.mt + ((long long)lp * N + t) * D;
    const double* S = s.st + ((long long)lp * N + t) * DD;
    double* ft = s.dEs + ((long long)lp * N + t) * W;
    if (MODEL == MODEL_DW || MODEL == MODEL_OU) {
        const double a = xp[t], bb = xp[N + t], mm = m[0], v = S[0], th = theta[0];
        const double m2 = mm * mm, E2 = m2 + v;
        if (MODEL == MODEL_DW) {
            const double c = 4.0 * th + a;
            const double E4 = m2 * m2 + 6 * m2 * v + 3 * v * v;
            ft[0] = c * E2 - 4.0 * E4 - bb * mm;               // double_well.py:251
        } else {
            ft[0] = E2 * (th - a) + mm * bb;                   // ornstein_uhlenbeck.py:223
        }
        return;
    }
    // Lorenz 63
    const double* A = xp + (long long)t * 9;
    const double* bt = xp + (long long)N * 9 + (long long)t * 3;
    double* fs = ft + 3;
    const double vS = theta[0], vR = theta[1], vB = theta[2];
    const double mx = m[0], my = m[1], mz = m[2];
    // the reference reads the UPPER triangle of S (lorenz_63.py:388-390, :601-606)
    const double Sxx = S[0], Sxy = S[1], Sxz = S[2], Syy = S[4], Syz = S[5], Szz = S[8];
    const double Exx = Sxx + mx * mx, Exy = Sxy + mx * my, Eyy = Syy + my * my;
    const double Exz = Sxz + mx * mz, Ezz = Szz + mz * mz, Eyz = Syz + my * mz;
    const double Exxz = Sxx * mz + 2 * Sxz * mx + (mx * mx) * mz;
    const double Exyz = Sxy * mz + Sxz * my + Syz * mx + mx * my * mz;
    // Efg_drift_theta, lorenz_63.py:622-631
    ft[0] = Eyy * (vS + A[1]) + Exx * (vS - A[0]) + Exy * (A[0] - 2 * vS - A[1]) + A[2] * (Eyz - Exz) +
                    bt[0] * (mx - my);
    ft[1] = vR * Exx - Exy - Exxz + A[3] * Exx + A[4] * Exy + A[5] * Exz - bt[1] * mx;
    ft[2] = -Exyz + vB * Ezz - A[6] * Exz - A[7] * Eyz - A[8] * Ezz + bt[2] * mz;
    // Efg_i = <r_i^2> of the quadratic residual r_i = c + l.x + s x_a x_b (see small_dim.cu: l63_energy)
    const double U[9] = {Sxx, Sxy, Sxz, Sxy, Syy, Syz, Sxz, Syz, Szz};
    const double l[9] = {A[0] - vS, A[1] + vS, A[2], A[3] + vR, A[4] - 1.0, A[5], A[6], A[7], A[8] - vB};
    const double sg[3] = {0.0, -1.0, 1.0};
    const int ib[3] = {0, 2, 1};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double s = sg[i];
        const int c = ib[i];
        double u[3] = {l[i * 3 + 0], l[i * 3 + 1], l[i * 3 + 2]};
        double mu = -bt[i] + u[0] * m[0] + u[1] * m[1] + u[2] * m[2];
        double extra = 0.0;
        if (i > 0) {
            mu += s * (m[0] * m[c] + U[c]);
            u[0] += s * m[c];
            u[c] += s * m[0];
            extra = U[0] * U[c * 3 + c] + U[c] * U[c];
        }
        double q = 0.0;
#pragma unroll
        for (int r = 0; r < 3; ++r) q += u[r] * (U[r * 3 + 0] * u[0] + U[r * 3 + 1] * u[1] + U[r * 3 + 2] * u[2]);
        fs[i] = mu * mu + q + extra;
    }
}

// ---- trapezoid over t for every component + final scalings: one CTA of 128 threads per problem ----
// Esde comes from esde_t exactly as finalize computes it (esde_of).  Component c is integrated by warp
// c % 4: lane l adds the intervals l, l + 32, ... in order, then a fixed xor tree; the order depends on N only.
__global__ void __launch_bounds__(ESDE_THREADS)
hyper_reduce_kernel(Batch b, Scratch s, int p0, int count, HyperOut o)
{
    __shared__ double sh[ESDE_THREADS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lp = blockIdx.x, p = p0 + lp, N = b.N, D = b.D;
    const int nth = hyper_ntheta(b.model, D), W = nth + (D == 1 ? 0 : D);
    const double* f = s.dEs + (long long)lp * N * W;
    const double* sg = b.sigma + p * b.sigma_stride;
    double* dth = o.dth ? o.dth + p * o.dth_stride : nullptr;
    double* dsig = o.dsig ? o.dsig + p * o.dsig_stride : nullptr;
    const double Esde = esde_of(b, p, s.esde_t + (long long)lp * N, sh);
    if (tid == 0 && o.Esde) o.Esde[p] = Esde;
    for (int c = warp; c < W; c += ESDE_THREADS / 32) {
        double tz = 0.0;
        for (int i = lane; i < N - 1; i += 32) tz += b.dt_model * (f[(long long)(i + 1) * W + c] + f[(long long)i * W + c]) / 2.0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) tz += __shfl_xor_sync(0xffffffffu, tz, off);
        if (lane != 0) continue;
        if (c < nth) {
            if (dth) dth[c] = (D == 1) ? (b.model == MODEL_DW ? 4.0 * tz : tz) / sg[0] : (1.0 / sg[c]) * tz;
        } else if (dsig) {
            const int i = c - nth;
            dsig[i * D + i] = -0.5 * (1.0 / sg[i]) * tz * (1.0 / sg[i]);
        }
    }
    if (dsig == nullptr) return;
    if (D == 1) {
        if (tid == 0) dsig[0] = -Esde / sg[0];
    } else {
        for (int e = tid; e < D * D; e += ESDE_THREADS)
            if (e / D != e % D) dsig[e] = 0.0;
    }
}

// dEobs_dr, 1-D likelihood (gaussian_like.py:194): one thread per observation
__global__ void obs_dr_kernel(int M, const long long* __restrict__ obs_t, const double* __restrict__ obs_y,
                              const double* __restrict__ R, const double* __restrict__ mt,
                              const double* __restrict__ st, double* __restrict__ dr)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= M) return;
    const long long t = obs_t[n];
    const double y = obs_y[n], m = mt[t], Ex2 = m * m + st[t];
    dr[t] = -0.5 * ((y * y) - 2.0 * y * m + Ex2 + 1.0) / R[0];
}

}  // namespace

void launch_obs_dr(int N, int M, const long long* obs_t, const double* obs_y, const double* R,
                   const double* mt, const double* st, double* dr, cudaStream_t stream)
{
    cudaMemsetAsync(dr, 0, sizeof(double) * N, stream);
    if (M > 0) obs_dr_kernel<<<(M + 127) / 128, 128, 0, stream>>>(M, obs_t, obs_y, R, mt, st, dr);
}

void launch_hyper_terms(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                        cudaStream_t st)
{
    if (b.model == MODEL_L96) {
        if (l96_tuned(b.D)) launch_l96_hyper(b, s, x, xs, p0, count, st);
        else launch_l96d_hyper(b, s, x, xs, p0, count, st);
        return;
    }
    const unsigned bl = (unsigned)(((long long)count * b.N + 127) / 128);
    if (b.model == MODEL_DW)      hyper_small_kernel<MODEL_DW><<<bl, 128, 0, st>>>(b, s, x, xs, p0, count);
    else if (b.model == MODEL_OU) hyper_small_kernel<MODEL_OU><<<bl, 128, 0, st>>>(b, s, x, xs, p0, count);
    else                          hyper_small_kernel<MODEL_L63><<<bl, 128, 0, st>>>(b, s, x, xs, p0, count);
}

void launch_hyper_reduce(const Batch& b, const Scratch& s, int p0, int count, const HyperOut& o, cudaStream_t st)
{
    hyper_reduce_kernel<<<count, ESDE_THREADS, 0, st>>>(b, s, p0, count, o);
}

}  // namespace vgpa
