// datagen.cu -- batched sample paths and noisy observations for ensembles (SURVEY 8 f4).
//
// Replaces, for B trajectories at once, the Euler-Maruyama loops of
//   DoubleWell.make_trajectory         src/dynamics/double_well.py:122-166
//   OrnsteinUhlenbeck.make_trajectory  src/dynamics/ornstein_uhlenbeck.py:128-161
//   Lorenz63.make_trajectory           src/dynamics/lorenz_63.py:181-233   (burn-in :196-199)
//   Lorenz96.make_trajectory           src/dynamics/lorenz_96.py:249-314   (burn-in :266-279)
// and StochasticProcess.collect_obs    src/dynamics/stochastic_process.py:130-230.
//
// The standard-normal draws are INPUTS, in the layout the reference draws them ((D, N) per path,
// (D, M) per observation set): the reference's seeds stay meaningful because the host (or any other
// generator) produces the stream and the device does the arithmetic.  Every operation is a single
// correctly rounded IEEE operation in the reference's evaluation order (no FMA contraction), so a
// path is bit-identical to the numpy loop given the same draws.  The recurrences are sequential in t:
// one thread per path for D = 1, 3, one 64-thread CTA per path for Lorenz 96 (D = 40, and any other
// 10 <= D <= 64; neighbour exchange through a double-buffered shared-memory state, one barrier per step).
#include "common.cuh"

namespace vgpa {
namespace {

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }

// lorenz_63.py:8-37
__device__ __forceinline__ void l63(const double x[3], double s, double r, double b, double f[3])
{
    f[0] = mul(s, sub(x[1], x[0]));
    f[1] = sub(mul(sub(r, x[2]), x[0]), x[1]);
    f[2] = sub(mul(x[0], x[1]), mul(b, x[2]));
}

__global__ void __launch_bounds__(64)
traj_small_kernel(TrajArgs a)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.B) return;
    const double* th = a.theta + p * a.theta_stride;
    const double* sg = a.sigma + p * a.sigma_stride;
    const double* z = a.z + p * a.z_stride;
    double* out = a.path + p * a.path_stride;
    const int N = a.N;
    const double dt = a.dt;
    if (a.D == 1) {
        const double sq = sqrt(mul(sg[0], dt));                  // np.sqrt(sigma * dt)
        const double theta = th[0];
        const double mu = (a.model == MODEL_OU) ? th[1] : 0.0;
        double x = a.x_init[p * a.x_init_stride];
        out[0] = x;
        for (int t = 1; t < N; ++t) {
            double f;
            if (a.model == MODEL_DW) f = mul(mul(mul(4.0, x), sub(theta, mul(x, x))), dt);   // double_well.py:158-159
            else f = mul(mul(theta, sub(mu, x)), dt);                                        // ornstein_uhlenbeck.py:155
            x = add(add(x, f), mul(sq, z[t]));
            out[t] = x;
        }
        return;
    }
    // Lorenz 63
    double x[3], f[3], sq[3];
    for (int i = 0; i < 3; ++i) sq[i] = sqrt(mul(sg[i], dt));    // cholesky(diag(sigma) * dt)
    if (a.x_init) {
        for (int i = 0; i < 3; ++i) x[i] = a.x_init[p * a.x_init_stride + i];
    } else {
        x[0] = x[1] = x[2] = 1.0;                                // lorenz_63.py:193-199
        for (int k = 0; k < 5000; ++k) {
            l63(x, th[0], th[1], th[2], f);
            for (int i = 0; i < 3; ++i) x[i] = add(x[i], mul(f[i], 1.0e-3));
        }
    }
    for (int i = 0; i < 3; ++i) out[i] = x[i];
    for (int t = 1; t < N; ++t) {
        l63(x, th[0], th[1], th[2], f);
        for (int i = 0; i < 3; ++i) {
            x[i] = add(add(x[i], mul(f[i], dt)), mul(sq[i], z[(long long)i * N + t]));       // lorenz_63.py:227
            out[(long long)t * 3 + i] = x[i];
        }
    }
}

// Lorenz 96, D = 40: thread i owns component i.
__global__ void __launch_bounds__(64)
traj_l96_kernel(TrajArgs a)
{
    constexpr int D = 40;
    __shared__ double xs[2][D];
    const int p = blockIdx.x, i = threadIdx.x;
    const bool on = i < D;
    const int N = a.N;
    const double u = a.theta[p * a.theta_stride];
    const double* z = a.z + p * a.z_stride + (long long)(on ? i : 0) * N;
    double* out = a.path + p * a.path_stride;
    const int ip1 = (i + 1) % D, im1 = (i + D - 1) % D, im2 = (i + D - 2) % D;
    double x = 0.0;
    int par = 0;
    // one Euler step of lorenz_96.py:85-101: ((x[i+1] - x[i-2]) * x[i-1] - x[i]) + u
    auto drift = [&](double xi) {
        if (on) xs[par][i] = xi;
        __syncthreads();
        double f = 0.0;
        if (on) f = add(sub(mul(sub(xs[par][ip1], xs[par][im2]), xs[par][im1]), xi), u);
        par ^= 1;
        return f;
    };
    if (a.x_init) {
        if (on) x = a.x_init[p * a.x_init_stride + i];
    } else {
        x = (i == D / 2) ? add(u, 1.0e-3) : u;                   // lorenz_96.py:269-275
        for (int k = 0; k < 5000; ++k) x = add(x, mul(drift(x), 1.0e-3));
    }
    const double sq = on ? sqrt(mul(a.sigma[p * a.sigma_stride + i], a.dt)) : 0.0;
    if (on) out[i] = x;
    double zn = (on && N > 1) ? z[1] : 0.0;
    for (int t = 1; t < N; ++t) {
        const double zt = zn;
        if (on && t + 1 < N) zn = z[t + 1];
        x = add(add(x, mul(drift(x), a.dt)), mul(sq, zt));       // lorenz_96.py:305-307
        if (on) out[(long long)t * D + i] = x;
    }
}

// Lorenz 96 at a run-time D <= 64 other than 40 (the D = 40 kernel above stays as it is): the same loop,
// thread i owns component i; the burn-in perturbs component int(D / 2) (lorenz_96.py:269-275).
__global__ void __launch_bounds__(64)
traj_l96d_kernel(TrajArgs a)
{
    __shared__ double xs[2][64];
    const int D = a.D, p = blockIdx.x, i = threadIdx.x;
    const bool on = i < D;
    const int N = a.N;
    const double u = a.theta[p * a.theta_stride];
    const double* z = a.z + p * a.z_stride + (long long)(on ? i : 0) * N;
    double* out = a.path + p * a.path_stride;
    const int ip1 = (i + 1) % D, im1 = (i + D - 1) % D, im2 = (i + D - 2) % D;
    double x = 0.0;
    int par = 0;
    auto drift = [&](double xi) {
        if (on) xs[par][i] = xi;
        __syncthreads();
        double f = 0.0;
        if (on) f = add(sub(mul(sub(xs[par][ip1], xs[par][im2]), xs[par][im1]), xi), u);
        par ^= 1;
        return f;
    };
    if (a.x_init) {
        if (on) x = a.x_init[p * a.x_init_stride + i];
    } else {
        x = (i == D / 2) ? add(u, 1.0e-3) : u;
        for (int k = 0; k < 5000; ++k) x = add(x, mul(drift(x), 1.0e-3));
    }
    const double sq = on ? sqrt(mul(a.sigma[p * a.sigma_stride + i], a.dt)) : 0.0;
    if (on) out[i] = x;
    double zn = (on && N > 1) ? z[1] : 0.0;
    for (int t = 1; t < N; ++t) {
        const double zt = zn;
        if (on && t + 1 < N) zn = z[t + 1];
        x = add(add(x, mul(drift(x), a.dt)), mul(sq, zt));       // lorenz_96.py:305-307
        if (on) out[(long long)t * D + i] = x;
    }
}

// stochastic_process.py:177-226: obs_y = path[obs_t] + sqrt(R) * xi, xi in (D, M) layout.
__global__ void __launch_bounds__(128)
collect_obs_kernel(ObsArgs a)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long per = (long long)a.M * a.D;
    if (gid >= per * a.B) return;
    const int p = (int)(gid / per);
    const int r = (int)(gid % per), j = r / a.D, i = r % a.D;
    const double y = a.path[p * a.path_stride + a.obs_t[j] * a.D + i];
    const double n = mul(sqrt(a.R[p * a.R_stride + i]), a.xi[p * a.xi_stride + (long long)i * a.M + j]);
    a.obs_y[p * a.obs_y_stride + r] = add(y, n);
}

}  // namespace

void launch_trajectories(const TrajArgs& a, cudaStream_t st)
{
    if (a.B <= 0) return;
    if (a.model == MODEL_L96 && a.D == 40) traj_l96_kernel<<<a.B, 64, 0, st>>>(a);
    else if (a.model == MODEL_L96) traj_l96d_kernel<<<a.B, 64, 0, st>>>(a);
    else traj_small_kernel<<<(a.B + 31) / 32, 32, 0, st>>>(a);
}

void launch_collect_obs(const ObsArgs& a, cudaStream_t st)
{
    const long long tot = (long long)a.B * a.M * a.D;
    if (tot <= 0) return;
    collect_obs_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(a);
}

}  // namespace vgpa
