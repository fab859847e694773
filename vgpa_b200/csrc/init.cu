// init.cu -- VarGP.initialization (variational.py:73-139) for a whole batch, in HBM: the
// starting point x0 = [A0 | b0] of every problem from a cubic spline through its observations,
// each state dimension separately, so that ensembles are created on the device instead of being
// uploaded (13 MB per Lorenz-96 problem).  SURVEY.md section 8 (f) item 2.
//
// The spline is scipy.interpolate.CubicSpline with its default 'not-a-knot' ends (the reference's
// dependency): first derivatives s at the knots from the tridiagonal system of
// CubicSpline.__init__ (n >= 4 knots; n = 3: the parabola through the points; n = 2: the line),
// then the Hermite cubic of CubicHermiteSpline evaluated as c3 + c2 d + c1 d^2 + c0 d^3.
// Knots: time_x = [tw[0], tw[obs_t], tw[-1]], values [y_first, y, y_last] (variational.py:86-104);
// tw[k] = t0 + k dt_model.
//   kernel 1: one thread per (problem, dimension) solves for the knot derivatives (Thomas
//             algorithm; scratch in global memory: 2 (M + 2) doubles per pair, M the handle's row capacity;
//             each problem has its own M[p] + 2 knots)
//   kernel 2: one thread per (problem, time index, dimension) evaluates the spline at tw[k] and
//             tw[k+1], forms b0 and the diagonal entry of A0 (the zeros of A0 come from a memset)
// A component a partially observed problem does not observe (vgpa_create_observed) has no spline: its mean path
// is the constant m0[p][d], so b0(t)_d = a_dd m0_d (DESIGN.md section 5.1).
#include "common.cuh"

namespace vgpa {
namespace {

// The knots of one problem: its n = M + 2 time points and the observations they take their values from
struct Knots {
    const long long* ot;   // the problem's M observation indices
    const double* oy;      // its M x D observation values
    int M, n;
};
__device__ __forceinline__ Knots knots_of(const Batch& b, int p)
{
    const int M = obs_count_of(b, p);
    return Knots{obs_t_of(b, p), b.obs_y + p * b.obs_y_stride, M, M + 2};
}
__device__ __forceinline__ double knot_x(const Batch& b, const Knots& kn, double t0, int j)
{
    const int n = kn.n;
    const long long idx = (j == 0) ? 0 : (j == n - 1 ? (long long)(b.N - 1) : kn.ot[j - 1]);
    return t0 + (double)idx * b.dt_model;
}
__device__ __forceinline__ double knot_y(const Batch& b, const Knots& kn, int d, int j)
{
    const int n = kn.n;
    const int o = (j == 0) ? 0 : (j == n - 1 ? kn.M - 1 : j - 1);
    return kn.oy[(long long)o * b.D + d];
}

__global__ void __launch_bounds__(128)
init_slopes_kernel(Batch b, int p0, int count, double t0, double* __restrict__ scratch, int* __restrict__ err)
{
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= count * b.D) return;
    const int lp = pair / b.D, d = pair - lp * b.D, p = p0 + lp;
    if (!((observed_of(b, p) >> d) & 1ull)) return;           // unobserved: no spline (init_x0_kernel writes m0)
    const Knots kn = knots_of(b, p);
    const int n = kn.n;
    double* s = scratch + (long long)pair * 2 * (b.M + 2);   // slots of the handle's capacity
    double* cp = s + n;
    for (int i = 0; i + 1 < n; ++i)
        if (!(knot_x(b, kn, t0, i + 1) > knot_x(b, kn, t0, i))) {   // scipy: x must be strictly increasing
            atomicExch(err, 1);
            return;
        }
    auto X = [&](int j) { return knot_x(b, kn, t0, j); };
    auto Y = [&](int j) { return knot_y(b, kn, d, j); };
    if (n == 2) {
        s[0] = s[1] = (Y(1) - Y(0)) / (X(1) - X(0));
        return;
    }
    if (n == 3) {
        const double dx0 = X(1) - X(0), dx1 = X(2) - X(1);
        const double sl0 = (Y(1) - Y(0)) / dx0, sl1 = (Y(2) - Y(1)) / dx1;
        const double b0 = 2 * sl0, b1 = 3 * (dx0 * sl1 + dx1 * sl0), b2 = 2 * sl1;
        const double s1 = (b1 - dx1 * b0 - dx0 * b2) / (dx0 + dx1);
        s[0] = b0 - s1; s[1] = s1; s[2] = b2 - s1;
        return;
    }
    {
        const double dx0 = X(1) - X(0), dx1 = X(2) - X(1), dd = X(2) - X(0);
        const double sl0 = (Y(1) - Y(0)) / dx0, sl1 = (Y(2) - Y(1)) / dx1;
        cp[0] = dd / dx1;
        s[0] = (((dx0 + 2 * dd) * dx1 * sl0 + dx0 * dx0 * sl1) / dd) / dx1;
    }
    for (int i = 1; i < n - 1; ++i) {
        const double dxm = X(i) - X(i - 1), dxp = X(i + 1) - X(i);
        const double slm = (Y(i) - Y(i - 1)) / dxm, slp = (Y(i + 1) - Y(i)) / dxp;
        const double den = 2 * (dxm + dxp) - dxp * cp[i - 1];
        cp[i] = dxm / den;
        s[i] = (3 * (dxp * slm + dxm * slp) - dxp * s[i - 1]) / den;
    }
    {
        const int i = n - 1;
        const double dxm = X(i) - X(i - 1), dxmm = X(i - 1) - X(i - 2), dd = X(i) - X(i - 2);
        const double slm = (Y(i) - Y(i - 1)) / dxm, slmm = (Y(i - 1) - Y(i - 2)) / dxmm;
        const double rhs = (dxm * dxm * slmm + (2 * dd + dxm) * dxmm * slm) / dd;
        s[i] = (rhs - dd * s[i - 1]) / (dxmm - dd * cp[i - 1]);
    }
    for (int i = n - 2; i >= 0; --i) s[i] -= cp[i] * s[i + 1];
}

__device__ __forceinline__ double spline_at(const Batch& b, const Knots& kn, const double* s, int d, double t0, int k)
{
    const int n = kn.n;
    // interval i: x[i] <= tw[k] < x[i+1], i.e. i = #{ observation indices <= k } (last interval closed)
    int lo = 0, hi = kn.M;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (kn.ot[mid] <= k) lo = mid + 1; else hi = mid;
    }
    int i = lo;
    if (i > n - 2) i = n - 2;
    const double xi = knot_x(b, kn, t0, i), xj = knot_x(b, kn, t0, i + 1);
    const double yi = knot_y(b, kn, d, i), yj = knot_y(b, kn, d, i + 1);
    const double h = xj - xi, slope = (yj - yi) / h;
    const double tt = (s[i] + s[i + 1] - 2 * slope) / h;
    const double c0 = tt / h, c1 = (slope - s[i]) / h - tt;
    const double dd = (t0 + (double)k * b.dt_model) - xi;
    return yi + s[i] * dd + c1 * (dd * dd) + c0 * (dd * dd * dd);
}

__global__ void __launch_bounds__(256)
init_x0_kernel(Batch b, int p0, int count, double t0, const double* __restrict__ scratch, double* __restrict__ x,
               long long xs)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int D = b.D, N = b.N;
    if (gid >= (long long)count * N * D) return;
    const int d = (int)(gid % D);
    const long long r = gid / D;
    const int k = (int)(r % N), lp = (int)(r / N), p = p0 + lp;
    const Knots kn = knots_of(b, p);
    const double* s = scratch + ((long long)lp * D + d) * 2 * (b.M + 2);
    double* xo = x + (long long)p * xs;
    const double ad = 0.5 * (b.sigma[p * b.sigma_stride + d] / 0.25);      // variational.py:95 / :122-126
    // An unobserved component has no spline: its mean path is the constant m0[p][d], so b0(t)_d = a_dd m0_d.
    const bool obs = (observed_of(b, p) >> d) & 1ull;
    const double m0 = obs ? spline_at(b, kn, s, d, t0, k) : b.m0[p * b.m0_stride + d];
    if (D == 1) {
        xo[k] = ad;
        xo[N + k] = m0;                                                     // :101
        return;
    }
    xo[((long long)k * D + d) * D + d] = ad;           // the rest of A0 was zero-filled by the launcher
    double bk = ad * m0;                                                    // :133 at the last index
    if (obs && k < N - 1) bk += (spline_at(b, kn, s, d, t0, k + 1) - m0) / b.dt_model;  // :121, :127 (self.dt = model.time_step, :57)
    xo[(long long)N * D * D + (long long)k * D + d] = bk;
}

}  // namespace

// x0 rows of problems p0 .. p0 + count - 1 into x (device, row stride xs); scratch: count * D * 2 (M + 2)
// doubles (device); err: one int (device), set when the knots are not strictly increasing.
void launch_initialization(const Batch& b, int p0, int count, double t0, double* scratch, double* x, long long xs,
                           int* err, cudaStream_t st)
{
    const int pairs = count * b.D;
    if (b.D > 1)   // A0 = diagonal: zero-fill the (N, D, D) block of every row at memset speed
        cudaMemset2DAsync(x + (long long)p0 * xs, sizeof(double) * xs, 0, sizeof(double) * (size_t)b.N * b.D * b.D,
                          (size_t)count, st);
    init_slopes_kernel<<<(pairs + 127) / 128, 128, 0, st>>>(b, p0, count, t0, scratch, err);
    const long long tot = (long long)count * b.N * b.D;
    init_x0_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(b, p0, count, t0, scratch, x, xs);
}

}  // namespace vgpa
