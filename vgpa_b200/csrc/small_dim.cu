// small_dim.cu -- D = 1 (Double Well, Ornstein-Uhlenbeck) and D = 3 (Lorenz 63)
// kernels.  With a state this small one inference problem fits in the registers
// of ONE thread, so the sequential sweeps run one thread per problem (a batch
// of B problems is B independent register-resident recurrences) and the
// time-parallel stage runs one thread per (problem, time index).
//
// Reference behaviour reproduced (paths relative to the reference root):
//   forward sweep   src/numerics/{euler,heun,runge_kutta2,runge_kutta4}.py solve_fwd
//   backward sweep  same files, solve_bwd; RHS in src/numerics/ode_solver.py:31-95
//   energies        src/dynamics/double_well.py:169-260, ornstein_uhlenbeck.py:165-232,
//                   lorenz_63.py:237-568
//   jumps           src/var_bayes/gaussian_like.py:155-243
//   gradient        src/var_bayes/variational.py:202-334
//   F               variational.py:199, utilities.py:144-201, gaussian_like.py:69-153
#include <cstdlib>

#include "common.cuh"
#include "l63_grad.cuh"

namespace vgpa {

// ---------------------------------------------------------------------------
// register-resident D x D helpers
// ---------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ void ld_vec(const double* __restrict__ g, double* r)
{
#pragma unroll
    for (int i = 0; i < D; ++i) r[i] = __ldg(g + i);
}

// ode_solver.py:44   -A m + b
template <int D>
__device__ __forceinline__ void fun_m(const double* m, const double* A, const double* b, double* o)
{
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) s += A[i * D + k] * m[k];
        o[i] = -s + b[i];
    }
}
// ode_solver.py:60   -A S - S A^T + Sigma   (Sigma diagonal)
template <int D>
__device__ __forceinline__ void fun_S(const double* S, const double* A, const double* sig, double* o)
{
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) {
            double p = 0.0, q = 0.0;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                p += A[i * D + k] * S[k * D + j];
                q += S[i * D + k] * A[j * D + k];
            }
            o[i * D + j] = -p - q + (i == j ? sig[i] : 0.0);
        }
}
// ode_solver.py:77   -g + A lam
template <int D>
__device__ __forceinline__ void fun_lam(const double* g, const double* A, const double* lam, double* o)
{
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) s += A[i * D + k] * lam[k];
        o[i] = -g[i] + s;
    }
}
// ode_solver.py:94   -G + Psi A + A^T Psi
template <int D>
__device__ __forceinline__ void fun_psi(const double* G, const double* A, const double* P, double* o)
{
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) {
            double p = 0.0, q = 0.0;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                p += P[i * D + k] * A[k * D + j];
                q += A[k * D + i] * P[k * D + j];
            }
            o[i * D + j] = -G[i * D + j] + p + q;
        }
}
template <int n>
__device__ __forceinline__ void axpy(const double* y, double a, const double* x, double* o)
{
#pragma unroll
    for (int i = 0; i < n; ++i) o[i] = y[i] + a * x[i];
}
template <int n>
__device__ __forceinline__ void mid(const double* p, const double* q, double* o)
{
#pragma unroll
    for (int i = 0; i < n; ++i) o[i] = 0.5 * (p[i] + q[i]);
}

// pull the line holding p into L2 (no register, no scoreboard): a thread-per-problem recurrence has a
// handful of private input streams and nothing but its own look-ahead to hide their DRAM latency
__device__ __forceinline__ void prefetch_l2(const void* p)
{
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
constexpr int PF_AHEAD = 16;   // time indices of look-ahead for the L2 prefetch
// Only small batches prefetch: they are latency bound (a few warps per SM).  With tens of thousands of
// threads in flight the prefetched lines are evicted before use and the extra requests cost bandwidth
// (measured: OU x 65536 5.1 -> 10.2 ms with prefetching, L63 x 4096 7.3 -> 5.7 ms).
constexpr int PF_MAX_BATCH = 8192;

// one step k -> k+1 of solve_fwd (the four solver files): Ak, bk at index k, An, bn at index k+1
template <int D, int METHOD>
__device__ __forceinline__ void fwd_step(const double* m, const double* S, const double* Ak, const double* bk,
                                         const double* An, const double* bn, const double* sig, double dt,
                                         double* mn, double* Sn)
{
    constexpr int DD = D * D;
    const double h = 0.5 * dt;
    (void)h; (void)An; (void)bn;
    if (METHOD == ODE_EULER) {  // euler.py:84-87
        double v1[D], k1[DD];
        fun_m<D>(m, Ak, bk, v1);
        axpy<D>(m, dt, v1, mn);
        fun_S<D>(S, Ak, sig, k1);
        axpy<DD>(S, dt, k1, Sn);
    } else if (METHOD == ODE_HEUN) {  // heun.py:91-106
        double v1[D], v2[D], vt[D], k1[DD], k2[DD], tmp[DD];
        fun_m<D>(m, Ak, bk, v1);
        axpy<D>(m, dt, v1, vt);
        fun_m<D>(vt, An, bn, v2);
#pragma unroll
        for (int i = 0; i < D; ++i) mn[i] = m[i] + h * (v1[i] + v2[i]);
        fun_S<D>(S, Ak, sig, k1);
        axpy<DD>(S, dt, k1, tmp);
        fun_S<D>(tmp, An, sig, k2);
#pragma unroll
        for (int i = 0; i < DD; ++i) Sn[i] = S[i] + h * (k1[i] + k2[i]);
    } else if (METHOD == ODE_RK2) {  // runge_kutta2.py:92,96 (inner stage: S in place of A)
        double am[DD], bm[D], v1[D], v2[D], vt[D], k1[DD], k2[DD], tmp[DD];
        mid<DD>(Ak, An, am);
        mid<D>(bk, bn, bm);
        fun_m<D>(m, Ak, bk, v1);
        axpy<D>(m, h, v1, vt);
        fun_m<D>(vt, am, bm, v2);
        axpy<D>(m, dt, v2, mn);
        fun_S<D>(S, S, sig, k1);
        axpy<DD>(S, h, k1, tmp);
        fun_S<D>(tmp, am, sig, k2);
        axpy<DD>(S, dt, k2, Sn);
    } else {  // runge_kutta4.py:93-108
        double am[DD], bm[D], v1[D], v2[D], v3[D], v4[D], vt[D];
        double k1[DD], k2[DD], k3[DD], k4[DD], tmp[DD];
        mid<DD>(Ak, An, am);
        mid<D>(bk, bn, bm);
        fun_m<D>(m, Ak, bk, v1);
        axpy<D>(m, h, v1, vt);
        fun_m<D>(vt, am, bm, v2);
        axpy<D>(m, h, v2, vt);
        fun_m<D>(vt, am, bm, v3);
        axpy<D>(m, dt, v3, vt);
        fun_m<D>(vt, An, bn, v4);
#pragma unroll
        for (int i = 0; i < D; ++i)
            mn[i] = m[i] + dt * (v1[i] + 2.0 * (v2[i] + v3[i]) + v4[i]) / 6.0;
        fun_S<D>(S, Ak, sig, k1);
        axpy<DD>(S, h, k1, tmp);
        fun_S<D>(tmp, am, sig, k2);
        axpy<DD>(S, h, k2, tmp);
        fun_S<D>(tmp, am, sig, k3);
        axpy<DD>(S, dt, k3, tmp);
        fun_S<D>(tmp, An, sig, k4);
#pragma unroll
        for (int i = 0; i < DD; ++i)
            Sn[i] = S[i] + dt * (k1[i] + 2.0 * (k2[i] + k3[i]) + k4[i]) / 6.0;
    }
}

// ---------------------------------------------------------------------------
// forward sweep: one thread per problem
// ---------------------------------------------------------------------------
template <int D, int METHOD>
__global__ void __launch_bounds__(64)
small_fwd_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0, int count)
{
    constexpr int DD = D * D;
    const int lp = blockIdx.x * blockDim.x + threadIdx.x;
    if (lp >= count) return;
    const int p = p0 + lp, N = b.N;
    if (b.active != nullptr && b.active[p] == 0) return;
    const bool pf = count <= PF_MAX_BATCH;
    const double* A = x + (long long)p * xs;
    const double* bo = A + (long long)N * DD;
    double sig[D], m[D], S[DD];
    ld_vec<D>(b.sigma + p * b.sigma_stride, sig);
    ld_vec<D>(b.m0 + p * b.m0_stride, m);
    ld_vec<DD>(b.s0 + p * b.s0_stride, S);
    double* mt = s.mt + (long long)lp * N * D;
    double* st = s.st + (long long)lp * N * DD;
#pragma unroll
    for (int i = 0; i < D; ++i) mt[i] = m[i];
#pragma unroll
    for (int i = 0; i < DD; ++i) st[i] = S[i];
    const double dt = b.dt, h = 0.5 * dt;
    // A(k), b(k) of the current index, of the next one (loaded a step ago) and of the one after
    // (load issued now): with one thread per problem nothing else hides the global-load latency
    double Ak[DD], bk[D], An[DD], bn[D], Af[DD], bf[D];
    ld_vec<DD>(A, Ak);
    ld_vec<D>(bo, bk);
    if (N > 1) {
        ld_vec<DD>(A + DD, An);
        ld_vec<D>(bo + D, bn);
    }
    for (int k = 0; k < N - 1; ++k) {
        {
            const int kf = (k + 2 < N) ? k + 2 : N - 1;
            ld_vec<DD>(A + (long long)kf * DD, Af);
            ld_vec<D>(bo + (long long)kf * D, bf);
            if (pf && (D > 1 || (k & 7) == 0) && k + PF_AHEAD < N) {   // D = 1: one 128-byte line lasts 16 indices
                prefetch_l2(A + (long long)(k + PF_AHEAD) * DD + DD - 1);
                prefetch_l2(bo + (long long)(k + PF_AHEAD) * D + D - 1);
            }
        }
        double mn[D], Sn[DD];
        fwd_step<D, METHOD>(m, S, Ak, bk, An, bn, sig, dt, mn, Sn);
#pragma unroll
        for (int i = 0; i < D; ++i) {
            m[i] = mn[i];
            bk[i] = bn[i];
            bn[i] = bf[i];
            mt[(long long)(k + 1) * D + i] = mn[i];
        }
#pragma unroll
        for (int i = 0; i < DD; ++i) {
            S[i] = Sn[i];
            Ak[i] = An[i];
            An[i] = Af[i];
            st[(long long)(k + 1) * DD + i] = Sn[i];
        }
    }
}

// ---------------------------------------------------------------------------
// staged forward sweep (large batches)
// ---------------------------------------------------------------------------
// One thread per problem as above, but with one thread per problem every global access of a warp
// touches 32 different lines (problems are N * D * (D + 1) doubles apart).  With tens of thousands
// of problems in flight that is what bounds the forward sweep (the L2 look-ahead of the small-batch
// kernel cannot be used: its lines are evicted before use).  Here a warp moves the streams of its 32
// problems through shared memory a block of TB time indices at a time.  A problem's block is
// contiguous in HBM, so the warp fetches it with coalesced 8-byte cp.async copies (lane e: element e
// of problem j's block, all copies of a block in flight at once) into row j of a buffer whose row
// pitch is odd (lane j then walks its own row without bank conflicts); m(t), S(t) take the same road
// back.  Measured (B200, F + gradient, forward sweep only): L63 x 16384 3.2 -> 1.8 ms, OU x 65536
// 1.98 -> 1.20 ms.  For batches of a few thousand problems (latency bound, not request bound) it is
// no faster (L63 x 4096: 1.64 vs 1.60 ms; OU x 1024: 0.51 vs 0.25 ms), and the same treatment of the
// backward sweep (six input streams, two output streams) was slower at every size tried (L63 x 4096
// 3.6 -> 4.7 ms, x 16384 6.3 -> 10.1 ms, OU x 65536 2.5 -> 2.9 ms): both stay on the register-prefetch
// kernels (profiles/README.md).
__host__ __device__ constexpr int odd_pitch(int n) { return n | 1; }

// 8-byte asynchronous global -> shared copy (SASS LDGSTS): no register, no scoreboard, so a warp has all
// the copies of a block in flight at once; waited for with stage_wait()
__device__ __forceinline__ void cp_async8(double* dst_smem, const double* src_gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst_smem)), "l"(src_gmem)
                 : "memory");
}
__device__ __forceinline__ void stage_wait()
{
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();
}
// rows j = 0 .. nprob-1 of len <= MAXLEN doubles: problem j at g + j * gstride <-> row j of buf
template <int MAXLEN>
__device__ __forceinline__ void stage_in(double* __restrict__ buf, int pitch, const double* __restrict__ g,
                                         long long gstride, int nprob, int len, int lane)
{
    for (int j = 0; j < nprob; ++j) {
        const double* src = g + (long long)j * gstride;
        double* dst = buf + j * pitch;
#pragma unroll
        for (int it = 0; it < (MAXLEN + 31) / 32; ++it) {
            const int e = lane + 32 * it;
            if (e < len) cp_async8(dst + e, src + e);
        }
    }
}
template <int MAXLEN>
__device__ __forceinline__ void stage_out(const double* __restrict__ buf, int pitch, double* __restrict__ g,
                                          long long gstride, int nprob, int len, int lane)
{
#pragma unroll 4
    for (int j = 0; j < nprob; ++j) {
        double* dst = g + (long long)j * gstride;
        const double* src = buf + j * pitch;
#pragma unroll
        for (int it = 0; it < (MAXLEN + 31) / 32; ++it) {
            const int e = lane + 32 * it;
            if (e < len) dst[e] = src[e];
        }
    }
}
// lines [p, p + bytes) into L2
__device__ __forceinline__ void prefetch_span(const double* p, int bytes)
{
    const char* c = reinterpret_cast<const char*>(p);
    for (int o = 0; o < bytes; o += 128) prefetch_l2(c + o);
    if (bytes > 0) prefetch_l2(c + bytes - 8);
}

template <int D, int METHOD, int TB>
__global__ void __launch_bounds__(32)
small_fwd_staged_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0, int count)
{
    constexpr int DD = D * D, NI = TB + 1;
    constexpr int PA = odd_pitch(NI * DD), PB = odd_pitch(NI * D), PS = odd_pitch(TB * DD), PM = odd_pitch(TB * D);
    extern __shared__ double stage_smem[];
    double* sA = stage_smem;
    double* sB = sA + 32 * PA;
    double* sS = sB + 32 * PB;
    double* sM = sS + 32 * PS;
    const int lane = threadIdx.x, lp0 = blockIdx.x * 32;
    const int nprob = min(32, count - lp0);
    const bool on = lane < nprob && (b.active == nullptr || b.active[p0 + lp0 + lane] != 0);
    const int lp = lp0 + (lane < nprob ? lane : 0), p = p0 + lp, N = b.N;
    const double* A0 = x + (long long)(p0 + lp0) * xs;      // problem 0 of this warp
    const double* b0 = A0 + (long long)N * DD;
    double* mt0 = s.mt + (long long)lp0 * N * D;
    double* st0 = s.st + (long long)lp0 * N * DD;
    double sig[D], m[D], S[DD];
    ld_vec<D>(b.sigma + p * b.sigma_stride, sig);
    ld_vec<D>(b.m0 + p * b.m0_stride, m);
    ld_vec<DD>(b.s0 + p * b.s0_stride, S);
    // (a skipped problem's scratch rows receive whatever its shared-memory row holds: nobody reads them)
    if (on) {
#pragma unroll
        for (int i = 0; i < D; ++i) mt0[(long long)lane * N * D + i] = m[i];
#pragma unroll
        for (int i = 0; i < DD; ++i) st0[(long long)lane * N * DD + i] = S[i];
    }
    const double dt = b.dt;
    for (int k0 = 0; k0 < N - 1; k0 += TB) {
        const int nb = min(TB, N - 1 - k0);      // steps k0 .. k0 + nb - 1 read indices k0 .. k0 + nb
        stage_in<NI * DD>(sA, PA, A0 + (long long)k0 * DD, xs, nprob, (nb + 1) * DD, lane);
        stage_in<NI * D>(sB, PB, b0 + (long long)k0 * D, xs, nprob, (nb + 1) * D, lane);
        if (on && k0 + TB < N - 1) {
            const int nn = min(TB, N - 1 - (k0 + TB)) + 1;
            prefetch_span(A0 + (long long)lane * xs + (long long)(k0 + TB) * DD, nn * DD * 8);
            prefetch_span(b0 + (long long)lane * xs + (long long)(k0 + TB) * D, nn * D * 8);
        }
        stage_wait();
        if (on) {
            const double* ra = sA + lane * PA;
            const double* rb = sB + lane * PB;
            double* rs = sS + lane * PS;
            double* rm = sM + lane * PM;
            for (int kk = 0; kk < nb; ++kk) {
                double Ak[DD], An[DD], bk[D], bn[D], mn[D], Sn[DD];
#pragma unroll
                for (int i = 0; i < DD; ++i) {
                    Ak[i] = ra[kk * DD + i];
                    An[i] = ra[(kk + 1) * DD + i];
                }
#pragma unroll
                for (int i = 0; i < D; ++i) {
                    bk[i] = rb[kk * D + i];
                    bn[i] = rb[(kk + 1) * D + i];
                }
                fwd_step<D, METHOD>(m, S, Ak, bk, An, bn, sig, dt, mn, Sn);
#pragma unroll
                for (int i = 0; i < D; ++i) {
                    m[i] = mn[i];
                    rm[kk * D + i] = mn[i];
                }
#pragma unroll
                for (int i = 0; i < DD; ++i) {
                    S[i] = Sn[i];
                    rs[kk * DD + i] = Sn[i];
                }
            }
        }
        __syncwarp();
        stage_out<TB * DD>(sS, PS, st0 + (long long)(k0 + 1) * DD, (long long)N * DD, nprob, nb * DD, lane);
        stage_out<TB * D>(sM, PM, mt0 + (long long)(k0 + 1) * D, (long long)N * D, nprob, nb * D, lane);
        __syncwarp();
    }
}
template <int D, int TB> constexpr size_t fwd_stage_bytes()
{
    return sizeof(double) * 32 * (odd_pitch((TB + 1) * D * D) + odd_pitch((TB + 1) * D) + odd_pitch(TB * D * D) + odd_pitch(TB * D));
}

// ---------------------------------------------------------------------------
// per-time-step SDE energy, its m/S gradients, and <f>, <df/dx>
// ---------------------------------------------------------------------------
struct Moments1 {  // gaussian_moments.py:57-74,108-122,155-167
    double E2, E3, E4, E6, Dm2, Dm3, Dm4, Dm6, Ds3, Ds4, Ds6;
    __device__ __forceinline__ Moments1(double m, double v)
    {
        const double m2 = m * m, m3 = m2 * m, m4 = m2 * m2, m5 = m4 * m, m6 = m3 * m3;
        const double v2 = v * v, v3 = v2 * v;
        E2 = m2 + v;
        E3 = m3 + 3 * m * v;
        E4 = m4 + 6 * m2 * v + 3 * v2;
        E6 = m6 + 15 * m4 * v + 45 * m2 * v2 + 15 * v3;
        Dm2 = 2 * m;
        Dm3 = 3 * (m2 + v);
        Dm4 = 4 * (m3 + 3 * m * v);
        Dm6 = 6 * (m5 + 10 * m3 * v + 15 * m * v2);
        Ds3 = 3 * m;
        Ds4 = 6 * (m2 + v);
        Ds6 = 15 * m4 + 90 * m2 * v + 45 * v2;
    }
};

// <f> and <df/dx> at one time index (needed by the energy output and again by
// the gradient assembly, which recomputes them instead of storing them).
template <int MODEL, int D>
__device__ __forceinline__ void drift_moments(const double* th, const double* m, const double* S,
                                              double* Ef, double* Edf)
{
    if (MODEL == MODEL_DW) {  // double_well.py:220,223
        const double E2 = m[0] * m[0] + S[0], E3 = m[0] * m[0] * m[0] + 3 * m[0] * S[0];
        Ef[0] = 4.0 * (th[0] * m[0] - E3);
        Edf[0] = 4.0 * (th[0] - 3.0 * E2);
    } else if (MODEL == MODEL_OU) {  // ornstein_uhlenbeck.py:211,214
        Ef[0] = -th[0] * m[0];
        Edf[0] = -th[0];
    } else {  // lorenz_63.py:319-326 (reads S[2,0] and S[1,0])
        const double vS = th[0], vR = th[1], vB = th[2];
        // (__dmul_rn: the product must not be contracted into whatever consumes <f>_0 -- the lane-parallel
        // kernels of l63_lanes.cu evaluate the same expressions and must give the same bits)
        Ef[0] = __dmul_rn(vS, m[1] - m[0]);
        Ef[1] = vR * m[0] - m[1] - S[2 * D + 0] - m[0] * m[2];
        Ef[2] = S[1 * D + 0] + m[0] * m[1] - vB * m[2];
        Edf[0] = -vS;        Edf[1] = vS;   Edf[2] = 0.0;
        Edf[3] = vR - m[2];  Edf[4] = -1.0; Edf[5] = -m[0];
        Edf[6] = m[1];       Edf[7] = m[0]; Edf[8] = -vB;
    }
}

// Lorenz 63: each residual r_i(x) = f_i(x) + (A x)_i - b_i is a quadratic
// polynomial  c + l.x + s x_a x_b  of the Gaussian state x ~ N(m, S), so with
// u = l + s (m_b e_a + m_a e_b),  mu = <r> = c + l.m + s (m_a m_b + S_ab):
//   <r^2>        = mu^2 + u'Su + s^2 (S_aa S_bb + S_ab^2)
//   d<r^2>/dm    = 2 mu u + 2 s ((Su)_b e_a + (Su)_a e_b)
//   d<r^2>/dS    = u u' + mu s (E_ab + E_ba) + s^2 (S_bb E_aa + S_aa E_bb + S_ab (E_ab + E_ba))
// This equals the reference's hand-expanded moment expressions
// (lorenz_63.py:393-566) EXCEPT that the reference differentiates w.r.t. each
// off-diagonal S_xy as ONE variable, i.e. its off-diagonal entries are twice the
// symmetric per-entry gradient; that factor is applied at the end (:564-566).
__device__ __forceinline__ void l63_energy(const double* th, const double* iS, const double* A,
                                           const double* bt, const double* m, const double* S,
                                           double& esde, double* dEm, double* dEs)
{
    const double vS = th[0], vR = th[1], vB = th[2];
    // the reference reads the UPPER triangle of S (lorenz_63.py:388-390)
    const double U[9] = {S[0], S[1], S[2], S[1], S[4], S[5], S[2], S[5], S[8]};
    const double l[9] = {A[0] - vS, A[1] + vS, A[2], A[3] + vR, A[4] - 1.0, A[5],
                         A[6], A[7], A[8] - vB};
    const double sg[3] = {0.0, -1.0, 1.0};
    const int ia[3] = {0, 0, 0}, ib[3] = {0, 2, 1};
    esde = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) dEm[i] = 0.0;
#pragma unroll
    for (int i = 0; i < 9; ++i) dEs[i] = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double s = sg[i];
        const int a = ia[i], c = ib[i];
        double u[3] = {l[i * 3 + 0], l[i * 3 + 1], l[i * 3 + 2]};
        double mu = -bt[i] + u[0] * m[0] + u[1] * m[1] + u[2] * m[2];
        double extra = 0.0;
        if (i > 0) {
            mu += s * (m[a] * m[c] + U[a * 3 + c]);
            u[a] += s * m[c];
            u[c] += s * m[a];
            extra = U[a * 3 + a] * U[c * 3 + c] + U[a * 3 + c] * U[a * 3 + c];
        }
        double Su[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) Su[r] = U[r * 3 + 0] * u[0] + U[r * 3 + 1] * u[1] + U[r * 3 + 2] * u[2];
        const double Er2 = mu * mu + (u[0] * Su[0] + u[1] * Su[1] + u[2] * Su[2]) + extra;
        const double w = 0.5 * iS[i];
        esde += w * Er2;
        double gm[3] = {2 * mu * u[0], 2 * mu * u[1], 2 * mu * u[2]};
        double G[9];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int q = 0; q < 3; ++q) G[r * 3 + q] = u[r] * u[q];
        if (i > 0) {
            gm[a] += 2 * s * Su[c];
            gm[c] += 2 * s * Su[a];
            const double off = mu * s + U[a * 3 + c];
            G[a * 3 + c] += off;
            G[c * 3 + a] += off;
            G[a * 3 + a] += U[c * 3 + c];
            G[c * 3 + c] += U[a * 3 + a];
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) dEm[r] += w * gm[r];
#pragma unroll
        for (int r = 0; r < 9; ++r) dEs[r] += w * G[r];
    }
    // off-diagonal convention of the reference (see above)
    dEs[1] *= 2.0; dEs[2] *= 2.0; dEs[3] *= 2.0; dEs[5] *= 2.0; dEs[6] *= 2.0; dEs[7] *= 2.0;
}

// Esde integrand and its m, S derivatives at one time index, D = 1
template <int MODEL>
__device__ __forceinline__ void energy1(double th, double sg, double At, double bt, double m, double S,
                                        double& e, double& dm, double& dS)
{
    if (MODEL == MODEL_DW) {  // double_well.py:214,243,248 (8*E6 in the energy, 16*Dm6 in the gradient)
        const Moments1 g(m, S);
        const double c = 4.0 * th + At, c2 = c * c, bb = bt;
        e = 8.0 * (g.E6 - c * g.E4 + bb * g.E3) + (c2 * g.E2) - (2.0 * bb * c * m) + bb * bb;
        dm = 0.5 * (16.0 * g.Dm6 - 8.0 * c * g.Dm4 + 8.0 * bb * g.Dm3 + c2 * g.Dm2 - 2.0 * bb * c) / sg;
        dS = 0.5 * (16.0 * g.Ds6 - 8.0 * c * g.Ds4 + 8.0 * bb * g.Ds3 + c2 * 1.0) / sg;
    } else {  // ornstein_uhlenbeck.py:205,217,221
        const double E2 = m * m + S, d = th - At, q1 = d * d;
        e = E2 * q1 + 2.0 * m * d * bt + bt * bt;
        dm = (m * q1 + th * bt - At * bt) / sg;
        dS = 0.5 * q1 / sg;
    }
}

template <int MODEL, int D>
__global__ void __launch_bounds__(128)
small_energy_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0, int count,
                    Extra ex)
{
    constexpr int DD = D * D;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int N = b.N;
    if (idx >= (long long)count * N) return;
    const int lp = (int)(idx / N), t = (int)(idx % N), p = p0 + lp;
    if (b.active != nullptr && b.active[p] == 0) return;
    const double* A = x + (long long)p * xs + (long long)t * DD;
    const double* bo = x + (long long)p * xs + (long long)N * DD + (long long)t * D;
    const double* th = b.theta + p * b.theta_stride;
    const double* sg = b.sigma + p * b.sigma_stride;
    double At[DD], bt[D], m[D], S[DD];
    ld_vec<DD>(A, At);
    ld_vec<D>(bo, bt);
    const long long oV = ((long long)lp * N + t) * D, oM = ((long long)lp * N + t) * DD;
#pragma unroll
    for (int i = 0; i < D; ++i) m[i] = s.mt[oV + i];
#pragma unroll
    for (int i = 0; i < DD; ++i) S[i] = s.st[oM + i];
    double e, dm[D], dS[DD];
    if constexpr (MODEL == MODEL_DW || MODEL == MODEL_OU) {
        energy1<MODEL>(th[0], sg[0], At[0], bt[0], m[0], S[0], e, dm[0], dS[0]);
    } else {
        double iS[3] = {1.0 / sg[0], 1.0 / sg[1], 1.0 / sg[2]};
        l63_energy(th, iS, At, bt, m, S, e, dm, dS);
    }
    s.esde_t[(long long)lp * N + t] = e;
#pragma unroll
    for (int i = 0; i < D; ++i) s.dEm[oV + i] = dm[i];
#pragma unroll
    for (int i = 0; i < DD; ++i) s.dEs[oM + i] = dS[i];
    if (ex.Efx != nullptr && lp == 0) {
        double Ef[D], Edf[DD];
        drift_moments<MODEL, D>(th, m, S, Ef, Edf);
#pragma unroll
        for (int i = 0; i < D; ++i) ex.Efx[(long long)t * D + i] = Ef[i];
#pragma unroll
        for (int i = 0; i < DD; ++i) ex.Edf[(long long)t * DD + i] = Edf[i];
    }
}

// ---------------------------------------------------------------------------
// backward sweep fused with the gradient assembly: one thread per problem.
// lam, Psi live in registers; dL/dA, dL/db are written as soon as lam[t],
// Psi[t] exist, so lam/Psi never go to HBM (unless ex.lamt asks for them).
// ---------------------------------------------------------------------------
template <int MODEL, int D>
__device__ __forceinline__ void grad_at(const double* th, const double* isg, double dtm,
                                        const double* At, const double* bt, const double* m,
                                        const double* S, const double* lam, const double* Psi,
                                        double* gA, double* gb)
{
    constexpr int DD = D * D;
    if (MODEL == MODEL_L63) {   // explicit rounding, shared with the lane-parallel kernel (l63_grad.cuh)
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double mm[3] = {m[0], m[1], m[2]};
            const double Ar[3] = {At[i * 3 + 0], At[i * 3 + 1], At[i * 3 + 2]};
            const double Pr[3] = {Psi[i * 3 + 0], Psi[i * 3 + 1], Psi[i * 3 + 2]};
            const L63Row r = l63_row_terms(i, th[0], th[1], th[2], mm, (i == 1) ? S[6] : S[3], Ar, bt[i], isg[i]);
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const double Sc[3] = {S[j], S[3 + j], S[6 + j]};
                gA[i * 3 + j] = l63_grad_a(r, Sc, Pr, m[j], lam[i], dtm);
            }
            gb[i] = l63_grad_b(r, lam[i], dtm);
        }
        return;
    }
    double Ef[D], Edf[DD], db[D];
    drift_moments<MODEL, D>(th, m, S, Ef, Edf);
#pragma unroll
    for (int i = 0; i < D; ++i) {  // variational.py:324-334
        double am = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) am += At[i * D + k] * m[k];
        db[i] = isg[i] * (-Ef[i] - am + bt[i]);
    }
#pragma unroll
    for (int i = 0; i < D; ++i) {
#pragma unroll
        for (int j = 0; j < D; ++j) {  // variational.py:312-322, :300-310
            double p1 = 0.0, p2 = 0.0;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                p1 += (isg[i] * (Edf[i * D + k] + At[i * D + k])) * S[k * D + j];
                p2 += Psi[i * D + k] * S[k * D + j];
            }
            gA[i * D + j] = dtm * ((p1 - db[i] * m[j]) - lam[i] * m[j] - 2.0 * p2);
        }
        gb[i] = dtm * (db[i] + lam[i]);  // variational.py:280,285
    }
}

// one step t -> t-1 of solve_bwd: (At, gt, Gt) at index t, (Am, gm, Gm) at index t-1; jm = jump of lambda
template <int D, int METHOD>
__device__ __forceinline__ void bwd_step(const double* lam, const double* Psi, const double* At, const double* gt,
                                         const double* Gt, const double* Am, const double* gm, const double* Gm,
                                         const double* jm, double dt, double* ln, double* Pn)
{
    constexpr int DD = D * D;
    const double h = 0.5 * dt;
    (void)h; (void)Am; (void)gm; (void)Gm;
    if (METHOD == ODE_EULER) {  // euler.py:146-149
        double v1[D], k1[DD];
        fun_lam<D>(gt, At, lam, v1);
        fun_psi<D>(Gt, At, Psi, k1);
#pragma unroll
        for (int i = 0; i < D; ++i) ln[i] = lam[i] - v1[i] * dt + jm[i];
#pragma unroll
        for (int i = 0; i < DD; ++i) Pn[i] = Psi[i] - k1[i] * dt;
    } else if (METHOD == ODE_HEUN) {  // heun.py:170-185
        double v1[D], v2[D], vt[D], k1[DD], k2[DD], tmp[DD];
        fun_lam<D>(gt, At, lam, v1);
        axpy<D>(lam, -dt, v1, vt);
        fun_lam<D>(gm, Am, vt, v2);
        fun_psi<D>(Gt, At, Psi, k1);
        axpy<DD>(Psi, -dt, k1, tmp);
        fun_psi<D>(Gm, Am, tmp, k2);
#pragma unroll
        for (int i = 0; i < D; ++i) ln[i] = lam[i] - h * (v1[i] + v2[i]) + jm[i];
#pragma unroll
        for (int i = 0; i < DD; ++i) Pn[i] = Psi[i] - h * (k1[i] + k2[i]);
    } else if (METHOD == ODE_RK2) {  // runge_kutta2.py:180-189
        double am[DD], gmid[D], Gmid[DD], v1[D], v2[D], vt[D], k1[DD], k2[DD], tmp[DD];
        mid<DD>(Am, At, am);
        mid<D>(gm, gt, gmid);
        mid<DD>(Gm, Gt, Gmid);
        fun_lam<D>(gt, At, lam, v1);
        axpy<D>(lam, -h, v1, vt);
        fun_lam<D>(gmid, am, vt, v2);
        fun_psi<D>(Gt, At, Psi, k1);
        axpy<DD>(Psi, -h, k1, tmp);
        fun_psi<D>(Gmid, am, tmp, k2);
#pragma unroll
        for (int i = 0; i < D; ++i) ln[i] = lam[i] - dt * v2[i] + jm[i];
#pragma unroll
        for (int i = 0; i < DD; ++i) Pn[i] = Psi[i] - dt * k2[i];
    } else {  // runge_kutta4.py:191-206
        double am[DD], gmid[D], Gmid[DD], v1[D], v2[D], v3[D], v4[D], vt[D];
        double k1[DD], k2[DD], k3[DD], k4[DD], tmp[DD];
        mid<DD>(Am, At, am);
        mid<D>(gm, gt, gmid);
        mid<DD>(Gm, Gt, Gmid);
        fun_lam<D>(gt, At, lam, v1);
        axpy<D>(lam, -h, v1, vt);
        fun_lam<D>(gmid, am, vt, v2);
        axpy<D>(lam, -h, v2, vt);
        fun_lam<D>(gmid, am, vt, v3);
        axpy<D>(lam, -dt, v3, vt);
        fun_lam<D>(gm, Am, vt, v4);
        fun_psi<D>(Gt, At, Psi, k1);
        axpy<DD>(Psi, -h, k1, tmp);
        fun_psi<D>(Gmid, am, tmp, k2);
        axpy<DD>(Psi, -h, k2, tmp);
        fun_psi<D>(Gmid, am, tmp, k3);
        axpy<DD>(Psi, -dt, k3, tmp);
        fun_psi<D>(Gm, Am, tmp, k4);
#pragma unroll
        for (int i = 0; i < D; ++i)
            ln[i] = lam[i] - dt * (v1[i] + 2.0 * (v2[i] + v3[i]) + v4[i]) / 6.0 + jm[i];
#pragma unroll
        for (int i = 0; i < DD; ++i)
            Pn[i] = Psi[i] - dt * (k1[i] + 2.0 * (k2[i] + k3[i]) + k4[i]) / 6.0;
    }
}

// jm_dense / js_dense: dense jump tables of the stand-alone sweep (BwdOde.__call__,
// bwd_ode.py:45); null in the batched path, where the jumps come from the observations.
struct SmallBwdArgs {
    const double* x; long long xs;
    double* grad; long long gs;
    const double* jm_dense; const double* js_dense;
};

template <int MODEL, int D, int METHOD>
__global__ void __launch_bounds__(64)
small_bwd_kernel(Batch b, Scratch s, SmallBwdArgs a, int p0, int count, Extra ex)
{
    constexpr int DD = D * D;
    const int lp = blockIdx.x * blockDim.x + threadIdx.x;
    if (lp >= count) return;
    const int p = p0 + lp, N = b.N;
    if (b.active != nullptr && b.active[p] == 0) return;
    const bool pf = count <= PF_MAX_BATCH;
    const bool dense = a.jm_dense != nullptr;
    const double* A = a.x + (long long)p * a.xs;
    const double* bo = A + (long long)N * DD;
    double* gA = a.grad ? a.grad + (long long)p * a.gs : nullptr;
    double* gb = a.grad ? gA + (long long)N * DD : nullptr;
    const double* mt = s.mt + (long long)lp * N * D;
    const double* st = s.st + (long long)lp * N * DD;
    const double* dEm = s.dEm + (long long)lp * N * D;
    const double* dEs = s.dEs + (long long)lp * N * DD;
    const double* th = dense ? nullptr : b.theta + p * b.theta_stride;
    const double* oy = dense ? nullptr : b.obs_y + p * b.obs_y_stride;
    const int* oidx = dense ? nullptr : obs_index_of(b, p);
    double isg[D], Rv[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        isg[i] = dense ? 0.0 : 1.0 / b.sigma[p * b.sigma_stride + i];
        Rv[i] = dense ? 1.0 : b.R[p * b.R_stride + i];
    }
    const bool keep = (ex.lamt != nullptr) && lp == 0;
    const double dt = b.dt, h = 0.5 * dt, dtm = b.dt_model;
    double lam[D], Psi[DD];
#pragma unroll
    for (int i = 0; i < D; ++i) lam[i] = 0.0;
#pragma unroll
    for (int i = 0; i < DD; ++i) Psi[i] = 0.0;
    // Register prefetch, as in the forward sweep: index t (current), t-1 (loaded a step ago) and
    // t-2 (load issued at the top of the step) for A, dE/dm, dE/dS; t and t-1 for m, S, b.
    double At[DD], gt[D], Gt[DD], Am[DD], gm[D], Gm[DD], Af[DD], gf[D], Gf[DD];
    double m[D], S[DD], bt[D], mp[D], Sp[DD], bp[D];
    ld_vec<DD>(A + (long long)(N - 1) * DD, At);
    ld_vec<D>(dEm + (long long)(N - 1) * D, gt);
    ld_vec<DD>(dEs + (long long)(N - 1) * DD, Gt);
    {
        const int t1 = (N >= 2) ? N - 2 : 0;
        ld_vec<DD>(A + (long long)t1 * DD, Am);
        ld_vec<D>(dEm + (long long)t1 * D, gm);
        ld_vec<DD>(dEs + (long long)t1 * DD, Gm);
    }
    if (gA != nullptr) {
        ld_vec<D>(mt + (long long)(N - 1) * D, m);
        ld_vec<DD>(st + (long long)(N - 1) * DD, S);
        ld_vec<D>(bo + (long long)(N - 1) * D, bt);
    }
    for (int t = N - 1; t >= 0; --t) {
        {
            const int t2 = (t >= 2) ? t - 2 : 0, t1 = (t >= 1) ? t - 1 : 0;
            ld_vec<DD>(A + (long long)t2 * DD, Af);
            ld_vec<D>(dEm + (long long)t2 * D, gf);
            ld_vec<DD>(dEs + (long long)t2 * DD, Gf);
            if (gA != nullptr) {
                ld_vec<D>(mt + (long long)t1 * D, mp);
                ld_vec<DD>(st + (long long)t1 * DD, Sp);
                ld_vec<D>(bo + (long long)t1 * D, bp);
            }
            if (pf && (D > 1 || (t & 7) == 0) && t >= PF_AHEAD) {
                const long long tp = t - PF_AHEAD;
                prefetch_l2(A + tp * DD);
                prefetch_l2(dEs + tp * DD);
                prefetch_l2(dEm + tp * D);
                if (gA != nullptr) {
                    prefetch_l2(st + tp * DD);
                    prefetch_l2(mt + tp * D);
                    prefetch_l2(bo + tp * D);
                }
            }
        }
        if (keep) {
#pragma unroll
            for (int i = 0; i < D; ++i) ex.lamt[(long long)t * D + i] = lam[i];
#pragma unroll
            for (int i = 0; i < DD; ++i) ex.psit[(long long)t * DD + i] = Psi[i];
        }
        if (gA != nullptr) {
            double ga[DD], gbv[D];
            grad_at<MODEL, D>(th, isg, dtm, At, bt, m, S, lam, Psi, ga, gbv);
#pragma unroll
            for (int i = 0; i < DD; ++i) gA[(long long)t * DD + i] = ga[i];
#pragma unroll
            for (int i = 0; i < D; ++i) gb[(long long)t * D + i] = gbv[i];
        }
        if (t == 0) break;
        // jump at index t-1 (gaussian_like.py:188,191 / :235,238); H = I, R diagonal
        double jm[D], js[D];
        const int n = dense ? -1 : oidx[t - 1];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            jm[i] = dense ? a.jm_dense[(long long)(t - 1) * D + i] : 0.0;
            js[i] = 0.0;
        }
        if (n >= 0) {
#pragma unroll
            for (int i = 0; i < D; ++i) {
                const double mprev = (gA != nullptr) ? mp[i] : mt[(long long)(t - 1) * D + i];
                jm[i] = -(oy[(long long)n * D + i] - mprev) / Rv[i];
                js[i] = 0.5 / Rv[i];
            }
        }
        double ln[D], Pn[DD];
        bwd_step<D, METHOD>(lam, Psi, At, gt, Gt, Am, gm, Gm, jm, dt, ln, Pn);
#pragma unroll
        for (int i = 0; i < D; ++i) Pn[i * D + i] += js[i];
        if (dense) {
#pragma unroll
            for (int i = 0; i < DD; ++i) Pn[i] += a.js_dense[(long long)(t - 1) * DD + i];
        }
#pragma unroll
        for (int i = 0; i < D; ++i) {
            lam[i] = ln[i];
            gt[i] = gm[i];
            gm[i] = gf[i];
            m[i] = mp[i];
            bt[i] = bp[i];
        }
#pragma unroll
        for (int i = 0; i < DD; ++i) {
            Psi[i] = Pn[i];
            At[i] = Am[i];
            Am[i] = Af[i];
            Gt[i] = Gm[i];
            Gm[i] = Gf[i];
            S[i] = Sp[i];
        }
    }
}

// ---------------------------------------------------------------------------
// F = E0 + Esde + Eobs : one CTA per problem, fixed-order reductions (bitwise
// reproducible, so a sharded batch returns the same F as a single-GPU one).
// block_sum and esde_of: common.cuh.
// ---------------------------------------------------------------------------

// The free energy of problem p from its Esde integrand f(t) and its moments (global or shared memory); every
// thread of the CTA (128 threads or more) calls it, every thread gets the value.  parts: E0, Esde, Eobs (or null).
__device__ __forceinline__ double free_energy_of(const Batch& b, int p, const double* f, const double* mt,
                                                 const double* st, double* sh, double* parts)
{
    constexpr int W = ESDE_THREADS;
    const int tid = threadIdx.x;
    const int D = b.D, M = obs_count_of(b, p), DD = D * D;
    const long long* ot = obs_t_of(b, p);
    const double Esde = esde_of(b, p, f, sh);
    double acc;
    // observation energy
    const double* oy = b.obs_y + p * b.obs_y_stride;
    const double* R = b.R + p * b.R_stride;
    double Eobs;
    const double LOG2PI = 1.8378770664093453;
    if (D == 1) {  // gaussian_like.py:69-96
        acc = 0.0;
        for (int n = tid; n < (tid < W ? M : 0); n += W) {
            const long long t = ot[n];
            const double y = oy[n], E2 = mt[t] * mt[t] + st[t];
            acc += (y * y) - 2.0 * y * mt[t] + E2;
        }
        const double sm = block_sum(acc, sh);
        Eobs = 0.5 * sm / R[0] + 0.5 * M * (LOG2PI + log(R[0]));
    } else {  // gaussian_like.py:98-153; S diagonal indexed by the observation ORDINAL n
        // H = the rows of the identity at the observed components O: the sums run over O, the count term has
        // D_o = |O|.  With O = every component the arithmetic is the identity operator's, bit for bit.
        const unsigned long long obs = observed_of(b, p);
        acc = 0.0;
        for (int q = tid; q < (tid < W ? M * D : 0); q += W) {
            const int n = q / D, i = q % D;
            if (!((obs >> i) & 1ull)) continue;
            const long long t = ot[n];
            const double z = (oy[(long long)n * D + i] - mt[t * D + i]) / sqrt(R[i]);
            acc += z * z + (1.0 / R[i]) * st[(long long)n * DD + (long long)i * D + i];
        }
        const double sm = block_sum(acc, sh);
        double ld = 0.0;
        int Do = 0;
        for (int i = 0; i < D; ++i)
            if ((obs >> i) & 1ull) {
                ld += log(sqrt(R[i]));
                ++Do;
            }
        Eobs = 0.5 * (sm + M * (Do * LOG2PI + 2.0 * ld));
    }
    const double E0 = b.E0[p * b.E0_stride];
    if (parts != nullptr && tid == 0) {
        parts[0] = E0;
        parts[1] = Esde;
        parts[2] = Eobs;
    }
    return E0 + Esde + Eobs;
}

__global__ void __launch_bounds__(128)
finalize_kernel(Batch b, Scratch s, double* __restrict__ F, int p0, int count, Extra ex)
{
    __shared__ double sh[128];
    const int lp = blockIdx.x, p = problem_at(b, p0 + lp);
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    const int N = b.N, D = b.D;
    const double Fp = free_energy_of(b, p, s.esde_t + (long long)lp * N, s.mt + (long long)lp * N * D,
                                     s.st + (long long)lp * N * D * D, sh, lp == 0 ? ex.parts : nullptr);
    if (threadIdx.x == 0) F[p] = Fp;
}

// ---------------------------------------------------------------------------
// D = 1 (DW, OU): time-parallel sweeps, one CTA of SCAN_THREADS threads per problem.
//
// With one thread per problem the sweeps above are a chain of N-1 dependent solver steps (~450 cycles
// each: OU x 1024, N = 1001 took 0.26 + 0.61 ms whatever the batch size).  But both moment ODEs are
// LINEAR in their state -- m' = -A m + b, S' = -2 A S + sigma, lam' and Psi' likewise
// (fwd_ode.py:41-75, bwd_ode.py:45-83) -- so one solver step is an affine map y -> P y + Q of each scalar,
// whatever the solver (the one exception: RK2's forward variance stage, runge_kutta2.py:92, passes S in
// place of A and is quadratic in S; see scan1_fwd_body).  The CTA first stages the problem's
// streams (A, b; backward also m, S, dE/dm, dE/dS) in shared memory with coalesced loads; then each thread
// takes a contiguous run of ~(N-1)/SCAN_THREADS steps and
//   1. finds the (P, Q) of every step of its run by applying THE SOLVER STEP ITSELF (fwd_step / bwd_step,
//      observation jumps included) to the states 0 and 1, and composes them;
//   2. a block scan composes the runs, giving each thread the state at the start of its run;
//   3. the thread walks its run again from that state with the solver step, storing m(t), S(t) (forward)
//      or assembling dL/dA(t), dL/db(t) (backward) exactly as the sequential kernels do.
// The chain is ~2 x 5 steps + the scan instead of 1000 steps, for ~3x the arithmetic.  Only the run-start
// states differ from the sequential kernels (rounding of the composed maps, ~1e-16 relative per step);
// inside a run the arithmetic is the sequential one.
// ---------------------------------------------------------------------------
constexpr int SCAN_MAX_BATCH = 16384;     // the separate sweeps (F only; RK2's backward sweep): above, one thread per problem
                                          // fills the FP64 pipe better.  The fused evaluation (scan1_eval_kernel) has no such
                                          // limit: measured faster than the sequential kernels at every batch size
                                          // (OU rk4 x 65536: 3.21 against 4.51 ms)
constexpr int SCAN_RK2_MAX_BATCH = 8192;  // RK2's forward sweep keeps one serial recurrence per problem (scan1_fwd_body): measured
                                          // against one thread per problem, OU rk2: 1024 problems 0.158 / 0.79 ms, 8192 1.00 / 1.11,
                                          // 16384 1.95 / 1.37, 65536 7.7 / 4.1
constexpr int SCAN_THREADS = 256;         // 128: same throughput, one problem 25 instead of 19 us (longer runs per thread)
// VGPA_SEQUENTIAL_D1=1 in the environment: D = 1 batches take the one-thread-per-problem kernels whatever their size
// (a diagnostic switch: A/B timings, and tests that compare the two kernel families on the same problems)
static bool scan_disabled()
{
    static const bool off = [] { const char* e = getenv("VGPA_SEQUENTIAL_D1"); return e != nullptr && e[0] == '1'; }();
    return off;
}
constexpr size_t SCAN_MAX_SMEM = 200 * 1024;

struct Affine { double P, Q; };           // y -> P y + Q
__device__ __forceinline__ Affine after(const Affine& later, const Affine& earlier)
{
    return {later.P * earlier.P, fma(later.P, earlier.Q, later.Q)};
}
// composition of the maps of threads 0 .. tid-1 (thread 0 first); identity for thread 0.
// sh: SCAN_THREADS / 32 slots.  Contains block barriers.
__device__ __forceinline__ Affine scan_exclusive(Affine f, Affine* sh)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const Affine o{__shfl_up_sync(0xffffffffu, f.P, d), __shfl_up_sync(0xffffffffu, f.Q, d)};
        if (lane >= d) f = after(f, o);
    }
    if (lane == 31) sh[w] = f;
    Affine e{__shfl_up_sync(0xffffffffu, f.P, 1), __shfl_up_sync(0xffffffffu, f.Q, 1)};
    if (lane == 0) e = {1.0, 0.0};
    __syncthreads();
    Affine pre{1.0, 0.0};
    for (int q = 0; q < w; ++q) pre = after(sh[q], pre);
    __syncthreads();
    return after(e, pre);
}
// Steps per thread.  ODD: thread r works on shared-memory doubles r L + j, and with an even L (8 for a grid of
// 1001 points) the 32 lanes of a warp fall on 2 of the 16 double-wide banks -- ncu showed 79 % of the kernel's
// shared-memory wavefronts were bank-conflict replays and the LSU pipe 87 % busy.  With an odd stride the lanes
// of each half-warp hit 16 different banks; a few threads at the end of the CTA stay idle instead.
__device__ __forceinline__ int run_length(int steps)
{
    return ((steps + SCAN_THREADS - 1) / SCAN_THREADS) | 1;
}
__device__ __forceinline__ void stage_array(double* __restrict__ dst, const double* __restrict__ src, int n)
{
    for (int i = threadIdx.x; i < n; i += SCAN_THREADS) dst[i] = __ldg(src + i);
}

// forward sweep of one problem: A, bo in shared memory; mt, st (N each) in shared or global memory.
// coef: 3 N doubles of shared memory, used by RK2 only.  RK2's variance stage passes S in place of A
// (runge_kutta2.py:92), which makes its step a QUADRATIC map S -> a S^2 + b S + c: no scan composes those.  Its
// coefficients still depend on A(t) only, so every thread finds them for its run (the solver step applied to
// S = 0, 1, -1), ONE thread then runs the 2-FMA recurrence over the whole grid (~25 cycles per step instead of the
// solver step's ~300) noting S at the start of every run, and the runs are walked from there as for the other
// solvers.  The mean is affine for every solver.
template <int METHOD>
__device__ __forceinline__ void scan1_fwd_body(const double* A, const double* bo, int N, double sig, double dt,
                                               double m0, double S0, double* mt, double* st, double* coef,
                                               Affine (*sh)[SCAN_THREADS / 32])
{
    __shared__ double run_start[SCAN_THREADS];
    const int tid = threadIdx.x;
    const int steps = N - 1, L = run_length(steps);
    const int k0 = min(tid * L, steps), k1 = min(k0 + L, steps);
    const double zero = 0.0, one = 1.0, minus = -1.0;
    Affine fm{1.0, 0.0}, fS{1.0, 0.0};
    for (int k = k0; k < k1; ++k) {
        double qm, qS, rm, rS;
        fwd_step<1, METHOD>(&zero, &zero, A + k, bo + k, A + k + 1, bo + k + 1, &sig, dt, &qm, &qS);
        fwd_step<1, METHOD>(&one, &one, A + k, bo + k, A + k + 1, bo + k + 1, &sig, dt, &rm, &rS);
        fm = after(Affine{rm - qm, qm}, fm);
        if constexpr (METHOD == ODE_RK2) {
            double um, uS;
            fwd_step<1, METHOD>(&zero, &minus, A + k, bo + k, A + k + 1, bo + k + 1, &sig, dt, &um, &uS);
            coef[3 * k + 0] = 0.5 * (rS + uS) - qS;      // a
            coef[3 * k + 1] = 0.5 * (rS - uS);           // b
            coef[3 * k + 2] = qS;                        // c
        } else {
            fS = after(Affine{rS - qS, qS}, fS);
        }
    }
    const Affine em = scan_exclusive(fm, sh[0]);         // (contains block barriers: coef is visible after it)
    double m = (tid == 0) ? m0 : fma(em.P, m0, em.Q);
    double S;
    if constexpr (METHOD == ODE_RK2) {
        if (tid == 0) {
            double Sq = S0;
            const double* c = coef;
            for (int r = 0, k = 0; k < steps; ++r) {
                run_start[r] = Sq;
                const int ke = min(k + L, steps);
#pragma unroll 4
                for (; k < ke; ++k, c += 3) Sq = fma(fma(c[0], Sq, c[1]), Sq, c[2]);
            }
        }
        __syncthreads();
        S = (k0 < k1) ? run_start[tid] : 0.0;
    } else {
        const Affine eS = scan_exclusive(fS, sh[1]);
        S = (tid == 0) ? S0 : fma(eS.P, S0, eS.Q);
    }
    if (tid == 0) {
        mt[0] = m0;
        st[0] = S0;
    }
    for (int k = k0; k < k1; ++k) {
        double mn, Sn;
        fwd_step<1, METHOD>(&m, &S, A + k, bo + k, A + k + 1, bo + k + 1, &sig, dt, &mn, &Sn);
        mt[k + 1] = mn;
        st[k + 1] = Sn;
        m = mn;
        S = Sn;
    }
}

// backward sweep and gradient of one problem: A, bo, mt, st, dEm, dEs in shared memory; gA, gb in global memory
template <int MODEL, int METHOD>
__device__ __forceinline__ void scan1_bwd_body(const Batch& b, int p, const double* A, const double* bo,
                                               const double* mt, const double* st, const double* dEm,
                                               const double* dEs, double* gA, double* gb,
                                               Affine (*sh)[SCAN_THREADS / 32])
{
    const int tid = threadIdx.x, N = b.N;
    const double* th = b.theta + p * b.theta_stride;
    const double* oy = b.obs_y + p * b.obs_y_stride;
    const int* oidx = obs_index_of(b, p);
    const double isg = 1.0 / b.sigma[p * b.sigma_stride], Rv = b.R[p * b.R_stride];
    const double dt = b.dt, dtm = b.dt_model;
    // step q = 0 .. N-2 takes index t = N-1-q to t-1
    const int steps = N - 1, L = run_length(steps);
    const int q0 = min(tid * L, steps), q1 = min(q0 + L, steps);
    const double zero = 0.0, one = 1.0;

    // jump of lambda and Psi at index t (gaussian_like.py:188,191), as in small_bwd_kernel
    auto jump = [&](int t, double& jm, double& js) {
        const int n = oidx[t];
        jm = 0.0;
        js = 0.0;
        if (n >= 0) {
            jm = -(oy[n] - mt[t]) / Rv;
            js = 0.5 / Rv;
        }
    };
    Affine fl{1.0, 0.0}, fP{1.0, 0.0};
    for (int q = q0; q < q1; ++q) {
        const int t = N - 1 - q;
        double jm, js, ql, qP, rl, rP;
        jump(t - 1, jm, js);
        bwd_step<1, METHOD>(&zero, &zero, A + t, dEm + t, dEs + t, A + t - 1, dEm + t - 1, dEs + t - 1, &jm, dt, &ql, &qP);
        bwd_step<1, METHOD>(&one, &one, A + t, dEm + t, dEs + t, A + t - 1, dEm + t - 1, dEs + t - 1, &jm, dt, &rl, &rP);
        qP += js;
        rP += js;
        fl = after(Affine{rl - ql, ql}, fl);
        fP = after(Affine{rP - qP, qP}, fP);
    }
    const Affine el = scan_exclusive(fl, sh[0]), eP = scan_exclusive(fP, sh[1]);
    double lam = (tid == 0) ? 0.0 : el.Q;      // the terminal state is zero: P * 0 + Q
    double Psi = (tid == 0) ? 0.0 : eP.Q;
    auto grad = [&](int t) {
        double ga, gbv;
        grad_at<MODEL, 1>(th, &isg, dtm, A + t, bo + t, mt + t, st + t, &lam, &Psi, &ga, &gbv);
        gA[t] = ga;
        gb[t] = gbv;
    };
    for (int q = q0; q < q1; ++q) {
        const int t = N - 1 - q;
        grad(t);
        double jm, js, ln, Pn;
        jump(t - 1, jm, js);
        bwd_step<1, METHOD>(&lam, &Psi, A + t, dEm + t, dEs + t, A + t - 1, dEm + t - 1, dEs + t - 1, &jm, dt, &ln, &Pn);
        lam = ln;
        Psi = Pn + js;
    }
    // index 0: the thread that took the last step (thread 0 when the grid has a single point)
    if ((steps == 0) ? (tid == 0) : (q0 < q1 && q1 == steps)) grad(0);
}

template <int METHOD>
__global__ void __launch_bounds__(SCAN_THREADS)
scan1_fwd_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0, int count)
{
    extern __shared__ double scan_sm[];
    __shared__ Affine sh[2][SCAN_THREADS / 32];
    const int lp = blockIdx.x;
    const int p = p0 + lp, N = b.N;
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    double* A = scan_sm;
    stage_array(A, x + (long long)p * xs, 2 * N);          // A then b, contiguous in x
    __syncthreads();
    scan1_fwd_body<METHOD>(A, A + N, N, b.sigma[p * b.sigma_stride], b.dt, b.m0[p * b.m0_stride], b.s0[p * b.s0_stride],
                           s.mt + (long long)lp * N, s.st + (long long)lp * N, A + 2 * N, sh);
}

template <int MODEL, int METHOD>
__global__ void __launch_bounds__(SCAN_THREADS)
scan1_bwd_kernel(Batch b, Scratch s, SmallBwdArgs a, int p0, int count)
{
    extern __shared__ double scan_sm[];
    __shared__ Affine sh[2][SCAN_THREADS / 32];
    const int lp = blockIdx.x;
    const int p = p0 + lp, N = b.N;
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    double* A = scan_sm;
    double* mt = A + 2 * N;
    double* st = mt + N;
    double* dEm = st + N;
    double* dEs = dEm + N;
    stage_array(A, a.x + (long long)p * a.xs, 2 * N);
    stage_array(mt, s.mt + (long long)lp * N, N);
    stage_array(st, s.st + (long long)lp * N, N);
    stage_array(dEm, s.dEm + (long long)lp * N, N);
    stage_array(dEs, s.dEs + (long long)lp * N, N);
    __syncthreads();
    double* gA = a.grad + (long long)p * a.gs;
    scan1_bwd_body<MODEL, METHOD>(b, p, A, A + N, mt, st, dEm, dEs, gA, gA + N, sh);
}

// The whole evaluation of one problem in ONE launch (F and the gradient wanted, no trajectories kept): forward
// sweep, Esde integrand and its derivatives, F, backward sweep and gradient, with m, S, dE/dm, dE/dS and the
// integrand living in shared memory only -- HBM sees x once (16 N bytes) and the gradient once.
template <int MODEL, int METHOD>
__global__ void __launch_bounds__(SCAN_THREADS)
scan1_eval_kernel(Batch b, const double* __restrict__ x, long long xs, double* __restrict__ F,
                  double* __restrict__ grad, long long gs, int p0, int count)
{
    extern __shared__ double scan_sm[];
    __shared__ Affine sh[2][SCAN_THREADS / 32];
    __shared__ double red[SCAN_THREADS];
    const int p = p0 + blockIdx.x, N = b.N, tid = threadIdx.x;
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    double* A = scan_sm;
    double* bo = A + N;
    double* mt = bo + N;
    double* st = mt + N;
    double* dEm = st + N;
    double* dEs = dEm + N;
    double* ft = dEs + N;
    stage_array(A, x + (long long)p * xs, 2 * N);
    const double sig = b.sigma[p * b.sigma_stride], th0 = b.theta[p * b.theta_stride];
    __syncthreads();
    scan1_fwd_body<METHOD>(A, bo, N, sig, b.dt, b.m0[p * b.m0_stride], b.s0[p * b.s0_stride], mt, st, dEm, sh);   // dEm, dEs, ft: free until the energy phase
    __syncthreads();
    for (int t = tid; t < N; t += SCAN_THREADS) energy1<MODEL>(th0, sig, A[t], bo[t], mt[t], st[t], ft[t], dEm[t], dEs[t]);
    __syncthreads();
    const double Fp = free_energy_of(b, p, ft, mt, st, red, nullptr);
    if (tid == 0) F[p] = Fp;
    double* gA = grad + (long long)p * gs;
    scan1_bwd_body<MODEL, METHOD>(b, p, A, bo, mt, st, dEm, dEs, gA, gA + N, sh);
}
// shared memory of the two kernels for a grid of N points; the launchers fall back to the sequential
// kernels when it does not fit
static inline size_t scan_fwd_bytes(int N, int method) { return sizeof(double) * (method == ODE_RK2 ? 5 : 2) * (size_t)N; }
static inline size_t scan_bwd_bytes(int N) { return sizeof(double) * 6 * (size_t)N; }
static inline size_t scan_eval_bytes(int N) { return sizeof(double) * 7 * (size_t)N; }

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
template <int D>
static void fwd_dispatch(const Batch& b, const Scratch& s, const double* x, long long xs, int p0,
                         int count, cudaStream_t st)
{
    if constexpr (D == 1) {
        const size_t sh = scan_fwd_bytes(b.N, b.method);
        if (count <= (b.method == ODE_RK2 ? SCAN_RK2_MAX_BATCH : SCAN_MAX_BATCH) && sh <= SCAN_MAX_SMEM && !scan_disabled()) {
            with_method(b.method, [&](auto m) {
                set_smem(scan1_fwd_kernel<m>, sh);
                scan1_fwd_kernel<m><<<count, SCAN_THREADS, sh, st>>>(b, s, x, xs, p0, count);
            });
            return;
        }
    }
    if (count > PF_MAX_BATCH) {   // large batches: streams staged through shared memory, one warp per CTA
        constexpr int TB = (D == 1) ? 16 : 8;
        const size_t sh = fwd_stage_bytes<D, TB>();
        const int bl = (count + 31) / 32;
        with_method(b.method, [&](auto m) {
            set_smem(small_fwd_staged_kernel<D, m, TB>, sh);
            small_fwd_staged_kernel<D, m, TB><<<bl, 32, sh, st>>>(b, s, x, xs, p0, count);
        });
        return;
    }
    // one thread per problem: small CTAs spread a small batch over more SMs (more load streams in flight)
    const int th = (count <= 148 * 64) ? 32 : 64, bl = (count + th - 1) / th;
    with_method(b.method, [&](auto m) { small_fwd_kernel<D, m><<<bl, th, 0, st>>>(b, s, x, xs, p0, count); });
}
void launch_small_fwd(const Batch& b, const Scratch& s, const double* x, long long xs, int p0,
                      int count, cudaStream_t st)
{
    if (b.D == 1) fwd_dispatch<1>(b, s, x, xs, p0, count, st);
    else if (l63_lanes_applies(b, count)) launch_l63_fwd_lanes(b, s, x, xs, p0, count, st);
    else          fwd_dispatch<3>(b, s, x, xs, p0, count, st);
}

// D = 1, F and gradient, nothing kept: one launch per pass.  False: not applicable (the caller runs the phases).
bool launch_small_fused(const Batch& b, const double* x, long long xs, double* F, double* g, long long gs,
                        int p0, int count, const Extra& ex, cudaStream_t st)
{
    const size_t sh = scan_eval_bytes(b.N);
    if (b.D != 1 || g == nullptr || sh > SCAN_MAX_SMEM || scan_disabled() ||
        (b.method == ODE_RK2 && count > SCAN_RK2_MAX_BATCH) ||
        ex.lamt != nullptr || ex.Efx != nullptr || ex.parts != nullptr)
        return false;
    with_method(b.method, [&](auto m) {
        const auto kernel = (b.model == MODEL_DW) ? scan1_eval_kernel<MODEL_DW, m> : scan1_eval_kernel<MODEL_OU, m>;
        set_smem(kernel, sh);
        kernel<<<count, SCAN_THREADS, sh, st>>>(b, x, xs, F, g, gs, p0, count);
    });
    return true;
}

void launch_small_energy(const Batch& b, const Scratch& s, const double* x, long long xs, int p0,
                         int count, const Extra& ex, cudaStream_t st)
{
    const long long tot = (long long)count * b.N;
    const int th = 128;
    const unsigned bl = (unsigned)((tot + th - 1) / th);
    if (b.model == MODEL_DW)      small_energy_kernel<MODEL_DW, 1><<<bl, th, 0, st>>>(b, s, x, xs, p0, count, ex);
    else if (b.model == MODEL_OU) small_energy_kernel<MODEL_OU, 1><<<bl, th, 0, st>>>(b, s, x, xs, p0, count, ex);
    else                          small_energy_kernel<MODEL_L63, 3><<<bl, th, 0, st>>>(b, s, x, xs, p0, count, ex);
}

template <int MODEL, int D>
static void bwd_dispatch(const Batch& b, const Scratch& s, const SmallBwdArgs& a, int p0, int count,
                         const Extra& ex, cudaStream_t st)
{
    if constexpr (D == 1) {
        const size_t sh = scan_bwd_bytes(b.N);
        if (a.grad != nullptr && a.jm_dense == nullptr && ex.lamt == nullptr && count <= SCAN_MAX_BATCH &&
            sh <= SCAN_MAX_SMEM && !scan_disabled()) {   // time-parallel
            with_method(b.method, [&](auto m) {
                set_smem(scan1_bwd_kernel<MODEL, m>, sh);
                scan1_bwd_kernel<MODEL, m><<<count, SCAN_THREADS, sh, st>>>(b, s, a, p0, count);
            });
            return;
        }
    }
    const int th = (count <= 148 * 64) ? 32 : 64, bl = (count + th - 1) / th;
    with_method(b.method, [&](auto m) { small_bwd_kernel<MODEL, D, m><<<bl, th, 0, st>>>(b, s, a, p0, count, ex); });
}
void launch_small_bwd(const Batch& b, const Scratch& s, const double* x, long long xs, double* g,
                      long long gs, int p0, int count, const Extra& ex, cudaStream_t st)
{
    SmallBwdArgs a{x, xs, g, gs, nullptr, nullptr};
    if (g != nullptr && ex.lamt == nullptr && l63_lanes_applies(b, count)) {
        launch_l63_bwd_lanes(b, s, x, xs, g, gs, p0, count, st);
        return;
    }
    if (b.model == MODEL_DW)      bwd_dispatch<MODEL_DW, 1>(b, s, a, p0, count, ex, st);
    else if (b.model == MODEL_OU) bwd_dispatch<MODEL_OU, 1>(b, s, a, p0, count, ex, st);
    else                          bwd_dispatch<MODEL_L63, 3>(b, s, a, p0, count, ex, st);
}

// Stand-alone backward sweep with dense jump tables, any supported D.
void launch_bwd_dense_l96(int method, int N, double dt, const double* A, const double* dEm,
                          const double* dEs, const double* jm, const double* js, double* lam,
                          double* psi, cudaStream_t st);
void launch_bwd_dense(int method, int D, int N, double dt, const double* A, const double* dEm,
                      const double* dEs, const double* jm, const double* js, double* lam,
                      double* psi, cudaStream_t st)
{
    if (D == 40) {
        launch_bwd_dense_l96(method, N, dt, A, dEm, dEs, jm, js, lam, psi, st);
        return;
    }
    if (D != 1 && D != 3) {   // Lorenz 96 at any other D
        launch_bwd_dense_l96d(method, D, N, dt, A, dEm, dEs, jm, js, lam, psi, st);
        return;
    }
    Batch b{};
    b.model = (D == 1) ? MODEL_OU : MODEL_L63;
    b.method = method; b.D = D; b.N = N; b.B = 1; b.dt = dt; b.dt_model = dt;
    Scratch s{};
    s.dEm = const_cast<double*>(dEm);
    s.dEs = const_cast<double*>(dEs);
    SmallBwdArgs a{A, 0, nullptr, 0, jm, js};
    Extra ex{};
    ex.lamt = lam; ex.psit = psi;
    if (D == 1) bwd_dispatch<MODEL_OU, 1>(b, s, a, 0, 1, ex, st);
    else        bwd_dispatch<MODEL_L63, 3>(b, s, a, 0, 1, ex, st);
}

// gaussian_like.py:188,191 (1-D) / :235,238 (n-D, diagonal R): -H^T R^-1 (y - H m) and 1/2 H^T R^-1 H for H the
// rows of the identity at the components set in `observed`; the other entries keep the launcher's zeros.
__global__ void jump_tables_kernel(int D, int N, int M, const long long* __restrict__ obs_t,
                                   const double* __restrict__ obs_y, const double* __restrict__ R,
                                   unsigned long long observed, const double* __restrict__ mt, double* __restrict__ jm,
                                   double* __restrict__ js)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= M * D) return;
    const int n = q / D, i = q % D;
    if (!((observed >> i) & 1ull)) return;
    const long long t = obs_t[n];
    jm[t * D + i] = -(obs_y[(long long)n * D + i] - mt[t * D + i]) / R[i];
    js[t * D * D + (long long)i * D + i] = 0.5 / R[i];
}
void launch_jump_tables(int D, int N, int M, const long long* obs_t, const double* obs_y, const double* R,
                        unsigned long long observed, const double* mt, double* jm, double* js, cudaStream_t st)
{
    cudaMemsetAsync(jm, 0, sizeof(double) * (size_t)N * D, st);
    cudaMemsetAsync(js, 0, sizeof(double) * (size_t)N * D * D, st);
    if (M > 0) jump_tables_kernel<<<(M * D + 127) / 128, 128, 0, st>>>(D, N, M, obs_t, obs_y, R, observed, mt, jm, js);
}

void launch_finalize(const Batch& b, const Scratch& s, double* F, int p0, int count, const Extra& ex,
                     cudaStream_t st)
{
    finalize_kernel<<<count, 128, 0, st>>>(b, s, F, p0, count, ex);
}

}  // namespace vgpa
