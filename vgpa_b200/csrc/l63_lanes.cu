// l63_lanes.cu -- Lorenz-63 (D = 3) forward and backward sweeps with SEVERAL LANES PER PROBLEM.
//
// One thread per problem (small_dim.cu) makes a warp issue ~200 dependent-ish FP64 instructions and
// ~24 fully divergent memory instructions per time index: a single problem takes 835 cycles per
// index in the forward and 2 100 in the backward sweep, and a batch of a few thousand problems
// (BASELINE configs[2]: 4096) puts one such warp on each SM.  Here a problem owns a group of 16
// lanes, lane (i, j) = (e >> 2, e & 3) of the group holding ONE entry of the 3 x 4 state
// [S | m] (forward) or [Psi | lam] (backward): column j < 3 is the matrix, column 3 the vector
// (row i = 3 of the group idles).  A right-hand-side evaluation is then three FMAs per lane, the
// operands a lane does not own arrive by width-16 shuffles, the matrices A(t) are read straight
// from global memory (every lane its row or columns: the loads of a group coalesce into a few
// sectors), and a batch of B problems runs on B / 2 warps -- all sub-partitions of the GPU for a
// few thousand problems.
//
// The arithmetic is the reference's (src/numerics/{euler,heun,runge_kutta2,runge_kutta4}.py,
// ode_solver.py:31-95, variational.py:202-334) in EXACTLY the operation order of small_dim.cu
// (fun_m / fun_S / fun_lam / fun_psi / fwd_step / bwd_step / grad_at), so a problem's results do not
// depend on which of the kernels served it (the batch-position tests compare them bit for bit).
#include "common.cuh"
#include "l63_grad.cuh"

namespace vgpa {
namespace {

constexpr int D = 3, DD = 9;
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double shfl16(double v, int src) { return __shfl_sync(FULL, v, src, 16); }

// A group walks a handful of private streams (A, b; in the backward sweep also m, S, dE/dm, dE/dS) one
// time index per step, and the step itself is short (~250 cycles): loading an index two steps ahead
// into registers, as the one-thread-per-problem kernels do, leaves every step waiting for DRAM (measured:
// 610 cycles per step for one problem).  So each warp stages its two problems' streams through shared
// memory in blocks of TB time indices with cp.async (8-byte copies: the streams are only 8-byte aligned),
// double buffered: block n + 1 is in flight while block n is consumed.  No CTA barrier: a CTA is one warp.
constexpr int TB = 8;             // time indices per block
constexpr int NI = TB + 1;        // ... plus the neighbour index the last step of a block reads

__device__ __forceinline__ void cp_async8(double* dst_smem, const double* src_gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst_smem)), "l"(src_gmem)
                 : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_wait()
{
    asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory");
    __syncwarp();
}
// `len` contiguous doubles g[0 .. len) -> dst[0 .. len), by the 16 lanes of a group
__device__ __forceinline__ void stage_span(double* dst, const double* __restrict__ g, int len, int e)
{
    for (int c = e; c < len; c += 16) cp_async8(dst + c, g + c);
}

// ---------------------------------------------------------------------------
// forward:  o = fun_m / fun_S of the 3 x 4 state X = [S | m] held one entry per lane
//   L[k]   : row i of the LEFT operand (A, or S itself in the inner covariance stage of RK2,
//            runge_kutta2.py:96 -- passed in by the caller)
//   column j of X arrives by shuffles from lanes (k, j)
//   j < 3 :  o_ij = -p_ij - q_ij + sigma_i delta_ij,  p = L X,  q_ij = p_ji (S is exactly symmetric in
//            small_dim.cu's fun_S too: q_ij there is the same products in the same order)
//   j = 3 :  o_i = -(L m)_i + b_i
// ---------------------------------------------------------------------------
__device__ __forceinline__ double fwd_fun(double X, const double (&L)[3], double sig_d, double bi, int i, int j)
{
    double p = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) p += L[k] * shfl16(X, 4 * k + j);
    const double q = shfl16(p, 4 * (j & 3) + i);     // p_ji (lanes of the vector column read an idle lane: unused)
    return (j < 3) ? (-p - q + sig_d) : (-p + bi);
}

// shared memory of one warp: [buffer][group][A: NI x 9 | b: NI x 3]
constexpr int FWD_PROB = NI * (DD + D);

template <int METHOD>
__global__ void __launch_bounds__(32)
l63_fwd_lanes_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0, int count)
{
    __shared__ double smem[2][2][FWD_PROB];
    const int lane = threadIdx.x, grp = lane >> 4, e = lane & 15, i = min(e >> 2, 2), j = e & 3;
    const bool live = (e >> 2) < 3;                                   // row 3 of the group idles
    const int lp_raw = 2 * (int)blockIdx.x + grp;
    const bool has = lp_raw < count;
    const int lp = has ? lp_raw : count - 1, p = p0 + lp, N = b.N;    // a padding group redoes the last problem, stores nothing
    const bool on = has && live && (b.active == nullptr || b.active[p] != 0);
    const double* A = x + (long long)p * xs;
    const double* bo = A + (long long)N * DD;
    double* mt = s.mt + (long long)lp * N * D;
    double* st = s.st + (long long)lp * N * DD;
    const double sig_d = (i == j) ? b.sigma[p * b.sigma_stride + i] : 0.0;
    double X = (j < 3) ? b.s0[p * b.s0_stride + 3 * i + j] : b.m0[p * b.m0_stride + i];
    double* out = (j < 3) ? st + 3 * i + j : mt + i;                  // my entry of index 0
    const int ostride = (j < 3) ? DD : D;
    if (on) out[0] = X;
    const double dt = b.dt, h = 0.5 * dt;
    (void)h;
    // block n covers steps t0 = n TB .. t0 + nb - 1 and reads indices t0 .. t0 + nb
    auto issue = [&](int n) {
        const int t0 = n * TB;
        if (t0 < N - 1) {
            const int ni = min(TB, N - 1 - t0) + 1;
            double* buf = smem[n & 1][grp];
            stage_span(buf, A + (long long)t0 * DD, ni * DD, e);
            stage_span(buf + NI * DD, bo + (long long)t0 * D, ni * D, e);
        }
        cp_commit();
    };
    issue(0);
    const int nblocks = (N - 1 + TB - 1) / TB;
    for (int n = 0; n < nblocks; ++n) {
        issue(n + 1);
        cp_wait<1>();                                                 // block n has landed (block n + 1 may be in flight)
        const double* sA = smem[n & 1][grp] + 3 * i;
        const double* sB = smem[n & 1][grp] + NI * DD + i;
        const int t0 = n * TB, nb = min(TB, N - 1 - t0);
        for (int tt = 0; tt < nb; ++tt) {
            double Ak[3], An[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                Ak[k] = sA[tt * DD + k];
                An[k] = sA[(tt + 1) * DD + k];
            }
            const double bk = sB[tt * D], bn = sB[(tt + 1) * D];
            double Xn;
            if (METHOD == ODE_EULER) {                  // euler.py:84-87
                const double o1 = fwd_fun(X, Ak, sig_d, bk, i, j);
                Xn = X + dt * o1;
            } else if (METHOD == ODE_HEUN) {            // heun.py:91-106
                const double o1 = fwd_fun(X, Ak, sig_d, bk, i, j);
                const double tmp = X + dt * o1;
                const double o2 = fwd_fun(tmp, An, sig_d, bn, i, j);
                Xn = X + h * (o1 + o2);
            } else if (METHOD == ODE_RK2) {             // runge_kutta2.py:92,96 (inner covariance stage: S in place of A)
                double am[3], L1[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) am[k] = 0.5 * (Ak[k] + An[k]);
                const double bm = 0.5 * (bk + bn);
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double sik = shfl16(X, 4 * i + k);          // row i of S
                    L1[k] = (j < 3) ? sik : Ak[k];
                }
                const double o1 = fwd_fun(X, L1, sig_d, bk, i, j);
                const double tmp = X + h * o1;
                const double o2 = fwd_fun(tmp, am, sig_d, bm, i, j);
                Xn = X + dt * o2;
            } else {                                    // runge_kutta4.py:93-108
                double am[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) am[k] = 0.5 * (Ak[k] + An[k]);
                const double bm = 0.5 * (bk + bn);
                const double o1 = fwd_fun(X, Ak, sig_d, bk, i, j);
                double tmp = X + h * o1;
                const double o2 = fwd_fun(tmp, am, sig_d, bm, i, j);
                tmp = X + h * o2;
                const double o3 = fwd_fun(tmp, am, sig_d, bm, i, j);
                tmp = X + dt * o3;
                const double o4 = fwd_fun(tmp, An, sig_d, bn, i, j);
                Xn = X + dt * (o1 + 2.0 * (o2 + o3) + o4) / 6.0;
            }
            X = Xn;
            if (on) out[(long long)(t0 + tt + 1) * ostride] = X;
        }
        __syncwarp();                                                 // the buffer is refilled by the next issue
    }
}

// ---------------------------------------------------------------------------
// backward:  o = fun_lam / fun_psi of Y = [Psi | lam]
//   j < 3 :  o_ij = -G_ij + p + q,  p = sum_k Psi_ik A_kj,  q = sum_k A_ki Psi_kj
//            (q is formed explicitly: small_dim.cu does, and Psi is symmetric only up to rounding)
//   j = 3 :  o_i = -g_i + sum_k A_ik lam_k
//   V1[k] : A_kj (column j of A) for j < 3, A_ik (row i) for j = 3;  V2[k] : A_ki (column i of A)
// ---------------------------------------------------------------------------
struct AOps {
    double V1[3], V2[3];
};
__device__ __forceinline__ void mid_aops(AOps& o, const AOps& lo, const AOps& hi)     // mid(Am, At) = 0.5 (Am + At)
{
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        o.V1[k] = 0.5 * (lo.V1[k] + hi.V1[k]);
        o.V2[k] = 0.5 * (lo.V2[k] + hi.V2[k]);
    }
}
// row i of Psi (lanes of the vector column: lam) as every lane needs it for the left products
__device__ __forceinline__ void row_of(double Y, int i, int j, double (&ya)[3])
{
#pragma unroll
    for (int k = 0; k < 3; ++k) ya[k] = shfl16(Y, (j < 3) ? 4 * i + k : 4 * k + 3);   // Psi_ik, or lam_k
}
__device__ __forceinline__ double bwd_fun(const double (&ya)[3], double Y, const AOps& a, double G, int j)
{
    double p = 0.0, q = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double yb = shfl16(Y, 4 * k + j);                         // Psi_kj
        p += ya[k] * a.V1[k];
        q += a.V2[k] * yb;
    }
    return (j < 3) ? (-G + p + q) : (-G + p);
}
__device__ __forceinline__ double bwd_fun(double Y, const AOps& a, double G, int i, int j)
{
    double ya[3];
    row_of(Y, i, j, ya);
    return bwd_fun(ya, Y, a, G, j);
}

// shared memory of one warp: [buffer][group][A | S | dE/dS : NI x 9 each | b | m | dE/dm : NI x 3 each];
// a block holds the contiguous index range [lo, top] of every stream, ascending (slot = index - lo)
constexpr int BWD_PROB = NI * (3 * DD + 3 * D);

template <int METHOD>
__global__ void __launch_bounds__(32)
l63_bwd_lanes_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, double* __restrict__ grad,
                     long long gs, int p0, int count)
{
    __shared__ double smem[2][2][BWD_PROB];
    const int lane = threadIdx.x, grp = lane >> 4, e = lane & 15, i = min(e >> 2, 2), j = e & 3, jc = (j < 3) ? j : 0;
    const bool live = (e >> 2) < 3;
    const int lp_raw = 2 * (int)blockIdx.x + grp;
    const bool has = lp_raw < count;
    const int lp = has ? lp_raw : count - 1, p = p0 + lp, N = b.N;
    const bool on = has && live && (b.active == nullptr || b.active[p] != 0);
    const double* A = x + (long long)p * xs;
    const double* bo = A + (long long)N * DD;
    double* gA = grad + (long long)p * gs;
    double* gb = gA + (long long)N * DD;
    const double* mt = s.mt + (long long)lp * N * D;
    const double* st = s.st + (long long)lp * N * DD;
    const double* dEm = s.dEm + (long long)lp * N * D;
    const double* dEs = s.dEs + (long long)lp * N * DD;
    const double* th = b.theta + p * b.theta_stride;
    const double* oy = b.obs_y + p * b.obs_y_stride;
    const int* oidx = obs_index_of(b, p);
    const double vS = th[0], vR = th[1], vB = th[2];
    const double isg_i = 1.0 / b.sigma[p * b.sigma_stride + i];
    const double Rv_i = b.R[p * b.R_stride + i];
    const double dt = b.dt, h = 0.5 * dt, dtm = b.dt_model;
    (void)h;
    double Y = 0.0;                                   // Psi_ij, or lam_i
    double* gdst = (j < 3) ? gA + 3 * i + j : gb + i;
    const int gstride = (j < 3) ? DD : D;
    const int sx = (i == 1) ? 6 : 3;                  // the entry of S the drift moment of row i reads (lorenz_63.py:319-326)
    // block n covers steps t = top .. top - nb + 1 (top = N - 1 - n TB) and reads indices top .. top - nb
    // (the index below the last step, clamped at 0); the streams run DOWNWARDS in time, so a block is the
    // contiguous range [lo, top] of every stream, stored so that slot u = top - index
    auto issue = [&](int n) {
        const int top = N - 1 - n * TB;
        if (top >= 0) {
            const int lo = max(top - TB, 0), ni = top - lo + 1;
            double* buf = smem[n & 1][grp];
            // stored ascending: slot of index idx = idx - lo
            stage_span(buf, A + (long long)lo * DD, ni * DD, e);
            stage_span(buf + NI * DD, st + (long long)lo * DD, ni * DD, e);
            stage_span(buf + 2 * NI * DD, dEs + (long long)lo * DD, ni * DD, e);
            stage_span(buf + 3 * NI * DD, bo + (long long)lo * D, ni * D, e);
            stage_span(buf + 3 * NI * DD + NI * D, mt + (long long)lo * D, ni * D, e);
            stage_span(buf + 3 * NI * DD + 2 * NI * D, dEm + (long long)lo * D, ni * D, e);
        }
        cp_commit();
    };
    issue(0);
    const int nblocks = (N + TB - 1) / TB;            // steps t = N - 1 .. 0 (the step at t = 0 only forms its gradient)
    for (int n = 0; n < nblocks; ++n) {
        issue(n + 1);
        cp_wait<1>();
        const int top = N - 1 - n * TB, lo = max(top - TB, 0);
        const double* sA = smem[n & 1][grp];
        const double* sS = sA + NI * DD;
        const double* sG = sA + 2 * NI * DD;
        const double* sb = sA + 3 * NI * DD;
        const double* sm = sb + NI * D;
        const double* sg = sb + 2 * NI * D;
        const int tend = max(top - TB + 1, 0);
        // operands of A and my entry of dE/dS (dE/dm) at index t: loaded at the top of a block, then handed down
        // from step to step (index t - 1 of one step is index t of the next)
        AOps at;
        double Gt;
        {
            const int u0 = top - lo;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                at.V1[k] = sA[u0 * DD + ((j < 3) ? 3 * k + j : 3 * i + k)];
                at.V2[k] = sA[u0 * DD + 3 * k + i];
            }
            Gt = (j < 3) ? sG[u0 * DD + 3 * i + j] : sg[u0 * D + i];
        }
        for (int t = top; t >= tend; --t) {
            const int u = t - lo, up = (t >= 1) ? u - 1 : u;           // slots of index t and t - 1
            double ya[3];
            row_of(Y, i, j, ya);                                       // shared by the gradient and the first stage
            // ---- gradient at index t (variational.py:280-334; grad_at of small_dim.cu) ----
            {
                double Ar[3], m[3], Sc[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    Ar[k] = sA[u * DD + 3 * i + k];
                    m[k] = sm[u * D + k];
                    Sc[k] = sS[u * DD + 3 * k + jc];
                }
                const double Sx = sS[u * DD + sx], bt = sb[u * D + i];
                const double lam_i = shfl16(Y, 4 * i + 3);
                const L63Row r = l63_row_terms(i, vS, vR, vB, m, Sx, Ar, bt, isg_i);
                const double mj = (j == 1) ? m[1] : (j == 2 ? m[2] : m[0]);      // (selects: no dynamic register indexing)
                const double ga = l63_grad_a(r, Sc, ya, mj, lam_i, dtm);          // (ya = row i of Psi for the matrix lanes)
                const double gbv = l63_grad_b(r, lam_i, dtm);
                if (on) gdst[(long long)t * gstride] = (j < 3) ? ga : gbv;
            }
            if (t == 0) break;
            // jump at index t-1 (gaussian_like.py:188,191 / :235,238); H = I, R diagonal
            double jmv = 0.0, jsv = 0.0;
            {
                const int no = oidx[t - 1];
                if (no >= 0) {
                    jmv = -(oy[(long long)no * D + i] - sm[up * D + i]) / Rv_i;
                    jsv = 0.5 / Rv_i;
                }
            }
            // ... and at index t - 1
            AOps am1;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                am1.V1[k] = sA[up * DD + ((j < 3) ? 3 * k + j : 3 * i + k)];
                am1.V2[k] = sA[up * DD + 3 * k + i];
            }
            const double Gm = (j < 3) ? sG[up * DD + 3 * i + j] : sg[up * D + i];
            double Yn;
            if (METHOD == ODE_EULER) {                  // euler.py:146-149
                const double o1 = bwd_fun(ya, Y, at, Gt, j);
                Yn = (j < 3) ? (Y - o1 * dt) : (Y - o1 * dt + jmv);
            } else if (METHOD == ODE_HEUN) {            // heun.py:170-185
                const double o1 = bwd_fun(ya, Y, at, Gt, j);
                const double tmp = Y + (-dt) * o1;
                const double o2 = bwd_fun(tmp, am1, Gm, i, j);
                Yn = (j < 3) ? (Y - h * (o1 + o2)) : (Y - h * (o1 + o2) + jmv);
            } else if (METHOD == ODE_RK2) {             // runge_kutta2.py:180-189
                AOps amid;
                mid_aops(amid, am1, at);
                const double Gmid = 0.5 * (Gm + Gt);
                const double o1 = bwd_fun(ya, Y, at, Gt, j);
                const double tmp = Y + (-h) * o1;
                const double o2 = bwd_fun(tmp, amid, Gmid, i, j);
                Yn = (j < 3) ? (Y - dt * o2) : (Y - dt * o2 + jmv);
            } else {                                    // runge_kutta4.py:191-206
                AOps amid;
                mid_aops(amid, am1, at);
                const double Gmid = 0.5 * (Gm + Gt);
                const double o1 = bwd_fun(ya, Y, at, Gt, j);
                double tmp = Y + (-h) * o1;
                const double o2 = bwd_fun(tmp, amid, Gmid, i, j);
                tmp = Y + (-h) * o2;
                const double o3 = bwd_fun(tmp, amid, Gmid, i, j);
                tmp = Y + (-dt) * o3;
                const double o4 = bwd_fun(tmp, am1, Gm, i, j);
                const double inc = dt * (o1 + 2.0 * (o2 + o3) + o4) / 6.0;
                Yn = (j < 3) ? (Y - inc) : (Y - inc + jmv);
            }
            if (i == j) Yn += jsv;
            Y = Yn;
            at = am1;
            Gt = Gm;
        }
        __syncwarp();                                                 // the buffer is refilled by the next issue
    }
}

}  // namespace

// number of problems up to which the lane-parallel kernels serve a Lorenz-63 batch (beyond it the batch
// fills the GPU with one thread per problem and the staged sweeps of small_dim.cu move fewer bytes per lane)
constexpr int L63_LANES_MAX = 8192;

bool l63_lanes_applies(const Batch& b, int count) { return b.model == MODEL_L63 && count <= L63_LANES_MAX; }

void launch_l63_fwd_lanes(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                          cudaStream_t st)
{
    const int th = 32, bl = (count + 1) / 2;     // one warp = one CTA = two problems
    with_method(b.method, [&](auto m) { l63_fwd_lanes_kernel<m><<<bl, th, 0, st>>>(b, s, x, xs, p0, count); });
}

void launch_l63_bwd_lanes(const Batch& b, const Scratch& s, const double* x, long long xs, double* grad, long long gs,
                          int p0, int count, cudaStream_t st)
{
    const int th = 32, bl = (count + 1) / 2;
    with_method(b.method, [&](auto m) { l63_bwd_lanes_kernel<m><<<bl, th, 0, st>>>(b, s, x, xs, grad, gs, p0, count); });
}

}  // namespace vgpa
