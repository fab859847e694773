// l96_sweeps.cu -- D = 40 forward and backward ODE sweeps, one CTA per inference
// problem, the whole sequential time loop on chip.
//
//   forward  : m' = -A m + b,  S' = -A S - S A^T + Sigma          (ode_solver.py:31-61)
//   backward : lam' = -dE/dm + A lam,  Psi' = -dE/dS + Psi A + A^T Psi  (:63-95)
//              with the observation jumps at obs_t (gaussian_like.py:200-243)
//              FUSED with the gradient assembly of VarGP.gradient
//              (variational.py:202-334): dL/dA[t], dL/db[t] are formed as soon
//              as lam[t], Psi[t] exist, so lam/Psi never travel to HBM.
//   solver tableaux exactly as src/numerics/{euler,heun,runge_kutta2,runge_kutta4}.py
//   (including runge_kutta2.py:96, where S stands in for A in the inner stage).
//
// CTA = 160 threads = 5 warps; warp w owns rows 8w..8w+7 of every matrix AND vector:
//   * its 8 x 40 tile-row of each 40 x 40 product runs on the FP64 tensor cores
//     (mma.sync m8n8k4 f64, SASS DMMA): per k-step one A fragment and five B fragments
//     from shared memory (skewed layout of common.cuh, sm_idx: conflict-free for the fragment
//     loads, the 16-byte accumulator accesses and the transposed reads) feed five DMMAs;
//     accumulators stay in registers;
//   * the mean / lambda recurrences (40 x 40 mat-vecs) ride in the same k-loop: the A
//     fragment already in registers times the vector entry, reduced over the four
//     lanes of a fragment row with two shuffles;
//   * operands that only their owner warp needs never touch shared memory: A(t) in the
//     forward sweep (left operand: fragments straight from global memory into registers)
//     and Psi in the backward sweep (registers, turned into fragments with shuffles);
//   * what every warp must see -- A(t), S(t) in the backward sweep -- arrives by 1-D bulk
//     async copies (TMA unit, SASS UBLKCP), eight 320-byte rows per warp, completing on
//     mbarriers one or two stages ahead of use.  (Explicit L2 prefetching further ahead
//     was measured and removed: with 444 CTAs streaming, prefetched lines were evicted
//     before use and DRAM traffic rose 60 % above the algorithmic bytes.)
// Symmetry: S and Psi are kept EXACTLY symmetric by forming P + P^T through a
// shared-memory transpose, so one product per RHS evaluation suffices.
#include "common.cuh"
#include "ptx.cuh"

namespace vgpa {
namespace {

constexpr int D = 40;
constexpr int MAT = SM_MAT;    // one matrix in the skewed layout of common.cuh (sm_idx): fragment loads,
                               // accumulator-layout 16-byte accesses and transposed reads all conflict-free
constexpr int ROWB = D * 8;    // bytes of one matrix row in HBM
constexpr int NMMA = 5;        // MMA warps = tile rows
constexpr int NTH = 32 * NMMA;

constexpr int SMALL_LAUNCH = 148;   // launches of at most one CTA per SM prefetch their streams into L2
constexpr int PF_STEPS = 4;         // ... this many time indices ahead

enum { K_CUR = 0, K_MID = 1, K_NEXT = 2 };

__host__ __device__ constexpr int n_stages(int m) { return m == ODE_EULER ? 1 : (m == ODE_RK4 ? 4 : 2); }
// which A (b / dE) a stage reads: the current index, the neighbour, their midpoint
__host__ __device__ constexpr int stage_kind(int m, int s)
{
    return m == ODE_EULER ? K_CUR
         : m == ODE_HEUN  ? (s == 0 ? K_CUR : K_NEXT)
         : m == ODE_RK2   ? (s == 0 ? K_CUR : K_MID)
                          : (s == 0 ? K_CUR : (s == 3 ? K_NEXT : K_MID));
}
// next stage operand = Y +/- next_coef * dt * k_s
__host__ __device__ constexpr double next_coef(int m, int s)
{
    return m == ODE_HEUN ? 1.0 : m == ODE_RK2 ? 0.5 : (s < 2 ? 0.5 : 1.0);
}
// weight of k_s in the final combination
__host__ __device__ constexpr double ksum_w(int m, int s)
{
    return m == ODE_RK2 ? (s == 0 ? 0.0 : 1.0) : m == ODE_RK4 ? ((s == 1 || s == 2) ? 2.0 : 1.0) : 1.0;
}
// Y_new = Y +/- final_step(ksum)
template <int METHOD>
__device__ __forceinline__ double final_step(double dt, double ksum)
{
    if (METHOD == ODE_HEUN) return (0.5 * dt) * ksum;
    if (METHOD == ODE_RK4) return dt * ksum / 6.0;
    return dt * ksum;
}

// D(8x8) += A(8x4) B(4x8) on the FP64 tensor cores.  Lane l = 4 g + q holds
// a = A[g][q], b = B[q][g], c0 = C[g][2q], c1 = C[g][2q+1].
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b)
{
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b));
}

// accumulator tile-row -> shared memory (each lane: two adjacent doubles per tile)
__device__ __forceinline__ void row_to_smem(double* __restrict__ T, int irow, int q, const double (&acc)[5][2])
{
#pragma unroll
    for (int J = 0; J < 5; ++J)
        *reinterpret_cast<double2*>(&T[sm_idx(irow, 8 * J + 2 * q)]) = make_double2(acc[J][0], acc[J][1]);
}

template <int KIND>
__device__ __forceinline__ double pick(double c, double n)
{
    return KIND == K_CUR ? c : (KIND == K_NEXT ? n : 0.5 * (c + n));
}

// every warp issues the bulk copies of its own 8 rows of a 40 x 40 matrix: the two rows of a row PAIR are
// contiguous in the skewed layout (sm_idx: offsets 0 and 40 of an 84-double group) as they are in HBM, so
// four 640-byte copies do (the bulk-copy instruction is what costs: eight 320-byte copies per warp and
// matrix were 9 % of the backward sweep's issued instructions)
__device__ __forceinline__ void load_rows(double* dst, const double* src, uint64_t* bar, int w, int lane)
{
    if (lane < 4) bulk_g2s(dst + sm_idx(8 * w + 2 * lane, 0), src + (8 * w + 2 * lane) * D, 2 * ROWB, bar);
}

// ===========================================================================
// forward sweep
// ===========================================================================
// In  P = A S  the drift matrix A is the LEFT operand, so a warp only ever needs its
// OWN eight rows of A(t) -- as DMMA A fragments and for the mean mat-vec.  A therefore
// never touches shared memory: each lane loads its ten fragment entries of A(t+1)
// straight from global memory (eight 32-byte row segments per warp instruction) at the
// top of step t -- a stage before their first use -- and keeps A(t), A(t+1) in registers.  Shared memory holds only S, the stage operand and the
// transpose exchange (42 KB), so four CTAs share an SM.
struct FwdSmem {
    double Sb[MAT], Hb[MAT];
    double Tb[MAT];
    double mv[D], vt[2][D], sig[D];
};

// tile-row product with the left operand in registers (fragment layout):
//   LK 0: a = A0[n]   LK 1: a = 0.5 (A0[n] + A1[n])
template <int LK>
__device__ __forceinline__ void mma_rowa(const double (&A0)[D / 4], const double (&A1)[D / 4],
                                         const double* __restrict__ X, const double* __restrict__ v, int g,
                                         int q, double (&acc)[5][2], double& yv)
{
#pragma unroll
    for (int J = 0; J < 5; ++J) acc[J][0] = acc[J][1] = 0.0;
    double y = 0.0;
    const int lb = sm_boff(q, g);
#pragma unroll
    for (int n = 0; n < D / 4; ++n) {
        const int k0 = 4 * n;
        const double a = LK == 0 ? A0[n] : 0.5 * (A0[n] + A1[n]);
        y = fma(a, v[k0 + q], y);
        double b[5];
#pragma unroll
        for (int J = 0; J < 5; ++J) b[J] = X[lb + (n >> 1) * SM_R8 + (n & 1) * SM_BH + 8 * J];
#pragma unroll
        for (int J = 0; J < 5; ++J) dmma(acc[J][0], acc[J][1], a, b[J]);
    }
    y += __shfl_xor_sync(0xffffffffu, y, 1);
    y += __shfl_xor_sync(0xffffffffu, y, 2);
    yv = y;
}

// RK2's inner covariance stage multiplies S by itself (runge_kutta2.py:96).  With S exactly symmetric the
// product is symmetric bit for bit: entry (j,i) is the same products accumulated in the same order as (i,j).
// So only the 15 tiles on or below the diagonal are computed, three per warp, and the warp that computes a
// tile also writes the stage operand at the tile and at its mirror image: 150 DMMAs instead of 250, and no
// exchange through shared memory.  Warp w computes tiles (a,b), (c,b), (c,d): per k-step two A fragments
// (tile rows a, c) and two B fragments (tile columns b, d) from S feed its three DMMAs.
struct SelfTiles { int a, b, c, d; };
__device__ constexpr SelfTiles kSelfTiles[NMMA] = {{0, 0, 1, 1}, {3, 3, 4, 4}, {2, 0, 3, 1}, {4, 1, 2, 2}, {3, 2, 4, 0}};

// H = S + (dt/2) (Sigma - 2 S S) on this warp's tiles and their mirror images, and the mean's stage
// operand of row irow: vt[0] = m + (dt/2) (b - A m), with A m from the fragments of A(t) in registers
__device__ __forceinline__ void rk2_self_stage(FwdSmem& sm, const SelfTiles& tl, const double (&A0)[D / 4], double bc,
                                               double dt, int irow, int g, int q)
{
    const double* X = sm.Sb;
    const int la = sm_idx(8 * tl.a + g, q), lc = sm_idx(8 * tl.c + g, q);
    const int lb = sm_boff(q, g) + 8 * tl.b, ld = sm_boff(q, g) + 8 * tl.d;
    double acc[3][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
    double y = 0.0;
#pragma unroll
    for (int n = 0; n < D / 4; ++n) {
        const int k0 = 4 * n, kb = (n >> 1) * SM_R8 + (n & 1) * SM_BH;
        y = fma(A0[n], sm.mv[k0 + q], y);
        const double fa = X[la + k0], fc = X[lc + k0], fb = X[lb + kb], fd = X[ld + kb];
        dmma(acc[0][0], acc[0][1], fa, fb);
        dmma(acc[1][0], acc[1][1], fc, fb);
        dmma(acc[2][0], acc[2][1], fc, fd);
    }
    y += __shfl_xor_sync(0xffffffffu, y, 1);
    y += __shfl_xor_sync(0xffffffffu, y, 2);
    const double cdt = next_coef(ODE_RK2, 0) * dt;
    if (q == 0) sm.vt[0][irow] = sm.mv[irow] + cdt * (-y + bc);
    const int tr[3] = {tl.a, tl.c, tl.c}, tc[3] = {tl.b, tl.b, tl.d};
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const int i = 8 * tr[t] + g, j0 = 8 * tc[t] + 2 * q;
        const double2 sv = *reinterpret_cast<const double2*>(&sm.Sb[sm_idx(i, j0)]);
        double out[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int j = j0 + e;
            const double kk = (i == j ? sm.sig[i] : 0.0) - (acc[t][e] + acc[t][e]);
            out[e] = (e == 0 ? sv.x : sv.y) + cdt * kk;
        }
        *reinterpret_cast<double2*>(&sm.Hb[sm_idx(i, j0)]) = make_double2(out[0], out[1]);
        if (tr[t] != tc[t]) {   // the mirror image (transposed 8-byte stores: conflict-free in this layout)
            sm.Hb[sm_idx(j0, i)] = out[0];
            sm.Hb[sm_idx(j0 + 1, i)] = out[1];
        }
    }
}

template <int METHOD>
__global__ void __launch_bounds__(NTH, 4)
l96_fwd_kernel(Batch b, Scratch s, const double* __restrict__ x, long long xs, int p0)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    FwdSmem& sm = *reinterpret_cast<FwdSmem*>(smem_raw);
    constexpr int NS = n_stages(METHOD);
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int irow = 8 * w + g;
    const int lp = blockIdx.x, p = problem_at(b, p0 + lp), N = b.N;
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
    const double* A = x + (long long)p * xs;
    const double* bo = A + (long long)N * D * D;
    double* mt = s.mt + (long long)lp * N * D;
    double* st = s.st + (long long)lp * N * D * D;
    const double dt = b.dt;

    // initial state: S0 -> Sb (and trajectory slot 0), m0 -> mv
    for (int e = tid; e < D * D; e += NTH) {
        const int i = e / D, j = e % D;
        const double v = b.s0[p * b.s0_stride + e];
        sm.Sb[sm_idx(i, j)] = v;
        st[e] = v;
    }
    if (tid < D) {
        const double v = b.m0[p * b.m0_stride + tid];
        sm.mv[tid] = v;
        mt[tid] = v;
        sm.sig[tid] = b.sigma[p * b.sigma_stride + tid];
    }
    // this lane's fragment entries (row irow, columns 4n + q) of A(k) and A(k+1), and b[irow]
    double Ac[D / 4], An[D / 4];
    const double* arow = A + (long long)irow * D + q;
#pragma unroll
    for (int n = 0; n < D / 4; ++n) {
        Ac[n] = arow[4 * n];
        An[n] = 0.0;
    }
    double bc = bo[irow], bn = 0.0;
    __syncthreads();

    const bool small_launch = gridDim.x <= SMALL_LAUNCH;
    const SelfTiles tl = kSelfTiles[w];
    for (int k = 0; k < N - 1; ++k) {
        // launches of at most one CTA per SM (a single SCG run) have nothing to hide the DRAM latency of
        // their only input stream behind: pull this warp's eight rows of A into L2, PF_STEPS indices ahead
        // Full waves look ahead ONE index only (7.6 MB in flight over 592 CTAs: nothing is evicted before
        // use), which turns the register loads of A(k+2) a step later into L2 hits.
        {
            const int ahead = small_launch ? PF_STEPS : 1;
            if (lane == 0 && k + 1 + ahead < N)
                bulk_prefetch_l2(A + (long long)(k + 1 + ahead) * D * D + (long long)(8 * w) * D, 8 * ROWB);
        }
        // A(k+1), b(k+1) for this step's later stages: loads stay in flight during stage 0
        {
            const double* an = arow + (long long)(k + 1) * D * D;
#pragma unroll
            for (int n = 0; n < D / 4; ++n) An[n] = an[4 * n];
            bn = bo[(long long)(k + 1) * D + irow];
        }
        double ksum[5][2];   // sum_s w_s k_s of this lane's covariance entries
        double kv = 0.0;     // same for row irow of the mean (replicated over q)
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            if (METHOD == ODE_RK2 && sidx == 0) {   // the covariance inner stage of RK2 uses S in place of A
                rk2_self_stage(sm, tl, Ac, bc, dt, irow, g, q);
                __syncthreads();  // Hb, vt[0] complete
                continue;
            }
            const int kind = stage_kind(METHOD, sidx);
            const double* X = (sidx == 0) ? sm.Sb : sm.Hb;
            const double* vX = (sidx == 0) ? sm.mv : sm.vt[(sidx - 1) & 1];
            double acc[5][2], yv;
            if (kind == K_CUR)        mma_rowa<0>(Ac, An, X, vX, g, q, acc, yv);
            else if (kind == K_NEXT)  mma_rowa<0>(An, An, X, vX, g, q, acc, yv);
            else                      mma_rowa<1>(Ac, An, X, vX, g, q, acc, yv);
            row_to_smem(sm.Tb, irow, q, acc);
            {   // mean stage for row irow: k = -Aop v + bop
                const double bv = kind == K_CUR ? bc : (kind == K_NEXT ? bn : 0.5 * (bc + bn));
                const double ks = -yv + bv;
                const double wt = ksum_w(METHOD, sidx);
                if (wt != 0.0) kv = (sidx == 0 || (METHOD == ODE_RK2)) ? wt * ks : kv + wt * ks;
                if (sidx < NS - 1 && q == 0) sm.vt[sidx & 1][irow] = sm.mv[irow] + (next_coef(METHOD, sidx) * dt) * ks;
            }
            __syncthreads();  // T complete
            {
                const int i = irow;
#pragma unroll
                for (int J = 0; J < 5; ++J) {
                    const int j0 = 8 * J + 2 * q;
                    const double2 sv = *reinterpret_cast<const double2*>(&sm.Sb[sm_idx(i, j0)]);
                    double out[2];
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int j = j0 + e;
                        const double kk = (i == j ? sm.sig[i] : 0.0) - (acc[J][e] + sm.Tb[sm_idx(j, i)]);
                        const double wt = ksum_w(METHOD, sidx);
                        if (wt != 0.0) ksum[J][e] = (sidx == 0 || (METHOD == ODE_RK2)) ? wt * kk : ksum[J][e] + wt * kk;
                        const double sold = e == 0 ? sv.x : sv.y;
                        if (sidx < NS - 1) out[e] = sold + (next_coef(METHOD, sidx) * dt) * kk;
                        else out[e] = sold + final_step<METHOD>(dt, ksum[J][e]);
                    }
                    if (sidx < NS - 1) {
                        *reinterpret_cast<double2*>(&sm.Hb[sm_idx(i, j0)]) = make_double2(out[0], out[1]);
                    } else {
                        *reinterpret_cast<double2*>(&sm.Sb[sm_idx(i, j0)]) = make_double2(out[0], out[1]);
                        *reinterpret_cast<double2*>(&st[(long long)(k + 1) * D * D + i * D + j0]) =
                            make_double2(out[0], out[1]);
                    }
                }
                if (sidx == NS - 1 && q == 0) {
                    const double mn = sm.mv[i] + final_step<METHOD>(dt, kv);
                    sm.mv[i] = mn;
                    mt[(long long)(k + 1) * D + i] = mn;
                }
            }
            __syncthreads();  // next operand (Hb / Sb, mv) visible; T reusable
        }
#pragma unroll
        for (int n = 0; n < D / 4; ++n) Ac[n] = An[n];
        bc = bn;
    }
}

// ===========================================================================
// backward sweep + gradient assembly
// ===========================================================================
// In  Q = X A  the multiplier X (Psi or a stage value of it) is the LEFT operand, so a
// warp only ever needs its OWN eight rows of X as A fragments.  Psi therefore never
// touches shared memory: it lives in registers in accumulator layout and is turned
// into A fragments with two shuffles per k-step (the four lanes of a fragment row
// hold the eight entries of a tile between them).  Shared memory holds only what
// other warps must see: the A(t) ring, S(t), the lambda vectors and a double-buffered
// transpose exchange -- which lets 3 CTAs share an SM and needs one barrier per stage.
struct BwdSmem {
    double Ab[2][MAT], Sb[MAT];
    double Tb[2][MAT];
    double mv[D], bv[D], lam[D], lt[2][D], isg[D], Rv[D];
    uint64_t barA[2], barS;
};

struct BwdArgs {
    const double* A;     // (N,D,D) of this launch's first problem (stride xs between problems)
    const double* bo;    // (N,D)   offsets (null when with_grad == 0)
    long long xs;
    const double* mt; const double* st;      // scratch (problem-major), may be null w/o grad
    const double* dEm; const double* dEs;    // (N,D), (N,D,D) per problem
    long long traj_v, traj_m;                // strides between problems of the above
    double* gA; double* gb; long long gs;    // gradient out (null: no gradient)
    const double* jm_dense; const double* js_dense;  // dense jump tables (stand-alone sweep) or null
    double* lam_out; double* psi_out;        // trajectories out (first problem only) or null
};

// tile-row product whose LEFT operand comes from registers (accumulator layout Xc):
//   MODE 0: a = X[irow][k]      MODE 2: a = isg * (A0[irow][k] + edf[k]) - 2 X[irow][k]
//   (edf: this lane's entries of row irow of the sparse Lorenz-96 Jacobian <df/dx>)
// RK: right operand plain (0) or midpoint (1);  VK: matrix of the fused mat-vec
// (3 = A0 of MODE 2, else K_CUR / K_NEXT / K_MID of (V0, V1)).
template <int MODE, int RK, int VK>
__device__ __forceinline__ void mma_rowx(const double (&Xc)[5][2], const double (&edf)[D / 4], const double* __restrict__ A0,
                                         const double* __restrict__ R0, const double* __restrict__ R1,
                                         const double* __restrict__ V0, const double* __restrict__ V1,
                                         const double* __restrict__ v, double isg_row, int irow, int g, int q,
                                         int lane, double (&acc)[5][2], double& yv)
{
#pragma unroll
    for (int J = 0; J < 5; ++J) acc[J][0] = acc[J][1] = 0.0;
    double y = 0.0;
    const int la = sm_idx(irow, q);
    const int lb = sm_boff(q, g);
    const int srcb = (lane & ~3) + (q >> 1);
    const bool odd = (q & 1) != 0;
    // the left-operand entry of k-step n+1 is fetched (two shuffles) before the DMMAs of k-step n are
    // issued, so that the shuffle latency hides behind the tensor work
    auto fetch = [&](int n) {
        const int src = srcb + ((n & 1) << 1);
        const double x0 = __shfl_sync(0xffffffffu, Xc[n >> 1][0], src);
        const double x1 = __shfl_sync(0xffffffffu, Xc[n >> 1][1], src);
        return odd ? x1 : x0;
    };
    double xnext = fetch(0);
#pragma unroll
    for (int n = 0; n < D / 4; ++n) {
        const int k0 = 4 * n;
        // entry (irow, k0 + q) sits in tile n/2 at lane 2*(n&1) + q/2 of this row group, slot q&1
        const double xv = xnext;
        if (n + 1 < D / 4) xnext = fetch(n + 1);
        double a, av = 0.0;
        if (MODE == 2) {
            av = A0[la + k0];
            a = fma(isg_row, av + edf[n], -2.0 * xv);   // Sigma^-1 (A + <df/dx>) - 2 Psi
        } else {
            a = xv;
        }
        if (VK == K_CUR) av = V0[la + k0];
        else if (VK == K_NEXT) av = V1[la + k0];
        else if (VK == K_MID) av = 0.5 * (V0[la + k0] + V1[la + k0]);
        y = fma(av, v[k0 + q], y);
        double b[5];
#pragma unroll
        for (int J = 0; J < 5; ++J) {
            const int o = lb + (n >> 1) * SM_R8 + (n & 1) * SM_BH + 8 * J;
            if (RK == 0) b[J] = R0[o];
            else b[J] = 0.5 * (R0[o] + R1[o]);
        }
#pragma unroll
        for (int J = 0; J < 5; ++J) dmma(acc[J][0], acc[J][1], a, b[J]);
    }
    y += __shfl_xor_sync(0xffffffffu, y, 1);
    y += __shfl_xor_sync(0xffffffffu, y, 2);
    yv = y;
}

// ROWS: per-problem observation schedules (obs_rows); ROWS = false is the shared-schedule kernel, unchanged
template <int METHOD, bool ROWS>
__global__ void __launch_bounds__(NTH, 3)
l96_bwd_kernel(Batch b, BwdArgs a, int p0)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    BwdSmem& sm = *reinterpret_cast<BwdSmem*>(smem_raw);
    constexpr int NS = n_stages(METHOD);
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int irow = 8 * w + g;   // the matrix / vector row of this lane
    const int lp = blockIdx.x, p = problem_at(b, p0 + lp), N = b.N;
    if (b.active != nullptr && b.active[p] == 0) return;   // the whole CTA: before any barrier
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
    const double dt = b.dt, dtm = b.dt_model;
    const bool small_launch = gridDim.x <= SMALL_LAUNCH;
    const double theta = (b.theta != nullptr) ? b.theta[p * b.theta_stride] : 0.0;

    if (tid == 0) {
        mbar_init(&sm.barA[0], 1);
        mbar_init(&sm.barA[1], 1);
        mbar_init(&sm.barS, 1);
        mbar_fence_init();
    }
    if (tid < D) {
        sm.lam[tid] = 0.0;                                  // lam[N-1] = 0
        sm.isg[tid] = (b.sigma != nullptr) ? 1.0 / b.sigma[p * b.sigma_stride + tid] : 0.0;
        sm.Rv[tid] = (b.R != nullptr) ? b.R[p * b.R_stride + tid] : 1.0;
    }
    // Psi (rows 8w..8w+7 in accumulator layout), dE/dS and dE/dm of the current index live in
    // registers; the neighbour index is prefetched into registers a step ahead
    double Pc[5][2], Hc[5][2], Gc[5][2], Gn[5][2];
    const double edf0[D / 4] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // unused by the MODE 0 products
    double gcv, gnv = 0.0;
#pragma unroll
    for (int J = 0; J < 5; ++J) {
        const double2 v = *reinterpret_cast<const double2*>(&dEs[(long long)(N - 1) * D * D + irow * D + 8 * J + 2 * q]);
        Gc[J][0] = v.x;
        Gc[J][1] = v.y;
        Gn[J][0] = Gn[J][1] = 0.0;
        Pc[J][0] = Pc[J][1] = 0.0;                          // Psi[N-1] = 0
        Hc[J][0] = Hc[J][1] = 0.0;
    }
    gcv = dEm[(long long)(N - 1) * D + irow];
    __syncthreads();
    {
        const int t = N - 1;
        if (tid == 0) mbar_arrive_expect_tx(&sm.barA[t & 1], D * ROWB);
        load_rows(sm.Ab[t & 1], A + (long long)t * D * D, &sm.barA[t & 1], w, lane);
        if (t >= 1) {
            if (tid == 0) mbar_arrive_expect_tx(&sm.barA[(t - 1) & 1], D * ROWB);
            load_rows(sm.Ab[(t - 1) & 1], A + (long long)(t - 1) * D * D, &sm.barA[(t - 1) & 1], w, lane);
        }
        if (with_grad) {
            if (tid == 0) {
                mbar_arrive_expect_tx(&sm.barS, D * ROWB + 2 * ROWB);
                bulk_g2s(sm.mv, mt + (long long)t * D, ROWB, &sm.barS);
                bulk_g2s(sm.bv, bo + (long long)t * D, ROWB, &sm.barS);
            }
            load_rows(sm.Sb, st + (long long)t * D * D, &sm.barS, w, lane);
        }
    }
    uint32_t parA[2] = {0u, 0u}, parS = 0u;
    mbar_wait(&sm.barA[(N - 1) & 1], parA[(N - 1) & 1]);
    parA[(N - 1) & 1] ^= 1u;
    int tsel = 0;   // which transpose buffer the next stage writes

    for (int t = N - 1; t >= 0; --t) {
        const int cur = t & 1, nxt = cur ^ 1;
        const double* Ac = sm.Ab[cur];
        const double* An = sm.Ab[nxt];
        if (keep) {  // lam[t], Psi[t] for vgpa_eval_full / the stand-alone sweep
#pragma unroll
            for (int J = 0; J < 5; ++J)
                *reinterpret_cast<double2*>(&a.psi_out[(long long)t * D * D + irow * D + 8 * J + 2 * q]) =
                    make_double2(Pc[J][0], Pc[J][1]);
            if (q == 0) a.lam_out[(long long)t * D + irow] = sm.lam[irow];
        }
        // Small launches only (at most one CTA per SM: nothing else hides HBM latency, which is what a
        // single problem then waits for): this warp's eight rows of the three streams, PF_STEPS
        // indices ahead, into L2.  With full waves the same prefetch was measured harmful (evictions);
        // the forward sweep does the same for its single stream.
        if (small_launch && lane == 0 && t >= PF_STEPS) {
            const long long o = (long long)(t - PF_STEPS) * D * D + (long long)(8 * w) * D;
            bulk_prefetch_l2(A + o, 8 * ROWB);
            bulk_prefetch_l2(dEs + o, 8 * ROWB);
            if (with_grad) bulk_prefetch_l2(st + o, 8 * ROWB);
        }
        // register prefetch of dE/dS[t-1], dE/dm[t-1] (consumed one or two stages later)
        if (t >= 1) {
#pragma unroll
            for (int J = 0; J < 5; ++J) {
                const double2 v = *reinterpret_cast<const double2*>(&dEs[(long long)(t - 1) * D * D + irow * D + 8 * J + 2 * q]);
                Gn[J][0] = v.x;
                Gn[J][1] = v.y;
            }
            gnv = dEm[(long long)(t - 1) * D + irow];
        }
        // ---- gradient at index t (variational.py:263-288) ----------------------
        if (with_grad) {
            mbar_wait(&sm.barS, parS);
            parS ^= 1u;
            double acc[5][2], am;
            const int i = irow;
            const int f1 = (i + 1) % D, b1 = (i + D - 1) % D, b2 = (i + D - 2) % D;
            // row i of <df/dx> (Jacobian of the Lorenz-96 drift at the mean, lorenz_96.py:34-83):
            // J[i][i] = -1, J[i][i+1] = m[i-1], J[i][i-2] = -m[i-1], J[i][i-1] = m[i+1] - m[i-2];
            // this lane keeps the entries that fall on its fragment columns k = 4n + q
            double edf[D / 4];
            {
                const double cf = sm.mv[b1], cb1 = sm.mv[f1] - sm.mv[b2];
#pragma unroll
                for (int n = 0; n < D / 4; ++n) {
                    const int k = 4 * n + q;
                    edf[n] = (k == i) ? -1.0 : (k == f1) ? cf : (k == b2) ? -cf : (k == b1) ? cb1 : 0.0;
                }
            }
            // W = (Sigma^-1 (A_t + <df/dx>) - 2 Psi_t) S_t   and   am = (A_t m_t)[irow]
            mma_rowx<2, 0, 3>(Pc, edf, Ac, sm.Sb, nullptr, nullptr, nullptr, sm.mv, sm.isg[irow], irow, g, q, lane, acc, am);
            // <f> of Lorenz 96 (lorenz_96.py:440-462)
            const double Ef = (sm.Sb[sm_idx(f1, b1)] - sm.Sb[sm_idx(b2, b1)]) + (sm.mv[f1] - sm.mv[b2]) * sm.mv[b1] -
                              sm.mv[i] + theta;
            const double db = sm.isg[i] * (-Ef - am + sm.bv[i]);   // variational.py:324-334
            const double ui = db + sm.lam[i];
            if (q == 0) gb[(long long)t * D + i] = dtm * ui;       // :280,285
#pragma unroll
            for (int J = 0; J < 5; ++J) {
                const int j0 = 8 * J + 2 * q;
                const double2 mj = *reinterpret_cast<const double2*>(&sm.mv[j0]);
                *reinterpret_cast<double2*>(&gA[(long long)t * D * D + i * D + j0]) =
                    make_double2(dtm * (acc[J][0] - ui * mj.x), dtm * (acc[J][1] - ui * mj.y));
            }
        }
        if (t == 0) break;
        // lam[t] (written at the end of the previous step, each warp its own rows) must be visible to every
        // warp before the first mat-vec; the gradient above only reads a warp's own rows of it, so the
        // barrier sits here and lets warps run ahead into the gradient of the next index
        __syncthreads();
        // ---- one backward step t -> t-1 ------------------------------------------
        bool next_ready = false;
        double ksum[5][2];
        double kv = 0.0;
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            const int kind = stage_kind(METHOD, sidx);
            if (kind != K_CUR && !next_ready) {
                mbar_wait(&sm.barA[nxt], parA[nxt]);
                parA[nxt] ^= 1u;
                next_ready = true;
            }
            if (sidx == 1 && stage_kind(METHOD, 1) == K_MID) __syncthreads();   // A_mid complete in slot cur
            const double* vX = (sidx == 0) ? sm.lam : sm.lt[(sidx - 1) & 1];
            double* Tw = sm.Tb[tsel];
            tsel ^= 1;
            double acc[5][2], yv;
            // Q = X Aop   and   yv = (Aop lam_op)[irow]
            if (sidx == 0) {
                if (kind == K_CUR)       mma_rowx<0, 0, K_CUR>(Pc, edf0, nullptr, Ac, nullptr, Ac, An, vX, 0.0, irow, g, q, lane, acc, yv);
                else if (kind == K_NEXT) mma_rowx<0, 0, K_NEXT>(Pc, edf0, nullptr, An, nullptr, Ac, An, vX, 0.0, irow, g, q, lane, acc, yv);
                else                     mma_rowx<0, 1, K_MID>(Pc, edf0, nullptr, Ac, An, Ac, An, vX, 0.0, irow, g, q, lane, acc, yv);
            } else {
                if (kind == K_CUR)       mma_rowx<0, 0, K_CUR>(Hc, edf0, nullptr, Ac, nullptr, Ac, An, vX, 0.0, irow, g, q, lane, acc, yv);
                else if (kind == K_NEXT) mma_rowx<0, 0, K_NEXT>(Hc, edf0, nullptr, An, nullptr, Ac, An, vX, 0.0, irow, g, q, lane, acc, yv);
                else                     mma_rowx<0, 0, K_CUR>(Hc, edf0, nullptr, Ac, nullptr, Ac, An, vX, 0.0, irow, g, q, lane, acc, yv);  // slot cur holds A_mid
            }
            row_to_smem(Tw, irow, q, acc);
            {
                const double gk = kind == K_CUR ? gcv : (kind == K_NEXT ? gnv : 0.5 * (gnv + gcv));
                const double ks = -gk + yv;  // ode_solver.py:77
                const double wt = ksum_w(METHOD, sidx);
                if (wt != 0.0) kv = (sidx == 0 || (METHOD == ODE_RK2)) ? wt * ks : kv + wt * ks;
                if (sidx < NS - 1 && q == 0) sm.lt[sidx & 1][irow] = sm.lam[irow] - (next_coef(METHOD, sidx) * dt) * ks;
            }
            __syncthreads();  // the only barrier of the stage: transpose buffer and next lambda operand complete
            if (sidx == 0 && NS > 1 && stage_kind(METHOD, 1) == K_MID) {
                // Every warp has finished its last product with A_t (gradient and stage 0): turn slot
                // cur into the midpoint A_mid = (A_t + A_{t-1}) / 2 IN PLACE, each warp its own eight
                // rows, so that the midpoint stages read one buffer (half the B-fragment traffic of
                // those stages and no per-fragment averaging).  The slot is refilled with A_{t-2}
                // after the last stage, as before.
                if (!next_ready) {
                    mbar_wait(&sm.barA[nxt], parA[nxt]);
                    parA[nxt] ^= 1u;
                    next_ready = true;
                }
                double* Aw = sm.Ab[cur];
#pragma unroll
                for (int n = 0; n < 5; ++n) {
                    const int c = lane + 32 * n, r = c / 20, ch = c - 20 * r;
                    const int o = sm_idx(8 * w + r, 2 * ch);
                    const double2 a2 = *reinterpret_cast<const double2*>(&Aw[o]);
                    const double2 b2 = *reinterpret_cast<const double2*>(&An[o]);
                    *reinterpret_cast<double2*>(&Aw[o]) = make_double2(0.5 * (a2.x + b2.x), 0.5 * (a2.y + b2.y));
                }
            }
            if (sidx == 0 && with_grad) {
                // S_t, m_t, b_t are dead (gradient written by every warp): fetch index t-1
                if (tid == 0) {
                    mbar_arrive_expect_tx(&sm.barS, D * ROWB + 2 * ROWB);
                    bulk_g2s(sm.mv, mt + (long long)(t - 1) * D, ROWB, &sm.barS);
                    bulk_g2s(sm.bv, bo + (long long)(t - 1) * D, ROWB, &sm.barS);
                }
                load_rows(sm.Sb, st + (long long)(t - 1) * D * D, &sm.barS, w, lane);
            }
            if (sidx == NS - 1 && t >= 2) {
                // slot `cur` is dead once every warp has finished the last product of the step
                if (!next_ready) {  // Euler: A_{t-1} has not been waited for yet
                    mbar_wait(&sm.barA[nxt], parA[nxt]);
                    parA[nxt] ^= 1u;
                    next_ready = true;
                }
                if (tid == 0) mbar_arrive_expect_tx(&sm.barA[cur], D * ROWB);
                load_rows(sm.Ab[cur], A + (long long)(t - 2) * D * D, &sm.barA[cur], w, lane);
            }
            {
                const int i = irow;
#pragma unroll
                for (int J = 0; J < 5; ++J) {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int j = 8 * J + 2 * q + e;
                        double gg;
                        if (kind == K_CUR) gg = Gc[J][e];
                        else if (kind == K_NEXT) gg = Gn[J][e];
                        else gg = 0.5 * (Gn[J][e] + Gc[J][e]);
                        const double kk = -gg + (acc[J][e] + Tw[sm_idx(j, i)]);  // ode_solver.py:94
                        const double wt = ksum_w(METHOD, sidx);
                        if (wt != 0.0) ksum[J][e] = (sidx == 0 || (METHOD == ODE_RK2)) ? wt * kk : ksum[J][e] + wt * kk;
                        if (sidx < NS - 1) Hc[J][e] = Pc[J][e] - (next_coef(METHOD, sidx) * dt) * kk;
                    }
                }
            }
        }
        if (!next_ready) {  // (t == 1 with Euler) keep the barrier phases in step
            mbar_wait(&sm.barA[nxt], parA[nxt]);
            parA[nxt] ^= 1u;
        }
        // ---- final combination + jump at index t-1 -----------------------------------
        const int n_obs = dense ? -1 : (ROWS ? obs_index_of(b, p)[t - 1] : b.obs_index[t - 1]);
        {
            const int i = irow;
#pragma unroll
            for (int J = 0; J < 5; ++J) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int j = 8 * J + 2 * q + e;
                    double pn = Pc[J][e] - final_step<METHOD>(dt, ksum[J][e]);
                    if (dense) pn += a.js_dense[(long long)(t - 1) * D * D + i * D + j];
                    else if (n_obs >= 0 && i == j) pn += 0.5 / sm.Rv[i];  // gaussian_like.py:238
                    Pc[J][e] = pn;
                    Gc[J][e] = Gn[J][e];  // dE/dS[t-1] becomes current
                }
            }
            double ln = sm.lam[i] - final_step<METHOD>(dt, kv);
            if (dense) ln += a.jm_dense[(long long)(t - 1) * D + i];
            else if (n_obs >= 0) {
                if (with_grad) mbar_wait(&sm.barS, parS);  // m[t-1] landed (parity unchanged)
                const double mprev = with_grad ? sm.mv[i] : mt[(long long)(t - 1) * D + i];
                ln += -(oy[(long long)n_obs * D + i] - mprev) / sm.Rv[i];  // :235
            }
            __syncwarp();
            if (q == 0) sm.lam[i] = ln;
            __syncwarp();   // the other lanes of row i read it in the gradient of index t-1
            gcv = gnv;
        }
    }
}

}  // namespace

void launch_l96_fwd(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count,
                    cudaStream_t st)
{
    const size_t sh = sizeof(FwdSmem);
    with_method(b.method, [&](auto m) {
        set_smem(l96_fwd_kernel<m>, sh);
        l96_fwd_kernel<m><<<count, NTH, sh, st>>>(b, s, x, xs, p0);
    });
}

static void bwd_launch(const Batch& b, const BwdArgs& a, int p0, int count, cudaStream_t st)
{
    const size_t sh = sizeof(BwdSmem);
    with_method(b.method, [&](auto m) {
        if (obs_rows(b)) {
            set_smem(l96_bwd_kernel<m, true>, sh);
            l96_bwd_kernel<m, true><<<count, NTH, sh, st>>>(b, a, p0);
        } else {
            set_smem(l96_bwd_kernel<m, false>, sh);
            l96_bwd_kernel<m, false><<<count, NTH, sh, st>>>(b, a, p0);
        }
    });
}

void launch_l96_bwd(const Batch& b, const Scratch& s, const double* x, long long xs, double* grad,
                    long long gs, int p0, int count, const Extra& ex, cudaStream_t st)
{
    const long long N = b.N;
    BwdArgs a{};
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

void launch_bwd_dense_l96(int method, int N, double dt, const double* A, const double* dEm,
                          const double* dEs, const double* jm, const double* js, double* lam,
                          double* psi, cudaStream_t st)
{
    Batch b{};
    b.model = MODEL_L96; b.method = method; b.D = D; b.N = N; b.B = 1; b.dt = dt; b.dt_model = dt;
    BwdArgs a{};
    a.A = A; a.xs = 0; a.dEm = dEm; a.dEs = dEs;
    a.jm_dense = jm; a.js_dense = js; a.lam_out = lam; a.psi_out = psi;
    bwd_launch(b, a, 0, 1, st);
}

}  // namespace vgpa
