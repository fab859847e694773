// api.cu -- the C ABI of libvgpa_b200.so (include/vgpa_b200.h): handle management,
// chunked three-phase evaluation (forward sweep -> time-parallel energy -> backward
// sweep fused with the gradient), the batched hyper-parameter gradients, host staging
// with copy/compute overlap.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/vgpa_b200.h"
#include "common.cuh"

using namespace vgpa;

namespace {

thread_local std::string g_create_error;

// Hand-over of large device blocks between handles (vgpa_scratch_cache): while it is enabled, the large blocks
// of a destroyed handle -- its trajectory scratch -- are kept and given to the next handle that asks for exactly
// the same size on the same device.  An ensemble optimised in resident sub-batches creates one evaluator per
// sub-batch, all of one shape; cudaFree of ~12 GB of scratch was measured at 0.02-0.4 s in a lone process and at
// up to 2 s when the processes of four or eight GPUs free at the same time (more than the optimisation of
// the sub-batch's tail).  Off by default: a destroyed handle returns its memory.
struct BlockCache {
    struct Blk { void* p; size_t bytes; int dev; };
    std::mutex mu;
    bool enabled = false;
    std::vector<Blk> blocks;
    static constexpr size_t MIN_BYTES = size_t(32) << 20;
    static constexpr size_t MAX_BLOCKS = 24;
    void* take(size_t n)
    {
        if (n < MIN_BYTES) return nullptr;
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lk(mu);
        for (size_t i = 0; i < blocks.size(); ++i)
            if (blocks[i].bytes == n && blocks[i].dev == dev) {
                void* p = blocks[i].p;
                blocks.erase(blocks.begin() + i);
                return p;
            }
        return nullptr;
    }
    bool put(void* p, size_t n)
    {
        if (n < MIN_BYTES) return false;
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lk(mu);
        if (!enabled || blocks.size() >= MAX_BLOCKS) return false;
        blocks.push_back({p, n, dev});
        return true;
    }
    long long purge()      // frees every cached block; returns the bytes released
    {
        std::vector<Blk> out;
        {
            std::lock_guard<std::mutex> lk(mu);
            out.swap(blocks);
        }
        int cur = 0;
        cudaGetDevice(&cur);
        long long total = 0;
        for (const Blk& b : out) {
            cudaSetDevice(b.dev);
            cudaFree(b.p);
            total += (long long)b.bytes;
        }
        cudaSetDevice(cur);
        return total;
    }
};
BlockCache g_block_cache;

// A device allocation that frees itself.  It is destroyed with its owner's device current: the block cache
// records the current device of a block it keeps.
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), bytes(std::exchange(o.bytes, 0)) {}
    DevBuf& operator=(DevBuf&& o) noexcept
    {
        std::swap(p, o.p);
        std::swap(bytes, o.bytes);
        return *this;
    }
    ~DevBuf() { release(); }
    cudaError_t alloc(size_t n)
    {
        release();
        if (n == 0) n = 8;
        if (void* c = g_block_cache.take(n)) {
            p = c;
            bytes = n;
            return cudaSuccess;
        }
        cudaError_t e = cudaMalloc(&p, n);
        if (e == cudaErrorMemoryAllocation && g_block_cache.purge() > 0) {   // the kept blocks are in the way
            cudaGetLastError();
            e = cudaMalloc(&p, n);
        }
        if (e == cudaSuccess) bytes = n;
        else p = nullptr;
        return e;
    }
    void release()
    {
        if (p && !g_block_cache.put(p, bytes)) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

// Staging of host arrays.  Each helper does nothing once `e` holds an error, so that a run of them stops at
// the first failure and `e` reports it.  The copies are plain cudaMemcpy (legacy default stream).
template <typename T = double>
void alloc(cudaError_t& e, DevBuf& dst, size_t n)
{
    if (e == cudaSuccess) e = dst.alloc(sizeof(T) * n);
}
template <typename T>
void to_device(cudaError_t& e, void* dst, const T* src, size_t n)
{
    if (e == cudaSuccess) e = cudaMemcpy(dst, src, sizeof(T) * n, cudaMemcpyHostToDevice);
}
template <typename T>
void upload(cudaError_t& e, DevBuf& dst, const T* src, size_t n)
{
    alloc<T>(e, dst, n);
    to_device(e, dst.p, src, n);
}
// dst NULL: an output the caller did not ask for
template <typename T>
void download(cudaError_t& e, T* dst, const void* src, size_t n)
{
    if (e == cudaSuccess && dst != nullptr) e = cudaMemcpy(dst, src, sizeof(T) * n, cudaMemcpyDeviceToHost);
}
// `rows` rows of `len` elements, `stride` apart (0 = one row shared by all), into a compact device buffer;
// *dstride: the row stride there
void stage_rows(cudaError_t& e, DevBuf& dst, const double* src, long long stride, long long len, int rows,
                long long* dstride)
{
    const int r = stride == 0 ? 1 : rows;
    alloc(e, dst, (size_t)len * r);
    if (e != cudaSuccess) return;
    *dstride = stride == 0 ? 0 : len;
    if (r == 1 || stride == len) e = cudaMemcpy(dst.p, src, sizeof(double) * (size_t)len * r, cudaMemcpyHostToDevice);
    else e = cudaMemcpy2D(dst.p, sizeof(double) * len, src, sizeof(double) * stride, sizeof(double) * len, r, cudaMemcpyHostToDevice);
}

// Trajectory scratch of one pass: `chunk` problems of N time points.
struct ScratchBufs {
    DevBuf mt, st, dEm, dEs, esde;
    cudaError_t alloc(long long chunk, long long N, long long D)
    {
        cudaError_t e = cudaSuccess;
        ::alloc(e, mt, chunk * N * D);
        ::alloc(e, st, chunk * N * D * D);
        ::alloc(e, dEm, chunk * N * D);
        ::alloc(e, dEs, chunk * N * D * D);
        ::alloc(e, esde, chunk * N);
        return e;
    }
    Scratch view(int* status) const
    {
        return Scratch{mt.as<double>(), st.as<double>(), dEm.as<double>(), dEs.as<double>(), esde.as<double>(), status};
    }
    size_t bytes() const { return mt.bytes + st.bytes + dEm.bytes + dEs.bytes + esde.bytes; }
};

std::string vformat(const char* fmt, va_list ap)
{
    char buf[512];
    vsnprintf(buf, sizeof buf, fmt, ap);
    return buf;
}

// The error of a call that has no handle (vgpa_last_error(NULL)); returns `code`.
int set_error(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    g_create_error = vformat(fmt, ap);
    va_end(ap);
    return code;
}
int set_cuda_error(cudaError_t e, const char* fn)
{
    return set_error(VGPA_ECUDA, "CUDA error in %s: %s", fn, cudaGetErrorString(e));
}

int n_theta(int model) { return model == VGPA_MODEL_L63 ? 3 : 1; }

}  // namespace

struct vgpa_handle {
    vgpa_desc d{};
    Batch batch{};
    int chunk = 0;
    long long n_x = 0;   // N * D * (D + 1)
    DevBuf theta, sigma, R, obs_t, obs_index, obs_count, obs_y, m0, s0, E0, observed, status;
    bool obs_rows = false;              // per-problem observation schedules (vgpa_create_obs_rows)
    int init_empty = -1, init_edge = -1;   // ... the first problem without observations / with one at index 0 or N - 1
    ScratchBufs sc;
    cudaEvent_t ev_done = nullptr;      // end of the last vgpa_eval_device (a call on ANOTHER stream waits for it: one scratch)
    // host-API staging: two slots of one chunk each
    DevBuf st_x[2], st_g[2], st_F;
    DevBuf plist2[2];                   // vgpa_set_active_list: compacted list of problem indices (device copies,
    int plist_flip = 0;                 //   alternating: the evaluation in flight may still read the previous one)
    cudaStream_t s_aux = nullptr;       //   non-blocking stream of the list upload
    cudaEvent_t plist_ev[2] = {nullptr, nullptr};   //   end of the last evaluation that read each copy
    bool plist_used[2] = {false, false};
    std::vector<int> plist_host;        // ... and the host copy
    int n_list = -1;                    // < 0: no list, every problem
    std::vector<int> status_map;        // status word k belongs to problem status_map[k] (the list of the compacted
                                        //   evaluation that wrote it); empty: to problem k
    cudaStream_t s_comp = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[2]{}, ev_comp[2]{}, ev_d2h[2]{};
    cudaStream_t last_stream = nullptr;
    bool status_dirty = false;
    long long launches = 0;
    std::string err;
    // optional per-kernel timing (bench.py roofline)
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> tev[4];
    size_t tev_used[4] = {0, 0, 0, 0};
    double t_ms[4] = {0, 0, 0, 0};
    long long t_n[4] = {0, 0, 0, 0};

    void tick(int kind, cudaStream_t st, bool begin)
    {
        if (!timing) return;
        if (begin) {
            if (tev_used[kind] == tev[kind].size()) {
                cudaEvent_t a, b;
                cudaEventCreate(&a);
                cudaEventCreate(&b);
                tev[kind].push_back({a, b});
            }
            cudaEventRecord(tev[kind][tev_used[kind]].first, st);
        } else {
            cudaEventRecord(tev[kind][tev_used[kind]].second, st);
            ++tev_used[kind];
        }
    }

    int fail(int code, const char* fmt, ...)
    {
        va_list ap;
        va_start(ap, fmt);
        err = vformat(fmt, ap);
        va_end(ap);
        return code;
    }
    int cuda_fail(cudaError_t e, const char* what)
    {
        return fail(VGPA_ECUDA, "CUDA error in %s: %s", what, cudaGetErrorString(e));
    }
};

#define CK(call, what)                                         \
    do {                                                       \
        cudaError_t e__ = (call);                              \
        if (e__ != cudaSuccess) return h->cuda_fail(e__, what); \
    } while (0)

namespace {

bool small_model(int model) { return model != VGPA_MODEL_L96; }

// Lorenz 96: the tuned kernels at D = 40, the run-time-D family (l96_dyn.cu) at every other D
void l96_fwd(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count, cudaStream_t st)
{
    if (l96_tuned(b.D)) launch_l96_fwd(b, s, x, xs, p0, count, st);
    else launch_l96d_fwd(b, s, x, xs, p0, count, st);
}
void l96_energy(const Batch& b, const Scratch& s, const double* x, long long xs, int p0, int count, const Extra& ex,
                cudaStream_t st)
{
    if (l96_tuned(b.D)) launch_l96_energy(b, s, x, xs, p0, count, ex, st);
    else launch_l96d_energy(b, s, x, xs, p0, count, ex, st);
}
void l96_bwd(const Batch& b, const Scratch& s, const double* x, long long xs, double* g, long long gs, int p0, int count,
             const Extra& ex, cudaStream_t st)
{
    if (l96_tuned(b.D)) launch_l96_bwd(b, s, x, xs, g, gs, p0, count, ex, st);
    else launch_l96d_bwd(b, s, x, xs, g, gs, p0, count, ex, st);
}

// one pass over problems [p0, p0 + count) with device buffers
void run_chunk(vgpa_handle* h, const double* d_x, long long xs, int want_grad, double* d_F, double* d_grad,
               long long gs, int p0, int count, const Extra& ex, cudaStream_t st)
{
    const Scratch sc = h->sc.view(h->status.as<int>() + p0);
    const Batch& b = h->batch;
    const bool small = small_model(b.model);
    h->tick(0, st, true);
    if (small && want_grad && launch_small_fused(b, d_x, xs, d_F, d_grad, gs, p0, count, ex, st)) {
        h->tick(0, st, false);      // the one launch is accounted to the first phase
        h->launches += 1;
        return;
    }
    if (small) launch_small_fwd(b, sc, d_x, xs, p0, count, st);
    else l96_fwd(b, sc, d_x, xs, p0, count, st);
    h->tick(0, st, false);
    h->tick(1, st, true);
    if (small) launch_small_energy(b, sc, d_x, xs, p0, count, ex, st);
    else l96_energy(b, sc, d_x, xs, p0, count, ex, st);
    h->tick(1, st, false);
    h->tick(2, st, true);
    launch_finalize(b, sc, d_F, p0, count, ex, st);
    h->tick(2, st, false);
    h->launches += 3;
    if (want_grad) {
        h->tick(3, st, true);
        if (small) launch_small_bwd(b, sc, d_x, xs, d_grad, gs, p0, count, ex, st);
        else l96_bwd(b, sc, d_x, xs, d_grad, gs, p0, count, ex, st);
        h->tick(3, st, false);
        h->launches += 1;
    }
}

// one pass of vgpa_hyper_device over problems [p0, p0 + count): the forward sweep, the energy stage with the
// hyper integrands (into the pass's dEs scratch, which nothing after them reads), F, the per-problem reduction
void run_hyper_chunk(vgpa_handle* h, const double* d_x, long long xs, double* d_F, const HyperOut& o, int p0, int count,
                     cudaStream_t st)
{
    const Scratch sc = h->sc.view(h->status.as<int>() + p0);
    const Batch& b = h->batch;
    const bool small = small_model(b.model);
    h->tick(0, st, true);
    if (small) launch_small_fwd(b, sc, d_x, xs, p0, count, st);
    else l96_fwd(b, sc, d_x, xs, p0, count, st);
    h->tick(0, st, false);
    h->tick(1, st, true);
    if (small) launch_small_energy(b, sc, d_x, xs, p0, count, Extra{}, st);
    launch_hyper_terms(b, sc, d_x, xs, p0, count, st);
    h->tick(1, st, false);
    h->tick(2, st, true);
    if (d_F != nullptr) launch_finalize(b, sc, d_F, p0, count, Extra{}, st);
    launch_hyper_reduce(b, sc, p0, count, o, st);
    h->tick(2, st, false);
    h->launches += (small ? 4 : 3) + (d_F != nullptr ? 1 : 0);
}

// The host-buffer entry points (vgpa_eval, vgpa_eval_full) always serve EVERY problem: the active set
// and the compacted list installed for vgpa_eval_device are suspended for the call (a masked problem
// would otherwise return whatever the staging buffers hold), and a device evaluation still pending on
// the caller's stream is waited for first (it shares the scratch and the status words).
struct HostCallScope {
    vgpa_handle* h;
    const int *active, *plist;
    explicit HostCallScope(vgpa_handle* h_) : h(h_), active(h_->batch.active), plist(h_->batch.plist)
    {
        if (h->status_dirty) cudaStreamSynchronize(h->last_stream);
        h->batch.active = nullptr;
        h->batch.plist = nullptr;
        h->status_map.clear();
    }
    ~HostCallScope()
    {
        h->batch.active = active;
        h->batch.plist = plist;
    }
};

int check_status(vgpa_handle* h)
{
    if (!h->status_dirty) return VGPA_OK;
    h->status_dirty = false;
    std::vector<int> st(h->d.B);
    // Every caller has synchronised the stream that wrote the status words.  The copy runs on the handle's private
    // NON-BLOCKING stream: a plain cudaMemcpy goes through the legacy default stream, which waits for every blocking
    // stream of the process -- e.g. for the evaluation another host thread has in flight on another handle
    // (ShardedBatchedSCG with concurrent sub-batches: two handles serialised each other at every status check).
    if (h->s_aux == nullptr) CK(cudaStreamCreateWithFlags(&h->s_aux, cudaStreamNonBlocking), "cudaStreamCreate");
    CK(cudaMemcpyAsync(st.data(), h->status.p, sizeof(int) * h->d.B, cudaMemcpyDeviceToHost, h->s_aux), "cudaMemcpyAsync(status)");
    CK(cudaStreamSynchronize(h->s_aux), "cudaStreamSynchronize(status)");
    for (int p = 0; p < h->d.B; ++p)
        if (st[p] != 0) {
            // under a compacted launch the status words are indexed by launch position
            const int prob = (p < (int)h->status_map.size()) ? h->status_map[p] : p;
            return h->fail(VGPA_ENOTPD, "Matrix is not positive definite: S(t) of problem %d at time index %d",
                           prob, st[p] - 1);
        }
    return VGPA_OK;
}

}  // namespace

extern "C" {

const char* vgpa_version(void) { return "vgpa_b200 0.1 (sm_100a)"; }

const char* vgpa_last_error(const vgpa_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

}  // extern "C"

namespace {

// vgpa_create, vgpa_create_obs_rows and vgpa_create_observed.  obs_t: the schedules, obs_t_stride elements apart (0 =
// one row shared by every problem); counts: B observation counts or NULL (desc->M each).  rows == false: vgpa_create's
// one schedule, desc->obs_t.  observed: the masks of the observed components, observed_stride words apart (0 = one
// mask shared by every problem), or NULL = every component.
int create_handle(const vgpa_desc* d, const int64_t* obs_t, int64_t obs_t_stride, const int32_t* counts, bool rows,
                  const uint64_t* observed, int64_t observed_stride, vgpa_handle** out)
{
    vgpa_handle* h = new vgpa_handle();
    h->d = *d;
    auto bail = [&](int rc) {
        g_create_error = h->err;
        vgpa_destroy(h);
        return rc;
    };
    // ---- validation (the ValueErrors of the reference constructors) ----
    if (d->model < 0 || d->model > 3) return bail(h->fail(VGPA_EINVAL, "Unknown stochastic model -> %d", d->model));
    if (d->method < 0 || d->method > 3)
        return bail(h->fail(VGPA_EINVAL, "Integration method is unknown -> %d", d->method));
    if (d->model == VGPA_MODEL_L96) {
        if (d->D < 10) return bail(h->fail(VGPA_EINVAL, " Lorenz96: Insufficient state vector dimensions: %d", d->D));
        if (d->D > 64)
            return bail(h->fail(VGPA_EINVAL, "Wrong state dimension %d for Lorenz 96 (supported: 10 <= D <= 64)", d->D));
    } else {
        const int needD = (d->model == VGPA_MODEL_L63) ? 3 : 1;
        if (d->D != needD) return bail(h->fail(VGPA_EINVAL, "Wrong state dimension %d for model %d (need %d)", d->D, d->model, needD));
    }
    if (d->N < 2) return bail(h->fail(VGPA_EINVAL, "Need at least two time points, got %d", d->N));
    if (d->M < 0 || d->B < 1) return bail(h->fail(VGPA_EINVAL, "Wrong sizes M=%d B=%d", d->M, d->B));
    if (!(d->dt > 0.0) || !(d->dt_model > 0.0))
        return bail(h->fail(VGPA_EINVAL, "Discrete time step should be strictly positive -> %g", d->dt));
    if (!rows) {
        if (d->M > 0 && d->obs_t == nullptr) return bail(h->fail(VGPA_EINVAL, "obs_t is NULL"));
        for (int n = 0; n < d->M; ++n) {
            if (d->obs_t[n] < 0 || d->obs_t[n] >= d->N || (n > 0 && d->obs_t[n] <= d->obs_t[n - 1]))
                return bail(h->fail(VGPA_EINVAL, "obs_t must be sorted unique indices in [0, N)"));
            // gaussian_like.py:137-146 indexes the covariance by the observation ordinal n
            if (n >= d->N) return bail(h->fail(VGPA_EINVAL, "more observations than time points"));
        }
    } else {
        if (d->obs_t != nullptr)
            return bail(h->fail(VGPA_EINVAL, "desc->obs_t must be NULL: the schedules are the obs_t argument"));
        if (d->M > 0 && obs_t == nullptr) return bail(h->fail(VGPA_EINVAL, "obs_t is NULL"));
        if (obs_t_stride < 0 || (obs_t_stride > 0 && obs_t_stride < d->M))
            return bail(h->fail(VGPA_EINVAL, "obs_t_stride %lld: 0 (one shared row) or at least M = %d", (long long)obs_t_stride,
                                d->M));
        for (int p = 0; p < d->B; ++p) {
            const int Mp = counts ? counts[p] : d->M;
            if (Mp < 0 || Mp > d->M)
                return bail(h->fail(VGPA_EINVAL, "M of problem %d is %d, outside [0, desc->M = %d]", p, Mp, d->M));
            const int64_t* ot = obs_t + p * obs_t_stride;
            for (int n = 0; n < Mp; ++n)
                if (ot[n] < 0 || ot[n] >= d->N || (n > 0 && ot[n] <= ot[n - 1]))
                    return bail(h->fail(VGPA_EINVAL, "obs_t of problem %d must be sorted unique indices in [0, N)", p));
            // VarGP.initialization's spline (variational.py:86-104) needs knots strictly inside the time window
            if (h->init_empty < 0 && Mp < 1) h->init_empty = p;
            if (h->init_edge < 0 && Mp > 0 && (ot[0] == 0 || ot[Mp - 1] == d->N - 1)) h->init_edge = p;
        }
    }
    if (observed != nullptr) {
        if (observed_stride < 0)
            return bail(h->fail(VGPA_EINVAL, "observed_stride %lld: 0 (one shared mask) or positive", (long long)observed_stride));
        for (int p = 0; p < d->B; ++p) {
            const uint64_t w = observed[p * observed_stride];
            if (w == 0) return bail(h->fail(VGPA_EINVAL, "the observation mask of problem %d has no bit set", p));
            if (d->D < 64 && (w >> d->D) != 0)
                return bail(h->fail(VGPA_EINVAL, "the observation mask of problem %d has a bit at or above D = %d", p, d->D));
        }
    }
    {
        const long long cnt = (d->sigma_stride == 0) ? 1 : d->B;
        for (long long q = 0; d->sigma && q < cnt; ++q)
            for (int i = 0; i < d->D; ++i)
                if (!(d->sigma[q * d->sigma_stride + i] > 0.0))
                    return bail(h->fail(VGPA_EINVAL, "The diffusion noise value should be strictly positive"));
    }
    if (cudaSetDevice(d->device) != cudaSuccess)
        return bail(h->fail(VGPA_ECUDA, "cudaSetDevice(%d) failed: no usable CUDA device", d->device));
    {
        cudaDeviceProp prop;
        cudaError_t e = cudaGetDeviceProperties(&prop, d->device);
        if (e != cudaSuccess) return bail(h->cuda_fail(e, "cudaGetDeviceProperties"));
        if (prop.major != 10)
            return bail(h->fail(VGPA_ECUDA, "device %d is sm_%d%d; this library is built for sm_100a only",
                                d->device, prop.major, prop.minor));
    }
    const int D = d->D, N = d->N, M = d->M, B = d->B;
    h->n_x = (long long)N * D * (D + 1);
    Batch& b = h->batch;
    b.model = d->model; b.method = d->method; b.D = D; b.N = N; b.M = M; b.B = B;
    b.dt = d->dt; b.dt_model = d->dt_model;
    // a per-problem parameter: one row shared by the batch (stride 0) or B rows `stride` apart
    auto upload_param = [&](DevBuf& buf, const double* src, long long stride, long long len, const double** dev,
                            long long* dev_stride, const char* name) -> int {
        if (src == nullptr) return h->fail(VGPA_EINVAL, "descriptor field %s is NULL", name);
        if (stride != 0 && stride < len) return h->fail(VGPA_EINVAL, "%s_stride %lld < %lld", name, stride, len);
        cudaError_t e = cudaSuccess;
        stage_rows(e, buf, src, stride, len, B, dev_stride);
        if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_create(params)");
        *dev = buf.as<double>();
        return VGPA_OK;
    };
    // Partially observed problems: the device copies of R and obs_y hold +inf and 0 at every unobserved (problem,
    // component), so that the sweeps' jumps -(y - m) / R and 0.5 / R are zeros there without a mask, and neither a NaN
    // nor any other value the caller left in those entries reaches the arithmetic.  B rows, or one when the values
    // and the masks are both shared.
    std::vector<double> R_obs, y_obs;
    const double* R_src = d->R;
    const double* y_src = d->obs_y;
    long long R_stride = d->R_stride, y_stride = d->obs_y_stride;
    auto mask_rows = [&](const double*& src, long long& stride, long long len, double fill, std::vector<double>& v) {
        if (observed == nullptr || src == nullptr || (stride != 0 && stride < len)) return;   // upload_param reports these
        const int rows = (stride == 0 && observed_stride == 0) ? 1 : B;
        v.resize((size_t)rows * len);
        for (int p = 0; p < rows; ++p) {
            const uint64_t w = observed[p * observed_stride];
            for (long long k = 0; k < len; ++k)
                v[(size_t)p * len + k] = ((w >> (k % D)) & 1) ? src[p * stride + k] : fill;
        }
        src = v.data();
        stride = rows == 1 ? 0 : len;
    };
    mask_rows(R_src, R_stride, D, INFINITY, R_obs);
    if (M > 0) mask_rows(y_src, y_stride, (long long)M * D, 0.0, y_obs);
    int rc;
#define UP_FROM(field, src, stride, len)                                                                      \
    if ((rc = upload_param(h->field, (src), (stride), (len), &b.field, &b.field##_stride, #field)) != VGPA_OK) \
        return bail(rc);
#define UP(field, len) UP_FROM(field, d->field, d->field##_stride, len)
    UP(theta, n_theta(d->model));
    UP(sigma, D);
    UP_FROM(R, R_src, R_stride, D);
    UP(m0, D);
    UP(s0, (long long)D * D);
    UP(E0, 1);
    if (M > 0) {
        UP_FROM(obs_y, y_src, y_stride, (long long)M * D);
    } else {
        b.obs_y = nullptr;
        b.obs_y_stride = 0;
    }
#undef UP
#undef UP_FROM
    if (observed != nullptr) {   // one word per problem on the device (a shared mask expanded)
        std::vector<unsigned long long> w(B);
        for (int p = 0; p < B; ++p) w[p] = observed[p * observed_stride];
        cudaError_t e = cudaSuccess;
        upload(e, h->observed, w.data(), w.size());
        if (e != cudaSuccess) return bail(h->cuda_fail(e, "upload(observed)"));
        b.observed = h->observed.as<unsigned long long>();
    }
    if (!rows) {
        std::vector<long long> ot(std::max(M, 1), 0);
        std::vector<int> oi(N, -1);
        for (int n = 0; n < M; ++n) {
            ot[n] = d->obs_t[n];
            oi[d->obs_t[n]] = n;
        }
        cudaError_t e = cudaSuccess;
        upload(e, h->obs_t, ot.data(), ot.size());
        upload(e, h->obs_index, oi.data(), oi.size());
        if (e != cudaSuccess) return bail(h->cuda_fail(e, "upload(obs_t)"));
        b.obs_t = h->obs_t.as<long long>();
        b.obs_index = h->obs_index.as<int>();
    } else {
        // (B, max(M, 1)) index rows, the (B, N) ordinal table the backward sweeps read at every step, B counts
        const long long Mc = std::max(M, 1);
        std::vector<long long> ot((size_t)B * Mc, 0);
        std::vector<int> oi((size_t)B * N, -1), cnt(B);
        for (int p = 0; p < B; ++p) {
            cnt[p] = counts ? counts[p] : M;
            const int64_t* src = obs_t + p * obs_t_stride;
            for (int n = 0; n < cnt[p]; ++n) {
                ot[(size_t)p * Mc + n] = src[n];
                oi[(size_t)p * N + src[n]] = n;
            }
        }
        cudaError_t e = cudaSuccess;
        upload(e, h->obs_t, ot.data(), ot.size());
        upload(e, h->obs_index, oi.data(), oi.size());
        upload(e, h->obs_count, cnt.data(), cnt.size());
        if (e != cudaSuccess) return bail(h->cuda_fail(e, "upload(obs_t)"));
        b.obs_t = h->obs_t.as<long long>();
        b.obs_index = h->obs_index.as<int>();
        b.obs_count = h->obs_count.as<int>();
        b.obs_t_stride = Mc;
        b.obs_index_stride = N;
        h->obs_rows = true;
    }
    // ---- scratch: trajectories for one chunk of problems ----
    const long long per = 8LL * N * (2LL * D + 2LL * D * D + 1);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    long long budget = d->scratch_bytes > 0 ? d->scratch_bytes : std::min<long long>(56LL << 30, (long long)(free_b * 0.35));
    long long chunk = std::max<long long>(1, std::min<long long>(B, budget / per));
    if (!small_model(d->model) && chunk < B) {
        if (d->scratch_bytes > 0 && l96_tuned(D)) {
            // caller-given budget: whole waves (multiples of 6 * 148: 3 backward / 4 forward CTAs per SM of the D = 40
            // kernels) when it allows
            const long long wave = 148 * 6;
            if (chunk >= wave) chunk = (chunk / wave) * wave;
            else if (chunk >= 148) chunk = (chunk / 148) * 148;
        } else {
            // default: as FEW passes as the budget allows, of EQUAL size.  Every pass ends in a partial wave of the
            // sweeps (one CTA per problem, a 1001-step recurrence each: the last CTAs run alone), so two passes of
            // 2048 problems beat four of 888 plus one of 544 by 2.3 % on the 4096-problem shard (measured; 54 GB
            // of scratch instead of 23)
            const long long passes = (B + chunk - 1) / chunk;
            chunk = (B + passes - 1) / passes;
        }
    }
    if (const char* ce = getenv("VGPA_CHUNK")) {   // experiments: explicit problems per pass
        const long long c = atoll(ce);
        if (c >= 1) chunk = std::min<long long>(c, B);
    }
    h->chunk = (int)chunk;
    {
        cudaError_t e = h->sc.alloc(chunk, N, D);
        alloc<int>(e, h->status, B);
        if (e == cudaSuccess) e = cudaMemset(h->status.p, 0, sizeof(int) * B);
        if (e != cudaSuccess) return bail(h->cuda_fail(e, "cudaMalloc(scratch)"));
    }
    {
        cudaError_t e;
        if ((e = cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking)) != cudaSuccess)
            return bail(h->cuda_fail(e, "cudaStreamCreate"));
        for (int q = 0; q < 2; ++q)
            if ((e = cudaEventCreateWithFlags(&h->ev_h2d[q], cudaEventDisableTiming)) != cudaSuccess ||
                (e = cudaEventCreateWithFlags(&h->ev_comp[q], cudaEventDisableTiming)) != cudaSuccess ||
                (e = cudaEventCreateWithFlags(&h->ev_d2h[q], cudaEventDisableTiming)) != cudaSuccess)
                return bail(h->cuda_fail(e, "cudaEventCreate"));
    }
    *out = h;
    return VGPA_OK;
}

}  // namespace

extern "C" {

int vgpa_create(const vgpa_desc* d, vgpa_handle** out)
{
    if (out) *out = nullptr;
    if (d == nullptr || out == nullptr) return set_error(VGPA_EINVAL, "vgpa_create: NULL argument");
    return create_handle(d, nullptr, 0, nullptr, false, nullptr, 0, out);
}

int vgpa_create_observed(const vgpa_desc* d, const int64_t* obs_t, int64_t obs_t_stride, const int32_t* M,
                         const uint64_t* observed, int64_t observed_stride, vgpa_handle** out)
{
    if (out) *out = nullptr;
    if (d == nullptr || out == nullptr) return set_error(VGPA_EINVAL, "vgpa_create_observed: NULL argument");
    if (obs_t_stride == 0 && M == nullptr && d->obs_t == nullptr) {   // one shared schedule: that of vgpa_create
        vgpa_desc one = *d;
        one.obs_t = obs_t;
        return create_handle(&one, nullptr, 0, nullptr, false, observed, observed_stride, out);
    }
    return create_handle(d, obs_t, obs_t_stride, M, true, observed, observed_stride, out);
}

int vgpa_create_obs_rows(const vgpa_desc* d, const int64_t* obs_t, int64_t obs_t_stride, const int32_t* M,
                         vgpa_handle** out)
{
    if (out) *out = nullptr;
    if (d == nullptr || out == nullptr) return set_error(VGPA_EINVAL, "vgpa_create_obs_rows: NULL argument");
    return vgpa_create_observed(d, obs_t, obs_t_stride, M, nullptr, 0, out);
}

void vgpa_destroy(vgpa_handle* h)
{
    if (!h) return;
    cudaSetDevice(h->d.device);
    cudaDeviceSynchronize();
    if (h->s_aux) cudaStreamDestroy(h->s_aux);
    for (int q = 0; q < 2; ++q)
        if (h->plist_ev[q]) cudaEventDestroy(h->plist_ev[q]);
    for (int q = 0; q < 2; ++q) {
        if (h->ev_h2d[q]) cudaEventDestroy(h->ev_h2d[q]);
        if (h->ev_comp[q]) cudaEventDestroy(h->ev_comp[q]);
        if (h->ev_d2h[q]) cudaEventDestroy(h->ev_d2h[q]);
    }
    for (int k = 0; k < 4; ++k)
        for (auto& pr : h->tev[k]) {
            cudaEventDestroy(pr.first);
            cudaEventDestroy(pr.second);
        }
    if (h->ev_done) cudaEventDestroy(h->ev_done);
    if (h->s_comp) cudaStreamDestroy(h->s_comp);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    delete h;   // frees the device buffers, with the handle's device current
}

int vgpa_eval_device(vgpa_handle* h, const double* d_x, int64_t x_stride, int want_grad, double* d_F,
                     double* d_grad, int64_t grad_stride, void* stream)
{
    if (!h) return VGPA_EINVAL;
    if (d_x == nullptr || d_F == nullptr) return h->fail(VGPA_EINVAL, "x / F is NULL");
    if (want_grad && d_grad == nullptr) return h->fail(VGPA_EINVAL, "want_grad set but grad is NULL");
    if (x_stride != 0 && x_stride < h->n_x) return h->fail(VGPA_EINVAL, "x_stride %lld < %lld", (long long)x_stride, h->n_x);
    if (want_grad && grad_stride < h->n_x && h->d.B > 1)
        return h->fail(VGPA_EINVAL, "grad_stride %lld < %lld", (long long)grad_stride, h->n_x);
    if (((uintptr_t)d_x & 15) || (x_stride & 1) || (want_grad && (((uintptr_t)d_grad & 15) || (grad_stride & 1))))
        return h->fail(VGPA_EINVAL, "device buffers must be 16-byte aligned with even strides");
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // The handle owns ONE scratch and one set of status words: an evaluation enqueued on another stream than the
    // previous one is ordered after it (same stream: stream order does it).
    if (h->ev_done != nullptr && h->status_dirty && st != h->last_stream)
        CK(cudaStreamWaitEvent(st, h->ev_done, 0), "cudaStreamWaitEvent");
    CK(cudaMemsetAsync(h->status.p, 0, sizeof(int) * h->d.B, st), "cudaMemsetAsync(status)");
    Extra ex{};
    const bool compacted = h->n_list >= 0 && h->batch.plist != nullptr;
    const int total = compacted ? h->n_list : h->d.B;   // launch positions
    if (compacted) h->status_map = h->plist_host;     // vgpa_sync names problems by this list, even if it changes first
    else h->status_map.clear();
    for (int p0 = 0; p0 < total; p0 += h->chunk) {
        const int count = std::min(h->chunk, total - p0);
        run_chunk(h, d_x, x_stride, want_grad, d_F, d_grad, grad_stride, p0, count, ex, st);
    }
    CK(cudaGetLastError(), "kernel launch");
    if (compacted) {   // this evaluation reads the current copy of the list
        const int q = h->plist_flip;
        if (h->plist_ev[q] == nullptr) CK(cudaEventCreateWithFlags(&h->plist_ev[q], cudaEventDisableTiming), "cudaEventCreate");
        CK(cudaEventRecord(h->plist_ev[q], st), "cudaEventRecord");
        h->plist_used[q] = true;
    }
    if (h->ev_done == nullptr) CK(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming), "cudaEventCreate");
    CK(cudaEventRecord(h->ev_done, st), "cudaEventRecord");
    h->last_stream = st;
    h->status_dirty = true;
    return VGPA_OK;
}

int vgpa_hyper_device(vgpa_handle* h, const double* d_x, int64_t x_stride, double* d_F, double* d_Esde,
                      double* d_dtheta, int64_t dtheta_stride, double* d_dsigma, int64_t dsigma_stride, void* stream)
{
    if (!h) return VGPA_EINVAL;
    if (d_x == nullptr) return h->fail(VGPA_EINVAL, "x is NULL");
    if (x_stride != 0 && x_stride < h->n_x) return h->fail(VGPA_EINVAL, "x_stride %lld < %lld", (long long)x_stride, h->n_x);
    if (((uintptr_t)d_x & 15) || (x_stride & 1))
        return h->fail(VGPA_EINVAL, "device buffers must be 16-byte aligned with even strides");
    const int D = h->d.D, B = h->d.B;
    const long long nth = hyper_ntheta(h->batch.model, D), nsig = (D == 1) ? 1 : (long long)D * D;
    if (d_dtheta != nullptr && dtheta_stride < nth && !(B == 1 && dtheta_stride == 0))
        return h->fail(VGPA_EINVAL, "dtheta_stride %lld < %lld", (long long)dtheta_stride, nth);
    if (d_dsigma != nullptr && dsigma_stride < nsig && !(B == 1 && dsigma_stride == 0))
        return h->fail(VGPA_EINVAL, "dsigma_stride %lld < %lld", (long long)dsigma_stride, nsig);
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // one scratch, one set of status words: ordered after the previous evaluation as in vgpa_eval_device
    if (h->ev_done != nullptr && h->status_dirty && st != h->last_stream)
        CK(cudaStreamWaitEvent(st, h->ev_done, 0), "cudaStreamWaitEvent");
    CK(cudaMemsetAsync(h->status.p, 0, sizeof(int) * B, st), "cudaMemsetAsync(status)");
    // every problem is served, its status word indexed by problem; the kernels take the Batch by value, so the
    // active set and the list are back in place for later calls as soon as the launches are enqueued
    const int *active = h->batch.active, *plist = h->batch.plist;
    h->batch.active = nullptr;
    h->batch.plist = nullptr;
    h->status_map.clear();
    const HyperOut o{d_Esde, d_dtheta, dtheta_stride, d_dsigma, dsigma_stride};
    for (int p0 = 0; p0 < B; p0 += h->chunk)
        run_hyper_chunk(h, d_x, x_stride, d_F, o, p0, std::min(h->chunk, B - p0), st);
    h->batch.active = active;
    h->batch.plist = plist;
    CK(cudaGetLastError(), "kernel launch");
    if (h->ev_done == nullptr) CK(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming), "cudaEventCreate");
    CK(cudaEventRecord(h->ev_done, st), "cudaEventRecord");
    h->last_stream = st;
    h->status_dirty = true;
    return VGPA_OK;
}

int vgpa_set_active(vgpa_handle* h, const int32_t* d_active)
{
    if (!h) return VGPA_EINVAL;
    h->batch.active = d_active;
    return VGPA_OK;
}

int vgpa_set_active_list(vgpa_handle* h, const int32_t* list, int32_t n)
{
    if (!h) return VGPA_EINVAL;
    if (list == nullptr || n < 0) {
        h->n_list = -1;
        h->batch.plist = nullptr;
        h->plist_host.clear();
        return VGPA_OK;
    }
    if (h->batch.model != MODEL_L96)
        return h->fail(VGPA_EINVAL, "vgpa_set_active_list: compacted launches exist for the Lorenz-96 kernels only "
                                    "(use vgpa_set_active for the small models)");
    if (n > h->d.B) return h->fail(VGPA_EINVAL, "vgpa_set_active_list: %d entries for %d problems", (int)n, h->d.B);
    for (int k = 0; k < n; ++k)
        if (list[k] < 0 || list[k] >= h->d.B)
            return h->fail(VGPA_EINVAL, "vgpa_set_active_list: entry %d = %d outside [0, %d)", k, (int)list[k], h->d.B);
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    // Upload on a private non-blocking stream into the buffer the evaluation in flight does NOT read: the call
    // waits for its own tiny copy only, never for the kernels already enqueued on the caller's stream.
    h->plist_flip ^= 1;
    DevBuf& buf = h->plist2[h->plist_flip];
    if (h->plist_used[h->plist_flip]) {    // an evaluation two list changes ago read this copy: it must be over
        CK(cudaEventSynchronize(h->plist_ev[h->plist_flip]), "cudaEventSynchronize");
        h->plist_used[h->plist_flip] = false;
    }
    const size_t bytes = sizeof(int) * (size_t)std::max(h->d.B, 1);
    if (buf.bytes < bytes) CK(buf.alloc(bytes), "cudaMalloc(list)");
    if (h->s_aux == nullptr) CK(cudaStreamCreateWithFlags(&h->s_aux, cudaStreamNonBlocking), "cudaStreamCreate");
    if (n > 0) {
        CK(cudaMemcpyAsync(buf.p, list, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, h->s_aux), "cudaMemcpyAsync(list)");
        CK(cudaStreamSynchronize(h->s_aux), "cudaStreamSynchronize");
    }
    h->plist_host.assign(list, list + n);
    h->n_list = n;
    h->batch.plist = buf.as<int>();
    return VGPA_OK;
}

long long vgpa_scratch_cache(int enable)
{
    {
        std::lock_guard<std::mutex> lk(g_block_cache.mu);
        g_block_cache.enabled = enable != 0;
    }
    return enable ? 0 : g_block_cache.purge();
}

int vgpa_sync(vgpa_handle* h)
{
    if (!h) return VGPA_EINVAL;
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    CK(cudaStreamSynchronize(h->last_stream), "cudaStreamSynchronize");
    return check_status(h);
}

int vgpa_eval(vgpa_handle* h, const double* x, int64_t x_stride, int want_grad, double* F, double* grad,
              int64_t grad_stride)
{
    if (!h) return VGPA_EINVAL;
    if (x == nullptr || F == nullptr) return h->fail(VGPA_EINVAL, "x / F is NULL");
    if (want_grad && grad == nullptr) return h->fail(VGPA_EINVAL, "want_grad set but grad is NULL");
    if (x_stride != 0 && x_stride < h->n_x) return h->fail(VGPA_EINVAL, "x_stride %lld < %lld", (long long)x_stride, h->n_x);
    if (want_grad && h->d.B > 1 && grad_stride < h->n_x)
        return h->fail(VGPA_EINVAL, "grad_stride %lld < %lld", (long long)grad_stride, h->n_x);
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    HostCallScope scope(h);
    // host buffers: short passes, so that the H2D copy of pass c + 1, the kernels of pass c and the D2H copy of
    // pass c - 1 overlap and the two staging slots per direction stay small (D = 40: 64 problems = 0.84 GB each)
    const int B = h->d.B, C = small_model(h->batch.model) ? h->chunk : std::min(h->chunk, 64);
    const long long nx = h->n_x;
    const bool shared_x = (x_stride == 0);
    // staging (lazily sized): per slot one chunk of x rows and gradient rows
    const size_t xbytes = sizeof(double) * (size_t)nx * (shared_x ? 1 : C);
    const int nslots = (B > C) ? 2 : 1;
    for (int q = 0; q < nslots; ++q) {
        if (h->st_x[q].bytes < xbytes) CK(h->st_x[q].alloc(xbytes), "cudaMalloc(x staging)");
        if (want_grad && h->st_g[q].bytes < sizeof(double) * (size_t)nx * C)
            CK(h->st_g[q].alloc(sizeof(double) * (size_t)nx * C), "cudaMalloc(grad staging)");
    }
    if (h->st_F.bytes < sizeof(double) * B) CK(h->st_F.alloc(sizeof(double) * B), "cudaMalloc(F)");
    CK(cudaMemsetAsync(h->status.p, 0, sizeof(int) * B, h->s_comp), "cudaMemsetAsync(status)");
    Extra ex{};
    int ci = 0;
    for (int p0 = 0; p0 < B; p0 += C, ++ci) {
        const int count = std::min(C, B - p0);
        const int q = ci & 1;
        // slot q: its previous gradients must have left and its previous x must be consumed
        if (ci >= 2) {
            CK(cudaStreamWaitEvent(h->s_h2d, h->ev_comp[q], 0), "cudaStreamWaitEvent");
            CK(cudaStreamWaitEvent(h->s_comp, h->ev_d2h[q], 0), "cudaStreamWaitEvent");
        }
        if (!shared_x || ci == 0) {
            if (shared_x) {
                CK(cudaMemcpyAsync(h->st_x[0].p, x, sizeof(double) * nx, cudaMemcpyHostToDevice, h->s_h2d), "H2D x");
            } else if (x_stride == nx) {
                CK(cudaMemcpyAsync(h->st_x[q].p, x + (long long)p0 * x_stride, sizeof(double) * nx * count,
                                   cudaMemcpyHostToDevice, h->s_h2d), "H2D x");
            } else {
                CK(cudaMemcpy2DAsync(h->st_x[q].p, sizeof(double) * nx, x + (long long)p0 * x_stride,
                                     sizeof(double) * x_stride, sizeof(double) * nx, count,
                                     cudaMemcpyHostToDevice, h->s_h2d), "H2D x");
            }
        }
        CK(cudaEventRecord(h->ev_h2d[q], h->s_h2d), "cudaEventRecord");
        CK(cudaStreamWaitEvent(h->s_comp, h->ev_h2d[q], 0), "cudaStreamWaitEvent");
        // kernels index problems globally (p0 + lp): offset the staged pointers accordingly
        const double* dx = shared_x ? h->st_x[0].as<double>() : h->st_x[q].as<double>() - (long long)p0 * nx;
        double* dg = want_grad ? h->st_g[q].as<double>() - (long long)p0 * nx : nullptr;
        run_chunk(h, dx, shared_x ? 0 : nx, want_grad, h->st_F.as<double>(), dg, nx, p0, count, ex, h->s_comp);
        CK(cudaGetLastError(), "kernel launch");
        CK(cudaEventRecord(h->ev_comp[q], h->s_comp), "cudaEventRecord");
        if (want_grad) {
            CK(cudaStreamWaitEvent(h->s_d2h, h->ev_comp[q], 0), "cudaStreamWaitEvent");
            if (grad_stride == nx || count == 1) {
                CK(cudaMemcpyAsync(grad + (long long)p0 * grad_stride, h->st_g[q].p, sizeof(double) * nx * count,
                                   cudaMemcpyDeviceToHost, h->s_d2h), "D2H grad");
            } else {
                CK(cudaMemcpy2DAsync(grad + (long long)p0 * grad_stride, sizeof(double) * grad_stride, h->st_g[q].p,
                                     sizeof(double) * nx, sizeof(double) * nx, count, cudaMemcpyDeviceToHost,
                                     h->s_d2h), "D2H grad");
            }
            CK(cudaEventRecord(h->ev_d2h[q], h->s_d2h), "cudaEventRecord");
        }
    }
    CK(cudaMemcpyAsync(F, h->st_F.p, sizeof(double) * B, cudaMemcpyDeviceToHost, h->s_comp), "D2H F");
    CK(cudaStreamSynchronize(h->s_comp), "cudaStreamSynchronize");
    CK(cudaStreamSynchronize(h->s_d2h), "cudaStreamSynchronize");
    h->status_dirty = true;
    return check_status(h);
}

int vgpa_eval_full(vgpa_handle* h, int64_t problem, const double* x, const vgpa_full_out* out)
{
    if (!h) return VGPA_EINVAL;
    if (x == nullptr || out == nullptr) return h->fail(VGPA_EINVAL, "x / out is NULL");
    if (problem < 0 || problem >= h->d.B) return h->fail(VGPA_EINVAL, "problem index %lld out of range", (long long)problem);
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    HostCallScope scope(h);
    const long long nx = h->n_x, N = h->d.N, D = h->d.D, nv = N * D, nm = N * D * D;
    DevBuf dx, dg, dF, dl, dp, def, dedf, dparts;
    cudaError_t e = cudaSuccess;
    upload(e, dx, x, nx);
    alloc(e, dg, nx);
    alloc(e, dF, h->d.B);
    alloc(e, dl, nv);
    alloc(e, dp, nm);
    alloc(e, def, nv);
    alloc(e, dedf, nm);
    alloc(e, dparts, 3);
    if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_eval_full setup");
    Extra ex{};
    ex.lamt = dl.as<double>(); ex.psit = dp.as<double>(); ex.Efx = def.as<double>(); ex.Edf = dedf.as<double>();
    ex.parts = dparts.as<double>();
    cudaMemsetAsync(h->status.p, 0, sizeof(int) * h->d.B, h->s_comp);
    // kernels address x / grad / F by global problem index
    run_chunk(h, dx.as<double>() - problem * nx, nx, 1, dF.as<double>(), dg.as<double>() - problem * nx, nx,
              (int)problem, 1, ex, h->s_comp);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->s_comp);
    if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_eval_full kernels");
    download(e, out->F, dF.as<double>() + problem, 1);
    download(e, out->parts, dparts.p, 3);
    download(e, out->grad, dg.p, nx);
    download(e, out->mt, h->sc.mt.p, nv);
    download(e, out->st, h->sc.st.p, nm);
    download(e, out->lamt, dl.p, nv);
    download(e, out->psit, dp.p, nm);
    download(e, out->Efx, def.p, nv);
    download(e, out->Edf, dedf.p, nm);
    download(e, out->dEsde_dm, h->sc.dEm.p, nv);
    download(e, out->dEsde_ds, h->sc.dEs.p, nm);
    if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_eval_full copy-back");
    h->status_dirty = true;
    return check_status(h);
}

// ---- stand-alone sweeps (FwdOde.__call__ / BwdOde.__call__) -------------------------
static int check_sweep_args(int method, int D, int N, double dt)
{
    if (method < 0 || method > 3) return set_error(VGPA_EINVAL, "Integration method is unknown");
    if (D != 1 && D != 3 && (D < 10 || D > 64))
        return set_error(VGPA_EINVAL, "unsupported state dimension %d (1, 3 or 10 <= D <= 64)", D);
    if (N < 2) return set_error(VGPA_EINVAL, "need at least two time points");
    if (!(dt > 0.0)) return set_error(VGPA_EINVAL, "Discrete time step should be strictly positive");
    return VGPA_OK;
}

int vgpa_solve_fwd(int device, int method, int D, int N, double dt, const double* A, const double* b,
                   const double* m0, const double* s0, const double* sigma, double* mt, double* st)
{
    if (int rc = check_sweep_args(method, D, N, dt)) return rc;
    if (!A || !b || !m0 || !s0 || !sigma || !mt || !st) return set_error(VGPA_EINVAL, "NULL argument");
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    const long long nv = (long long)N * D, nm = (long long)N * D * D;
    DevBuf dx, dm0, ds0, dsig, dmt, dst;
    cudaError_t e = cudaSuccess;
    alloc(e, dx, nm + nv);
    to_device(e, dx.as<double>(), A, nm);
    to_device(e, dx.as<double>() + nm, b, nv);
    upload(e, dm0, m0, D);
    upload(e, ds0, s0, (size_t)D * D);
    upload(e, dsig, sigma, D);
    alloc(e, dmt, nv);
    alloc(e, dst, nm);
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_solve_fwd");
    Batch bt{};
    bt.model = (D >= 10) ? MODEL_L96 : (D == 3 ? MODEL_L63 : MODEL_OU);
    bt.method = method; bt.D = D; bt.N = N; bt.B = 1; bt.dt = dt; bt.dt_model = dt;
    bt.sigma = dsig.as<double>(); bt.m0 = dm0.as<double>(); bt.s0 = ds0.as<double>();
    Scratch sc{};
    sc.mt = dmt.as<double>(); sc.st = dst.as<double>();
    if (D >= 10) l96_fwd(bt, sc, dx.as<double>(), 0, 0, 1, nullptr);
    else launch_small_fwd(bt, sc, dx.as<double>(), 0, 0, 1, nullptr);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    download(e, mt, dmt.p, nv);
    download(e, st, dst.p, nm);
    return e == cudaSuccess ? VGPA_OK : set_cuda_error(e, "vgpa_solve_fwd");
}

int vgpa_solve_bwd(int device, int method, int D, int N, double dt, const double* A, const double* dEm,
                   const double* dEs, const double* jm, const double* js, double* lam, double* psi)
{
    if (int rc = check_sweep_args(method, D, N, dt)) return rc;
    if (!A || !dEm || !dEs || !jm || !js || !lam || !psi) return set_error(VGPA_EINVAL, "NULL argument");
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    const long long nv = (long long)N * D, nm = (long long)N * D * D;
    DevBuf dA, dgm, dgs, djm, djs, dl, dp;
    cudaError_t e = cudaSuccess;
    upload(e, dA, A, nm);
    upload(e, dgm, dEm, nv);
    upload(e, dgs, dEs, nm);
    upload(e, djm, jm, nv);
    upload(e, djs, js, nm);
    alloc(e, dl, nv);
    alloc(e, dp, nm);
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_solve_bwd");
    launch_bwd_dense(method, D, N, dt, dA.as<double>(), dgm.as<double>(), dgs.as<double>(), djm.as<double>(),
                     djs.as<double>(), dl.as<double>(), dp.as<double>(), nullptr);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    download(e, lam, dl.p, nv);
    download(e, psi, dp.p, nm);
    return e == cudaSuccess ? VGPA_OK : set_cuda_error(e, "vgpa_solve_bwd");
}

int vgpa_model_energy(int device, int model, int D, int N, double dt_model, const double* theta,
                      const double* sigma, const double* A, const double* b, const double* m, const double* S,
                      double* Esde, double* Ef, double* Edf, double* dEm, double* dEs, double* dEth, double* dEsig)
{
    if (model < 0 || model > 3) return set_error(VGPA_EINVAL, "Unknown stochastic model");
    const bool okD = (model == VGPA_MODEL_L96) ? (D >= 10 && D <= 64) : (D == ((model == VGPA_MODEL_L63) ? 3 : 1));
    if (!okD || N < 2 || !(dt_model > 0.0)) return set_error(VGPA_EINVAL, "Wrong dimensions for model.energy");
    if (!theta || !sigma || !A || !b || !m || !S || !Esde || !Ef || !Edf || !dEm || !dEs)
        return set_error(VGPA_EINVAL, "NULL argument");
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    const long long nv = (long long)N * D, nm = (long long)N * D * D;
    const int nth = n_theta(model);
    DevBuf dx, dth, dsig, dmt, dst, dgm, dgs, des, def, dedf, dparts, dzero, dF, dstat, dterms, dhth, dhsig;
    const bool hyper = (dEth != nullptr) || (dEsig != nullptr);
    const int nhth = hyper_ntheta(model, D);
    const long long nsig = (D == 1) ? 1 : (long long)D * D;
    cudaError_t e = cudaSuccess;
    alloc(e, dx, nm + nv);
    to_device(e, dx.as<double>(), A, nm);
    to_device(e, dx.as<double>() + nm, b, nv);
    upload(e, dth, theta, nth);
    upload(e, dsig, sigma, D);
    upload(e, dmt, m, nv);
    upload(e, dst, S, nm);
    alloc(e, dgm, nv);
    alloc(e, dgs, nm);
    alloc(e, des, N);
    alloc(e, def, nv);
    alloc(e, dedf, nm);
    alloc(e, dparts, 3);
    alloc(e, dzero, 1);
    alloc(e, dF, 1);
    alloc<int>(e, dstat, 1);
    if (e == cudaSuccess) e = cudaMemset(dzero.p, 0, sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(dstat.p, 0, sizeof(int));
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_model_energy");
    Batch bt{};
    bt.model = model; bt.method = ODE_EULER; bt.D = D; bt.N = N; bt.M = 0; bt.B = 1;
    bt.dt = dt_model; bt.dt_model = dt_model;
    bt.theta = dth.as<double>(); bt.sigma = dsig.as<double>(); bt.R = dsig.as<double>();
    bt.E0 = dzero.as<double>();
    Scratch sc{};
    sc.mt = dmt.as<double>(); sc.st = dst.as<double>(); sc.dEm = dgm.as<double>(); sc.dEs = dgs.as<double>();
    sc.esde_t = des.as<double>(); sc.status = dstat.as<int>();
    Extra ex{};
    ex.Efx = def.as<double>(); ex.Edf = dedf.as<double>(); ex.parts = dparts.as<double>();
    if (model == VGPA_MODEL_L96) l96_energy(bt, sc, dx.as<double>(), 0, 0, 1, ex, nullptr);
    else launch_small_energy(bt, sc, dx.as<double>(), 0, 0, 1, ex, nullptr);
    launch_finalize(bt, sc, dF.as<double>(), 0, 1, ex, nullptr);
    if (hyper) {   // the launchers of vgpa_hyper_device with B = 1; the integrands go to a buffer of their own
        alloc(e, dterms, (size_t)N * (nhth + (D == 1 ? 0 : D)));
        alloc(e, dhth, nhth);
        alloc(e, dhsig, nsig);
        if (e != cudaSuccess) return set_cuda_error(e, "vgpa_model_energy");
        Scratch hs = sc;
        hs.dEs = dterms.as<double>();
        launch_hyper_terms(bt, hs, dx.as<double>(), 0, 0, 1, nullptr);
        launch_hyper_reduce(bt, hs, 0, 1, HyperOut{nullptr, dhth.as<double>(), 0, dhsig.as<double>(), 0}, nullptr);
    }
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    double parts[3] = {0, 0, 0};
    int stat = 0;
    download(e, parts, dparts.p, 3);
    download(e, &stat, dstat.p, 1);
    download(e, dEth, dhth.p, nhth);
    download(e, dEsig, dhsig.p, nsig);
    download(e, Ef, def.p, nv);
    download(e, Edf, dedf.p, nm);
    download(e, dEm, dgm.p, nv);
    download(e, dEs, dgs.p, nm);
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_model_energy");
    if (stat != 0) return set_error(VGPA_ENOTPD, "Matrix is not positive definite: S(t) at time index %d", stat - 1);
    *Esde = parts[1];
    return VGPA_OK;
}

}  // extern "C"

// vgpa_obs_energy and vgpa_obs_energy_observed: the components whose bit of `observed` is clear are left out of Eobs
// and keep zero jumps.
static int obs_energy(int device, int D, int N, int M, const int64_t* obs_t, const double* obs_y, const double* R,
                      uint64_t observed, const double* mt, const double* st, double* Eobs, double* jm, double* js,
                      double* dr)
{
    if ((D != 1 && D != 3 && (D < 10 || D > 64)) || N < 2 || M < 0 || M > N)
        return set_error(VGPA_EINVAL, "Wrong dimensions for the likelihood");
    if ((M > 0 && (!obs_t || !obs_y)) || !R || !mt || !st || !Eobs || !jm || !js) return set_error(VGPA_EINVAL, "NULL argument");
    for (int n = 0; n < M; ++n)
        if (obs_t[n] < 0 || obs_t[n] >= N) return set_error(VGPA_EINVAL, "observation index out of range");
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    const long long nv = (long long)N * D, nm = (long long)N * D * D;
    DevBuf dot, doy, dR, dmt, dst, djm, djs, des, dparts, dzero, dF, ddr, dobs;
    std::vector<long long> ot(std::max(M, 1), 0);
    for (int n = 0; n < M; ++n) ot[n] = obs_t[n];
    const unsigned long long word = observed;
    cudaError_t e = cudaSuccess;
    upload(e, dot, ot.data(), ot.size());
    upload(e, dobs, &word, 1);
    alloc(e, doy, (size_t)std::max(M, 1) * D);
    if (M > 0) to_device(e, doy.p, obs_y, (size_t)M * D);
    upload(e, dR, R, D);
    upload(e, dmt, mt, nv);
    upload(e, dst, st, nm);
    alloc(e, djm, nv);
    alloc(e, djs, nm);
    alloc(e, des, N);
    alloc(e, dparts, 3);
    alloc(e, dzero, 1);
    alloc(e, dF, 1);
    if (e == cudaSuccess) e = cudaMemset(dzero.p, 0, sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(des.p, 0, sizeof(double) * N);
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_obs_energy");
    Batch bt{};
    bt.model = (D == 1) ? MODEL_OU : (D == 3 ? MODEL_L63 : MODEL_L96);
    bt.D = D; bt.N = N; bt.M = M; bt.B = 1; bt.dt = 1.0; bt.dt_model = 1.0;
    bt.sigma = dR.as<double>(); bt.R = dR.as<double>(); bt.E0 = dzero.as<double>();
    bt.obs_t = dot.as<long long>(); bt.obs_y = doy.as<double>(); bt.observed = dobs.as<unsigned long long>();
    Scratch sc{};
    sc.mt = dmt.as<double>(); sc.st = dst.as<double>(); sc.esde_t = des.as<double>();
    Extra ex{};
    ex.parts = dparts.as<double>();
    launch_finalize(bt, sc, dF.as<double>(), 0, 1, ex, nullptr);
    launch_jump_tables(D, N, M, dot.as<long long>(), doy.as<double>(), dR.as<double>(), observed, dmt.as<double>(),
                       djm.as<double>(), djs.as<double>(), nullptr);
    if (dr != nullptr && D == 1) {
        alloc(e, ddr, N);
        if (e != cudaSuccess) return set_cuda_error(e, "vgpa_obs_energy");
        launch_obs_dr(N, M, dot.as<long long>(), doy.as<double>(), dR.as<double>(), dmt.as<double>(), dst.as<double>(),
                      ddr.as<double>(), nullptr);
    }
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    double parts[3] = {0, 0, 0};
    download(e, parts, dparts.p, 3);
    if (e == cudaSuccess && dr != nullptr) {
        if (D == 1) download(e, dr, ddr.p, N);
        else std::fill(dr, dr + (size_t)N * M * M, 0.0);   // the reference's n-D branch returns zeros (gaussian_like.py:226)
    }
    download(e, jm, djm.p, nv);
    download(e, js, djs.p, nm);
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_obs_energy");
    *Eobs = parts[2];
    return VGPA_OK;
}

extern "C" {

int vgpa_obs_energy(int device, int D, int N, int M, const int64_t* obs_t, const double* obs_y, const double* R,
                    const double* mt, const double* st, double* Eobs, double* jm, double* js, double* dr)
{
    return obs_energy(device, D, N, M, obs_t, obs_y, R, ~0ull, mt, st, Eobs, jm, js, dr);
}

int vgpa_obs_energy_observed(int device, int D, int N, int M, const int64_t* obs_t, const double* obs_y, const double* R,
                             uint64_t observed, const double* mt, const double* st, double* Eobs, double* jm, double* js)
{
    if (observed == 0) return set_error(VGPA_EINVAL, "the observation mask has no bit set");
    if (D >= 1 && D < 64 && (observed >> D) != 0)
        return set_error(VGPA_EINVAL, "the observation mask has a bit at or above D = %d", D);
    return obs_energy(device, D, N, M, obs_t, obs_y, R, observed, mt, st, Eobs, jm, js, nullptr);
}

static int init_check(vgpa_handle* h, const double* x, int64_t x_stride)
{
    if (x == nullptr) return h->fail(VGPA_EINVAL, "x is NULL");
    if (x_stride < h->n_x) return h->fail(VGPA_EINVAL, "x_stride %lld < %lld", (long long)x_stride, h->n_x);
    if (h->d.M < 1) return h->fail(VGPA_EINVAL, "initialization needs at least one observation");
    if (h->init_empty >= 0)
        return h->fail(VGPA_EINVAL, "initialization needs at least one observation: problem %d has none", h->init_empty);
    if (h->init_edge >= 0)
        return h->fail(VGPA_EINVAL, "`x` must be strictly increasing sequence: an observation of problem %d sits at the first "
                                    "or last grid index", h->init_edge);
    return VGPA_OK;
}

int vgpa_initialization(vgpa_handle* h, double t0, double* d_x, int64_t x_stride, void* stream)
{
    if (!h) return VGPA_EINVAL;
    if (int rc = init_check(h, d_x, x_stride)) return rc;
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int B = h->d.B, D = h->d.D, n = h->d.M + 2;
    DevBuf scratch, err;
    cudaError_t e = cudaSuccess;
    alloc(e, scratch, (size_t)B * D * 2 * n);
    alloc<int>(e, err, 1);
    if (e == cudaSuccess) e = cudaMemsetAsync(err.p, 0, sizeof(int), st);
    if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_initialization");
    launch_initialization(h->batch, 0, B, t0, scratch.as<double>(), d_x, x_stride, err.as<int>(), st);
    h->launches += 2;
    int bad = 0;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, err.p, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);   // the scratch is released on return
    if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_initialization");
    if (bad) return h->fail(VGPA_EINVAL, "`x` must be strictly increasing sequence: an observation sits at the first or last grid index");
    return VGPA_OK;
}

int vgpa_initialization_host(vgpa_handle* h, double t0, double* x, int64_t x_stride)
{
    if (!h) return VGPA_EINVAL;
    if (int rc = init_check(h, x, x_stride)) return rc;
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    const int B = h->d.B, D = h->d.D, n = h->d.M + 2;
    const long long nx = h->n_x;
    const int C = std::max(1, std::min(B, 64));
    DevBuf scratch, err, dx;
    cudaError_t e = cudaSuccess;
    alloc(e, scratch, (size_t)C * D * 2 * n);
    alloc<int>(e, err, 1);
    alloc(e, dx, (size_t)C * nx);
    if (e == cudaSuccess) e = cudaMemset(err.p, 0, sizeof(int));
    if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_initialization_host");
    for (int p0 = 0; p0 < B && e == cudaSuccess; p0 += C) {
        const int count = std::min(C, B - p0);
        // kernels index problems globally: offset the staging pointer accordingly
        launch_initialization(h->batch, p0, count, t0, scratch.as<double>(), dx.as<double>() - (long long)p0 * nx, nx,
                              err.as<int>(), h->s_comp);
        h->launches += 2;
        e = cudaGetLastError();
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(x + (long long)p0 * x_stride, sizeof(double) * x_stride, dx.p, sizeof(double) * nx,
                                  sizeof(double) * nx, count, cudaMemcpyDeviceToHost, h->s_comp);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->s_comp);
    }
    int bad = 0;
    download(e, &bad, err.p, 1);
    if (e != cudaSuccess) return h->cuda_fail(e, "vgpa_initialization_host");
    if (bad) return h->fail(VGPA_EINVAL, "`x` must be strictly increasing sequence: an observation sits at the first or last grid index");
    return VGPA_OK;
}

// ---- batched sample paths and observations (SURVEY 8 f4; datagen.cu) -------------------------
static int model_dim(int model) { return model == VGPA_MODEL_L96 ? 40 : (model == VGPA_MODEL_L63 ? 3 : 1); }
static int traj_ntheta(int model) { return model == VGPA_MODEL_L63 ? 3 : (model == VGPA_MODEL_OU ? 2 : 1); }

static int check_traj_args(int model, int D, int N, int B, double dt, const void* theta, const void* sigma,
                           const void* x_init, const void* z, const void* path, int64_t z_stride, int64_t path_stride)
{
    if (model < 0 || model > 3) return set_error(VGPA_EINVAL, "Unknown stochastic model");
    if (model == VGPA_MODEL_L96 && D < 10) return set_error(VGPA_EINVAL, " Lorenz96: Insufficient state vector dimensions: %d", D);
    if (model == VGPA_MODEL_L96 && D > 64)
        return set_error(VGPA_EINVAL, "Wrong state dimension %d for Lorenz 96 (supported: 10 <= D <= 64)", D);
    if (model != VGPA_MODEL_L96 && D != model_dim(model))
        return set_error(VGPA_EINVAL, "Wrong state dimension %d for model %d (need %d)", D, model, model_dim(model));
    if (N < 1 || B < 1) return set_error(VGPA_EINVAL, "need N >= 1 time points and B >= 1 paths");
    if (!(dt > 0.0)) return set_error(VGPA_EINVAL, "Discrete time step should be strictly positive");
    if (!theta || !sigma || !z || !path) return set_error(VGPA_EINVAL, "NULL argument");
    if (D == 1 && !x_init) return set_error(VGPA_EINVAL, "x_init is required for the 1-D models");
    if ((z_stride != 0 && z_stride < (int64_t)N * D) || (B > 1 && path_stride < (int64_t)N * D))
        return set_error(VGPA_EINVAL, "z_stride / path_stride shorter than one path");
    return VGPA_OK;
}

int vgpa_make_trajectory_device_dim(int device, int model, int D, int N, int B, double dt, const double* d_theta,
                                    int64_t theta_stride, const double* d_sigma, int64_t sigma_stride, const double* d_x_init,
                                    int64_t x_init_stride, const double* d_z, int64_t z_stride, double* d_path,
                                    int64_t path_stride, void* stream)
{
    if (int rc = check_traj_args(model, D, N, B, dt, d_theta, d_sigma, d_x_init, d_z, d_path, z_stride, path_stride)) return rc;
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    TrajArgs a{model, D, N, B, dt, d_theta, theta_stride, d_sigma, sigma_stride, d_x_init, x_init_stride,
               d_z, z_stride, d_path, path_stride};
    launch_trajectories(a, static_cast<cudaStream_t>(stream));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? VGPA_OK : set_cuda_error(e, "vgpa_make_trajectory_device");
}

int vgpa_make_trajectory_device(int device, int model, int N, int B, double dt, const double* d_theta, int64_t theta_stride,
                                const double* d_sigma, int64_t sigma_stride, const double* d_x_init, int64_t x_init_stride,
                                const double* d_z, int64_t z_stride, double* d_path, int64_t path_stride, void* stream)
{
    return vgpa_make_trajectory_device_dim(device, model, model_dim(model), N, B, dt, d_theta, theta_stride, d_sigma,
                                           sigma_stride, d_x_init, x_init_stride, d_z, z_stride, d_path, path_stride, stream);
}

int vgpa_make_trajectory_dim(int device, int model, int D, int N, int B, double dt, const double* theta,
                             int64_t theta_stride, const double* sigma, int64_t sigma_stride, const double* x_init,
                             int64_t x_init_stride, const double* z, int64_t z_stride, double* path, int64_t path_stride)
{
    if (int rc = check_traj_args(model, D, N, B, dt, theta, sigma, x_init, z, path, z_stride, path_stride)) return rc;
    if ((theta_stride != 0 && theta_stride < traj_ntheta(model)) || (sigma_stride != 0 && sigma_stride < D) ||
        (x_init && x_init_stride != 0 && x_init_stride < D))
        return set_error(VGPA_EINVAL, "theta_stride / sigma_stride / x_init_stride shorter than one entry (0 = shared)");
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    const int64_t len = (int64_t)N * D;
    DevBuf dth, dsg, dxi, dz, dp;
    TrajArgs a{};
    a.model = model; a.D = D; a.N = N; a.B = B; a.dt = dt;
    cudaError_t e = cudaSuccess;
    stage_rows(e, dth, theta, theta_stride, traj_ntheta(model), B, &a.theta_stride);
    stage_rows(e, dsg, sigma, sigma_stride, D, B, &a.sigma_stride);
    if (x_init) stage_rows(e, dxi, x_init, x_init_stride, D, B, &a.x_init_stride);
    stage_rows(e, dz, z, z_stride, len, B, &a.z_stride);
    alloc(e, dp, (size_t)len * B);
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_make_trajectory");
    a.theta = dth.as<double>(); a.sigma = dsg.as<double>(); a.x_init = x_init ? dxi.as<double>() : nullptr;
    a.z = dz.as<double>(); a.path = dp.as<double>(); a.path_stride = len;
    launch_trajectories(a, nullptr);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess)
        e = cudaMemcpy2D(path, sizeof(double) * (B > 1 ? path_stride : len), dp.p, sizeof(double) * len, sizeof(double) * len, B,
                         cudaMemcpyDeviceToHost);
    return e == cudaSuccess ? VGPA_OK : set_cuda_error(e, "vgpa_make_trajectory");
}

int vgpa_make_trajectory(int device, int model, int N, int B, double dt, const double* theta, int64_t theta_stride,
                         const double* sigma, int64_t sigma_stride, const double* x_init, int64_t x_init_stride,
                         const double* z, int64_t z_stride, double* path, int64_t path_stride)
{
    return vgpa_make_trajectory_dim(device, model, model_dim(model), N, B, dt, theta, theta_stride, sigma, sigma_stride,
                                    x_init, x_init_stride, z, z_stride, path, path_stride);
}

static int check_obs_args(int D, int N, int M, int B, const int64_t* obs_t /* host, or NULL = not checked */)
{
    if (D != 1 && D != 3 && (D < 10 || D > 64))
        return set_error(VGPA_EINVAL, "unsupported state dimension %d (1, 3 or 10 <= D <= 64)", D);
    if (N < 1 || M < 0 || B < 1) return set_error(VGPA_EINVAL, "need N >= 1, M >= 0, B >= 1");
    for (int j = 0; obs_t && j < M; ++j)
        if (obs_t[j] < 0 || obs_t[j] >= N) return set_error(VGPA_EINVAL, "observation index outside the time grid");
    return VGPA_OK;
}

int vgpa_collect_obs_device(int device, int D, int N, int M, int B, const int64_t* d_obs_t, const double* d_R, int64_t R_stride,
                            const double* d_path, int64_t path_stride, const double* d_xi, int64_t xi_stride,
                            double* d_obs_y, int64_t obs_y_stride, void* stream)
{
    if (int rc = check_obs_args(D, N, M, B, nullptr)) return rc;
    if (!d_obs_t || !d_R || !d_path || !d_xi || !d_obs_y) return set_error(VGPA_EINVAL, "NULL argument");
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    ObsArgs a{D, N, M, B, reinterpret_cast<const long long*>(d_obs_t), d_R, R_stride, d_path, path_stride, d_xi, xi_stride,
              d_obs_y, obs_y_stride};
    launch_collect_obs(a, static_cast<cudaStream_t>(stream));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? VGPA_OK : set_cuda_error(e, "vgpa_collect_obs_device");
}

int vgpa_collect_obs(int device, int D, int N, int M, int B, const int64_t* obs_t, const double* R, int64_t R_stride,
                     const double* path, int64_t path_stride, const double* xi, int64_t xi_stride, double* obs_y,
                     int64_t obs_y_stride)
{
    if (!obs_t || !R || !path || !xi || !obs_y) return set_error(VGPA_EINVAL, "NULL argument");
    if (int rc = check_obs_args(D, N, M, B, obs_t)) return rc;
    if (M == 0) return VGPA_OK;
    if ((R_stride != 0 && R_stride < D) || (path_stride != 0 && path_stride < (int64_t)N * D) ||
        (xi_stride != 0 && xi_stride < (int64_t)M * D) || (B > 1 && obs_y_stride < (int64_t)M * D))
        return set_error(VGPA_EINVAL, "R_stride / path_stride / xi_stride / obs_y_stride shorter than one entry (0 = shared)");
    if (cudaSetDevice(device) != cudaSuccess) return set_error(VGPA_ECUDA, "cudaSetDevice failed");
    const int64_t plen = (int64_t)N * D, olen = (int64_t)M * D;
    DevBuf dt_, dR, dp, dx, dy;
    ObsArgs a{};
    a.D = D; a.N = N; a.M = M; a.B = B;
    cudaError_t e = cudaSuccess;
    upload(e, dt_, obs_t, M);
    stage_rows(e, dR, R, R_stride, D, B, &a.R_stride);
    stage_rows(e, dp, path, path_stride, plen, B, &a.path_stride);
    stage_rows(e, dx, xi, xi_stride, olen, B, &a.xi_stride);
    alloc(e, dy, (size_t)olen * B);
    if (e != cudaSuccess) return set_cuda_error(e, "vgpa_collect_obs");
    a.obs_t = dt_.as<long long>(); a.R = dR.as<double>(); a.path = dp.as<double>(); a.xi = dx.as<double>();
    a.obs_y = dy.as<double>(); a.obs_y_stride = olen;
    launch_collect_obs(a, nullptr);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess)
        e = cudaMemcpy2D(obs_y, sizeof(double) * (B > 1 ? obs_y_stride : olen), dy.p, sizeof(double) * olen, sizeof(double) * olen,
                         B, cudaMemcpyDeviceToHost);
    return e == cudaSuccess ? VGPA_OK : set_cuda_error(e, "vgpa_collect_obs");
}

void* vgpa_host_alloc(int64_t bytes)
{
    void* p = nullptr;
    if (bytes <= 0 || cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void vgpa_host_free(void* p)
{
    if (p) cudaFreeHost(p);
}

// Host copy on several threads: what a caller with an ordinary (pageable) x uses to fill a page-locked
// staging buffer; one core copies ~10 GB/s, which for a 13 MB x is a tenth of a single-problem evaluation.
void vgpa_host_copy(void* dst, const void* src, int64_t bytes, int threads)
{
    if (!dst || !src || bytes <= 0) return;
    const int64_t min_part = 1 << 20;
    int n = (int)std::min<int64_t>(std::max(threads, 1), (bytes + min_part - 1) / min_part);
    if (n <= 1) {
        std::memcpy(dst, src, (size_t)bytes);
        return;
    }
    const int64_t part = ((bytes + n - 1) / n + 63) & ~int64_t(63);
    std::vector<std::thread> pool;
    pool.reserve(n - 1);
    for (int i = 1; i < n; ++i) {
        const int64_t off = part * i;
        if (off >= bytes) break;
        const int64_t len = std::min(part, bytes - off);
        pool.emplace_back([=]() { std::memcpy((char*)dst + off, (const char*)src + off, (size_t)len); });
    }
    std::memcpy(dst, src, (size_t)std::min(part, bytes));
    for (auto& t : pool) t.join();
}

int vgpa_host_equal(const void* a, const void* b, int64_t bytes, int threads)
{
    if (bytes <= 0) return 1;
    if (!a || !b) return 0;
    const int64_t min_part = 1 << 20;
    const int n = (int)std::min<int64_t>(std::max(threads, 1), (bytes + min_part - 1) / min_part);
    if (n <= 1) return std::memcmp(a, b, (size_t)bytes) == 0;
    const int64_t part = ((bytes + n - 1) / n + 63) & ~int64_t(63);
    std::vector<int> same(n, 1);
    std::vector<std::thread> pool;
    pool.reserve(n - 1);
    for (int i = 1; i < n; ++i) {
        const int64_t off = part * i;
        if (off >= bytes) break;
        const int64_t len = std::min(part, bytes - off);
        int* out = &same[i];
        pool.emplace_back([=]() { *out = std::memcmp((const char*)a + off, (const char*)b + off, (size_t)len) == 0; });
    }
    same[0] = std::memcmp(a, b, (size_t)std::min(part, bytes)) == 0;
    for (auto& t : pool) t.join();
    for (int v : same)
        if (!v) return 0;
    return 1;
}

int vgpa_set_timing(vgpa_handle* h, int enable)
{
    if (!h) return VGPA_EINVAL;
    h->timing = enable != 0;
    return VGPA_OK;
}

int vgpa_get_timing(vgpa_handle* h, double ms[4], int64_t launches[4])
{
    if (!h || !ms || !launches) return VGPA_EINVAL;
    CK(cudaSetDevice(h->d.device), "cudaSetDevice");
    CK(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
    for (int k = 0; k < 4; ++k) {
        for (size_t q = 0; q < h->tev_used[k]; ++q) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, h->tev[k][q].first, h->tev[k][q].second) == cudaSuccess) {
                h->t_ms[k] += t;
                h->t_n[k] += 1;
            }
        }
        h->tev_used[k] = 0;
        ms[k] = h->t_ms[k];
        launches[k] = h->t_n[k];
        h->t_ms[k] = 0;
        h->t_n[k] = 0;
    }
    return VGPA_OK;
}

int64_t vgpa_launch_count(const vgpa_handle* h) { return h ? h->launches : 0; }
int64_t vgpa_chunk_size(const vgpa_handle* h) { return h ? h->chunk : 0; }
int64_t vgpa_scratch_in_use(const vgpa_handle* h)
{
    if (!h) return 0;
    return (int64_t)h->sc.bytes();
}

}  // extern "C"
