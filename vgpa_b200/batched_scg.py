"""
BatchedSCG: the reference's scaled-conjugate-gradient optimiser
(src/numerics/optim_scg.py:75-285) run for B independent problems AT ONCE with the
variational parameters, gradients and search directions resident in HBM.

SURVEY.md 8(f) item 1: the host SCG costs a 13 MB host<->device round trip of x and
grad F per evaluation (L96), which caps the end-to-end rate at PCIe speed.  Here the
per-problem control flow is vectorised over B on the host (B scalars per quantity),
while every length-n operation -- the two free-energy/gradient evaluations of an
iteration (vgpa_eval_device) and the optimiser's dot products, AXPYs and direction
updates (vgpa_bdot / baxpy / bdir / bcopy / bstats) -- runs on the device.  PyTorch
only owns the device buffers.

Memory: FIVE (B, n) buffers -- x, the trial point, the gradient, the trial gradient and the search
direction (65.6 MB per Lorenz-96 problem).  The reference's grad_old is not kept: it only enters
through g_new . g_old (taken as trial-gradient . gradient just before the gradient is replaced) and
through sum |g_old| (a scalar per problem).  Host synchronisations: three per iteration (the
direction's dot products; the curvature evaluation with its dot product; the trial evaluation with
every reduction the rest of the iteration can need, computed for all active rows at once).  Thinned-out
Lorenz-96 ensembles are evaluated through compacted launches (vgpa_set_active_list), so the survivors
still fill whole waves.  `ShardedBatchedSCG` runs an ensemble over the GPUs of a node in resident
sub-batches and gathers the results.

Per problem the arithmetic is the reference's, so each problem's `fx` trace follows
the reference's SCG (tests/test_gpu_batched_scg.py: 1e-6 on the common prefix, against the traces
the unmodified reference recorded).
"""
import numpy as np

from ._lib import lib, raise_for


class BatchedSCG:
    SIGMA0 = 1.0e-3
    BETA_MIN, BETA_MAX = 1.0e-15, 1.0e+100

    def __init__(self, evaluator, options=None):
        """evaluator: a vgpa_b200.BatchEvaluator (B problems, n_x parameters each)."""
        opts = options or {}
        self.ev = evaluator
        self.nit = opts.get("max_it", 150)
        self.x_tol = opts.get("x_tol", 1.0e-6)
        self.f_tol = opts.get("f_tol", 1.0e-8)
        self.display = opts.get("display", False)
        self.stats = None
        self.host_syncs = 0

    # -- device helpers ----------------------------------------------------------
    def _setup(self, X0, adopt=False):
        import torch
        self.torch = torch
        ev = self.ev
        B, n = ev.B, ev.n_x
        dev = torch.device("cuda", ev.device)
        if adopt and isinstance(X0, torch.Tensor) and X0.is_cuda and X0.shape == (B, n) and X0.is_contiguous():
            self.X = X0                              # the caller's device buffer becomes x (no sixth buffer)
        else:
            X = torch.as_tensor(X0, dtype=torch.float64)
            if X.dim() == 1:
                X = X.unsqueeze(0).expand(B, n)
            self.X = X.to(dev).contiguous().clone()
        z = lambda: torch.empty((B, n), dtype=torch.float64, device=dev)
        self.XT, self.Gn, self.GT, self.Dd = z(), z(), z(), z()
        self.Fd = torch.empty(B, dtype=torch.float64, device=dev)
        self.sc = torch.zeros(8 * B, dtype=torch.float64, device=dev)       # reduction outputs: dot (3B) | stats (2B) | stats (2B)
        self.coef = torch.empty(B, dtype=torch.float64, device=dev)         # per-problem scalars in
        self.mask = torch.empty(B, dtype=torch.int32, device=dev)
        self.act = torch.ones(B, dtype=torch.int32, device=dev)              # active set of the evaluations
        self.actv = torch.ones(B, dtype=torch.int32, device=dev)             # ... of the vector kernels
        self._actv_ptr = None                                                # None = every row
        self.stream = torch.cuda.current_stream(dev).cuda_stream
        self.B, self.n = B, n
        self._use_list = ev.model == "L96"
        self.host_syncs = 0

    def _eval_async(self, X, G, who=None):
        """Enqueue F (device, self.Fd) and grad at the rows of X.  `who` (B booleans): the problems that
        need this evaluation; the others are skipped -- Lorenz-96 through a compacted launch list (the
        survivors fill whole waves), the small models through per-problem flags -- and their F entries
        and gradient rows keep their previous content (every use below is masked by the same condition)."""
        ev = self.ev
        partial = who is not None and not who.all()
        if partial and self._use_list:
            ev.set_active(None)
            ev.set_active_list(np.flatnonzero(who))
        elif partial:
            self.act.copy_(self.torch.from_numpy(np.ascontiguousarray(who.astype(np.int32))))
            ev.set_active(self.act.data_ptr())
        else:
            ev.set_active(None)
            if self._use_list:
                ev.set_active_list(None)
        ev.eval_device(X.data_ptr(), self.n, self.Fd.data_ptr(), G.data_ptr(), self.n, self.stream)

    def _finish_eval(self):
        """Wait for the enqueued work (one host synchronisation), check the evaluation's status."""
        try:
            self.ev.sync()
        finally:
            self.ev.set_active(None)
            if self._use_list:
                self.ev.set_active_list(None)
        self.host_syncs += 1

    def _rows(self, active):
        """Rows the vector kernels below work on: the problems still being optimised (a superset is
        harmless: every use of their results is masked on the host)."""
        if active.all():
            self._actv_ptr = None
        else:
            self.actv.copy_(self.torch.from_numpy(np.ascontiguousarray(active.astype(np.int32))))
            self._actv_ptr = self.actv.data_ptr()

    def _dot_async(self, x, y, z=None):
        """sc[0:B] = x.y, sc[B:2B] = x.z, sc[2B:3B] = x.x (enqueued)."""
        raise_for(lib.vgpa_bdot(self.B, self.n, x.data_ptr(), y.data_ptr(), z.data_ptr() if z is not None else None,
                                self.n, self.sc.data_ptr(), self._actv_ptr, self.stream))

    def _stats_async(self, x, slot):
        """sc[(3 + 2 slot) B ...] = max|x|, sum|x| (enqueued); slot 0 or 1."""
        off = (3 + 2 * slot) * self.B * 8
        raise_for(lib.vgpa_bstats(self.B, self.n, x.data_ptr(), self.n, self.sc.data_ptr() + off, self._actv_ptr, self.stream))

    def _fetch(self, with_F=False):
        """The reduction outputs (and F) on the host: (dot3 (3, B), stats0 (2, B), stats1 (2, B)[, F (B,)])."""
        r = self.sc.cpu().numpy()
        B = self.B
        out = (r[:3 * B].reshape(3, B).copy(), r[3 * B:5 * B].reshape(2, B).copy(), r[5 * B:7 * B].reshape(2, B).copy())
        return out + (self.Fd.cpu().numpy().copy(),) if with_F else out

    def _axpy(self, a, x, y, out):
        self.coef.copy_(self.torch.from_numpy(np.ascontiguousarray(a)))
        raise_for(lib.vgpa_baxpy(self.B, self.n, self.coef.data_ptr(), x.data_ptr(), y.data_ptr(), out.data_ptr(),
                                 self.n, self._actv_ptr, self.stream))

    def _copy_where(self, m, src, dst):
        self.mask.copy_(self.torch.from_numpy(np.ascontiguousarray(m.astype(np.int32))))
        raise_for(lib.vgpa_bcopy(self.B, self.n, self.mask.data_ptr(), src.data_ptr(), dst.data_ptr(), self.n,
                                 self.stream))

    def _direction(self, mode, gamma):
        self.mask.copy_(self.torch.from_numpy(np.ascontiguousarray(mode.astype(np.int32))))
        self.coef.copy_(self.torch.from_numpy(np.ascontiguousarray(gamma)))
        raise_for(lib.vgpa_bdir(self.B, self.n, self.mask.data_ptr(), self.coef.data_ptr(), self.Dd.data_ptr(),
                                self.Gn.data_ptr(), self.n, self.stream))

    # -- the optimiser -------------------------------------------------------------
    def __call__(self, X0, adopt=False):
        """Returns (X (B, n) device tensor, fx (B,) numpy).  self.stats holds the per-problem
        traces: fx, dfx, beta of shape (max_it, B), MaxIt (B,), f_eval, df_eval (B,).
        adopt=True: a contiguous (B, n) CUDA tensor X0 is optimised in place (no copy of it is made)."""
        self._setup(X0, adopt)
        B, nit = self.B, self.nit
        eps = np.finfo(float).eps
        st = {"MaxIt": np.full(B, nit), "fx": np.zeros((nit, B)), "dfx": np.zeros((nit, B)),
              "beta": np.zeros((nit, B)), "f_eval": np.zeros(B), "df_eval": np.zeros(B), "evaluations": 0}
        self.stats = st
        self._eval_async(self.X, self.Gn)
        self._stats_async(self.Gn, 0)
        self._finish_eval()
        _, s0, _, f_now = self._fetch(True)
        st["evaluations"] += 1
        st["f_eval"] += 1
        st["df_eval"] += 1
        f_old = f_now.copy()
        sum_gn = s0[1].copy()                                         # sum |grad_new|
        sum_go = sum_gn.copy()                                        # sum |grad_old| (grad_old = grad_new at the start)
        self._direction(np.full(B, 2), np.zeros(B))                  # d = -grad
        active = np.ones(B, dtype=bool)
        success = np.ones(B, dtype=bool)
        n_success = np.zeros(B, dtype=np.int64)
        beta = np.ones(B)
        kappa, theta, mu = np.zeros(B), np.zeros(B), np.zeros(B)
        fx_out = f_now.copy()

        for j in range(nit):
            if not active.any():
                break
            self._rows(active)
            S = success & active
            if S.any():
                # first / second directional derivatives along d  (optim_scg.py:137-170)
                self._dot_async(self.Dd, self.Gn)
                self.host_syncs += 1
                d3, _, _ = self._fetch()
                dg, dd = d3[0], d3[2]
                flip = S & (dg >= 0.0)
                if flip.any():
                    self._direction(np.where(flip, 2, 0), np.zeros(B))
                    self._dot_async(self.Dd, self.Gn)
                    self.host_syncs += 1
                    d3, _, _ = self._fetch()
                    dg, dd = np.where(flip, d3[0], dg), np.where(flip, d3[2], dd)
                mu = np.where(S, dg, mu)
                kappa = np.where(S, dd, kappa)
                tiny = S & (kappa < eps)
                if tiny.any():                                        # optim_scg.py:148-156
                    st["MaxIt"][tiny] = j + 1
                    fx_out[tiny] = f_now[tiny]
                    active &= ~tiny
                    S &= ~tiny
                sigma = np.where(S, self.SIGMA0 / np.sqrt(np.where(kappa > 0, kappa, 1.0)), 0.0)
                self._axpy(sigma, self.Dd, self.X, self.XT)           # x_plus = x + sigma d
                self._eval_async(self.XT, self.GT, S)                 # df(x_plus, eval_fun=True)
                self._dot_async(self.Dd, self.GT)
                self._finish_eval()
                d3, _, _ = self._fetch()
                st["evaluations"] += 1
                st["f_eval"][S] += 1
                st["df_eval"][S] += 1
                theta = np.where(S, (d3[0] - mu) / np.where(S, sigma, 1.0), theta)
            # effective curvature and step length  (optim_scg.py:173-186)
            delta = theta + beta * kappa
            neg = active & (delta <= 0.0)
            delta = np.where(neg, beta * kappa, delta)
            beta = np.where(neg, beta - theta / np.where(kappa != 0, kappa, 1.0), beta)
            alpha = np.where(active, -(mu / np.where(delta != 0, delta, 1.0)), 0.0)
            self._axpy(alpha, self.Dd, self.X, self.XT)               # x_new = x + alpha d
            self._eval_async(self.XT, self.GT, active)                # f(x_new); its gradient is kept
            # every reduction the rest of the iteration can need, for all active rows, behind the SAME
            # synchronisation: g_trial . g (the Polak-Ribiere numerator needs g_new . g_old AFTER the move,
            # i.e. trial gradient . current gradient), g_trial . g_trial, sum |g_trial|, max |d|
            self._dot_async(self.GT, self.Gn)
            self._stats_async(self.GT, 0)
            self._stats_async(self.Dd, 1)
            self._finish_eval()
            d3, sGT, sD, f_new = self._fetch(True)
            st["evaluations"] += 1
            st["f_eval"][active] += 1
            # comparison ratio  (optim_scg.py:192-204)
            with np.errstate(divide="ignore", invalid="ignore"):
                Delta = 2.0 * (f_new - f_old) / (alpha * mu)
            succ = active & (Delta >= 0.0)
            fail = active & ~succ
            success = np.where(active, succ, success)
            n_success = n_success + succ
            self._copy_where(succ, self.XT, self.X)
            f_now = np.where(succ, f_new, np.where(fail, f_old, f_now))
            # statistics: the reference records sum|g| of the gradient at the PREVIOUS accepted
            # point on success and of grad_old on failure (optim_scg.py:197-209)
            st["fx"][j] = np.where(active, f_now, st["fx"][j - 1] if j else f_now)
            st["beta"][j] = beta
            st["dfx"][j] = np.where(succ, sum_gn, sum_go)
            if self.display and j % 10 == 0:
                print(f" {j}: mean fx={np.mean(f_now):.3f}\tactive={int(active.sum())}")
            # termination and the move to the new point  (optim_scg.py:217-247)
            move = np.zeros(B, dtype=bool)
            gg_all = ggo = np.zeros(B)
            if succ.any():
                maxd = sD[0]
                done = succ & (np.abs(alpha) * maxd <= self.x_tol) & (np.abs(f_new - f_old) <= self.f_tol)
                st["MaxIt"][done] = j + 1
                fx_out[done] = f_new[done]
                active &= ~done
                move = succ & ~done
                f_old = np.where(move, f_new, f_old)
                ggo, gg_all = d3[0], d3[2]                            # (new grad_new) . (new grad_old), |new grad_new|^2
                sum_go = np.where(move, sum_gn, sum_go)               # grad_old = grad_new
                sum_gn = np.where(move, sGT[1], sum_gn)               # grad_new = df(x) (x == x_new)
                self._copy_where(move, self.GT, self.Gn)
                st["f_eval"][move] += 1                               # the reference re-evaluates f(x), df(x)
                st["df_eval"][move] += 1
                zero = move & np.isclose(gg_all, 0.0)
                st["MaxIt"][zero] = j + 1
                fx_out[zero] = f_now[zero]
                active &= ~zero
            # scale update  (optim_scg.py:250-257)
            beta = np.where(active & (Delta < 0.25), np.minimum(4.0 * beta, self.BETA_MAX), beta)
            beta = np.where(active & (Delta > 0.75), np.maximum(0.5 * beta, self.BETA_MIN), beta)
            # search direction: Polak-Ribiere, restart after n successes  (optim_scg.py:262-274)
            restart = active & (n_success == self.n)
            n_success = np.where(restart, 0, n_success)
            pr = active & ~restart & move
            with np.errstate(divide="ignore", invalid="ignore"):
                gamma = np.where(pr, np.maximum((ggo - gg_all) / mu, 0.0), 0.0)
            mode = np.where(restart, 2, np.where(pr, 1, 0))
            if mode.any():
                self._direction(mode, gamma)
        fx_out = np.where(active, f_old, fx_out)                      # max_it reached: optim_scg.py:281
        st["host_syncs"] = self.host_syncs
        return self.X, fx_out


def save_ensemble(name, output):
    """Write the results of an ensemble run, keyed like the reference's Simulation.save
    (src/var_bayes/simulation.py:248-311: one gzip-compressed dataset per key of `output`, scalars as
    1-D arrays) with a leading problem axis: fx (B,), at (K, N, D, D) / bt (K, N, D) for the K problems
    whose optimised parameters were kept (`kept`), plus the per-problem optimiser statistics.  HDF5
    (`<name>.h5`) when h5py is installed, else `<name>.npz` with the same keys; vgpa_b200.simulation.load
    reads either."""
    from pathlib import Path
    stem = str(name).strip().replace(" ", "_")
    data = {k: np.atleast_1d(v) if np.isscalar(v) else np.asarray(v) for k, v in output.items()}
    try:
        import h5py
    except ImportError:
        h5py = None
    if h5py is not None:
        out = Path(stem + ".h5")
        with h5py.File(out, "w") as fh:
            for key, val in data.items():
                fh.create_dataset(key, data=val, shape=val.shape, compression="gzip")
    else:
        out = Path(stem + ".npz")
        np.savez_compressed(out, **data)
    return out


_release_thread = None


def _release_now():
    """Switch the scratch hand-over off, free what it still holds and what torch's allocator caches."""
    import torch
    lib.vgpa_scratch_cache(0)
    torch.cuda.empty_cache()


def _start_release():
    """_release_now on a background thread: tens of GB of cudaFree take up to seconds when every rank of a node
    frees at the same time, and nothing the caller is waiting for depends on it."""
    global _release_thread
    import threading
    _join_release()
    _release_thread = threading.Thread(target=_release_now, name="vgpa-scratch-release")
    _release_thread.start()


def _join_release():
    """Wait for a release still in flight (its memory is about to be needed)."""
    global _release_thread
    if _release_thread is not None:
        _release_thread.join()
        _release_thread = None


class ShardedBatchedSCG:
    """An ensemble of `total` independent optimisations over the GPUs of one node (one process per GPU,
    contiguous blocks of problems as in vgpa_b200.ensemble) in device-resident sub-batches: per sub-batch
    the starting points come from the on-device initialisation (or from `x0_fn`), BatchedSCG optimises
    them in place, and only the per-problem results (fx, iteration and evaluation counts, optionally the
    optimised parameters of selected problems) leave the device.  The one collective is the final gather
    (NCCL under torch.distributed; no process group: a single GPU).

    make_evaluator(lo, hi) -> BatchEvaluator for the problems [lo, hi) on this rank's device.
    sub_batch: problems resident at once (None: as many as fit `mem_fraction` of the free HBM with the
    optimiser's five (B, n) buffers and the evaluator's scratch)."""

    def __init__(self, total, make_evaluator, options=None, sub_batch=None, rank=None, world=None, group=None,
                 mem_fraction=0.85):
        from .ensemble import shard_bounds
        import torch.distributed as dist
        if rank is None or world is None:
            if dist.is_available() and dist.is_initialized():
                rank, world = dist.get_rank(group), dist.get_world_size(group)
            else:
                rank, world = 0, 1
        self.total, self.rank, self.world, self.group = int(total), rank, world, group
        self.lo, self.hi = shard_bounds(total, rank, world)
        self.make_evaluator, self.options = make_evaluator, dict(options or {})
        self.sub_batch, self.mem_fraction = sub_batch, mem_fraction
        self.result = None

    def _pick_sub_batch(self, n_x, device, scratch_per_problem):
        """Problems resident at once: the optimiser's five (B, n) buffers plus the evaluator's scratch (which
        holds the trajectories of up to one pass = up to the whole sub-batch) within `mem_fraction` of the free HBM."""
        import torch
        free, _ = torch.cuda.mem_get_info(device)
        per_problem = 5 * 8 * n_x + scratch_per_problem + 64
        return max(1, int(free * self.mem_fraction // per_problem))

    def run(self, t0=0.0, x0_fn=None, keep=(), concurrent=1, hyper=False):
        """Optimise the local block.  x0_fn(lo, hi, X) fills the (hi - lo, n) device tensor X with starting
        points (default: the on-device VarGP.initialization).  keep: global problem indices whose optimised
        x is returned (host).  concurrent: sub-batches optimised AT THE SAME TIME, each by its own host thread
        on its own CUDA stream with its own evaluator -- the problems of a sub-batch converge at different
        iterations, and the thinned-out tail of one sub-batch (latency bound: a few problems cost as much per
        evaluation as a full wave) can overlap the full waves of another.  (Measured on one B200, Lorenz-96:
        1776 problems as two sub-batches of 888, 177-200 optimisations/s one after the other, 217-235 concurrently;
        888 problems as one sub-batch 229, as two concurrent halves 176 -- concurrency only pays between sub-batches
        that each fill the GPU, so the default stays 1.)  hyper=True: each sub-batch also computes model.energy's
        hyper-parameter gradients at its optimised x (one vgpa_hyper_device call before x is freed), returned
        as Esde (total,), dEsde_dtheta (total, n_theta) and dEsde_dsigma_diag (total, D) -- the diagonal only,
        dEsde_dsigma is diagonal (the full D x D of 32768 Lorenz-96 problems is 420 MB).  Returns the dict that `save` writes,
        identical on every rank (except `kept` entries, which each rank holds for its own problems until the
        gather)."""
        import time
        import torch
        import torch.distributed as dist
        keep = set(int(k) for k in keep)
        n_local = self.hi - self.lo
        concurrent = max(1, int(concurrent))
        fx = np.zeros(n_local)
        n_it = np.zeros(n_local, dtype=np.int64)
        f_eval = np.zeros(n_local)
        kept = {}
        hyp = None
        sub = self.sub_batch
        if sub is None and n_local > 0:   # from the evaluator's shape: what fits the free HBM, shared by the workers
            ev = self.make_evaluator(self.lo, min(self.hi, self.lo + 1))
            dev = torch.device("cuda", ev.device)
            # evaluator scratch: 2 (D + D^2) N + N doubles per problem of a pass
            scratch = 8 * ev.N * (2 * ev.D * (ev.D + 1) + 1)
            n_x = ev.n_x
            ev.close()
            sub = min(n_local, max(1, self._pick_sub_batch(n_x, dev, scratch) // concurrent))
        ranges = [(p, min(self.hi, p + sub)) for p in range(self.lo, self.hi, max(sub or 1, 1))]

        def work(rng_):
            lo_, hi_ = rng_
            t_create = time.perf_counter()
            ev = self.make_evaluator(lo_, hi_)
            t_create = time.perf_counter() - t_create
            dev = torch.device("cuda", ev.device)
            torch.cuda.set_device(dev)
            stream = torch.cuda.Stream(dev) if concurrent > 1 else torch.cuda.current_stream(dev)
            try:
                with torch.cuda.stream(stream):
                    b = ev.B
                    t_x0 = time.perf_counter()
                    X = torch.empty((b, ev.n_x), dtype=torch.float64, device=dev)
                    if x0_fn is None:
                        ev.initialization_device(X.data_ptr(), ev.n_x, float(t0), stream.cuda_stream)
                        ev.sync()
                    else:
                        x0_fn(lo_, hi_, X)
                    stream.synchronize()
                    t_x0 = time.perf_counter() - t_x0
                    opt = BatchedSCG(ev, self.options)
                    t_opt = time.perf_counter()
                    Xf, fxb = opt(X, adopt=True)
                    stream.synchronize()
                    t_opt = time.perf_counter() - t_opt
                    res = {"range": rng_, "optimise_seconds": t_opt, "create_seconds": t_create, "x0_seconds": t_x0, "fx": fxb, "n_it": opt.stats["MaxIt"], "f_eval": opt.stats["f_eval"],
                           "evaluations": opt.stats["evaluations"] * b, "syncs": opt.host_syncs,
                           "kept": {k: Xf[k - lo_].cpu().numpy() for k in keep if lo_ <= k < hi_}}
                    if hyper:
                        res["hyper"] = self._hyper_at(ev, Xf, stream)
                    t_free = time.perf_counter()
                    del opt, Xf, X
                return res
            finally:
                ev.close()
                if "res" in locals():
                    res["free_seconds"] = time.perf_counter() - t_free

        # Evaluators of one shape follow each other: the library hands the scratch of a closed one to the next
        # (vgpa_scratch_cache) instead of freeing and re-allocating tens of GB per sub-batch, and torch's allocator
        # does the same for the optimiser's buffers.  What is still kept at the end is released on a background
        # thread AFTER the gather: the results are complete, and a cudaFree of that size takes up to seconds when
        # every rank of a node frees at the same time (a release started before the gather only made the gather
        # wait for it: measured).
        _join_release()
        lib.vgpa_scratch_cache(1)
        t_ = time.perf_counter()
        def work_retry(rng_):
            # Sub-batches of one shape reuse the torch allocator's cached buffers and the library's kept scratch.
            # When the shape changes (the last, smaller sub-batch) what is kept may be in the way: release, retry.
            try:
                return work(rng_)
            except torch.cuda.OutOfMemoryError:
                lib.vgpa_scratch_cache(0)
                torch.cuda.empty_cache()
                lib.vgpa_scratch_cache(1)
                return work(rng_)

        try:
            if concurrent == 1 or len(ranges) <= 1:
                results = [work_retry(r_) for r_ in ranges]
            else:
                from concurrent.futures import ThreadPoolExecutor
                with ThreadPoolExecutor(max_workers=concurrent) as pool:
                    results = list(pool.map(work_retry, ranges))
        except BaseException:
            _release_now()
            raise
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        seconds = time.perf_counter() - t_
        evaluations, syncs, optimise_seconds, create_seconds, x0_seconds = 0, 0, 0.0, 0.0, 0.0
        for r in results:
            sl = slice(r["range"][0] - self.lo, r["range"][1] - self.lo)
            fx[sl], n_it[sl], f_eval[sl] = r["fx"], r["n_it"], r["f_eval"]
            evaluations += r["evaluations"]
            syncs += r["syncs"]
            optimise_seconds += r["optimise_seconds"]
            create_seconds += r["create_seconds"]
            x0_seconds += r["x0_seconds"]
            kept.update(r["kept"])
            if hyper:
                if hyp is None:
                    hyp = {k: np.zeros((n_local,) + v.shape[1:]) for k, v in r["hyper"].items()}
                for k, v in r["hyper"].items():
                    hyp[k][sl] = v
        # gather of the per-problem results (the only collective)
        def gather(v):
            if self.world == 1 or not (dist.is_available() and dist.is_initialized()):
                return v
            from .ensemble import gather_free_energies
            return gather_free_energies(np.asarray(v, dtype=np.float64), self.total, self.group)
        t_g = time.perf_counter()
        out = {"fx": gather(fx), "n_it": gather(n_it.astype(np.float64)).astype(np.int64), "f_eval": gather(f_eval),
               "rank_seconds": seconds, "rank_optimise_seconds": optimise_seconds, "rank_problem_evaluations": evaluations, "rank_host_syncs": syncs,
               "sub_batch": sub, "concurrent": concurrent, "kept": kept}
        if hyper:
            for k, v in hyp.items():     # gathered like fx, one column at a time
                out[k] = gather(v) if v.ndim == 1 else np.stack([gather(v[:, j]) for j in range(v.shape[1])], axis=1)
        out["rank_phase_seconds"] = {"create_evaluators": round(create_seconds, 4), "starting_points": round(x0_seconds, 4),
                                     "optimise": round(optimise_seconds, 4), "whole_loop": round(seconds, 4),
                                     "close_evaluators": round(sum(r.get("free_seconds", 0.0) for r in results), 4),
                                     "release": "scratch (vgpa_scratch_cache) and torch cache: on a background thread, after the gather",
                                     "gather": round(time.perf_counter() - t_g, 4)}
        self.result = out
        _start_release()
        return out

    @staticmethod
    def _hyper_at(ev, X, stream):
        """Esde, dEsde_dtheta and the diagonal of dEsde_dsigma of every problem of `ev` at the rows of X (host arrays)."""
        import torch
        b, D, nth = ev.B, ev.D, ev.n_theta
        nsig = 1 if D == 1 else D * D
        Esde = torch.empty(b, dtype=torch.float64, device=X.device)
        dth = torch.empty((b, nth), dtype=torch.float64, device=X.device)
        dsig = torch.empty((b, nsig), dtype=torch.float64, device=X.device)
        ev.hyper_device(X.data_ptr(), ev.n_x, None, Esde.data_ptr(), dth.data_ptr(), nth, dsig.data_ptr(), nsig,
                        stream.cuda_stream)
        ev.sync()
        diag = dsig if D == 1 else dsig[:, ::D + 1]
        return {"Esde": Esde.cpu().numpy(), "dEsde_dtheta": dth.cpu().numpy(), "dEsde_dsigma_diag": diag.cpu().numpy()}

    def save(self, name, N, D):
        """Rank-local file `<name>_rank<r>` in the reference's key convention (save_ensemble)."""
        r = self.result
        ks = sorted(r["kept"])
        out = {"fx": r["fx"], "n_it": r["n_it"], "f_eval": r["f_eval"], "problem": np.array(ks, dtype=np.int64)}
        for k in ("Esde", "dEsde_dtheta", "dEsde_dsigma_diag"):
            if k in r:
                out[k] = r[k]
        if ks:
            xs = np.stack([r["kept"][k] for k in ks])
            if D == 1:
                out["at"], out["bt"] = xs[:, :N], xs[:, N:]
            else:
                out["at"] = xs[:, :N * D * D].reshape(len(ks), N, D, D)
                out["bt"] = xs[:, N * D * D:].reshape(len(ks), N, D)
        return save_ensemble(f"{name}_rank{self.rank}", out)
