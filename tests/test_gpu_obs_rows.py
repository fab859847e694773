"""
Per-problem observation schedules (vgpa_create_obs_rows; BatchEvaluator with a list of obs_t arrays).

Each batch gets four schedules assigned round-robin: none (M_p = 0), one observation, a dense one with adjacent indices
and observations at index 0 and at N - 1 (whose jump is never applied), and a sparse one.  Then, for every kernel
family (the CASES table of test_gpu_layouts.py, plus Lorenz 96 at D = 13 and D = 64):

  - every F and gradient row is, bit for bit, the row of the same problem in a handle of the same B and pass split in
    which every problem carries that row's schedule (the launchers pick the kernel family by the problem count, so
    the same B means the same family);
  - sampled rows match the oracle at 1e-9.

Also: the degenerate forms (stride 0 with no counts; identical rows) give the shared handle's bits; the host entry
point across its staging passes, padded and shared device rows, active flags and compacted lists with sentinel bits,
forced pass splits, the hyper-parameter gradients, vgpa_eval_full, a LinAlgError naming the problem, initialisation
against the oracle and its errors, and the batched optimisers on ragged batches.
"""
import numpy as np
import pytest

from conftest import grad_err
from oracle import Problem
from test_gpu_l96_dims import L96Batch, DT as L96_DT
from test_gpu_layouts import CASES, SENT, _alloc, _Batch, _eval_device, _expect, _fill, _rows, _sample_rows

pytestmark = pytest.mark.gpu
TOL = 1e-9


def schedules(N):
    """Four schedules on an N-point grid: none, one, dense with both ends and adjacent indices, sparse."""
    dense = sorted({0, 1, 2, *range(5, N - 3, 3), N - 2, N - 1})
    sparse = list(range(3, N - 1, max(7, N // 20)))
    return [np.zeros(0, dtype=np.int64), np.array([N // 2]), np.array(dense), np.array(sparse)]


class Ragged:
    """A batch of `base` (theta, sigma, R, m0, s0, E0, x per problem) with per-problem schedules: problem p observes at
    scheds[kind[p]], and its value at time index t is Y[p, t]."""

    def __init__(self, base, dt, dt_model, scheds=None, kind=None, seed=0):
        self.base, self.dt, self.dt_model = base, dt, dt_model
        self.model, self.method, self.D, self.N, self.B = base.model, base.method, base.D, base.N, base.B
        self.scheds = schedules(self.N) if scheds is None else scheds
        self.kind = np.arange(self.B) % len(self.scheds) if kind is None else np.asarray(kind)
        oy = base.obs_y                                      # (B, M0, D): values near the model's path
        rng = np.random.default_rng([seed, self.B, self.N])
        t = np.arange(self.N)
        self.Y = oy[:, t % oy.shape[1]] + 0.05 * rng.standard_normal((self.B, self.N, self.D))
        self.X, self.n_x = base.X, base.n_x

    def sched(self, p):
        return self.scheds[self.kind[p]]

    def _kw(self, idx):
        b = self.base
        s0 = np.asarray(b.s0).reshape(b.B, -1)
        return dict(model=self.model, method=self.method, N=self.N, dt=self.dt, theta=b.theta[idx], sigma=b.sigma[idx],
                    R=b.R[idx], m0=b.m0[idx], s0=s0[idx], E0=np.asarray(b.E0)[idx], B=len(idx),
                    dt_model=self.dt_model, D=self.D)

    def evaluator(self, idx=None, **kw):
        """The ragged handle (of the problems idx)."""
        from vgpa_b200.engine import BatchEvaluator
        idx = np.arange(self.B) if idx is None else np.asarray(idx)
        return BatchEvaluator(obs_t=[self.sched(p) for p in idx], obs_y=[self.Y[p, self.sched(p)] for p in idx],
                              **self._kw(idx), **kw)

    def same(self, k, idx=None, **kw):
        """A shared-schedule handle of the same problems: every one observes at scheds[k]."""
        from vgpa_b200.engine import BatchEvaluator
        idx = np.arange(self.B) if idx is None else np.asarray(idx)
        s = self.scheds[k]
        return BatchEvaluator(obs_t=s, obs_y=self.Y[idx][:, s], **self._kw(idx), **kw)

    def problem(self, p):
        b, D = self.base, self.D
        s = self.sched(p)
        return Problem(model=self.model, method=self.method, D=D, N=self.N, dt=self.dt, theta=b.theta[p],
                       sigma=b.sigma[p], R=b.R[p], obs_t=s, obs_y=self.Y[p, s].reshape(s.size, D), m0=b.m0[p],
                       s0=np.asarray(b.s0[p]).reshape(D, D) if D > 1 else np.asarray(b.s0[p]).ravel(),
                       E0=float(np.asarray(b.E0)[p]), dt_model=self.dt_model)


def from_case(model, method, N, B, seed=1):
    bt = _Batch(model, method, N, B, seed=seed)
    g = bt.g
    return Ragged(bt, float(g["dt"]), Problem.from_golden(g).dt_model, seed=seed)


def from_l96(D, N, B, method="rk2", oracle=None, seed=0):
    bt = L96Batch(D, N, B, method, seed=seed, oracle=oracle)
    bt.model = "L96"
    return Ragged(bt, L96_DT, L96_DT, seed=seed)


def dev_eval(ev, X, want_grad=True):
    """Compact device evaluation: F (B,) and gradient (B, n_x) as int64 CPU tensors (gradient None for F only)."""
    import torch
    B, n = ev.B, ev.n_x
    Xt = torch.from_numpy(np.ascontiguousarray(X)).cuda()
    F = torch.empty(B, dtype=torch.float64, device="cuda")
    G = torch.empty((B, n), dtype=torch.float64, device="cuda") if want_grad else None
    ev.eval_device(Xt.data_ptr(), n, F.data_ptr(), G.data_ptr() if want_grad else None, n,
                   torch.cuda.current_stream().cuda_stream)
    ev.sync()
    return F.view(torch.int64).cpu(), (G.view(torch.int64).cpu() if want_grad else None)


def assert_rows_match_same_schedule(rg, F, G, want_grad=True, **kw):
    """Every row of the ragged evaluation (F, G) against the handle in which all problems carry its schedule."""
    import torch
    for k in range(len(rg.scheds)):
        rows = np.flatnonzero(rg.kind == k)
        if rows.size == 0:
            continue
        with rg.same(k, **kw) as ev:
            Fk, Gk = dev_eval(ev, rg.X, want_grad)
        r = torch.from_numpy(rows)
        assert torch.equal(F[r], Fk[r]), (k, rows[:8])
        if want_grad:
            assert torch.equal(G[r], Gk[r]), (k, rows[:8])


def assert_oracle(oracle, rg, F, G, rows, want_grad=True):
    import torch
    Fh = F.view(torch.float64).numpy()
    F_o, G_o = oracle.eval_batch([rg.problem(i) for i in rows], rg.X[rows], want_grad=want_grad)
    for k, i in enumerate(rows):
        assert abs(Fh[i] - F_o[k]) <= TOL * abs(F_o[k]), (i, rg.sched(i).size, Fh[i], F_o[k])
        if want_grad:
            assert grad_err(G[i].view(torch.float64).numpy(), G_o[k], rg.N, rg.D) < TOL, i


# ---- 1. every kernel family ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-{c[1]}-N{c[2] or 1001}-B{c[3]}-{c[6]}")
def test_every_kernel_family(oracle, case):
    model, method, N, B, want_grad, per_pass, _ = case
    rg = from_case(model, method, N, B)
    kw = dict(scratch_bytes=per_pass * rg.base.per_problem_bytes() + 64) if per_pass else {}
    with rg.evaluator(**kw) as ev:
        if per_pass:
            assert ev.chunk_size < B
        chunk = ev.chunk_size
        F, G = dev_eval(ev, rg.X, want_grad)
    assert_rows_match_same_schedule(rg, F, G, want_grad, **kw)
    rows = sorted(r for r in set(_sample_rows(B, chunk)) | {1, 2, 3} if r < B)
    assert_oracle(oracle, rg, F, G, rows, want_grad)


@pytest.mark.parametrize("D,N,B,method", [(13, 101, 9, "rk2"), (64, 61, 5, "rk4"), (13, 41, 6, "euler")])
def test_l96_run_time_d(oracle, D, N, B, method):
    rg = from_l96(D, N, B, method, oracle=oracle)
    with rg.evaluator() as ev:
        F, G = dev_eval(ev, rg.X)
    assert_rows_match_same_schedule(rg, F, G)
    assert_oracle(oracle, rg, F, G, range(B))


# ---- 2. degenerate forms ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model,method,N,B", [("OU", "rk4", 1001, 7), ("L63", "rk2", 61, 7), ("L96", "rk2", 101, 5),
                                              ("DW", "heun", 4000, 5)])
def test_degenerate_forms_give_the_shared_bits(model, method, N, B, monkeypatch):
    import ctypes as C
    import torch
    from vgpa_b200 import _lib
    rg = from_case(model, method, N, B)
    k = 3
    with rg.same(k) as ev:
        F0, G0 = dev_eval(ev, rg.X)
    # identical rows through vgpa_create_obs_rows' per-problem path
    rg_eq = Ragged(rg.base, rg.dt, rg.dt_model, scheds=rg.scheds, kind=np.full(B, k))
    rg_eq.Y = rg.Y
    with rg_eq.evaluator() as ev:
        F1, G1 = dev_eval(ev, rg.X)
    assert torch.equal(F0, F1) and torch.equal(G0, G1)
    # vgpa_create_obs_rows with stride 0 and no counts stands for vgpa_create
    create = _lib.lib.vgpa_create
    calls = []

    def via_obs_rows(d, out):
        desc = d._obj
        ot = C.cast(desc.obs_t, C.c_void_p).value
        desc.obs_t = None
        calls.append(1)
        return _lib.lib.vgpa_create_obs_rows(d, ot, 0, None, out)

    monkeypatch.setattr(_lib.lib, "vgpa_create", via_obs_rows)
    with rg.same(k) as ev:
        F2, G2 = dev_eval(ev, rg.X)
    monkeypatch.setattr(_lib.lib, "vgpa_create", create)
    assert calls
    assert torch.equal(F0, F2) and torch.equal(G0, G2)


# ---- 3. entry points ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["L96-13", "L96-40", "OU"])
def test_host_entry_point_across_staging_passes(oracle, which):
    import torch
    rg = from_l96(13, 41, 70, "rk2", oracle=oracle) if which == "L96-13" else \
        from_case("L96", "rk2", 21, 70) if which == "L96-40" else from_case("OU", "rk2", 201, 150)
    with rg.evaluator() as ev:
        Fd, Gd = dev_eval(ev, rg.X)
        Fh, Gh = ev.eval(rg.X)
    assert torch.equal(torch.from_numpy(Fh.view(np.int64)), Fd)
    assert torch.equal(torch.from_numpy(Gh.view(np.int64)), Gd)


@pytest.mark.parametrize("which", ["OU-fused", "DW-scan1-bwd", "L63-lanes", "L96-40", "L96-13"])
def test_device_layouts_and_masks(oracle, which):
    import torch
    rg = {"OU-fused": lambda: from_case("OU", "rk4", 1001, 7),
          "DW-scan1-bwd": lambda: from_case("DW", "heun", 4000, 5),
          "L63-lanes": lambda: from_case("L63", "rk2", 61, 7),
          "L96-40": lambda: from_case("L96", "rk2", 101, 6),
          "L96-13": lambda: from_l96(13, 41, 6, "heun", oracle=oracle)}[which]()
    B, n = rg.B, rg.n_x
    X = torch.from_numpy(rg.X).cuda()
    with rg.evaluator() as ev:
        F0, G0 = (t.cuda() for t in dev_eval(ev, rg.X))

        def run(Xt, xs, gs):
            xb = _fill(Xt, B, n, xs)
            Fb, gb = _alloc(B, 1, 1), _alloc(B, n, gs)
            _eval_device(ev, xb.view(torch.float64), xs, Fb.view(torch.float64), gb.view(torch.float64), gs, 1)
            return Fb, gb

        xs, gs = n + 4, n + 2
        Fb, gb = run(X, xs, gs)                                     # padded rows
        assert torch.equal(Fb, _expect(F0.view(B, 1), B, 1, 1)) and torch.equal(gb, _expect(G0, B, n, gs))
        j = 2                                                       # one x shared by every problem
        Fs, Gs = (t.cuda() for t in dev_eval(ev, np.repeat(rg.X[j:j + 1], B, axis=0)))
        Fb, gb = run(X[j:j + 1], 0, gs)
        assert torch.equal(Fb, _expect(Fs.view(B, 1), B, 1, 1)) and torch.equal(gb, _expect(Gs, B, n, gs))
        on = np.zeros(B, dtype=bool)                                # masked: skipped rows keep their sentinels
        if rg.model == "L96":
            lst = np.array([B - 1, 1, 3, 2])
            on[lst] = True
            ev.set_active_list(lst)
        else:
            on[[0, 2, 3]] = True
            flags = torch.from_numpy(on.astype(np.int32)).cuda()
            ev.set_active(flags.data_ptr())
        Fb, gb = run(X, xs, gs)
        ev.set_active_list(None) if rg.model == "L96" else ev.set_active(None)
        which_rows = torch.from_numpy(on).cuda()
        assert torch.equal(Fb, _expect(F0.view(B, 1), B, 1, 1, which_rows))
        assert torch.equal(gb, _expect(G0, B, n, gs, which_rows))
        assert int(gb[-1]) == SENT


@pytest.mark.parametrize("which", ["L96-40", "L96-13", "OU", "L63"])
def test_forced_pass_split(oracle, which):
    import torch
    rg = {"L96-40": lambda: from_case("L96", "rk4", 21, 9), "L96-13": lambda: from_l96(13, 41, 9, "rk4", oracle=oracle),
          "OU": lambda: from_case("OU", "rk4", 1001, 9), "L63": lambda: from_case("L63", "euler", 61, 9)}[which]()
    per = 8 * rg.N * (2 * rg.D + 2 * rg.D * rg.D + 1)
    with rg.evaluator() as ev:
        F0, G0 = dev_eval(ev, rg.X)
    with rg.evaluator(scratch_bytes=2 * per + 64) as ev:
        assert ev.chunk_size == 2
        F1, G1 = dev_eval(ev, rg.X)
    if which.startswith("L96"):   # Lorenz 96: the sweeps' results do not depend on the pass split
        assert torch.equal(F0, F1) and torch.equal(G0, G1)
    assert_rows_match_same_schedule(rg, F1, G1, scratch_bytes=2 * per + 64)


@pytest.mark.parametrize("which", ["OU", "DW", "L63", "L96-40", "L96-13"])
def test_hyper_device(oracle, which):
    rg = {"OU": lambda: from_case("OU", "rk4", 1001, 8), "DW": lambda: from_case("DW", "rk2", 1001, 8),
          "L63": lambda: from_case("L63", "rk2", 61, 8), "L96-40": lambda: from_case("L96", "rk2", 101, 8),
          "L96-13": lambda: from_l96(13, 41, 8, "rk2", oracle=oracle)}[which]()
    with rg.evaluator() as ev:
        F, _ = dev_eval(ev, rg.X, want_grad=False)
        h = ev.hyper(rg.X)
    assert np.array_equal(h["F"].view(np.int64), F.numpy())
    for k in range(len(rg.scheds)):
        rows = np.flatnonzero(rg.kind == k)
        with rg.same(k) as ev:
            hk = ev.hyper(rg.X)
        for key in ("F", "Esde", "dEsde_dtheta", "dEsde_dsigma"):
            assert np.array_equal(h[key][rows].view(np.int64), hk[key][rows].view(np.int64)), (k, key)


@pytest.mark.parametrize("which", ["OU", "L63", "L96-40", "L96-13"])
def test_eval_full(oracle, which):
    rg = {"OU": lambda: from_case("OU", "rk4", 1001, 4), "L63": lambda: from_case("L63", "rk2", 61, 4),
          "L96-40": lambda: from_case("L96", "rk2", 101, 4),
          "L96-13": lambda: from_l96(13, 41, 4, "rk2", oracle=oracle)}[which]()
    with rg.evaluator() as ev:
        for p in (2, 3):                                   # the dense and the sparse schedule
            out = ev.eval_full(rg.X[p], problem=p)
            ref = oracle.eval(rg.problem(p), rg.X[p], full=True)
            for key in ("F", "E0", "Esde", "Eobs"):
                assert abs(out[key] - ref[key]) <= TOL * max(abs(ref[key]), 1e-300), (p, key)
            assert grad_err(out["grad"], ref["grad"], rg.N, rg.D) < TOL, p
            for key in ("mt", "st", "lamt", "psit", "dEsde_dm", "dEsde_ds"):
                a, b = np.ravel(out[key]), np.ravel(ref[key])
                assert np.max(np.abs(a - b)) <= TOL * max(np.max(np.abs(b)), 1e-300), (p, key)


def test_not_positive_definite_names_the_problem(oracle):
    from numpy.linalg import LinAlgError
    rg = from_l96(13, 41, 4, "euler", oracle=oracle)
    X = rg.X.copy()
    N, D = rg.N, rg.D
    X[3, :N * D * D] = -200.0 * np.tile(np.eye(D).ravel(), N)
    X[3, :N * D * D] += 50.0 * np.random.default_rng(0).standard_normal(N * D * D)
    with rg.evaluator() as ev:
        with pytest.raises(LinAlgError, match="problem 3 "):
            ev.eval(X)


# ---- 4. initialisation --------------------------------------------------------------------------------------------
def interior(N):
    """Schedules that VarGP.initialization accepts: 1, 2, 3 and many observations, none at the ends."""
    return [np.array([N // 3]), np.array([2, N - 3]), np.array([3, 4, N // 2]), np.arange(1, N - 1, 4)]


@pytest.mark.parametrize("which", ["DW", "OU", "L63", "L96-40", "L96-13"])
def test_initialization(oracle, which):
    import torch
    base = {"DW": lambda: _Batch("DW", "euler", 401, 8, seed=2), "OU": lambda: _Batch("OU", "rk4", 401, 8, seed=2),
            "L63": lambda: _Batch("L63", "rk2", 61, 8, seed=2), "L96-40": lambda: _Batch("L96", "rk2", 41, 8, seed=2),
            "L96-13": lambda: L96Batch(13, 41, 8, "rk2", oracle=oracle)}[which]()
    if which == "L96-13":
        base.model = "L96"
        rg = Ragged(base, L96_DT, L96_DT, scheds=interior(base.N))
    else:
        rg = Ragged(base, float(base.g["dt"]), Problem.from_golden(base.g).dt_model, scheds=interior(base.N))
    with rg.evaluator() as ev:
        X0 = ev.initialization(0.0)
        Xd = torch.full((rg.B, rg.n_x + 2), float("nan"), dtype=torch.float64, device="cuda")
        ev.initialization_device(Xd.data_ptr(), rg.n_x + 2, 0.0, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    assert np.array_equal(Xd[:, :rg.n_x].cpu().numpy().view(np.int64), X0.view(np.int64))
    for p in range(rg.B):
        assert grad_err(X0[p], oracle.initialization(rg.problem(p), 0.0), rg.N, rg.D) < TOL, p


@pytest.mark.parametrize("bad,match", [("none", "problem 2 has none"), ("first", "problem 2 sits"),
                                       ("last", "problem 2 sits")])
def test_initialization_errors_name_the_problem(bad, match):
    base = _Batch("OU", "rk4", 101, 4, seed=2)
    N = base.N
    sc = interior(N)
    sc[2] = {"none": np.zeros(0, dtype=np.int64), "first": np.array([0, 5]), "last": np.array([5, N - 1])}[bad]
    rg = Ragged(base, float(base.g["dt"]), Problem.from_golden(base.g).dt_model, scheds=sc)
    with rg.evaluator() as ev:
        with pytest.raises(ValueError, match=match):
            ev.initialization(0.0)


# ---- 5. optimisers ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["L63", "DW"])
def test_batched_scg_traces_equal_same_schedule_batches(which):
    from vgpa_b200.batched_scg import BatchedSCG
    rg = from_case("L63", "rk2", 61, 8) if which == "L63" else from_case("DW", "rk4", 401, 8)
    opts = {"max_it": 25, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    with rg.evaluator() as ev:
        opt = BatchedSCG(ev, opts)
        _, fx = opt(rg.X)
        st = opt.stats
    for k in range(len(rg.scheds)):
        rows = np.flatnonzero(rg.kind == k)
        with rg.same(k) as ev:
            opt = BatchedSCG(ev, opts)
            _, fxk = opt(rg.X)
            sk = opt.stats
        assert np.array_equal(st["MaxIt"][rows], sk["MaxIt"][rows]), k
        assert np.array_equal(st["fx"][:, rows].view(np.int64), sk["fx"][:, rows].view(np.int64)), k
        assert np.array_equal(fx[rows].view(np.int64), fxk[rows].view(np.int64)), k


def test_sharded_batched_scg_on_ragged_lists():
    from vgpa_b200.batched_scg import BatchedSCG, ShardedBatchedSCG
    base = _Batch("L63", "rk2", 61, 6, seed=4)
    rg = Ragged(base, float(base.g["dt"]), Problem.from_golden(base.g).dt_model, scheds=interior(base.N))
    opts = {"max_it": 8, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    ens = ShardedBatchedSCG(rg.B, lambda lo, hi: rg.evaluator(np.arange(lo, hi)), opts, sub_batch=2)
    res = ens.run(t0=0.0, hyper=True)
    assert res["fx"].shape == (rg.B,) and np.all(np.isfinite(res["fx"]))
    assert res["dEsde_dtheta"].shape == (rg.B, 3) and res["Esde"].shape == (rg.B,)
    for lo in range(0, rg.B, 2):                           # each sub-batch is its own ragged handle
        idx = np.arange(lo, lo + 2)
        with rg.evaluator(idx) as ev:
            _, fx = BatchedSCG(ev, opts)(ev.initialization(0.0))
        assert np.array_equal(res["fx"][idx].view(np.int64), fx.view(np.int64)), lo
