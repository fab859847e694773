"""
Lorenz 96 at state dimensions other than 40 (10 <= D <= 64): the run-time-D kernel family of l96_dyn.cu.

  - F and gradient against the oracle at 1e-9 for D in {10, 13, 24, 39, 41, 64}, every solver, plus one long
    recurrence (D = 64, RK4, N = 1001); every problem of a batch has its own theta, Sigma, R, observations, m0, s0,
    E0 and x;
  - vgpa_eval_full, the stand-alone operators and the hyper-parameter gradients against the oracle;
  - bits: a problem's F and gradient do not depend on its batch position, the pass split, active sets, compacted
    lists, padded strides or a shared x; skipped rows and padding keep their sentinel bits;
  - initialisation, sample paths (bit for bit), observations, BatchedSCG against a host SCG on the oracle,
    ShardedBatchedSCG(hyper=True), argument errors and the LinAlgError of a non-positive-definite S(t).
The oracle's Lorenz-96 code takes its D from the problem; at D = 40 it is pinned to the reference's goldens.
"""
import os
from pathlib import Path

import numpy as np
import pytest

from conftest import grad_err, rel_err
from oracle import Problem

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
TOL = 1e-9
DT = 0.01


def l96_path(D, N, dt, theta, sigma, z):
    """Lorenz96.make_trajectory (lorenz_96.py:249-314) in numpy, given its draws z (D, N): the burn-in from
    theta * ones(D) with int(D / 2) perturbed, then Euler-Maruyama; one IEEE operation per numpy operation."""
    f = lambda x: (np.roll(x, -1) - np.roll(x, 2)) * np.roll(x, 1) - x + theta
    x = theta * np.ones(D)
    x[int(D / 2.0)] += 1.0e-3
    for _ in range(5000):
        x = x + f(x) * 1.0e-3
    out = np.empty((N, D))
    out[0] = x
    sq = np.sqrt(np.asarray(sigma) * dt)
    for t in range(1, N):
        x = x + f(x) * dt + sq * z[:, t]
        out[t] = x
    return out


class L96Batch:
    """B Lorenz-96 problems of dimension D on an N-point grid that differ in every per-problem input."""

    def __init__(self, D, N, B, method="rk2", seed=0, oracle=None):
        rng = np.random.default_rng([seed, D, N, B])
        self.D, self.N, self.B, self.method = D, N, B, method
        u = np.linspace(0.0, 1.0, B)[:, None]
        path = l96_path(D, N, DT, 8.0, np.ones(D), rng.standard_normal((D, N)))
        self.obs_t = np.arange(5, N - 2, 10, dtype=np.int64)
        M = self.obs_t.size
        self.theta = 8.0 * (1.0 + 0.02 * u)
        self.sigma = (0.7 + 0.6 * u) * (1.0 + 0.1 * rng.random((B, D)))
        self.R = (0.8 + 0.4 * u) * np.ones((B, D))
        self.obs_y = path[self.obs_t][None] + 0.3 * rng.standard_normal((B, M, D))
        self.m0 = path[0][None] + 0.1 * rng.standard_normal((B, D))
        self.s0 = np.stack([(0.2 + 0.05 * k) * np.eye(D) for k in u[:, 0]])
        self.E0 = 3.0 + u[:, 0]
        self.n_x = N * D * (D + 1)
        orc = oracle
        X = []
        for i in range(B):
            x0 = orc.initialization(self.problem(i))
            X.append(x0 * (1.0 + 0.01 * rng.standard_normal(x0.size)))
        self.X = np.stack(X)

    def problem(self, i):
        D = self.D
        return Problem(model="L96", method=self.method, D=D, N=self.N, dt=DT, theta=self.theta[i], sigma=self.sigma[i],
                       R=self.R[i], obs_t=self.obs_t, obs_y=self.obs_y[i], m0=self.m0[i], s0=self.s0[i],
                       E0=float(self.E0[i]), dt_model=DT)

    def evaluator(self, rows=None, **kw):
        from vgpa_b200.engine import BatchEvaluator
        r = np.arange(self.B) if rows is None else np.asarray(rows)
        return BatchEvaluator("L96", self.method, self.N, DT, theta=self.theta[r], sigma=self.sigma[r], R=self.R[r],
                              obs_t=self.obs_t, obs_y=self.obs_y[r], m0=self.m0[r], s0=self.s0[r].reshape(len(r), -1),
                              E0=self.E0[r], B=len(r), dt_model=DT, D=self.D, **kw)


def _check(oracle, bt, F, G, rows):
    for i in rows:
        Fo, Go = oracle.eval(bt.problem(i), bt.X[i])
        assert abs(F[i] - Fo) <= TOL * abs(Fo), (bt.D, i, F[i], Fo)
        assert grad_err(G[i], Go, bt.N, bt.D) < TOL, (bt.D, i)


@pytest.mark.parametrize("method", ["euler", "heun", "rk2", "rk4"])
@pytest.mark.parametrize("D", [10, 13, 24, 39, 41, 64])
def test_parity_with_oracle(oracle, D, method):
    N = {"euler": 51, "heun": 81, "rk2": 101, "rk4": 201}[method]
    bt = L96Batch(D, N, 5, method, oracle=oracle)
    with bt.evaluator() as ev:
        F, G = ev.eval(bt.X)
    _check(oracle, bt, F, G, (0, 2, 4))


def test_long_recurrence_d64_rk4(oracle):
    bt = L96Batch(64, 1001, 2, "rk4", oracle=oracle)
    with bt.evaluator() as ev:
        F, G = ev.eval(bt.X)
    _check(oracle, bt, F, G, (0, 1))


@pytest.mark.parametrize("D", [13, 64])
def test_eval_full(oracle, D):
    bt = L96Batch(D, 61, 3, "rk4", oracle=oracle)
    with bt.evaluator() as ev:
        got = ev.eval_full(bt.X[1], problem=1)
    ref = oracle.eval(bt.problem(1), bt.X[1], full=True)
    for k in ("mt", "st", "lamt", "psit", "Efx", "Edf", "dEsde_dm", "dEsde_ds"):
        assert rel_err(np.asarray(got[k]).ravel(), ref[k].ravel()) < TOL, k
    assert abs(got["F"] - ref["F"]) <= TOL * abs(ref["F"])
    for k in ("E0", "Esde", "Eobs"):
        assert abs(got[k] - ref[k]) <= TOL * max(abs(ref[k]), 1e-300), k
    assert grad_err(got["grad"], ref["grad"], bt.N, D) < TOL


@pytest.mark.parametrize("D", [10, 64])
def test_standalone_operators(oracle, D):
    from vgpa_b200 import engine
    bt = L96Batch(D, 41, 1, "rk2", oracle=oracle)
    prob, x = bt.problem(0), bt.X[0]
    N = bt.N
    ref = oracle.eval(prob, x, full=True)
    A, b = x[:N * D * D].reshape(N, D, D), x[N * D * D:].reshape(N, D)
    mt, st = engine.solve_fwd("rk2", A, b, bt.m0[0], bt.s0[0], bt.sigma[0], DT)
    assert rel_err(mt, ref["mt"]) < TOL and rel_err(st, ref["st"]) < TOL
    Eobs, jm, js = engine.obs_energy(bt.obs_t, bt.obs_y[0], bt.R[0], ref["mt"], ref["st"])
    assert abs(Eobs - ref["Eobs"]) <= TOL * abs(ref["Eobs"])
    lam, psi = engine.solve_bwd("rk2", A, ref["dEsde_dm"], ref["dEsde_ds"], jm, js, DT)
    assert rel_err(lam, ref["lamt"]) < TOL and rel_err(psi, ref["psit"]) < TOL
    Esde, Ef, Edf, dm, ds, dth, dsig = engine.model_energy("L96", bt.theta[0], bt.sigma[0], A, b, ref["mt"], ref["st"],
                                                          DT, hyper=True)
    assert abs(Esde - ref["Esde"]) <= TOL * abs(ref["Esde"])
    for got, k in ((Ef, "Efx"), (Edf, "Edf"), (dm, "dEsde_dm"), (ds, "dEsde_ds")):
        assert rel_err(got, ref[k]) < TOL, k
    o_th, o_sig = oracle.energy_hyper(prob, x, ref["mt"], ref["st"])
    assert rel_err(dth, o_th) < TOL and rel_err(dsig, o_sig) < TOL


@pytest.mark.parametrize("D", [12, 41])
def test_hyper_gradients(oracle, D):
    import torch
    bt = L96Batch(D, 61, 4, "rk2", oracle=oracle)
    with bt.evaluator() as ev:
        h = ev.hyper(bt.X)
        F, Esde, dth, dsig = h["F"], h["Esde"], h["dEsde_dtheta"], h["dEsde_dsigma"]
        X = torch.as_tensor(bt.X, device="cuda")
        Fd = torch.empty(bt.B, dtype=torch.float64, device="cuda")
        ev.eval_device(X.data_ptr(), bt.n_x, Fd.data_ptr())
        ev.sync()
    assert np.array_equal(np.asarray(F).view(np.int64), Fd.cpu().numpy().view(np.int64))
    for i in range(bt.B):
        full = oracle.eval(bt.problem(i), bt.X[i], want_grad=False, full=True)
        o_th, o_sig = oracle.energy_hyper(bt.problem(i), bt.X[i], full["mt"], full["st"])
        assert rel_err(dth[i], o_th) < TOL and rel_err(np.asarray(dsig[i]).ravel(), o_sig.ravel()) < TOL, i
        S = np.asarray(dsig[i]).reshape(D, D)
        assert np.all(S[~np.eye(D, dtype=bool)] == 0.0)
        assert abs(np.sum(bt.sigma[i] * np.diag(S)) + Esde[i]) <= 1e-12 * abs(Esde[i])


def _dev_eval(ev, X, xs, gs, B, n):
    """vgpa_eval_device into sentinel-filled buffers with a guard row; returns (F, G) host copies (bits)."""
    import torch
    F = torch.full((B + 1,), float("nan"), dtype=torch.float64, device="cuda")
    G = torch.full(((B + 1) * gs,), float("nan"), dtype=torch.float64, device="cuda")
    ev.eval_device(X.data_ptr(), xs, F.data_ptr(), G.data_ptr(), gs)
    ev.sync()
    return F.cpu().numpy(), G.cpu().numpy().reshape(B + 1, gs)


@pytest.mark.parametrize("D", [13, 41])
def test_bits_do_not_depend_on_layout(oracle, D):
    import torch
    B, N = 7, 31
    bt = L96Batch(D, N, B, "rk2", seed=3, oracle=oracle)
    n = bt.n_x
    per = 8 * N * (2 * D + 2 * D * D + 1)
    X = torch.as_tensor(bt.X, device="cuda").contiguous()
    nan_bits = np.float64("nan").view(np.int64)
    with bt.evaluator(scratch_bytes=3 * per) as ev:         # passes of 3, 3 and a ragged 1
        assert ev.chunk_size == 3
        F0, G0 = _dev_eval(ev, X, n, n, B, n)
        _check(oracle, bt, F0, G0, (0, 3, 6))
        # padded strides
        Xp = torch.zeros((B, n + 6), dtype=torch.float64, device="cuda")
        Xp[:, :n] = X
        F1, G1 = _dev_eval(ev, Xp, n + 6, n + 4, B, n)
        assert np.array_equal(F1[:B].view(np.int64), F0[:B].view(np.int64))
        assert np.array_equal(G1[:B, :n].view(np.int64), G0[:B, :n].view(np.int64))
        assert np.all(G1[:B, n:].view(np.int64) == nan_bits) and np.all(G1[B].view(np.int64) == nan_bits)
        # compacted unsorted list across passes: listed rows equal, the others keep their sentinels
        lst = [5, 1, 6, 2]
        ev.set_active_list(lst)
        F2, G2 = _dev_eval(ev, X, n, n, B, n)
        ev.set_active_list(None)
        for p in range(B):
            if p in lst:
                assert F2[p].view(np.int64) == F0[p].view(np.int64) and np.array_equal(G2[p].view(np.int64), G0[p].view(np.int64))
            else:
                assert F2[p].view(np.int64) == nan_bits and np.all(G2[p].view(np.int64) == nan_bits)
        # active flags
        act = torch.tensor([1, 0, 1, 0, 0, 1, 1], dtype=torch.int32, device="cuda")
        ev.set_active(act.data_ptr())
        F3, G3 = _dev_eval(ev, X, n, n, B, n)
        ev.set_active(None)
        for p in range(B):
            ok = bool(act[p])
            assert (F3[p].view(np.int64) == F0[p].view(np.int64)) if ok else (F3[p].view(np.int64) == nan_bits)
    # batch position: the problems reversed, one pass
    rev = np.arange(B)[::-1].copy()
    with bt.evaluator(rows=rev) as ev:
        F4, G4 = _dev_eval(ev, X[torch.as_tensor(rev, device="cuda")].contiguous(), n, n, B, n)
    assert np.array_equal(F4[:B][::-1].view(np.int64), F0[:B].view(np.int64))
    assert np.array_equal(G4[:B][::-1].view(np.int64), G0[:B].view(np.int64))
    # a shared x (stride 0) equals B copies of it
    with bt.evaluator() as ev:
        F5, G5 = _dev_eval(ev, X[2].contiguous(), 0, n, B, n)
        F6, G6 = _dev_eval(ev, X[2:3].expand(B, n).contiguous(), n, n, B, n)
    assert np.array_equal(F5.view(np.int64), F6.view(np.int64)) and np.array_equal(G5.view(np.int64), G6.view(np.int64))


def test_initialization(oracle):
    bt = L96Batch(24, 71, 3, "rk2", oracle=oracle)
    with bt.evaluator() as ev:
        X0 = ev.initialization(0.0)
    for i in range(bt.B):
        assert grad_err(X0[i], oracle.initialization(bt.problem(i)), bt.N, bt.D) < TOL, i


@pytest.mark.parametrize("D", [10, 41, 64])
def test_sample_paths_and_observations(oracle, D):
    from vgpa_b200 import engine
    N, B = 301, 3
    rng = np.random.default_rng(D)
    z = rng.standard_normal((B, D, N))
    theta = np.array([[8.0], [7.5], [9.0]])
    sig = 0.5 + rng.random((B, D))
    paths = engine.make_trajectories("L96", N, DT, theta, sig, z)
    assert paths.shape == (B, N, D)
    for p in range(B):
        ref = l96_path(D, N, DT, theta[p, 0], sig[p], z[p])
        assert np.array_equal(paths[p].view(np.int64), ref.view(np.int64)), p
    obs_t = np.arange(10, N, 25)
    R = 0.3 + rng.random(D)
    xi = rng.standard_normal((B, D, obs_t.size))
    obs = engine.collect_observations(paths, obs_t, R, xi)
    for p in range(B):
        assert np.array_equal(obs[p], oracle.collect_obs(paths[p], obs_t, R, xi[p])), p


def test_lorenz96_object_at_d20():
    from vgpa_b200.dynamics import Lorenz96
    m = Lorenz96([1.0] * 20, 8.0, r_seed=3, dim_d=20)
    m.make_trajectory(0.0, 2.0, 0.01, device=0)
    dev = m.sample_path.copy()
    m2 = Lorenz96([1.0] * 20, 8.0, r_seed=3, dim_d=20)
    m2.make_trajectory(0.0, 2.0, 0.01)
    assert dev.shape == (201, 20) and np.array_equal(dev, m2.sample_path)


def test_lorenz96_d20_vargp_scg_converges():
    """Lorenz96([1.0] * 20, 8.0, dim_d=20) with its own observations, VarGP built from it as Simulation.build does:
    free_energy, gradient and the host SCG run to convergence on the GPU."""
    from vgpa_b200 import SCG, BwdOde, FwdOde, GaussianLikelihood, Lorenz96, PriorKL0, VarGP
    D, dt = 20, 0.01
    m = Lorenz96([1.0] * D, 8.0, r_seed=5, dim_d=D)
    m.make_trajectory(0.0, 1.0, dt)
    obs_t, obs_y, obs_noise = m.collect_obs(8, 1.0)
    m0 = m.sample_path[0] + 0.1 * m.rng.standard_normal(D)
    vgpa = VarGP(m, m0, 0.2 * np.eye(D), FwdOde(dt, "rk2", False), BwdOde(dt, "rk2", False),
                 GaussianLikelihood(obs_y, obs_t, obs_noise, None, False), PriorKL0(np.ones(D), 0.5 * np.eye(D), False),
                 obs_y, obs_t)
    x0 = vgpa.initialization()
    F0, g0 = vgpa.free_energy(x0), vgpa.gradient(x0)
    assert np.isfinite(F0) and g0.shape == x0.shape and np.all(np.isfinite(g0))
    opts = {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    scg = SCG(vgpa.free_energy, vgpa.gradient, opts)
    x, fx = scg(x0.copy())
    assert int(scg.stats["MaxIt"]) < opts["max_it"] and fx < F0
    vgpa.close()


def test_batched_scg_matches_host_scg(oracle):
    from vgpa_b200.batched_scg import BatchedSCG
    from vgpa_b200.scg import SCG
    bt = L96Batch(12, 101, 3, "rk2", seed=5, oracle=oracle)
    opts = {"max_it": 60, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    with bt.evaluator() as ev:
        opt = BatchedSCG(ev, opts)
        X, fx = opt(bt.X)
        st = opt.stats
    for p in range(bt.B):
        prob = bt.problem(p)
        f = lambda x: oracle.eval(prob, x, want_grad=False)[0]
        df = lambda x, eval_fun=False: oracle.eval(prob, x)[1]
        scg = SCG(f, df, opts)
        x1, f1 = scg(bt.X[p].copy())
        n = min(int(scg.stats["MaxIt"]), int(st["MaxIt"][p]))
        ref, new = scg.stats["fx"][:n], st["fx"][:n, p]
        assert np.max(np.abs(new - ref) / np.maximum(np.abs(ref), 1.0)) < 1e-6, p
        assert abs(fx[p] - f1) <= 1e-6 * max(abs(f1), 1.0), p


def test_sharded_hyper_keys(oracle):
    from vgpa_b200.batched_scg import ShardedBatchedSCG
    bt = L96Batch(12, 61, 4, "rk2", seed=6, oracle=oracle)
    opts = {"max_it": 5, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    ens = ShardedBatchedSCG(bt.B, lambda lo, hi: bt.evaluator(rows=np.arange(lo, hi)), opts, sub_batch=2)
    res = ens.run(t0=0.0, hyper=True)
    assert res["dEsde_dtheta"].shape == (bt.B, 12) and res["dEsde_dsigma_diag"].shape == (bt.B, 12)
    assert res["Esde"].shape == (bt.B,)


@pytest.mark.parametrize("D", [9, 65])
def test_out_of_range_dimensions_raise(oracle, D):
    from vgpa_b200 import engine
    from vgpa_b200.dynamics import Lorenz96
    with pytest.raises(ValueError):
        Lorenz96([1.0] * D, 8.0, dim_d=D)
    with pytest.raises(ValueError):
        engine.BatchEvaluator("L96", "rk2", 11, DT, theta=8.0, sigma=np.ones(D), R=np.ones(D), obs_t=[5],
                              obs_y=np.zeros(D), m0=np.zeros(D), s0=np.eye(D).ravel(), E0=0.0, D=D)
    N = 11
    with pytest.raises(ValueError):
        engine.solve_fwd("rk2", np.zeros((N, D, D)), np.zeros((N, D)), np.zeros(D), np.eye(D), np.ones(D), DT)
    with pytest.raises(ValueError):
        engine.make_trajectories("L96", N, DT, [8.0], np.ones(D), np.zeros((1, D, N)))


def test_not_positive_definite_is_linalg_error(oracle):
    from numpy.linalg import LinAlgError
    bt = L96Batch(13, 41, 3, "euler", oracle=oracle)
    X = bt.X.copy()
    N, D = bt.N, bt.D
    X[1, :N * D * D] = -200.0 * np.tile(np.eye(D).ravel(), N)            # S(t) leaves the PD cone
    X[1, :N * D * D] += 50.0 * np.random.default_rng(0).standard_normal(N * D * D)
    with bt.evaluator() as ev:
        with pytest.raises(LinAlgError, match="problem 1 "):
            ev.eval(X)


def test_reference_lorenz96_d20_dropin():
    """The reference's own Lorenz96(..., dim_d=20) and its FwdOde, BwdOde, GaussianLikelihood and PriorKL0 objects
    drive vgpa_b200.VarGP; one evaluation at a dense perturbation of x0 must match the reference's own VarGP to 1e-9
    (skips without the reference tree: VGPA_REFERENCE or baseline/_ref)."""
    import contextlib
    import io
    import sys
    try:
        from baseline.refload import import_reference
        ref = import_reference()
        from src.dynamics.lorenz_96 import Lorenz96 as RefL96
    except ImportError as e:
        pytest.skip(f"the unmodified reference is not importable here: {e}")
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import make_golden as mg
    from vgpa_b200.variational import VarGP
    D, dt = 20, 0.01
    with contextlib.redirect_stdout(io.StringIO()):
        model = RefL96([1.0] * D, 8.0, mg.SEED, dim_d=D)
        model.make_trajectory(0.0, 0.4, dt)
        obs_t, obs_y, obs_noise = model.collect_obs(8, 1.0, None)
    m0 = model.sample_path[0] + 0.1 * model.rng.standard_normal(D)
    s0 = 0.2 * np.eye(D)
    args = (model, m0, s0, ref["FwdOde"](dt, "rk2", False), ref["BwdOde"](dt, "rk2", False),
            ref["GaussianLikelihood"](obs_y, obs_t, obs_noise, None, False),
            ref["PriorKL0"](1.0 * np.ones(D), 0.5 * np.eye(D), False), obs_y, obs_t)
    ref_vgpa, vgpa = ref["VarGP"](*args), VarGP(*args)
    x0 = ref_vgpa.initialization()
    x = mg.perturb(x0, D, vgpa.dim_n, np.random.default_rng([mg.SEED, 20]))
    F_ref, g_ref = ref_vgpa.free_energy(x), ref_vgpa.gradient(x)
    F, g = vgpa.free_energy(x), vgpa.gradient(x)
    assert abs(F - F_ref) <= TOL * abs(F_ref)
    assert grad_err(g, g_ref, vgpa.dim_n, D) < TOL
    vgpa.close()
