"""
Partially observed problems on the device (vgpa_create_observed, vgpa_obs_energy_observed, BatchEvaluator(observed=...),
GaussianLikelihood(operator=...), VarGP, Simulation).

  1. Oracle parity for every kernel family with D > 1 (the CASES of test_gpu_layouts.py for L63 and L96 D = 40, plus
     run-time-D L96 at D = 13 and 64), with masks of one component, all but one, alternating and random ones, assigned
     per problem: F and every gradient block at 1e-9.
  2. A full mask gives the bits of a handle without one: F, gradient, vgpa_eval_full and x0.
  3. Independent of the oracle: a masked handle against an unmasked one with R_i = 1e100 off the mask (1e-12).
  4. NaN in unobserved obs_y columns and R entries gives the bits of zeros there.
  5. Per-problem masks: every row is, bit for bit, the row of a handle of the same B (and pass split) in which every
     problem carries that row's mask, also with ragged schedules; active flags and an unsorted compacted list give
     the listed rows of the full evaluation.
  6. vgpa_hyper_device: F as vgpa_eval, dEsde as the unmasked handle.
  7. Initialisation: observed components as the unmasked handle, unobserved b0 = a_dd m0_d, host VarGP agrees.
  8. The stand-alone likelihood against the oracle.
  9. Simulation end to end with the JSON's operator, both optimisers; BatchedSCG against a host SCG on the oracle.
"""
import sys

import numpy as np
import pytest

from conftest import GOLDEN, grad_err, rel_err
from partial_obs_oracle import PartialObsOracle
from test_gpu_l96_dims import L96Batch
from test_gpu_layouts import _Batch, _sample_rows

sys.path.insert(0, str(GOLDEN))
import make_golden as mg  # noqa: E402

pytestmark = pytest.mark.gpu
TOL = 1e-9


def mask_pool(D, seed=0):
    """One component, all but one, alternating, and two random masks (as bit words)."""
    rng = np.random.default_rng([seed, D])
    rand = [int(sum(1 << int(i) for i in rng.choice(D, rng.integers(1, D), replace=False))) for _ in range(2)]
    return [1 << (D // 2), ((1 << D) - 1) & ~(1 << 1), sum(1 << i for i in range(0, D, 2))] + rand


def bits(w, D):
    return [i for i in range(D) if (w >> i) & 1]


# (model, method, N, B, problems per pass (0: one pass), family): the D > 1 families of test_gpu_layouts.CASES
FAMILIES = [
    ("L63", "rk2", 61, 7, 0, "lanes"),
    ("L63", "heun", 30, 8193, 0, "staged-fwd-one-thread-bwd"),
    ("L63", "euler", 61, 11, 3, "lanes-passes"),
    ("L96", "rk2", 101, 5, 0, "small-launch"),
    ("L96", "rk4", 21, 1800, 900, "full-wave"),
]


def _family(case, seed=1):
    model, method, N, B, per_pass, _ = case
    bt = _Batch(model, method, N, B, seed=seed)
    kw = dict(scratch_bytes=per_pass * bt.per_problem_bytes() + 64) if per_pass else {}
    return bt, kw


def _ev(bt, **over):
    """A handle over the problems of a test_gpu_layouts batch, any of its inputs replaced."""
    from test_gpu_parity import evaluator_from_golden
    kw = dict(B=bt.B, N=bt.N, obs_t=bt.obs_t, theta=bt.theta, sigma=bt.sigma, R=bt.R, obs_y=bt.obs_y, m0=bt.m0,
              s0=bt.s0, E0=bt.E0)
    kw.update(over)
    return evaluator_from_golden(bt.g, **kw)


@pytest.fixture(scope="module")
def masked(oracle):
    """The oracle with a component-selecting operator (partial_obs_oracle.py)."""
    return PartialObsOracle(oracle)


@pytest.mark.parametrize("case", FAMILIES, ids=lambda c: f"{c[0]}-{c[1]}-B{c[3]}-{c[5]}")
def test_oracle_parity_and_rows_of_every_family(masked, case):
    bt, kw = _family(case)
    D, B = bt.D, bt.B
    pool = mask_pool(D)
    kind = np.arange(B) % len(pool)
    words = [pool[k] for k in kind]
    with _ev(bt, observed=[bits(w, D) for w in words], **kw) as ev:
        chunk = ev.chunk_size
        F, G = ev.eval(bt.X)
    for i in _sample_rows(B, chunk) + [k for k in range(len(pool)) if k < B]:
        Fo, go = masked.eval(bt.problem(i), words[i], bt.X[i])
        assert abs(F[i] - Fo) <= TOL * abs(Fo), (i, F[i], Fo)
        assert grad_err(G[i], go, bt.N, D) < TOL, i
    # every row is the row of a handle in which every problem carries that row's mask
    for k, w in enumerate(pool):
        rows = np.flatnonzero(kind == k)
        if rows.size == 0:
            continue
        with _ev(bt, observed=bits(w, D), **kw) as ev1:
            F1, G1 = ev1.eval(bt.X)
        assert np.array_equal(F[rows], F1[rows]), k
        assert np.array_equal(G[rows], G1[rows]), k


@pytest.mark.parametrize("D", [13, 64])
def test_oracle_parity_at_run_time_d(oracle, masked, D):
    bt = L96Batch(D, 41, 6, method="heun" if D == 13 else "rk2", oracle=oracle)
    pool = mask_pool(D)
    words = [pool[p % len(pool)] for p in range(bt.B)]
    with bt.evaluator(observed=[bits(w, D) for w in words]) as ev:
        F, G = ev.eval(bt.X)
    for i in range(bt.B):
        Fo, go = masked.eval(bt.problem(i), words[i], bt.X[i])
        assert abs(F[i] - Fo) <= TOL * abs(Fo), (i, F[i], Fo)
        assert grad_err(G[i], go, bt.N, D) < TOL, i
    w = pool[2]
    with bt.evaluator(observed=bits(w, D)) as ev1:
        F1, G1 = ev1.eval(bt.X)
    rows = [p for p in range(bt.B) if words[p] == w]
    assert np.array_equal(F[rows], F1[rows]) and np.array_equal(G[rows], G1[rows])


SMALL = [FAMILIES[0], FAMILIES[3]]


@pytest.mark.parametrize("case", SMALL, ids=lambda c: f"{c[0]}-{c[5]}")
def test_full_mask_gives_the_identity_bits(case):
    bt, kw = _family(case)
    D = bt.D
    with _ev(bt, **kw) as ev0, _ev(bt, observed=np.ones(D, dtype=bool), **kw) as ev1:
        F0, G0 = ev0.eval(bt.X)
        F1, G1 = ev1.eval(bt.X)
        assert np.array_equal(F0, F1) and np.array_equal(G0, G1)
        a, b = ev0.eval_full(bt.X[1], problem=1), ev1.eval_full(bt.X[1], problem=1)
        for k in ("F", "E0", "Esde", "Eobs", "grad", "mt", "st", "lamt", "psit", "Efx", "Edf", "dEsde_dm", "dEsde_ds"):
            assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(ev0.initialization(), ev1.initialization())


@pytest.mark.parametrize("case", SMALL, ids=lambda c: f"{c[0]}-{c[5]}")
def test_mask_is_the_large_noise_limit(case):
    """Tied to the golden-pinned identity path without the oracle: an unobserved component is one observed with
    infinite noise."""
    bt, kw = _family(case)
    D, M = bt.D, bt.obs_t.size
    for w in mask_pool(D)[:3]:
        hidden = [i for i in range(D) if not (w >> i) & 1]
        R_big = bt.R.copy()
        R_big[:, hidden] = 1e100
        with _ev(bt, observed=bits(w, D), **kw) as evm, _ev(bt, R=R_big, **kw) as evu:
            Fm, Gm = evm.eval(bt.X)
            Fu, Gu = evu.eval(bt.X)
            fm, fu = evm.eval_full(bt.X[0], 0), evu.eval_full(bt.X[0], 0)
        for p in range(bt.B):
            assert grad_err(Gm[p], Gu[p], bt.N, D) < 1e-12, (w, p)
            count = 0.5 * M * np.sum(np.log(2 * np.pi) + np.log(R_big[p, hidden]))
            assert abs(Fm[p] + count - Fu[p]) <= 1e-12 * abs(Fu[p]), (w, p)
        assert rel_err(fm["lamt"], fu["lamt"]) < 1e-12 and rel_err(fm["psit"], fu["psit"]) < 1e-12


@pytest.mark.parametrize("case", SMALL, ids=lambda c: f"{c[0]}-{c[5]}")
def test_unobserved_inputs_are_never_read(case):
    bt, kw = _family(case)
    D = bt.D
    words = [mask_pool(D)[p % 3] for p in range(bt.B)]
    seen = np.array([[(w >> i) & 1 for i in range(D)] for w in words], dtype=bool)
    out = []
    for fill in (0.0, np.nan):
        y = np.where(seen[:, None, :], bt.obs_y, fill)
        R = np.where(seen, bt.R, fill)
        with _ev(bt, observed=seen, obs_y=y, R=R, **kw) as ev:
            F, G = ev.eval(bt.X)
            full = ev.eval_full(bt.X[2], 2)
            out.append((F, G, full, ev.initialization()))
    (F0, G0, f0, x0), (F1, G1, f1, x1) = out
    assert np.isfinite(F1).all()
    assert np.array_equal(F0, F1) and np.array_equal(G0, G1) and np.array_equal(x0, x1)
    for k in ("F", "Eobs", "grad", "lamt", "psit"):
        assert np.array_equal(f0[k], f1[k]), k


def test_ragged_schedules_passes_active_flags_and_lists():
    """Per-problem masks with per-problem schedules and a forced pass split: rows as in one-mask handles; active
    flags and an unsorted compacted list give the listed rows of the full evaluation."""
    import torch
    bt, _ = _family(("L96", "rk2", 61, 12, 0, ""))
    D, B, N = bt.D, bt.B, bt.N
    kw = dict(scratch_bytes=5 * bt.per_problem_bytes() + 64)
    scheds = [np.array([5, 17, 30]), np.array([9]), np.arange(3, N - 2, 4), np.zeros(0, dtype=np.int64)]
    obs_t = [scheds[p % 4] for p in range(B)]
    rng = np.random.default_rng(5)
    obs_y = [bt.obs_y[p, :1] + 0.1 * rng.standard_normal((t.size, D)) for p, t in enumerate(obs_t)]
    pool = mask_pool(D, seed=3)
    words = [pool[p % len(pool)] for p in range(B)]
    X = bt.X
    with _ev(bt, obs_t=obs_t, obs_y=obs_y, observed=[bits(w, D) for w in words], **kw) as ev:
        assert ev.chunk_size < B
        F, G = ev.eval(X)
        Xd = torch.from_numpy(X).cuda()
        Fd = torch.full((B,), -7.0, dtype=torch.float64, device="cuda")
        Gd = torch.full((B, bt.n_x), -7.0, dtype=torch.float64, device="cuda")
        listed = [9, 2, 7, 0, 11]
        act = torch.zeros(B, dtype=torch.int32, device="cuda")
        act[listed] = 1
        ev.set_active(act.data_ptr())
        ev.set_active_list(listed)
        ev.eval_device(Xd.data_ptr(), bt.n_x, Fd.data_ptr(), Gd.data_ptr())
        ev.sync()
        ev.set_active_list(None)
        ev.set_active(None)
        Fl, Gl = Fd.cpu().numpy(), Gd.cpu().numpy()
    assert np.array_equal(Fl[listed], F[listed]) and np.array_equal(Gl[listed], G[listed])
    rest = [p for p in range(B) if p not in listed]
    assert (Fl[rest] == -7.0).all() and (Gl[rest] == -7.0).all()
    for k, w in enumerate(pool):
        rows = [p for p in range(B) if words[p] == w]
        with _ev(bt, obs_t=obs_t, obs_y=obs_y, observed=bits(w, D), **kw) as ev1:
            F1, G1 = ev1.eval(X)
        assert np.array_equal(F[rows], F1[rows]) and np.array_equal(G[rows], G1[rows]), k


@pytest.mark.parametrize("case", SMALL, ids=lambda c: f"{c[0]}-{c[5]}")
def test_hyper_path_follows_the_mask(case):
    bt, kw = _family(case)
    D = bt.D
    words = [mask_pool(D)[p % 3] for p in range(bt.B)]
    with _ev(bt, observed=[bits(w, D) for w in words], **kw) as ev, _ev(bt, **kw) as ev0:
        F, _ = ev.eval(bt.X)
        h, h0 = ev.hyper(bt.X), ev0.hyper(bt.X)
    assert np.array_equal(h["F"], F)
    for k in ("Esde", "dEsde_dtheta", "dEsde_dsigma"):
        assert np.array_equal(h[k], h0[k]), k


@pytest.mark.parametrize("case", SMALL, ids=lambda c: f"{c[0]}-{c[5]}")
def test_initialization_of_unobserved_components(masked, case):
    bt, kw = _family(case)
    D, N = bt.D, bt.N
    words = [mask_pool(D)[p % 3] for p in range(bt.B)]
    with _ev(bt, observed=[bits(w, D) for w in words], **kw) as ev, _ev(bt, **kw) as ev0:
        X, X0 = ev.initialization(), ev0.initialization()
    nA = N * D * D
    assert np.array_equal(X[:, :nA], X0[:, :nA])
    for p, w in enumerate(words):
        b, b0 = X[p, nA:].reshape(N, D), X0[p, nA:].reshape(N, D)
        seen = bits(w, D)
        hidden = [i for i in range(D) if i not in seen]
        assert np.array_equal(b[:, seen], b0[:, seen]), p
        ad = 0.5 * (bt.sigma[p, hidden] / 0.25)
        assert np.array_equal(b[:, hidden], np.broadcast_to(ad * bt.m0[p, hidden], (N, len(hidden)))), p
        assert grad_err(X[p], masked.initialization(bt.problem(p), w), N, D) < TOL, p


@pytest.mark.parametrize("model,cols", [("L63", [0, 2]), ("L96", list(range(1, 40, 3)))])
def test_standalone_likelihood_matches_the_oracle(masked, model, cols):
    from vgpa_b200.likelihood import GaussianLikelihood
    bt, _ = _family(FAMILIES[0] if model == "L63" else FAMILIES[3])
    D, N, M = bt.D, bt.N, bt.obs_t.size
    rng = np.random.default_rng(7)
    mt = rng.standard_normal((N, D))
    st = np.abs(rng.standard_normal((N, D, D))) + np.eye(D)
    Rsel = 0.5 + rng.random(len(cols))
    lik = GaussianLikelihood(bt.obs_y[0][:, cols], bt.obs_t, np.diag(Rsel), cols, single_dim=False)
    E = lik(mt, st)
    jm, js, dr = lik.gradients(mt, st)
    assert jm.shape == (N, D) and js.shape == (N, D, D) and dr.shape == (N, M, M)
    R = np.full(D, np.nan)                   # unobserved entries: never read
    R[cols] = Rsel
    prob = bt.problem(0)
    prob.R = R
    word = sum(1 << c for c in cols)
    Eo = masked.eobs(prob, word, mt, st)
    jmo, jso = masked.jumps(prob, word, mt)
    assert abs(E - Eo) <= TOL * abs(Eo)
    assert rel_err(jm, jmo) < TOL and rel_err(js, jso) < TOL
    hidden = [i for i in range(D) if i not in cols]
    assert not jm[:, hidden].any() and not js[:, hidden][:, :, hidden].any()


def _simulate(model, method, tf, operator, optimizer, max_it):
    from vgpa_b200 import Simulation
    params = mg.config(model, method, tf)
    params["Observations"]["operator"] = operator
    sim = Simulation("t")
    sim.setup(params)
    vg = sim.build()
    x_host, x_gpu = vg.initialization(), vg.initialization_gpu()
    vg.close()
    sim.run(max_it=max_it, display=False, optimizer=optimizer)
    return sim, x_host, x_gpu


@pytest.mark.parametrize("model,method,tf,operator,max_it", [
    ("L63", "rk2", 4.0, [0], 200),
    ("L96", "rk2", 1.0, list(range(0, 40, 2)), 60),
])
def test_simulation_with_the_json_operator(model, method, tf, operator, max_it, capsys):
    runs = {opt: _simulate(model, method, tf, operator, opt, max_it) for opt in ("host", "device")}
    capsys.readouterr()
    (h, xh, xg), (d, _, _) = runs["host"], runs["device"]
    D = h.m_data["model"].sample_path.shape[1]
    N = h.m_data["model"].sample_path.shape[0]
    assert grad_err(xg, xh, N, D) < TOL                     # host VarGP.initialization against the device rows
    fh, fd = np.asarray(h.scg_stats["fx"]), np.asarray(d.scg_stats["fx"])
    n = min(int(h.scg_stats["MaxIt"]), int(d.scg_stats["MaxIt"]))
    assert n > 5
    assert np.max(np.abs(fd[:n] - fh[:n]) / np.maximum(np.abs(fh[:n]), 1.0)) < 1e-6
    assert fh[n - 1] < fh[0] and np.isfinite(h.output["fx"])
    assert {"mt", "st", "lamt", "psit"} <= set(h.output)


def test_batched_scg_follows_a_host_scg_on_the_oracle(masked):
    """A masked L63 batch under BatchedSCG: problem 0's trace against the host SCG driven by the oracle."""
    from vgpa_b200.batched_scg import BatchedSCG
    from vgpa_b200.scg import SCG
    bt, _ = _family(FAMILIES[0])
    D = bt.D
    words = [mask_pool(D)[p % 3] for p in range(bt.B)]
    opts = {"max_it": 40, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    with _ev(bt, observed=[bits(w, D) for w in words]) as ev:
        opt = BatchedSCG(ev, opts)
        opt(bt.X)
        trace = opt.stats["fx"][:, 0].copy()
        n_dev = int(opt.stats["MaxIt"][0])
        del opt
    prob, w0 = bt.problem(0), words[0]
    host = SCG(lambda x: masked.eval(prob, w0, x, want_grad=False)[0], lambda x, **kw: masked.eval(prob, w0, x)[1], opts)
    host(bt.X[0].copy())
    ref = np.asarray(host.stats["fx"])
    n = min(n_dev, int(host.stats["MaxIt"]))
    assert n > 5
    assert np.max(np.abs(trace[:n] - ref[:n]) / np.maximum(np.abs(ref[:n]), 1.0)) < 1e-6
