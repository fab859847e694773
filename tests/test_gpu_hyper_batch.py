"""
Batched hyper-parameter gradients (vgpa_hyper_device, BatchEvaluator.hyper / hyper_device, ShardedBatchedSCG.run(hyper=True)):
dEsde/dtheta, dEsde/dSigma, Esde and F of every problem of a handle, on the device.

  - every kernel family of the F-only evaluation (the forward sweeps chosen by model, method, N and problems per pass)
    against the oracle at 1e-9, problem by problem, at the oracle's own m(t), S(t); the golden problems as rows of a
    batch against the unmodified reference (hyper_*.npz);
  - sum_i sigma_i dEsde/dSigma_ii = -Esde (Esde is homogeneous of degree -1 in Sigma), off-diagonals exactly 0;
  - dEsde/dtheta is dF/dtheta at fixed x for DW, OU and L63 (m, S, E0 and Eobs do not depend on theta): central
    differences of F between handles at theta +- h;
  - bits: F is what vgpa_eval_device returns; a problem's outputs do not depend on its batch position, its neighbours,
    the pass split, an installed active set or compacted list;
  - layouts: shared x, padded output rows, NULL outputs, sentinel-filled buffers with a guard row;
  - argument checks, a LinAlgError naming the problem, and the ensemble driver's new keys.
"""
from pathlib import Path

import numpy as np
import pytest

from conftest import rel_err
from test_gpu_layouts import _Batch, _alloc, _expect, _fill, _load, _not_pd_x, _rows, _sample_rows, _stream
from test_gpu_parity import evaluator_from_golden

ROOT = Path(__file__).resolve().parents[1]
TOL = 1e-9

# (model, method, N (None: the golden grid), B, problems per pass (0: one pass), kernel family of the forward sweep)
CASES = [
    ("OU", "rk4", 1001, 7, 0, "scan1-fwd"),
    ("OU", "rk2", 6000, 3, 0, "serial-fwd"),
    ("OU", "rk2", 201, 8193, 0, "staged-fwd"),
    ("DW", "euler", 101, 16385, 0, "staged-fwd"),
    ("DW", "rk4", None, 9, 4, "scan1-fwd-passes"),
    ("L63", "rk2", 61, 7, 0, "lanes-fwd"),
    ("L63", "euler", 61, 11, 3, "lanes-passes"),
    ("L63", "heun", 30, 8193, 0, "staged-fwd"),
    ("L96", "rk2", 101, 5, 0, "small-launch"),
    ("L96", "rk4", 21, 1800, 900, "full-wave-ragged"),
]
IDS = [f"{c[0]}-{c[1]}-N{c[2] or 1001}-B{c[3]}-{c[5]}" for c in CASES]


def _nsig(D):
    return 1 if D == 1 else D * D


class _Out:
    """Sentinel-filled device buffers for the four outputs of B problems (row strides nth + pad, nsig + pad)."""

    def __init__(self, ev, pad=0):
        self.B, self.nth, self.ns = ev.B, ev.n_theta, _nsig(ev.D)
        self.ts, self.ss = self.nth + pad, self.ns + pad
        self.F, self.E = _alloc(self.B, 1, 1), _alloc(self.B, 1, 1)
        self.th, self.sg = _alloc(self.B, self.nth, self.ts), _alloc(self.B, self.ns, self.ss)

    def run(self, ev, x, xs, want=("F", "E", "th", "sg")):
        p = {k: (getattr(self, k).data_ptr() if k in want else None) for k in ("F", "E", "th", "sg")}
        ev.hyper_device(x.data_ptr(), xs, p["F"], p["E"], p["th"], self.ts, p["sg"], self.ss, _stream())
        ev.sync()
        return self

    def host(self):
        import torch
        f = lambda buf, n, s: _rows(buf, self.B, n, s).contiguous().view(torch.float64).cpu().numpy()
        return f(self.F, 1, 1)[:, 0], f(self.E, 1, 1)[:, 0], f(self.th, self.nth, self.ts), f(self.sg, self.ns, self.ss)

    def bits(self):
        return [b.cpu().numpy() for b in (self.F, self.E, self.th, self.sg)]


def _hyper(ev, X):
    """Compact hyper outputs of ev at X ((B, n) CUDA tensor) as host arrays F, Esde, dth (B, nth), dsig (B, nsig)."""
    return _Out(ev).run(ev, _fill(X, ev.B, ev.n_x, ev.n_x).view(X.dtype), ev.n_x).host()


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _check_oracle(oracle, bt, rows, F, Esde, dth, dsig):
    D = bt.D
    for i in rows:
        prob = bt.problem(i)
        full = oracle.eval(prob, bt.X[i], want_grad=False, full=True)
        o_th, o_sig = oracle.energy_hyper(prob, bt.X[i], full["mt"], full["st"])
        assert abs(F[i] - full["F"]) <= TOL * abs(full["F"]), i
        assert abs(Esde[i] - full["Esde"]) <= TOL * abs(full["Esde"]), i
        assert rel_err(dth[i], np.atleast_1d(o_th)) < TOL, i
        assert rel_err(dsig[i], np.atleast_1d(o_sig).ravel()) < TOL, i
        assert D == 1 or dsig[i].size == D * D


def _check_identity(bt, Esde, dsig):
    """sum_i sigma_i dEsde/dSigma_ii = -Esde; for D > 1 the off-diagonal entries are exactly +0.0."""
    D = bt.D
    for i in range(bt.B):
        diag = dsig[i] if D == 1 else dsig[i].reshape(D, D).diagonal()
        s = float(np.dot(bt.sigma[i], diag))
        assert abs(s + Esde[i]) <= 1e-12 * abs(Esde[i]), i
    if D > 1:
        off = dsig.reshape(bt.B, D, D)[:, ~np.eye(D, dtype=bool)]
        assert not _bits(off).any()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_every_forward_family_against_oracle(oracle, case):
    import torch
    model, method, N, B, per_pass, _ = case
    bt = _Batch(model, method, N, B, seed=5)
    n = bt.n_x
    kw = dict(scratch_bytes=per_pass * bt.per_problem_bytes() + 64) if per_pass else {}
    X = torch.from_numpy(bt.X).cuda()
    with bt.evaluator(**kw) as ev:
        if per_pass:
            assert ev.chunk_size < B
        chunk = ev.chunk_size
        F, Esde, dth, dsig = _hyper(ev, X)
        # F: the bits of the F-only evaluation of the same x
        Fe = torch.empty(B, dtype=torch.float64, device="cuda")
        ev.eval_device(X.data_ptr(), n, Fe.data_ptr(), None, None, _stream())
        ev.sync()
        assert np.array_equal(_bits(F), _bits(Fe.cpu().numpy()))
    rows = _sample_rows(B, chunk)
    _check_oracle(oracle, bt, rows, F, Esde, dth, dsig)
    _check_identity(bt, Esde, dsig)

    # the same problems in reverse order (other positions, other neighbours, the same kernel family) and, where the
    # case has passes, another pass split: the same bits problem by problem
    rev = np.arange(B)[::-1].copy()
    splits = [kw] + ([dict(scratch_bytes=(per_pass // 2 + 1) * bt.per_problem_bytes() + 64)] if per_pass else [])
    for kw2 in splits:
        with bt.evaluator(rev, **kw2) as ev2:
            if kw2 is not kw:
                assert ev2.chunk_size not in (chunk, B)
            got = _hyper(ev2, torch.from_numpy(bt.X[rev]).cuda())
        for a, b in zip((F, Esde, dth, dsig), got):
            assert np.array_equal(_bits(a), _bits(b[::-1]))


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["DW", "OU", "L63", "L96"])
def test_golden_row_inside_a_batch_matches_reference(model):
    """The golden eval_<model>_rk2 problem as row 1 of a batch of 3 whose other rows have other x."""
    import torch
    g = np.load(ROOT / "tests" / "golden" / f"eval_{model}_rk2.npz")
    h = np.load(ROOT / "tests" / "golden" / f"hyper_{model}.npz")
    rng = np.random.default_rng(2)
    X = np.stack([g["x"] * (1.0 + 0.01 * rng.standard_normal(g["x"].size)), g["x"], g["x"] * 1.01])
    with evaluator_from_golden(g, B=3) as ev:
        out = ev.hyper(torch.from_numpy(X).cuda())
        out_host = ev.hyper(X)
    for k in out:
        assert np.array_equal(_bits(out[k]), _bits(out_host[k])), k
    assert abs(out["F"][1] - float(g["F"])) <= TOL * abs(float(g["F"]))
    assert abs(out["Esde"][1] - float(g["Esde"])) <= TOL * abs(float(g["Esde"]))
    assert rel_err(out["dEsde_dtheta"][1], h["dEsde_dtheta"]) < TOL
    assert rel_err(out["dEsde_dsigma"][1], h["dEsde_dsigma"]) < TOL
    D = int(g["D"])
    if D == 1:
        assert out["dEsde_dtheta"].shape == (3,) and out["dEsde_dsigma"].shape == (3,)
    else:
        assert out["dEsde_dtheta"].shape == (3, h["dEsde_dtheta"].size) and out["dEsde_dsigma"].shape == (3, D, D)


@pytest.mark.gpu
@pytest.mark.parametrize("model,method,N", [("DW", "heun", 1001), ("OU", "rk4", 1001), ("L63", "rk2", 61)])
def test_dtheta_is_dF_dtheta(model, method, N):
    """Central differences of F between two handles at theta +- h e_k, problem by problem, to relative 1e-6."""
    import torch
    bt = _Batch(model, method, N, 4, seed=8)
    X = torch.from_numpy(bt.X).cuda()
    with bt.evaluator() as ev:
        _, _, dth, _ = _hyper(ev, X)
    theta0 = bt.theta.copy()
    for k in range(theta0.shape[1]):
        hk = 1e-5 * np.maximum(1.0, np.abs(theta0[:, k]))
        Fs = []
        for sgn in (1.0, -1.0):
            bt.theta = theta0.copy()
            bt.theta[:, k] += sgn * hk
            with bt.evaluator() as evh:
                Fs.append(evh.eval(bt.X, want_grad=False)[0])
        bt.theta = theta0
        fd = (Fs[0] - Fs[1]) / (2.0 * hk)
        assert np.all(np.abs(dth[:, k] - fd) <= 1e-6 * np.abs(fd)), (k, dth[:, k], fd)


@pytest.mark.gpu
@pytest.mark.parametrize("model,method,N,B", [("OU", "rk4", 1001, 7), ("L63", "rk2", 61, 7), ("L96", "rk2", 41, 6)])
def test_layouts_masks_and_null_outputs(model, method, N, B):
    import torch
    bt = _Batch(model, method, N, B, seed=3)
    n = bt.n_x
    X = torch.from_numpy(bt.X).cuda()
    with bt.evaluator() as ev:
        ref = _Out(ev).run(ev, _fill(X, B, n, n).view(torch.float64), n)
        F0 = _rows(ref.F, B, 1, 1).clone()
        # padded x and padded output rows: the same bits in the rows, sentinels everywhere else
        xb = _fill(X, B, n, n + 4)
        x_before = xb.clone()
        pad = _Out(ev, pad=3).run(ev, xb.view(torch.float64), n + 4)
        assert torch.equal(xb, x_before)
        shapes = (("F", 1, 1, 1), ("E", 1, 1, 1), ("th", ref.nth, ref.nth, pad.ts), ("sg", ref.ns, ref.ns, pad.ss))
        for k, w, s0, s in shapes:
            assert torch.equal(getattr(pad, k), _expect(_rows(getattr(ref, k), B, w, s0), B, w, s)), k
        # NULL outputs: the others as before, the buffers not passed untouched
        for want in (("th",), ("F", "sg"), ("E",)):
            part = _Out(ev, pad=3).run(ev, xb.view(torch.float64), n + 4, want)
            for k, w, s0, s in shapes:
                exp = _expect(_rows(getattr(ref, k), B, w, s0), B, w, s) if k in want else _alloc(B, w, s)
                assert torch.equal(getattr(part, k), exp), (want, k)
        # one x shared by every problem: the compact call at the broadcast x
        j = B // 2
        Xj = X[j:j + 1]
        bc = _Out(ev).run(ev, _fill(Xj.expand(B, n).contiguous(), B, n, n).view(torch.float64), n)
        sh = _Out(ev).run(ev, _fill(Xj, B, n, 0).view(torch.float64), 0)
        assert all(np.array_equal(a, b) for a, b in zip(bc.bits(), sh.bits()))
        # an active set / compacted list: every problem is still served, and it stays installed for eval_device
        rng = np.random.default_rng(1)
        if model == "L96":
            lst = rng.permutation(B)[:B // 2]
            ev.set_active_list(lst)
            on = np.zeros(B, dtype=bool)
            on[lst] = True
        else:
            on = rng.random(B) < 0.5
            on[0], on[-1] = True, False
            flags = torch.from_numpy(on.astype(np.int32)).cuda()
            ev.set_active(flags.data_ptr())
        masked = _Out(ev).run(ev, _fill(X, B, n, n).view(torch.float64), n)
        assert all(np.array_equal(a, b) for a, b in zip(masked.bits(), ref.bits()))
        Fm = _alloc(B, 1, 1)
        ev.eval_device(X.data_ptr(), n, Fm.data_ptr(), None, None, _stream())
        ev.sync()
        assert torch.equal(Fm, _expect(F0, B, 1, 1, torch.from_numpy(on).cuda()))
        ev.set_active(None)
        ev.set_active_list(None)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["eval_DW_rk4", "eval_L63_heun", "eval_L96_rk2"])
def test_argument_checks(name):
    import torch
    g = _load(name)
    B = 2
    rng = np.random.default_rng(12)
    X = np.stack([g["x"] * (1.0 + 0.01 * rng.standard_normal(g["x"].size)) for _ in range(B)])
    with evaluator_from_golden(g, B=B) as ev:
        n, nth, ns = ev.n_x, ev.n_theta, _nsig(ev.D)
        ref = ev.hyper(X)
        Xd = _fill(torch.from_numpy(X).cuda(), B, n, n + 2)
        out = _Out(ev)
        x, th, sg = Xd.data_ptr(), out.th.data_ptr(), out.sg.data_ptr()
        bad = [(x, n + 1, nth, ns),            # odd x stride
               (x + 8, n + 2, nth, ns),        # x rows 8 bytes off the 16-byte alignment
               (x, n - 2, nth, ns),            # 0 < x stride < n_x
               (x, n + 2, nth - 1 if nth > 1 else 0, ns),   # dtheta stride below one row with B > 1
               (x, n + 2, nth, ns - 1 if ns > 1 else 0)]    # dsigma stride below one row with B > 1
        for xp, xs, ts, ss in bad:
            with pytest.raises(ValueError):
                ev.hyper_device(xp, xs, None, None, th, ts, sg, ss, _stream())
            assert np.array_equal(ev.hyper(X)["dEsde_dtheta"], ref["dEsde_dtheta"])   # the handle still works
    with evaluator_from_golden(g, B=1) as ev1:             # one problem: output strides of 0 are accepted
        ref1 = ev1.hyper(X[0])
        x1 = torch.from_numpy(X[:1]).cuda()
        o = _Out(ev1)
        ev1.hyper_device(x1.data_ptr(), n, None, None, o.th.data_ptr(), 0, o.sg.data_ptr(), 0, _stream())
        ev1.sync()
        _, _, th1, sg1 = o.host()
        assert np.array_equal(th1.ravel(), np.ravel(ref1["dEsde_dtheta"]))
        assert np.array_equal(sg1.ravel(), np.ravel(ref1["dEsde_dsigma"]))


@pytest.mark.gpu
def test_not_positive_definite_names_the_problem():
    g = _load("eval_L96_euler")
    N, D, B = int(g["N"]), int(g["D"]), 6
    X = np.stack([g["x"]] * B)
    X[3] = _not_pd_x(g)
    good = np.stack([g["x"]] * B)
    with evaluator_from_golden(g, B=B, scratch_bytes=2 * 8 * N * (2 * D + 2 * D * D + 1) + 64) as ev:
        assert ev.chunk_size == 2
        with pytest.raises(np.linalg.LinAlgError, match=r"problem 3 at"):
            ev.hyper(X)
        ev.set_active_list([5, 3, 0])                      # problem 3 at list position 1: the call serves every problem
        with pytest.raises(np.linalg.LinAlgError, match=r"problem 3 at"):
            ev.hyper(X)
        ev.set_active_list(None)
        out = ev.hyper(good)
        assert np.all(np.abs(out["F"] - float(g["F"])) <= TOL * abs(float(g["F"])))
        assert np.all(np.abs(out["Esde"] - float(g["Esde"])) <= TOL * abs(float(g["Esde"])))


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("eval_L63_heun", 5), ("eval_L96_euler", 3)])
def test_ensemble_driver_returns_and_saves_hyper_keys(tmp_path, name, B):
    from oracle import prior_kl0
    from vgpa_b200.batched_scg import ShardedBatchedSCG
    from vgpa_b200.engine import BatchEvaluator
    from vgpa_b200.simulation import load
    g = _load(name)
    model, method = str(g["model"]), str(g["method"])
    D, N = int(g["D"]), int(g["N"])
    rng = np.random.default_rng([4, D])
    obs_y = np.stack([g["obs_y"] + 0.05 * rng.standard_normal(g["obs_y"].shape) for _ in range(B)])
    E0 = float(prior_kl0(g["m0"], g["s0"], g["mu0"], g["tau0"], False))
    common = dict(model=model, method=method, N=N, dt=float(g["dt"]), theta=g["theta"], sigma=g["sigma"], R=g["R"],
                  obs_t=g["obs_t"], m0=g["m0"], s0=g["s0"], E0=E0, dt_model=float(g["dt"]))
    opts = {"max_it": 4, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
    make = lambda lo, hi: BatchEvaluator(obs_y=obs_y[lo:hi], B=hi - lo, **common)
    ens = ShardedBatchedSCG(B, make, opts)
    plain = ens.run(keep=range(B))
    assert not {"Esde", "dEsde_dtheta", "dEsde_dsigma_diag"} & set(plain)
    res = ens.run(keep=range(B), hyper=True)
    assert np.array_equal(res["fx"], plain["fx"])
    Xk = np.stack([res["kept"][k] for k in range(B)])
    with make(0, B) as ev:
        ref = ev.hyper(Xk)
    assert res["Esde"].shape == (B,) and res["dEsde_dtheta"].shape == (B, ev.n_theta)
    assert res["dEsde_dsigma_diag"].shape == (B, D)
    assert np.array_equal(_bits(res["Esde"]), _bits(ref["Esde"]))
    assert np.array_equal(_bits(res["dEsde_dtheta"]), _bits(ref["dEsde_dtheta"]))
    assert np.array_equal(_bits(res["dEsde_dsigma_diag"]), _bits(np.stack([np.diag(s) for s in ref["dEsde_dsigma"]])))
    z = load(ens.save(str(tmp_path / "ens"), N, D))
    for k in ("Esde", "dEsde_dtheta", "dEsde_dsigma_diag"):
        assert np.array_equal(z[k], res[k]), k


def test_library_exports_and_header_declares_hyper_device():
    """CPU: the built library exports vgpa_hyper_device and the public header declares it."""
    import ctypes
    from vgpa_b200._lib import LIB_PATH
    assert hasattr(ctypes.CDLL(str(LIB_PATH)), "vgpa_hyper_device")
    header = (ROOT / "include" / "vgpa_b200.h").read_text()
    assert "int vgpa_hyper_device(vgpa_handle *h, const double *d_x, int64_t x_stride, double *d_F," in header
