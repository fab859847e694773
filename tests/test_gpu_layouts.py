"""
Row layouts of the device entry points.  The rest of the suite hands the kernels rows exactly n_x apart, so a kernel
that confuses the x stride, the gradient stride and n_x passes it.  Here every kernel family (the launchers choose one
by model, method, N and the problems per pass) runs with padded, shared (stride 0) and masked rows:

  - every F and gradient row must equal, bit for bit, the row of the same problem from the compact evaluation
    (dispatch depends on the problem count, N and the method, never on a stride);
  - padding, guard rows after the last row, rows of skipped problems and the gradient buffer of F-only calls
    keep a sentinel NaN bit pattern (compared as int64);
  - sampled rows of the compact evaluation match the oracle at 1e-9.

Every buffer holds at least B rows at max(stride, n_x) plus a guard row, so a kernel using a wrong stride reads
sentinels or writes inside the buffer: a layout error shows up as data, never as an access outside an allocation.
Also here: the host entry point with strided buffers, initialisation into strided rows, the argument checks of the
device entry point, the problem named by a LinAlgError, and the SCG vector kernels against exact arithmetic.
"""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import golden_eval_files, grad_err
from oracle import Problem, prior_kl0
from test_gpu_edge import _x_prefix
from test_gpu_parity import evaluator_from_golden

pytestmark = pytest.mark.gpu
TOL = 1e-9
SENT = 0x7FF40BADF00D0001          # a signalling-NaN payload: any kernel that reads it as a value changes its bits
GUARD = 1                          # rows after the last one


def _load(name):
    return np.load(str(next(p for p in golden_eval_files() if name in p)))


def _lib():
    from vgpa_b200._lib import lib, raise_for
    return lib, raise_for


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _sentinel(n):
    import torch
    return torch.full((int(n),), SENT, dtype=torch.int64, device="cuda")


def _alloc(B, n, stride):
    """A sentinel-filled int64 device buffer for B rows of n values `stride` apart (stride 0: one shared row),
    sized for B rows at max(stride, n) plus the guard rows whatever the stride."""
    return _sentinel((B + GUARD) * max(stride, n))


def _rows(buf, B, n, stride):
    """The (B, n) rows of a buffer (stride 0: the one shared row, (1, n))."""
    if stride == 0:
        return buf[:n].view(1, n)
    return buf[:B * stride].view(B, stride)[:, :n]


def _fill(X, B, n, stride):
    """X (B, n) or (1, n) float64 device tensor into a fresh sentinel buffer laid out with `stride`."""
    import torch
    buf = _alloc(B, n, stride)
    _rows(buf, B, n, stride).copy_(X.view(torch.int64)[:1] if stride == 0 else X.view(torch.int64))
    return buf


def _expect(ref, B, n, stride, which=None):
    """The buffer a layout should leave: rows `which` (all when None) of ref (B, n) int64, sentinel elsewhere."""
    buf = _alloc(B, n, stride)
    v = _rows(buf, B, n, stride)
    if which is None:
        v.copy_(ref)
    else:
        v[which] = ref[which]
    return buf


def _eval_device(ev, x, xs, F, g, gs, want_grad):
    """vgpa_eval_device, the gradient buffer passed even when want_grad == 0 (it must stay untouched then)."""
    lib, raise_for = _lib()
    raise_for(lib.vgpa_eval_device(ev._h, x.data_ptr(), xs, int(want_grad), F.data_ptr(), g.data_ptr(), gs,
                                   _stream()), ev._h)
    ev.sync()


def _x_at(g, N):
    """An evaluation point on a grid of N points: the golden x cut to N points, or repeated in time beyond its own."""
    N0, D = int(g["N"]), int(g["D"])
    if N <= N0:
        return _x_prefix(g, N)
    x = g["x"]
    A = np.resize(x[:N0 * D * D].reshape(N0, -1), (N, D * D))
    b = np.resize(x[N0 * D * D:].reshape(N0, -1), (N, D))
    return np.concatenate([A.ravel(), b.ravel()])


class _Batch:
    """B problems of one shape that differ in theta, sigma, R, obs_y, m0, s0, E0 and x (seeded)."""

    def __init__(self, model, method, N, B, seed=0):
        g = _load(f"eval_{model}_{method}")
        D = int(g["D"])
        N = int(g["N"]) if N is None else int(N)
        rng = np.random.default_rng([seed, B, N, D])
        u = np.linspace(0.0, 1.0, B)[:, None]
        self.g, self.model, self.method, self.D, self.N, self.B = g, model, method, D, N, B
        self.obs_t = g["obs_t"][g["obs_t"] < N - 1]
        M = self.obs_t.size
        self.theta = np.atleast_2d(g["theta"]) * (1.0 + 0.02 * u)
        self.sigma = np.atleast_2d(g["sigma"]) * (0.7 + 0.6 * u)
        self.R = np.atleast_2d(g["R"]) * (0.8 + 0.4 * u)
        self.obs_y = g["obs_y"][:M].reshape(1, M, D) + 0.1 * rng.standard_normal((B, M, D))
        self.m0 = np.atleast_2d(g["m0"]).reshape(1, D) + 0.05 * rng.standard_normal((B, D))
        self.s0 = np.asarray(g["s0"], dtype=float).reshape(1, D * D) * (1.0 + 0.3 * u)
        E0 = float(prior_kl0(g["m0"], g["s0"], g["mu0"], g["tau0"], D == 1))
        self.E0 = E0 + 0.01 * u.ravel()
        x = _x_at(g, N)
        self.X = x * (1.0 + 0.01 * rng.standard_normal((B, x.size)))
        self.n_x = x.size

    def evaluator(self, idx=None, **kw):
        idx = np.arange(self.B) if idx is None else np.asarray(idx)
        return evaluator_from_golden(self.g, B=idx.size, N=self.N, obs_t=self.obs_t, theta=self.theta[idx],
                                     sigma=self.sigma[idx], R=self.R[idx], obs_y=self.obs_y[idx], m0=self.m0[idx],
                                     s0=self.s0[idx], E0=self.E0[idx], **kw)

    def problem(self, i):
        D = self.D
        return Problem(model=self.model, method=self.method, D=D, N=self.N, dt=float(self.g["dt"]),
                       theta=self.theta[i], sigma=self.sigma[i], R=self.R[i], obs_t=self.obs_t, obs_y=self.obs_y[i],
                       m0=self.m0[i], s0=self.s0[i].reshape(D, D) if D > 1 else self.s0[i], E0=float(self.E0[i]),
                       dt_model=Problem.from_golden(self.g).dt_model)

    def per_problem_bytes(self):
        D = self.D
        return 8 * self.N * (2 * D + 2 * D * D + 1)


# (model, method, N (None: the golden grid), B, gradient, problems per pass (0: one pass), kernel family)
CASES = [
    ("OU", "rk4", 1001, 7, True, 0, "scan1-fused"),
    ("OU", "rk4", 1001, 7, False, 0, "scan1-fwd-energy-finalize"),
    ("DW", "heun", 4000, 5, True, 0, "scan1-fwd-scan1-bwd"),
    ("OU", "euler", 5000, 3, True, 0, "scan1-fwd-serial-bwd"),
    ("OU", "rk2", 6000, 3, True, 0, "serial-fwd-serial-bwd"),
    ("OU", "rk2", 201, 8193, True, 0, "staged-fwd-scan1-bwd"),
    ("DW", "euler", 101, 16385, False, 0, "staged-fwd-F-only"),
    ("DW", "rk4", None, 9, True, 4, "scan1-fused-passes"),
    ("L63", "rk2", 61, 7, True, 0, "lanes-fwd-bwd"),
    ("L63", "rk4", 61, 7, False, 0, "lanes-fwd"),
    ("L63", "heun", 30, 8193, True, 0, "staged-fwd-serial-bwd"),
    ("L63", "euler", 61, 11, True, 3, "lanes-passes"),
    ("L96", "rk2", 101, 5, True, 0, "small-launch"),
    ("L96", "rk4", 21, 1800, True, 900, "full-wave-ragged"),
]


def _sample_rows(B, chunk):
    """First and last problem, both sides of the first warp boundary and of every pass boundary, one interior row."""
    rows = {0, 31, 32, B - 1, (B * 5) // 8}
    for p0 in range(chunk, B, chunk):
        rows |= {p0 - 1, p0}
    return sorted(r for r in rows if 0 <= r < B)


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-{c[1]}-N{c[2] or 1001}-B{c[3]}-{c[6]}")
def test_layouts_of_every_kernel_family(oracle, case):
    import torch
    model, method, N, B, want_grad, per_pass, _ = case
    bt = _Batch(model, method, N, B, seed=1)
    n = bt.n_x
    kw = dict(scratch_bytes=per_pass * bt.per_problem_bytes() + 64) if per_pass else {}
    X = torch.from_numpy(bt.X).cuda()
    rng = np.random.default_rng(3)
    with bt.evaluator(**kw) as ev:
        assert ev.n_x == n
        if per_pass:
            assert ev.chunk_size < B
        chunk = ev.chunk_size

        def run(Xt, xs, gs):
            xb = _fill(Xt, B, n, xs)
            x_before = xb.clone()
            Fb, gb = _alloc(B, 1, 1), _alloc(B, n, gs)
            _eval_device(ev, xb.view(torch.float64), xs, Fb.view(torch.float64), gb.view(torch.float64), gs,
                         want_grad)
            assert torch.equal(xb, x_before)                 # x is read only
            return Fb, gb

        def check(Fb, gb, F_ref, G_ref, gs, which=None):
            assert torch.equal(Fb, _expect(F_ref, B, 1, 1, which))
            if want_grad:
                assert torch.equal(gb, _expect(G_ref, B, n, gs, which))
            else:                                           # F only: the gradient buffer is not touched
                assert torch.equal(gb, _alloc(B, n, gs))

        # V0 compact: the reference of the other layouts
        F0b, G0b = run(X, n, n)
        F0, G0 = _rows(F0b, B, 1, 1).clone(), _rows(G0b, B, n, n).clone()
        check(F0b, G0b, F0, G0, n)
        F0h = F0.view(torch.float64).cpu().numpy().ravel()
        rows = _sample_rows(B, chunk)
        G0s = G0[rows].view(torch.float64).cpu().numpy() if want_grad else None
        F_o, G_o = oracle.eval_batch([bt.problem(i) for i in rows], bt.X[rows], want_grad=want_grad)
        for k, i in enumerate(rows):
            assert abs(F0h[i] - F_o[k]) <= TOL * abs(F_o[k]), i
            if want_grad:
                assert grad_err(G0s[k], G_o[k], bt.N, bt.D) < TOL, i

        # V1 padded rows, different paddings for x and the gradient
        xs, gs = n + 4, n + 2
        check(*run(X, xs, gs), F0, G0, gs)

        # V2 one x shared by every problem: the compact evaluation of the broadcast x
        j = B // 2
        Xj = X[j:j + 1]
        Fbc, Gbc = run(Xj.expand(B, n).contiguous(), n, n)
        check(*run(Xj, 0, gs), _rows(Fbc, B, 1, 1), _rows(Gbc, B, n, n), gs)
        del Fbc, Gbc

        # V3 masked problems, padded rows
        if model == "L96":
            lst = rng.permutation(B)[:max(2, (2 * B) // 3)]          # unsorted; several passes when chunked
            assert per_pass == 0 or lst.size > chunk
            ev.set_active_list(lst)
            on = np.zeros(B, dtype=bool)
            on[lst] = True
        else:
            on = rng.random(B) < 0.6
            on[0], on[-1] = True, False
            flags = torch.from_numpy(on.astype(np.int32)).cuda()
            ev.set_active(flags.data_ptr())
        Fm, Gm = run(X, xs, gs)
        if model == "L96":
            ev.set_active_list(None)
        else:
            ev.set_active(None)
        check(Fm, Gm, F0, G0, gs, which=torch.from_numpy(on).cuda())

        if model == "L96" and B > 148:
            # the sampled rows again in handles of 5 problems: launches of 5 CTAs (small_launch in the sweeps)
            for k in range(0, len(rows), 5):
                idx = rows[k:k + 5]
                with bt.evaluator(idx) as ev5:
                    F5, G5 = ev5.eval(bt.X[idx])
                assert np.array_equal(F5.view(np.int64), F0[idx].cpu().numpy().ravel())
                assert np.array_equal(G5.view(np.int64), G0[idx].cpu().numpy())


@pytest.mark.parametrize("name", ["eval_DW_heun", "eval_OU_rk2", "eval_L63_rk4", "eval_L96_euler"])
def test_shared_constants_equal_repeated_rows(name):
    """Each per-problem constant given as B identical rows (stride = its length) or once (stride 0)."""
    g = _load(name)
    B = 3
    rng = np.random.default_rng(4)
    X = np.stack([g["x"] * (1.0 + 0.01 * rng.standard_normal(g["x"].size)) for _ in range(B)])
    rep = {k: np.stack([np.asarray(g[k], dtype=float)] * B) for k in ("theta", "sigma", "R", "obs_y", "m0", "s0")}
    D = int(g["D"])
    E0 = float(prior_kl0(g["m0"], g["s0"], g["mu0"], g["tau0"], D == 1))
    with evaluator_from_golden(g, B=B) as ev_s, evaluator_from_golden(g, B=B, E0=np.full(B, E0), **rep) as ev_r:
        F_s, G_s = ev_s.eval(X)
        F_r, G_r = ev_r.eval(X)
    assert np.array_equal(F_s, F_r) and np.array_equal(G_s, G_r)


def _host_rows(B, n, stride):
    """A sentinel-filled host buffer of B rows `stride` apart (plus a guard row) and its float64 view."""
    buf = np.full((B + GUARD) * max(stride, n), SENT, dtype=np.int64)
    return buf, buf.view(np.float64)


def _host_eval_strided(ev, X, xs, gs):
    lib, raise_for = _lib()
    B, n = ev.B, ev.n_x
    xb, xf = _host_rows(B, n, xs)
    if xs == 0:
        xf[:n] = X[0]
    else:
        xf[:B * xs].reshape(B, xs)[:, :n] = X
    x_before = xb.copy()
    Fb, Ff = _host_rows(B, 1, 1)
    gb, gf = _host_rows(B, n, gs)
    raise_for(lib.vgpa_eval(ev._h, xf.ctypes.data, xs, 1, Ff.ctypes.data, gf.ctypes.data, gs), ev._h)
    assert np.array_equal(xb, x_before)
    return Fb, gb


def _host_expect(ref, B, n, stride):
    buf, f = _host_rows(B, n, stride)
    if stride == 0:
        f[:n] = ref[0]
    else:
        f[:B * stride].reshape(B, stride)[:, :n] = ref
    return buf


@pytest.mark.parametrize("name,B,per_pass,xs_pad,gs_pad", [
    ("eval_L96_rk2", 70, 0, 2, 4),          # host passes of 64 + 6: both staging slots, 2-D copies both ways
    ("eval_L63_heun", 9, 4, 4, 2),          # passes of 4 problems
    ("eval_OU_rk4", 1, 0, 2, 2),            # one problem: the gradient row is one plain copy
    ("eval_L96_rk4", 70, 0, None, 4),       # one x shared by every problem, padded gradient rows
], ids=["L96-B70", "L63-passes", "OU-B1", "L96-shared-x"])
def test_host_entry_point_with_strided_buffers(name, B, per_pass, xs_pad, gs_pad):
    g = _load(name)
    rng = np.random.default_rng(6)
    X = np.stack([g["x"] * (1.0 + 0.01 * rng.standard_normal(g["x"].size)) for _ in range(B)])
    D, N = int(g["D"]), int(g["N"])
    kw = dict(scratch_bytes=per_pass * 8 * N * (2 * D + 2 * D * D + 1) + 64) if per_pass else {}
    with evaluator_from_golden(g, B=B, **kw) as ev:
        if per_pass:
            assert ev.chunk_size < B
        n = ev.n_x
        if xs_pad is None:
            X = X[:1]
            F_ref, G_ref = ev.eval(X[0])
        else:
            F_ref, G_ref = ev.eval(X)
        xs = 0 if xs_pad is None else n + xs_pad
        Fb, gb = _host_eval_strided(ev, X, xs, n + gs_pad)
    assert np.array_equal(Fb, _host_expect(F_ref[:, None], B, 1, 1))
    assert np.array_equal(gb, _host_expect(G_ref, B, n, n + gs_pad))


@pytest.mark.parametrize("name,pad", [("eval_OU_heun", 2), ("eval_L63_rk2", 4), ("eval_L96_rk4", 6)])
def test_initialization_into_strided_rows(name, pad):
    import torch
    lib, raise_for = _lib()
    g = _load(name)
    B = 3
    rng = np.random.default_rng(7)
    obs = np.stack([g["obs_y"] + 0.2 * rng.standard_normal(g["obs_y"].shape) for _ in range(B)])
    with evaluator_from_golden(g, B=B, obs_y=obs) as ev:
        n = ev.n_x
        xs = n + pad
        ref = ev.initialization(0.0)
        assert not np.array_equal(ref[0], ref[1])
        # device rows
        buf = _alloc(B, n, xs)
        ev.initialization_device(buf.data_ptr(), xs, 0.0, _stream())
        torch.cuda.synchronize()
        exp = _expect(torch.from_numpy(ref).cuda().view(torch.int64), B, n, xs)
        assert torch.equal(buf, exp)
        # host rows
        hb, hf = _host_rows(B, n, xs)
        raise_for(lib.vgpa_initialization_host(ev._h, 0.0, hf.ctypes.data_as(C.POINTER(C.c_double)), xs), ev._h)
    assert np.array_equal(hb, _host_expect(ref, B, n, xs))


@pytest.mark.parametrize("name", ["eval_DW_rk4", "eval_OU_euler", "eval_L63_heun", "eval_L96_rk2"])
def test_device_entry_point_argument_contract(name):
    import torch
    lib, raise_for = _lib()
    g = _load(name)
    B = 2
    rng = np.random.default_rng(12)
    X = np.stack([g["x"] * (1.0 + 0.01 * rng.standard_normal(g["x"].size)) for _ in range(B)])
    with evaluator_from_golden(g, B=B) as ev:
        n = ev.n_x
        F_ref, G_ref = ev.eval(X)
        Xd = _fill(torch.from_numpy(X).cuda(), B, n, n + 2)
        F = _alloc(B, 1, 1)
        G = _alloc(B, n, n + 2)
        x, f, gp = Xd.data_ptr(), F.data_ptr(), G.data_ptr()
        bad = [(x, n + 1, gp, n),            # odd x stride
               (x, n, gp, n + 1),            # odd gradient stride
               (x, n, gp + 8, n),            # gradient rows 8 bytes off the 16-byte alignment
               (x, n - 2, gp, n),            # 0 < x stride < n_x
               (x, n, gp, n - 2)]            # gradient stride < n_x with B > 1
        for xp, xs, gptr, gs in bad:
            with pytest.raises(ValueError):
                ev.eval_device(xp, xs, f, gptr, gs, _stream())
            ev.eval_device(x, n + 2, f, gp, n + 2, _stream())    # the handle still evaluates correctly
            ev.sync()
            assert np.array_equal(_rows(F, B, 1, 1).view(torch.float64).cpu().numpy().ravel(), F_ref)
            assert np.array_equal(_rows(G, B, n, n + 2).view(torch.float64).cpu().numpy(), G_ref)
        xh = np.zeros((B, n + 2))
        Fh, Gh = np.zeros(B), np.zeros((B, n))
        rc = lib.vgpa_eval(ev._h, xh.ctypes.data, n - 2, 1, Fh.ctypes.data, Gh.ctypes.data, n)
        with pytest.raises(ValueError):
            raise_for(rc, ev._h)
        assert np.array_equal(ev.eval(X)[0], F_ref)
    # one problem: its gradient row needs no stride
    with evaluator_from_golden(g, B=1) as ev1:
        F1, G1 = ev1.eval(X[0])
        x1 = _fill(torch.from_numpy(X[:1]).cuda(), 1, n, n)
        F = _alloc(1, 1, 1)
        G = _alloc(1, n, n)
        ev1.eval_device(x1.data_ptr(), n, F.data_ptr(), G.data_ptr(), 0, _stream())
        ev1.sync()
        assert torch.equal(G, _expect(torch.from_numpy(G1).cuda().view(torch.int64), 1, n, n))
        assert F[0].item() == int(F1.view(np.int64)[0])


def _not_pd_x(g):
    """The x of test_not_positive_definite_is_linalg_error: S(t) leaves the positive-definite cone."""
    N, D = int(g["N"]), int(g["D"])
    x = g["x"].copy()
    x[:N * D * D] = -200.0 * np.tile(np.eye(D).ravel(), N)
    x[:N * D * D] += 50.0 * np.random.default_rng(0).standard_normal(N * D * D)
    return x


def test_linalg_error_names_the_problem():
    """A LinAlgError names the problem whose S(t) failed, not its launch position, also under a compacted list;
    the host entry points evaluate every problem whatever list is installed, and name problems as such."""
    import torch
    g = _load("eval_L96_euler")
    N, D, B = int(g["N"]), int(g["D"]), 6
    X = np.stack([g["x"]] * B)
    X[3] = _not_pd_x(g)
    good = np.stack([g["x"]] * B)
    F_g = float(g["F"])
    with evaluator_from_golden(g, B=B, scratch_bytes=2 * 8 * N * (2 * D + 2 * D * D + 1) + 64) as ev:
        assert ev.chunk_size == 2
        n = ev.n_x
        Xd, good_d = torch.from_numpy(X).cuda(), torch.from_numpy(good).cuda()
        F = torch.empty(B, dtype=torch.float64, device="cuda")
        G = torch.empty((B, n), dtype=torch.float64, device="cuda")

        def device_eval(x):
            ev.eval_device(x.data_ptr(), n, F.data_ptr(), G.data_ptr(), n, _stream())
            ev.sync()

        def all_good(listed=range(B)):
            device_eval(good_d)
            assert all(abs(F[p].item() - F_g) <= TOL * abs(F_g) for p in listed)
            Fh, _ = ev.eval(good)
            assert np.all(np.abs(Fh - F_g) <= TOL * abs(F_g))

        with pytest.raises(np.linalg.LinAlgError, match=r"problem 3 at"):
            ev.eval(X)
        all_good()
        with pytest.raises(np.linalg.LinAlgError, match=r"problem 3 at"):
            device_eval(Xd)
        all_good()
        ev.set_active_list([5, 3, 0])                      # problem 3 sits at launch position 1
        with pytest.raises(np.linalg.LinAlgError, match=r"problem 3 at"):
            device_eval(Xd)
        all_good([5, 3, 0])
        ev.set_active_list([1, 2, 4, 5])                   # problem 3 is not listed: a host call still evaluates it
        with pytest.raises(np.linalg.LinAlgError, match=r"problem 3 at"):
            ev.eval(X)
        with pytest.raises(np.linalg.LinAlgError, match=r"problem 3 at"):
            ev.eval_full(X[3], problem=3)
        device_eval(Xd)                                    # ... and a device call does not
        all_good([1, 2, 4, 5])
        ev.set_active_list(None)


# ---- the SCG vector kernels (vecops.cu) -----------------------------------------------------------------------

VEC_SHAPES = [(B, n) for B in (1, 3) for n in (1, 255, 256, 257, 8191, 8192, 8193, 3 * 8192 + 5, 64 * 8192 + 1)]
VEC_SHAPES += [(B, n) for B in (592, 593) for n in (1, 255, 256, 257, 8193)]     # one slice per row at these B


def _vec_rows(V, stride):
    """(B, n) float64 numpy rows into a sentinel-filled device buffer, `stride` apart."""
    import torch
    B, n = V.shape
    buf = _alloc(B, n, stride)
    _rows(buf, B, n, stride).copy_(torch.from_numpy(np.ascontiguousarray(V)).cuda().view(torch.int64))
    return buf


def _host_vec_expect(V, stride):
    B, n = V.shape
    buf, f = _host_rows(B, n, stride)
    f[:B * stride].reshape(B, stride)[:, :n] = V
    return buf


def _check_vecops(B, n, rng):
    import torch
    lib, raise_for = _lib()
    st = _stream()
    s = n + 3
    x, y, z, d, gg = (rng.integers(-8, 9, size=(B, n)).astype(np.float64) for _ in range(5))
    active = rng.random(B) < 0.7
    active[0] = True
    act = torch.from_numpy(active.astype(np.int32)).cuda()
    xb, yb, zb = _vec_rows(x, s), _vec_rows(y, s), _vec_rows(z, s)
    f = lambda t: t.data_ptr()

    def out_of(buf):
        torch.cuda.synchronize()
        return buf.cpu().numpy()

    def vec_expect(V, keep=None, old=None):
        V = V.copy()
        if keep is not None:
            V[~keep] = old[~keep]
        return _host_vec_expect(V, s)

    dots = np.stack([(x * y).sum(1), (x * z).sum(1), (x * x).sum(1)])        # exact: integer partial sums
    for zp, act_p, on in ((zb, None, np.ones(B, bool)), (None, act, active)):
        out = _sentinel(3 * B + GUARD)
        raise_for(lib.vgpa_bdot(B, n, f(xb), f(yb), f(zp) if zp is not None else None, s, f(out),
                                f(act_p) if act_p is not None else None, st))
        exp = np.full(3 * B + GUARD, SENT, dtype=np.int64)
        ref = dots.copy()
        if zp is None:
            ref[1] = 0.0
        exp[:3 * B].reshape(3, B)[:, on] = ref[:, on].view(np.int64)
        assert np.array_equal(out_of(out), exp), ("bdot", B, n)
    stats = np.stack([np.abs(x).max(1), np.abs(x).sum(1)])
    out = _sentinel(2 * B + GUARD)
    raise_for(lib.vgpa_bstats(B, n, f(xb), s, f(out), f(act), st))
    exp = np.full(2 * B + GUARD, SENT, dtype=np.int64)
    exp[:2 * B].reshape(2, B)[:, active] = stats[:, active].view(np.int64)
    assert np.array_equal(out_of(out), exp), ("bstats", B, n)

    a = rng.choice([0.5, -0.5, 2.0, -3.0], size=B)
    a_d = torch.from_numpy(a).cuda()
    ob = _vec_rows(gg, s)                          # previous contents: kept in the rows of inactive problems
    raise_for(lib.vgpa_baxpy(B, n, f(a_d), f(xb), f(yb), f(ob), s, f(act), st))
    assert np.array_equal(out_of(ob), vec_expect(y + a[:, None] * x, active, gg)), ("baxpy", B, n)

    mode = rng.integers(0, 3, size=B).astype(np.int32)
    gamma = 2.0 ** rng.integers(-3, 4, size=B).astype(np.float64)
    mode_d, gamma_d = torch.from_numpy(mode).cuda(), torch.from_numpy(gamma).cuda()
    db, gb = _vec_rows(d, s), _vec_rows(gg, s)
    raise_for(lib.vgpa_bdir(B, n, f(mode_d), f(gamma_d), f(db), f(gb), s, st))
    dn = np.where((mode == 1)[:, None], gamma[:, None] * d - gg, np.where((mode == 2)[:, None], -gg, d))
    assert np.array_equal(out_of(db), vec_expect(dn)), ("bdir", B, n)
    assert np.array_equal(out_of(gb), vec_expect(gg)), ("bdir reads g only", B, n)

    mask = (rng.random(B) < 0.5).astype(np.int32)
    mask_d = torch.from_numpy(mask).cuda()
    dst = _vec_rows(d, s)
    raise_for(lib.vgpa_bcopy(B, n, f(mask_d), f(zb), f(dst), s, st))
    assert np.array_equal(out_of(dst), vec_expect(z, mask != 0, d)), ("bcopy", B, n)
    for buf, V in ((xb, x), (yb, y), (zb, z)):
        assert np.array_equal(out_of(buf), vec_expect(V)), ("inputs untouched", B, n)


def test_vector_kernels_exact_on_integers():
    """Integer data in [-8, 8], a in {+-0.5, 2, -3}, gamma a power of two: every partial sum, y + a x and
    gamma d - g is exact in fp64 whatever the summation order, so the kernels must match numpy bit for bit.
    Shapes span every slice count of slices() (1, 3, 64 slices per row); row stride n + 3 with sentinels."""
    rng = np.random.default_rng(21)
    # small call, a call whose slice partials outgrow the thread's partial buffer, small call again
    _check_vecops(3, 257, rng)
    _check_vecops(40000, 2, rng)
    _check_vecops(3, 257, rng)
    for B, n in VEC_SHAPES:
        _check_vecops(B, n, rng)


@pytest.mark.parametrize("n", [1, 257, 8193, 3 * 8192 + 5, 64 * 8192 + 1])
def test_vector_dot_against_exact_sum(n):
    """Random floats in [1, 2): x.y within 1e-12 sum|x_i y_i| of math.fsum -- one dropped or doubled element
    is off by at least 1."""
    import torch
    lib, raise_for = _lib()
    B = 3
    rng = np.random.default_rng(n)
    x, y = (1.0 + rng.random((B, n)) for _ in range(2))
    s = n + 3
    xb, yb = _vec_rows(x, s), _vec_rows(y, s)
    out = torch.empty(3 * B, dtype=torch.float64, device="cuda")
    raise_for(lib.vgpa_bdot(B, n, xb.data_ptr(), yb.data_ptr(), None, s, out.data_ptr(), None, _stream()))
    got = out.cpu().numpy()
    for p in range(B):
        for k, v in ((0, y[p]), (2, x[p])):
            exact = math.fsum(x[p] * v)
            assert abs(got[k * B + p] - exact) <= 1e-12 * float(np.abs(x[p] * v).sum()), (p, k)
