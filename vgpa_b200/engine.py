"""
Batch evaluator: the Python face of a `vgpa_handle` (include/vgpa_b200.h).

One `BatchEvaluator` holds B independent inference problems of the same shape
(model, ODE method, D, N, observation times) on one GPU and evaluates the
variational free energy and its gradient for all of them in one call -- what
`VarGP.free_energy` + `VarGP.gradient` (reference src/var_bayes/variational.py:141-289)
do for a single problem.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import MODELS, METHODS, MODEL_DIM, VgpaDesc, model_dim, VgpaFullOut, dptr, f64, lib, raise_for


def _rows(a, B, n, name):
    """n values shared by the B problems, or B x n: returns the flat array and its row stride (0 = shared)."""
    a = f64(a).reshape(-1)
    if a.size == n:
        return a, 0
    if a.size == B * n:
        return a, n
    raise ValueError(f"{name}: expected {n} or {B}x{n} values, got {a.size}")


def _is_schedule_list(obs_t):
    """True for per-problem schedules: a list or tuple whose entries are index arrays (not ints)."""
    return isinstance(obs_t, (list, tuple)) and len(obs_t) > 0 and any(np.ndim(o) > 0 for o in obs_t)


def _schedule_rows(obs_t, obs_y, B, D):
    """Per-problem schedules: B index arrays and B (M_p, D) value arrays ((M_p,) too for D = 1), padded to the
    largest M_p.  Returns the (B, max(M, 1)) int64 index rows, the (B, M, D) values, the B counts and M."""
    if len(obs_t) != B:
        raise ValueError(f"obs_t: expected {B} per-problem index arrays, got {len(obs_t)}")
    if not isinstance(obs_y, (list, tuple)) or len(obs_y) != B:
        raise ValueError(f"obs_y: per-problem obs_t needs a matching sequence of {B} (M_p, D) arrays")
    ts, ys = [], []
    for p, (t, y) in enumerate(zip(obs_t, obs_y)):
        t = np.asarray(t)
        if t.ndim != 1 or (t.size and not np.issubdtype(t.dtype, np.integer)):
            raise ValueError(f"obs_t of problem {p}: expected a 1-D array of integer indices, got shape {t.shape}")
        y = np.asarray(y, dtype=np.float64)
        if D == 1 and y.ndim == 1:
            y = y.reshape(-1, 1)
        if y.shape != (t.size, D):
            raise ValueError(f"obs_y of problem {p}: expected shape ({t.size}, {D}), got {y.shape}")
        ts.append(t.astype(np.int64))
        ys.append(y)
    counts = np.array([t.size for t in ts], dtype=np.int32)
    M = int(counts.max())
    rows = np.zeros((B, max(M, 1)), dtype=np.int64)
    vals = np.zeros((B, M, D))
    for p, (t, y) in enumerate(zip(ts, ys)):
        rows[p, :t.size] = t
        vals[p, :t.size] = y
    return rows, vals, counts, M


def _mask_word(sel, D, what):
    """One observation mask: a (D,) bool array or a 1-D sequence of distinct component indices -> the bit word."""
    a = np.asarray(sel)
    if a.ndim != 1:
        raise ValueError(f"{what}: expected a ({D},) bool array or a list of component indices, got shape {a.shape}")
    if a.dtype == np.bool_:
        if a.size != D:
            raise ValueError(f"{what}: a bool mask needs {D} entries, got {a.size}")
        idx = np.flatnonzero(a)
    else:
        if a.size and not np.issubdtype(a.dtype, np.integer):
            raise ValueError(f"{what}: component indices must be integers, got {a.dtype}")
        idx = a.astype(np.int64)
        if np.any((idx < 0) | (idx >= D)):
            raise ValueError(f"{what}: component index out of range [0, {D}): {idx.tolist()}")
        if np.unique(idx).size != idx.size:
            raise ValueError(f"{what}: duplicate component index in {idx.tolist()}")
    if idx.size == 0:
        raise ValueError(f"{what}: no component is observed")
    return int(sum(1 << int(i) for i in idx))


def observed_words(observed, B, D):
    """The observed components as bit words (bit i = component i): one mask shared by the batch -- a (D,) bool
    array or a 1-D list of component indices -- or one per problem -- a (B, D) bool array or a list of B index
    lists.  Returns (uint64 array, stride in words: 0 shared, 1 per problem)."""
    a = observed if isinstance(observed, np.ndarray) else None
    per = (a is not None and a.ndim == 2) or (
        a is None and isinstance(observed, (list, tuple)) and len(observed) > 0 and any(np.ndim(o) > 0 for o in observed))
    if not per:
        return np.array([_mask_word(observed, D, "observed")], dtype=np.uint64), 0
    if len(observed) != B:
        raise ValueError(f"observed: expected {B} per-problem masks, got {len(observed)}")
    return np.array([_mask_word(o, D, f"observed of problem {p}") for p, o in enumerate(observed)], dtype=np.uint64), 1


class BatchEvaluator:
    """
    :param model:  "DW" | "OU" | "L63" | "L96"   (simulation.py:20)
    :param method: "euler" | "heun" | "rk2" | "rk4" (utilities.py:12)
    :param N: number of time-grid points; dt: sweep step; dt_model: model.time_step
    :param theta, sigma (D diag), R (D diag), obs_y (M,D), m0 (D), s0 (D,D), E0:
           one value set shared by the batch, or B of them stacked on axis 0
    :param obs_t: (M,) sorted unique observation indices, shared by the batch; or a list of B such index arrays,
           one schedule per problem (their counts may differ, 0 included), with obs_y a matching list of B
           (M_p, D) arrays ((M_p,) accepted for D = 1).  A list or tuple is read as per-problem schedules as soon
           as one entry is not a scalar: a nested list such as [[3, 6]] is one schedule per problem (here B = 1),
           not a flattened shared schedule, and needs obs_y as a list too.  A flat list or any numpy array keeps
           the shared meaning.
    :param D: state dimension; None = the model's (L96: 40).  L96 takes any 10 <= D <= 64
    :param observed: the observed state components; None = all.  One set shared by the batch -- a (D,) bool
           array or a 1-D list of component indices -- or one per problem -- a (B, D) bool array or a list of B
           index lists.  obs_y and R keep their D columns; those of unobserved components are ignored.  An
           unobserved component contributes nothing to Eobs and its jumps, and initialization() gives it the
           constant mean path m0 (vgpa_create_observed).
    """

    def __init__(self, model, method, N, dt, theta, sigma, R, obs_t, obs_y, m0, s0, E0,
                 B=1, dt_model=None, device=0, scratch_bytes=0, D=None, observed=None):
        key = str(model).upper()
        if key not in MODELS:
            raise ValueError(f" Unknown stochastic model -> {key}")
        mkey = str(method).lower()
        if mkey not in METHODS:
            raise ValueError(f" Integration method is unknown -> {method}.")
        D = model_dim(key, D)
        self.model, self.method, self.D, self.N, self.B = key, mkey, D, int(N), int(B)
        self.n_x = self.N * D * (D + 1)
        self.device = int(device)
        keep = {}
        rows = _is_schedule_list(obs_t)
        if rows:
            obs_t, obs_y, counts, M = _schedule_rows(obs_t, obs_y, self.B, D)
            keep["counts"] = counts
        else:
            obs_t = np.ascontiguousarray(np.asarray(obs_t, dtype=np.int64).ravel())
            M = obs_t.size
        if observed is not None:
            keep["observed"], obs_stride = observed_words(observed, self.B, D)
        nth = 3 if key == "L63" else 1
        d = VgpaDesc()
        d.model, d.method, d.D, d.N, d.M, d.B = MODELS[key], METHODS[mkey], D, self.N, M, self.B
        d.device = self.device
        d.dt = float(dt)
        d.dt_model = float(dt if dt_model is None else dt_model)
        for name, val, n in (("theta", theta, nth), ("sigma", sigma, D), ("R", R, D), ("obs_y", obs_y, M * D),
                             ("m0", m0, D), ("s0", s0, D * D), ("E0", E0, 1)):
            if name == "obs_y" and M == 0:
                continue
            arr, stride = _rows(val, self.B, n, name)
            keep[name] = arr
            setattr(d, name, dptr(arr))
            setattr(d, name + "_stride", stride)
        keep["obs_t"] = obs_t
        d.scratch_bytes = int(scratch_bytes)
        self._h = C.c_void_p()
        if observed is not None:
            rc = lib.vgpa_create_observed(C.byref(d), obs_t.ctypes.data, obs_t.shape[1] if rows else 0,
                                          counts.ctypes.data if rows else None, keep["observed"].ctypes.data,
                                          obs_stride, C.byref(self._h))
        elif rows:   # every problem its own schedule, padded to M rows
            rc = lib.vgpa_create_obs_rows(C.byref(d), obs_t.ctypes.data, obs_t.shape[1], counts.ctypes.data,
                                          C.byref(self._h))
        else:
            d.obs_t = obs_t.ctypes.data_as(C.POINTER(C.c_int64))
            rc = lib.vgpa_create(C.byref(d), C.byref(self._h))
        raise_for(rc, None)
        self._keep = keep

    # -- lifetime ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            lib.vgpa_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- evaluation ---------------------------------------------------------
    def eval(self, X, want_grad=True, F_out=None, G_out=None):
        """Host buffers.  X: (n_x,) shared by all problems, or (B, n_x).
        Returns (F (B,), grad (B, n_x) or None)."""
        X = np.asarray(X)
        if X.dtype != np.float64 or not X.flags.c_contiguous:
            X = f64(X)
        if X.size == self.n_x:
            xs = 0
        elif X.size == self.B * self.n_x:
            xs = self.n_x
        else:
            raise ValueError(f"x: expected {self.n_x} or {self.B}x{self.n_x} values, got {X.size}")
        F = np.empty(self.B) if F_out is None else F_out
        G = None
        if want_grad:
            G = np.empty((self.B, self.n_x)) if G_out is None else G_out
        rc = lib.vgpa_eval(self._h, X.ctypes.data, xs, 1 if want_grad else 0, F.ctypes.data,
                           G.ctypes.data if want_grad else None, self.n_x)
        raise_for(rc, self._h)
        return F, G

    def eval_device(self, x_ptr, x_stride, F_ptr, grad_ptr=None, grad_stride=None, stream=0):
        """Device pointers (ints), asynchronous on `stream`; call sync() afterwards."""
        rc = lib.vgpa_eval_device(self._h, x_ptr, x_stride, 1 if grad_ptr else 0, F_ptr, grad_ptr,
                                  self.n_x if grad_stride is None else grad_stride, stream or None)
        raise_for(rc, self._h)

    def sync(self):
        raise_for(lib.vgpa_sync(self._h), self._h)

    @property
    def n_theta(self):
        """Entries of dEsde_dtheta per problem: 1 (DW, OU), 3 (L63), D (L96, lorenz_96.py:431)."""
        return {"DW": 1, "OU": 1, "L63": 3, "L96": self.D}[self.model]

    def hyper_device(self, x_ptr, x_stride, F_ptr=None, Esde_ptr=None, dtheta_ptr=None, dtheta_stride=None,
                     dsigma_ptr=None, dsigma_stride=None, stream=0):
        """model.energy's hyper-parameter gradients for every problem at its x row (vgpa_hyper_device): device
        pointers (ints), asynchronous on `stream`; call sync() afterwards.  Any output may be None; default strides
        are compact rows (n_theta and 1 or D*D values)."""
        nsig = 1 if self.D == 1 else self.D * self.D
        rc = lib.vgpa_hyper_device(self._h, x_ptr, x_stride, F_ptr, Esde_ptr, dtheta_ptr,
                                   self.n_theta if dtheta_stride is None else dtheta_stride, dsigma_ptr,
                                   nsig if dsigma_stride is None else dsigma_stride, stream or None)
        raise_for(rc, self._h)

    def hyper(self, X):
        """F, Esde, dEsde_dtheta and dEsde_dsigma of every problem at its x: X (n_x,) shared by all problems or
        (B, n_x), a host array or a CUDA tensor.  Returns a dict of host arrays; each problem's entries have the
        shapes StochasticProcess.energy returns: F, Esde (B,); dEsde_dtheta (B,) for D = 1, else (B, n_theta);
        dEsde_dsigma (B,) for D = 1, else (B, D, D)."""
        import torch
        dev = torch.device("cuda", self.device)
        Xt = torch.as_tensor(X, dtype=torch.float64, device=dev)
        if Xt.numel() == self.n_x:
            Xt, xs = Xt.reshape(1, self.n_x).contiguous(), 0
        elif Xt.numel() == self.B * self.n_x:
            Xt, xs = Xt.reshape(self.B, self.n_x).contiguous(), self.n_x
        else:
            raise ValueError(f"x: expected {self.n_x} or {self.B}x{self.n_x} values, got {Xt.numel()}")
        B, D, nth = self.B, self.D, self.n_theta
        F, Esde = (torch.empty(B, dtype=torch.float64, device=dev) for _ in range(2))
        dth = torch.empty((B, nth), dtype=torch.float64, device=dev)
        dsig = torch.empty((B, 1 if D == 1 else D * D), dtype=torch.float64, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        self.hyper_device(Xt.data_ptr(), xs, F.data_ptr(), Esde.data_ptr(), dth.data_ptr(), nth, dsig.data_ptr(),
                          dsig.shape[1], stream)
        self.sync()
        out = {"F": F.cpu().numpy(), "Esde": Esde.cpu().numpy(), "dEsde_dtheta": dth.cpu().numpy(),
               "dEsde_dsigma": dsig.cpu().numpy()}
        if D == 1:
            out["dEsde_dtheta"], out["dEsde_dsigma"] = out["dEsde_dtheta"][:, 0], out["dEsde_dsigma"][:, 0]
        else:
            out["dEsde_dsigma"] = out["dEsde_dsigma"].reshape(B, D, D)
        return out

    def set_active(self, mask_ptr=None):
        """Device pointer to B int32 flags (0 = skip the problem in the following eval_device calls:
        its F and gradient row stay untouched), or None for every problem."""
        raise_for(lib.vgpa_set_active(self._h, mask_ptr), self._h)

    def set_active_list(self, problems=None):
        """Compacted launches (Lorenz-96 only): evaluate exactly these problem indices in the following
        eval_device calls, chunked by list position -- a thinned-out ensemble keeps whole waves.  None: off."""
        if problems is None:
            raise_for(lib.vgpa_set_active_list(self._h, None, -1), self._h)
            return
        lst = np.ascontiguousarray(problems, dtype=np.int32)
        raise_for(lib.vgpa_set_active_list(self._h, lst.ctypes.data, int(lst.size)), self._h)

    def initialization(self, t0=0.0):
        """VarGP.initialization for every problem of the batch, computed on the GPU: (B, n_x) host array."""
        X = np.empty((self.B, self.n_x))
        raise_for(lib.vgpa_initialization_host(self._h, float(t0), dptr(X), self.n_x), self._h)
        return X

    def initialization_device(self, x_ptr, x_stride=None, t0=0.0, stream=0):
        """The same into DEVICE rows x_ptr + p * x_stride (an ensemble's starting points never leave HBM)."""
        rc = lib.vgpa_initialization(self._h, float(t0), x_ptr, self.n_x if x_stride is None else x_stride,
                                     stream or None)
        raise_for(rc, self._h)

    def eval_full(self, x, problem=0):
        """Everything the reference caches or passes between stages, for one problem."""
        x = f64(x).reshape(-1)
        if x.size != self.n_x:
            raise ValueError(f"x: expected {self.n_x} values, got {x.size}")
        N, D = self.N, self.D
        nv, nm = N * D, N * D * D
        bufs = dict(F=np.zeros(1), parts=np.zeros(3), grad=np.empty(self.n_x), mt=np.empty(nv),
                    st=np.empty(nm), lamt=np.empty(nv), psit=np.empty(nm), Efx=np.empty(nv),
                    Edf=np.empty(nm), dEsde_dm=np.empty(nv), dEsde_ds=np.empty(nm))
        out = VgpaFullOut(**{k: dptr(v) for k, v in bufs.items()})
        rc = lib.vgpa_eval_full(self._h, int(problem), dptr(x), C.byref(out))
        raise_for(rc, self._h)
        vs = (N,) if D == 1 else (N, D)
        ms = (N,) if D == 1 else (N, D, D)
        res = {k: bufs[k].reshape(ms if k in ("st", "psit", "Edf", "dEsde_ds") else vs)
               for k in ("mt", "st", "lamt", "psit", "Efx", "Edf", "dEsde_dm", "dEsde_ds")}
        res.update(F=float(bufs["F"][0]), E0=bufs["parts"][0], Esde=bufs["parts"][1],
                   Eobs=bufs["parts"][2], grad=bufs["grad"])
        return res

    def set_timing(self, enable=True):
        raise_for(lib.vgpa_set_timing(self._h, 1 if enable else 0), self._h)

    def get_timing(self):
        """{kind: (total_ms, launches)} since the last call; kinds fwd/energy/finalize/bwd."""
        ms = np.zeros(4)
        n = np.zeros(4, dtype=np.int64)
        raise_for(lib.vgpa_get_timing(self._h, dptr(ms), n.ctypes.data_as(C.POINTER(C.c_int64))), self._h)
        return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(("fwd", "energy", "finalize", "bwd"))}

    # -- introspection ------------------------------------------------------
    @property
    def launch_count(self):
        return int(lib.vgpa_launch_count(self._h))

    @property
    def chunk_size(self):
        return int(lib.vgpa_chunk_size(self._h))

    @property
    def scratch_bytes(self):
        return int(lib.vgpa_scratch_in_use(self._h))


# -- operator-level entry points (one problem, host buffers) -------------------
def solve_fwd(method, A, b, m0, s0, sigma_diag, dt, device=0):
    """FwdOde.__call__ (fwd_ode.py:45): returns mt (N,D), st (N,D,D) (1-D: (N,), (N,))."""
    b = f64(b)
    single = b.ndim == 1
    N = b.shape[0]
    D = 1 if single else b.shape[1]
    A, m0, s0, sg = f64(A), f64(np.atleast_1d(m0)), f64(np.atleast_1d(s0)), f64(np.atleast_1d(sigma_diag))
    if A.size != N * D * D or m0.size != D or s0.size != D * D or sg.size != D:
        raise ValueError("solve_fwd: inconsistent shapes")
    mt, st = np.empty(N * D), np.empty(N * D * D)
    rc = lib.vgpa_solve_fwd(device, METHODS[str(method).lower()], D, N, float(dt), dptr(A), dptr(b),
                            dptr(m0), dptr(s0), dptr(sg), dptr(mt), dptr(st))
    raise_for(rc, None)
    return (mt, st) if single else (mt.reshape(N, D), st.reshape(N, D, D))


def solve_bwd(method, A, dEsde_dm, dEsde_ds, dEobs_dm, dEobs_ds, dt, device=0):
    """BwdOde.__call__ (bwd_ode.py:45): returns lam (N,D), psi (N,D,D)."""
    g = f64(dEsde_dm)
    single = g.ndim == 1
    N = g.shape[0]
    D = 1 if single else g.shape[1]
    A, G, jm, js = f64(A), f64(dEsde_ds), f64(dEobs_dm), f64(dEobs_ds)
    if A.size != N * D * D or G.size != N * D * D or jm.size != N * D or js.size != N * D * D:
        raise ValueError("solve_bwd: inconsistent shapes")
    lam, psi = np.empty(N * D), np.empty(N * D * D)
    rc = lib.vgpa_solve_bwd(device, METHODS[str(method).lower()], D, N, float(dt), dptr(A), dptr(g),
                            dptr(G), dptr(jm), dptr(js), dptr(lam), dptr(psi))
    raise_for(rc, None)
    return (lam, psi) if single else (lam.reshape(N, D), psi.reshape(N, D, D))


def model_energy(model, theta, sigma_diag, A, b, m, S, dt_model, device=0, hyper=False):
    """model.energy(A, b, m, S, obs_t) of the reference's StochasticProcess classes.
    Returns Esde, Ef, Edf, dEsde_dm, dEsde_ds (+ dEsde_dtheta, dEsde_dsigma with hyper=True)."""
    key = str(model).upper()
    b = f64(b)
    N = b.shape[0]
    D = model_dim(key, (b.size // N) if key == "L96" else None)
    A, m, S = f64(A), f64(m), f64(S)
    th, sg = f64(np.atleast_1d(theta)), f64(np.atleast_1d(sigma_diag))
    if A.size != N * D * D or m.size != N * D or S.size != N * D * D or b.size != N * D or sg.size != D:
        raise ValueError("model_energy: inconsistent shapes")
    Esde = np.zeros(1)
    Ef, Edf, dm, ds = np.empty(N * D), np.empty(N * D * D), np.empty(N * D), np.empty(N * D * D)
    nth = {"DW": 1, "OU": 1, "L63": 3, "L96": D}[key]
    dth = np.zeros(nth) if hyper else None
    dsig = np.zeros(1 if D == 1 else D * D) if hyper else None
    rc = lib.vgpa_model_energy(device, MODELS[key], D, N, float(dt_model), dptr(th), dptr(sg), dptr(A),
                               dptr(b), dptr(m), dptr(S), dptr(Esde), dptr(Ef), dptr(Edf), dptr(dm), dptr(ds),
                               dptr(dth) if hyper else None, dptr(dsig) if hyper else None)
    raise_for(rc, None)
    if D == 1:
        out = (float(Esde[0]), Ef, Edf, dm, ds)
        return out + (float(dth[0]), float(dsig[0])) if hyper else out
    out = (float(Esde[0]), Ef.reshape(N, D), Edf.reshape(N, D, D), dm.reshape(N, D), ds.reshape(N, D, D))
    return out + (dth, dsig.reshape(D, D)) if hyper else out


def obs_energy(obs_t, obs_y, R_diag, m, s, device=0, with_dr=False, observed=None):
    """GaussianLikelihood.__call__ / .gradients: returns Eobs, dEobs_dm, dEobs_ds (+ dEobs_dr).  observed: the bit
    word of the observed components (vgpa_obs_energy_observed; obs_y (M, D) and R (D,) with ignored entries at the
    others), None = all; dEobs_dr is not available with a mask."""
    m = f64(m)
    single = m.ndim == 1
    N = m.shape[0]
    D = 1 if single else m.shape[1]
    s, oy, R = f64(s), f64(obs_y), f64(np.atleast_1d(R_diag))
    ot = np.ascontiguousarray(np.asarray(obs_t, dtype=np.int64).ravel())
    M = ot.size
    if s.size != N * D * D or oy.size != M * D or R.size != D:
        raise ValueError("obs_energy: inconsistent shapes")
    E = np.zeros(1)
    jm, js = np.empty(N * D), np.empty(N * D * D)
    dr = np.empty(N if single else N * M * M) if with_dr else None
    if observed is not None:
        if with_dr:
            raise ValueError("obs_energy: dEobs_dr is not computed for a component-selecting operator")
        rc = lib.vgpa_obs_energy_observed(device, D, N, M, ot.ctypes.data_as(C.POINTER(C.c_int64)), dptr(oy), dptr(R),
                                          int(observed), dptr(m), dptr(s), dptr(E), dptr(jm), dptr(js))
    else:
        rc = lib.vgpa_obs_energy(device, D, N, M, ot.ctypes.data_as(C.POINTER(C.c_int64)), dptr(oy), dptr(R),
                                 dptr(m), dptr(s), dptr(E), dptr(jm), dptr(js), dptr(dr) if with_dr else None)
    raise_for(rc, None)
    if single:
        out = (float(E[0]), jm, js)
        return out + (dr,) if with_dr else out
    out = (float(E[0]), jm.reshape(N, D), js.reshape(N, D, D))
    return out + (dr.reshape(N, M, M),) if with_dr else out


# -- batched data generation (SURVEY 8 f4; host buffers) ------------------------------
def make_trajectories(model, N, dt, theta, sigma_diag, z, x_init=None, device=0):
    """B sample paths by the Euler-Maruyama loop of <Model>.make_trajectory, on the GPU.
    z: (B, D, N) standard-normal draws in the reference's (D, N) layout ((B, N) for the 1-D models);
    theta: DW [theta], OU [theta, mu], L63 [sigma, rho, beta], L96 [F]; x_init: state at t0 (required
    for DW / OU; None for L63 / L96 = the reference's burn-in).  Returns (B, N, D) ((B, N) for D = 1)."""
    key = str(model).upper()
    if key not in MODELS:
        raise ValueError(f" Unknown stochastic model -> {key}")
    N = int(N)
    z = f64(z)
    # L96: D from the draws' (B, D, N) shape (a single path's (D, N) too), 40 when that is ambiguous
    D = model_dim(key, z.shape[-2] if key == "L96" and z.ndim >= 2 else None)
    if z.size % (N * D) or z.size == 0:
        raise ValueError(f"z: expected B x {D} x {N} values, got {z.size}")
    B = z.size // (N * D)
    nth = {"DW": 1, "OU": 2, "L63": 3, "L96": 1}[key]
    th, ths = _rows(theta, B, nth, "theta")
    sg, sgs = _rows(sigma_diag, B, D, "sigma")
    xi, xis = (None, 0) if x_init is None else _rows(x_init, B, D, "x_init")
    path = np.empty((B, N) if D == 1 else (B, N, D))
    rc = lib.vgpa_make_trajectory_dim(device, MODELS[key], D, N, B, float(dt), th.ctypes.data, ths, sg.ctypes.data, sgs,
                                  None if xi is None else xi.ctypes.data, xis, z.ctypes.data, N * D,
                                  path.ctypes.data, N * D)
    raise_for(rc, None)
    return path


def collect_observations(path, obs_t, R_diag, xi, device=0):
    """B noisy observation sets (StochasticProcess.collect_obs) on the GPU.
    path: (B, N, D) or (B, N), or one path shared by the sets ((N, D) / (N,) with xi giving B);
    xi: (B, D, M) draws ((B, M) for D = 1).  Returns (B, M, D) ((B, M) for D = 1)."""
    ot = np.ascontiguousarray(np.asarray(obs_t, dtype=np.int64).ravel())
    M = ot.size
    R = f64(np.atleast_1d(R_diag))
    xi = f64(xi)
    path = f64(path)
    D = R.shape[-1]
    if M == 0 or xi.size % (M * D):
        raise ValueError(f"xi: expected B x {D} x {M} values, got {xi.size}")
    B = xi.size // (M * D)
    if path.ndim == (1 if D == 1 else 2):     # one path shared by the B sets
        N, ps = path.shape[0], 0
    elif path.ndim == (2 if D == 1 else 3) and path.shape[0] == B:
        N, ps = path.shape[1], path.shape[1] * D
    else:
        raise ValueError(f"path: expected (N, D) or (B, N, D) with B = {B}, got {path.shape}")
    Rr, Rs = _rows(R, B, D, "R")
    out = np.empty((B, M) if D == 1 else (B, M, D))
    rc = lib.vgpa_collect_obs(device, D, N, M, B, ot.ctypes.data, Rr.ctypes.data, Rs, path.ctypes.data, ps,
                              xi.ctypes.data, M * D, out.ctypes.data, M * D)
    raise_for(rc, None)
    return out
