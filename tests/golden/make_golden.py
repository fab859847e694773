#!/usr/bin/env python
"""
Generate the golden fixtures under tests/golden/ by running the UNMODIFIED
reference (vrettasm/VGPA: a checkout named by VGPA_REFERENCE, or baseline/_ref).
The reference is not part of this repository; its outputs are, as the .npz
files this script writes.

Run (with the reference checkout):

    python tests/golden/make_golden.py            # per-evaluation fixtures
    python tests/golden/make_golden.py --scg      # + SCG convergence traces
    python tests/golden/make_golden.py --l96-full # + L96 N=1001 known answers
    python tests/golden/make_golden.py --no-eval --l96-mid   # L96 N=101, M=8: all intermediates
    python tests/golden/make_golden.py --no-eval --scg-full   # full SCG runs at the BASELINE shapes

What is recorded per case (all float64, reference layouts):
  inputs : model, method, D, N, dt, theta, sigma(diag), obs_t, obs_y, R(diag),
           m0, s0, mu0, tau0, x (the evaluation point)
  outputs: F, E0, Esde, Eobs, grad, mt, st, lamt, psit, Efx, Edf,
           dEsde_dm, dEsde_ds

Reference call sites reproduced here: Simulation.setup
(src/var_bayes/simulation.py:92-176) and the object construction of
Simulation.run (src/var_bayes/simulation.py:189-212).
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time
import types
from pathlib import Path

import numpy as np

REF = Path(os.environ.get("VGPA_REFERENCE", Path(__file__).resolve().parents[2] / "baseline" / "_ref"))
HERE = Path(__file__).resolve().parent
SEED = 31415926535


def _import_reference():
    if not REF.exists():
        raise SystemExit("the reference tree is missing: set VGPA_REFERENCE to a checkout of vrettasm/VGPA")
    sys.dont_write_bytecode = True
    sys.path.insert(0, str(REF))
    # h5py is only used by Simulation.save/load (simulation.py:1,293,336).
    sys.modules.setdefault("h5py", types.ModuleType("h5py"))
    from src.var_bayes.simulation import Simulation          # noqa
    from src.var_bayes.fwd_ode import FwdOde                  # noqa
    from src.var_bayes.bwd_ode import BwdOde                  # noqa
    from src.var_bayes.gaussian_like import GaussianLikelihood  # noqa
    from src.var_bayes.prior_kl0 import PriorKL0              # noqa
    from src.var_bayes.variational import VarGP               # noqa
    from src.numerics.optim_scg import SCG                    # noqa
    return dict(Simulation=Simulation, FwdOde=FwdOde, BwdOde=BwdOde,
                GaussianLikelihood=GaussianLikelihood, PriorKL0=PriorKL0,
                VarGP=VarGP, SCG=SCG)


def base_params(model, method, tf, sys_noise, obs_noise, density, theta):
    return {"Output_Name": "golden", "Model": model, "Ode-method": method,
            "Random-Seed": SEED,
            "Time-window": {"t0": 0.0, "tf": tf, "dt": 0.01},
            "Noise": {"sys": sys_noise, "obs": obs_noise},
            "Observations": {"density": density, "operator": None},
            "Drift": {"theta": theta},
            "Prior": {"tau0": 0.5, "mu0": 1.0}}


# name -> params (shipped JSON values; L63/L96 with Noise.sys as a list, see
# SURVEY.md F6: the shipped scalar crashes the reference).
def config(model, method, tf=None):
    if model == "DW":
        return base_params("DW", method, tf or 10.0, 0.8, 0.04, 2, 1.0)
    if model == "OU":
        return base_params("OU", method, tf or 10.0, 0.8, 0.04, 2, 2.0)
    if model == "L63":
        return base_params("L63", method, tf or 20.0, [10.0] * 3, 2.0, 5,
                           [10.0, 28.0, 2.6667])
    if model == "L96":
        return base_params("L96", method, tf or 4.0, [4.0] * 40, 1.0, 8, 8.0)
    raise ValueError(model)


def build(ref, params):
    """Simulation.setup + the constructor block of Simulation.run."""
    with contextlib.redirect_stdout(io.StringIO()):
        sim = ref["Simulation"]("golden")
        sim.setup(params, None)
    md = sim.m_data
    dt = md["time_window"]["dt"]
    fwd = ref["FwdOde"](dt, md["ode_solver"], md["single_dim"])
    bwd = ref["BwdOde"](dt, md["ode_solver"], md["single_dim"])
    lik = ref["GaussianLikelihood"](md["obs_y"], md["obs_t"], md["obs_noise"],
                                    md["obs_setup"]["operator"], md["single_dim"])
    kl0 = ref["PriorKL0"](md["mu0"], md["tau0"], md["single_dim"])
    vgpa = ref["VarGP"](md["model"], md["m0"], md["s0"], fwd, bwd, lik, kl0,
                        md["obs_y"], md["obs_t"])
    return sim, vgpa


def perturb(x0, D, N, rng):
    """A dense evaluation point: the reference's x0 plus dense noise on A (so
    that A, A^T mix-ups and off-diagonal paths are exercised) and on b."""
    x = x0.copy()
    na = N * D * D
    x[:na] += 0.15 * rng.standard_normal(na)
    x[na:] += 0.25 * rng.standard_normal(N * D)
    return x


def evaluate(vgpa, x):
    """free_energy + gradient + every intermediate the path produces."""
    md = vgpa.model
    F = vgpa.free_energy(x)
    g = vgpa.gradient(x)
    out = vgpa.arg_out
    D, N = vgpa.dim_d, vgpa.dim_n
    if D == 1:
        A, b = x[:N], x[N:]
    else:
        A, b = x[:N * D * D].reshape(N, D, D), x[N * D * D:].reshape(N, D)
    Esde, (Efx, Edf), (dm, ds, *_) = md.energy(A, b, out["mt"], out["st"], vgpa.obs_t)
    Eobs = vgpa.likelihood(out["mt"], out["st"])
    E0 = vgpa.kl0(out["m0"], out["s0"])
    return dict(F=np.float64(F), E0=np.float64(E0), Esde=np.float64(Esde),
                Eobs=np.float64(Eobs), grad=g, mt=out["mt"], st=out["st"],
                lamt=out["lamt"], psit=out["psit"], Efx=np.asarray(Efx),
                Edf=np.asarray(Edf), dEsde_dm=np.asarray(dm), dEsde_ds=np.asarray(ds))


def inputs_of(sim, vgpa, params, x):
    md = sim.m_data
    D, N = vgpa.dim_d, vgpa.dim_n
    sig = np.atleast_1d(np.asarray(md["model"].sigma, dtype=float))
    sig = np.diag(sig).copy() if sig.ndim == 2 else sig
    R = np.atleast_1d(np.asarray(md["obs_noise"], dtype=float))
    R = np.diag(R).copy() if R.ndim == 2 else R
    return dict(model=params["Model"], method=params["Ode-method"].lower(),
                D=np.int64(D), N=np.int64(N), dt=np.float64(params["Time-window"]["dt"]),
                tf=np.float64(params["Time-window"]["tf"]),
                theta=np.atleast_1d(np.asarray(md["model"].theta, dtype=float)),
                sigma=sig, R=R,
                obs_t=np.asarray(md["obs_t"], dtype=np.int64),
                obs_y=np.asarray(md["obs_y"], dtype=float),
                m0=np.atleast_1d(np.asarray(md["m0"], dtype=float)),
                s0=np.atleast_2d(np.asarray(md["s0"], dtype=float)),
                mu0=np.atleast_1d(np.asarray(md["mu0"], dtype=float)),
                tau0=np.atleast_2d(np.asarray(md["tau0"], dtype=float)),
                x=x)


EVAL_CASES = [  # (model, tf) -- every solver is generated for each
    ("DW", 10.0), ("OU", 10.0), ("L63", 2.0), ("L96", 0.2)]
METHODS = ["euler", "heun", "rk2", "rk4"]


def make_eval(ref):
    for model, tf in EVAL_CASES:
        for method in METHODS:
            params = config(model, method, tf)
            sim, vgpa = build(ref, params)
            x0 = vgpa.initialization()
            rng = np.random.default_rng([SEED, 7])
            x = perturb(x0, vgpa.dim_d, vgpa.dim_n, rng)
            t0 = time.perf_counter()
            out = evaluate(vgpa, x)
            el = time.perf_counter() - t0
            rec = inputs_of(sim, vgpa, params, x)
            rec.update(out)
            # F at the unperturbed x0 as an extra known answer.
            rec["x0"] = x0
            rec["F_x0"] = np.float64(vgpa.free_energy(x0))
            rec["gnorm_x0"] = np.float64(np.linalg.norm(vgpa.gradient(x0)))
            name = HERE / f"eval_{model}_{method}.npz"
            np.savez_compressed(name, **rec)
            print(f"{name.name}: N={vgpa.dim_n} F={out['F']:.12g} "
                  f"|g|={np.linalg.norm(out['grad']):.6g} ({el:.2f}s)")


def make_l96_mid(ref):
    """L96 at tf = 1.0 (N = 101 grid points, M = 8 observations), RK2 and RK4: the multi-observation
    jump logic of the backward sweep and the sn_diag quirk (SURVEY F5) pinned at the INTERMEDIATE level
    (lamt, psit, ...) for D = 40, which the tf = 0.2 fixtures (M = 1) cannot do.  The (N, D, D) arrays
    are stored at a subset of time indices (every observation index, its neighbours, both ends and
    every 8th index) to keep the fixture small; F, the gradient and the (N, D) arrays are complete."""
    for method in ("rk2", "rk4"):
        params = config("L96", method, 1.0)
        sim, vgpa = build(ref, params)
        x0 = vgpa.initialization()
        x = perturb(x0, vgpa.dim_d, vgpa.dim_n, np.random.default_rng([SEED, 13]))
        t0 = time.perf_counter()
        out = evaluate(vgpa, x)
        el = time.perf_counter() - t0
        N = vgpa.dim_n
        obs_t = np.asarray(sim.m_data["obs_t"], dtype=np.int64)
        keep = set(range(0, N, 8)) | {0, 1, N - 2, N - 1}
        for t in obs_t:
            keep |= {int(t) - 1, int(t), int(t) + 1}
        t_idx = np.array(sorted(k for k in keep if 0 <= k < N), dtype=np.int64)
        rec = inputs_of(sim, vgpa, params, x)
        for k, v in out.items():
            rec[k] = v[t_idx] if (isinstance(v, np.ndarray) and v.ndim == 3) else v
        rec["t_idx"] = t_idx
        if method != "rk2":      # the evaluation point does not depend on the solver: stored once, in mid_L96_rk2.npz
            assert np.array_equal(x, np.load(HERE / "mid_L96_rk2.npz")["x"])
            del rec["x"]
        name = HERE / f"mid_L96_{method}.npz"
        np.savez_compressed(name, **rec)
        print(f"{name.name}: N={N} M={obs_t.size} F={out['F']:.12g} kept {t_idx.size} of {N} indices ({el:.2f}s)")


def make_scg(ref, which):
    """SCG convergence traces with the reference's own optimiser."""
    jobs = {"DW": (config("DW", "euler"), 500), "OU": (config("OU", "rk4"), 500),
            "L63": (config("L63", "heun", 2.0), 500),
            "L96": (config("L96", "rk2", 0.2), 12)}
    for key in which:
        params, max_it = jobs[key]
        sim, vgpa = build(ref, params)
        opts = {"max_it": max_it, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
        scg = ref["SCG"](vgpa.free_energy, vgpa.gradient, opts)
        x0 = vgpa.initialization()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            x, fx = scg(x0.copy())
        el = time.perf_counter() - t0
        st = scg.stats
        n = int(st["MaxIt"])
        rec = inputs_of(sim, vgpa, params, x0)
        rec.update(dict(max_it=np.int64(max_it), n_it=np.int64(n), fx_final=np.float64(fx),
                        trace_fx=st["fx"][:n].copy(), trace_dfx=st["dfx"][:n].copy(),
                        trace_beta=st["beta"][:n].copy(), f_eval=np.float64(st["f_eval"]),
                        df_eval=np.float64(st["df_eval"]), x_final=x))
        name = HERE / f"scg_{key}.npz"
        np.savez_compressed(name, **rec)
        print(f"{name.name}: it={n} fx={fx:.12g} f_eval={st['f_eval']} ({el:.1f}s)")


def make_scg_full(ref, which):
    """Full SCG optimisations to convergence with the reference's own optimiser at the BASELINE
    shapes: configs[3] (L96 D=40, tf=10 -> N=1001, RK2; about 18 minutes of CPU) and configs[2]
    (L63, tf=20 -> N=2002, Heun as shipped; about 3 minutes).  Only the trace is stored."""
    jobs = {"L96": ("rk2", 10.0), "L63": ("heun", 20.0)}
    for key in which:
        method, tf = jobs[key]
        sim, vgpa = build(ref, config(key, method, tf))
        opts = {"max_it": 500, "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False}
        scg = ref["SCG"](vgpa.free_energy, vgpa.gradient, opts)
        x0 = vgpa.initialization()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            x, fx = scg(x0.copy())
        el = time.perf_counter() - t0
        st = scg.stats
        n = int(st["MaxIt"])
        name = HERE / f"scg_{key}_full.npz"
        np.savez_compressed(name, model=key, method=method, tf=np.float64(tf), max_it=np.int64(500),
                            n_it=np.int64(n), fx_final=np.float64(fx), trace_fx=st["fx"][:n].copy(),
                            trace_dfx=st["dfx"][:n].copy(), trace_beta=st["beta"][:n].copy(),
                            f_eval=np.float64(st["f_eval"]), df_eval=np.float64(st["df_eval"]),
                            ref_seconds=np.float64(el))
        print(f"{name.name}: it={n} fx={fx:.12g} f_eval={st['f_eval']} ({el:.1f}s)")


def make_scg_rosenbrock(ref):
    """The reference's SCG on an analytic test function (no VGPA involved): pins the
    repo's own optimiser (vgpa_b200/scg.py) on the CPU."""
    def f(x):
        return float(np.sum(100.0 * (x[1:] - x[:-1] ** 2) ** 2 + (1.0 - x[:-1]) ** 2))

    def df(x, eval_fun=False):
        g = np.zeros_like(x)
        g[:-1] = -400.0 * x[:-1] * (x[1:] - x[:-1] ** 2) - 2.0 * (1.0 - x[:-1])
        g[1:] += 200.0 * (x[1:] - x[:-1] ** 2)
        return g
    x0 = np.array([-1.2, 1.0, 0.7, -0.4, 1.5, 0.2])
    scg = ref["SCG"](f, df, {"max_it": 400, "x_tol": 1.0e-10, "f_tol": 1.0e-14, "display": False})
    with contextlib.redirect_stdout(io.StringIO()):
        x, fx = scg(x0.copy())
    st = scg.stats
    n = int(st["MaxIt"])
    np.savez_compressed(HERE / "scg_rosenbrock.npz", x0=x0, x_final=x, fx_final=np.float64(fx),
                        n_it=np.int64(n), trace_fx=st["fx"][:n].copy(), trace_dfx=st["dfx"][:n].copy(),
                        trace_beta=st["beta"][:n].copy(), f_eval=np.float64(st["f_eval"]),
                        df_eval=np.float64(st["df_eval"]))
    print(f"scg_rosenbrock.npz: it={n} fx={fx:.6g}")


def make_l96_full(ref):
    """Known answers at the north-star shape (L96 D=40, tf=10 -> N=1001, RK2):
    F(x0), |grad F(x0)| and sparse samples of the gradient.  x0 itself is not
    stored (13 MB); the repo's own host mirror regenerates it bit-for-bit and
    the fixture carries a checksum to prove that."""
    params = config("L96", "rk2", 10.0)
    sim, vgpa = build(ref, params)
    x0 = vgpa.initialization()
    t0 = time.perf_counter()
    F = vgpa.free_energy(x0)
    g = vgpa.gradient(x0)
    el = time.perf_counter() - t0
    idx = np.linspace(0, g.size - 1, 4096).astype(np.int64)
    rec = inputs_of(sim, vgpa, params, np.zeros(1))
    rec.update(dict(F_x0=np.float64(F), gnorm_x0=np.float64(np.linalg.norm(g)),
                    g_idx=idx, g_samples=g[idx].copy(), g_absmax=np.float64(np.abs(g).max()),
                    x0_sum=np.float64(x0.sum()), x0_abs_sum=np.float64(np.abs(x0).sum()),
                    x0_idx=idx, x0_samples=x0[idx].copy(), ref_seconds=np.float64(el)))
    del rec["x"]
    name = HERE / "known_L96_N1001.npz"
    np.savez_compressed(name, **rec)
    print(f"{name.name}: F={F!r} |g|={np.linalg.norm(g)!r} ({el:.1f}s)")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--scg", nargs="*", default=None,
                    help="also write SCG traces (default: DW OU L63 L96)")
    ap.add_argument("--l96-full", action="store_true")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--rosenbrock", action="store_true")
    ap.add_argument("--l96-mid", action="store_true", help="L96 N=101, M=8 with all intermediates (RK2, RK4)")
    ap.add_argument("--scg-full", nargs="*", default=None,
                    help="full SCG runs at the BASELINE shapes (default: L63 L96; ~20 min of CPU)")
    a = ap.parse_args()
    ref = _import_reference()
    if not a.no_eval:
        make_eval(ref)
    if a.scg is not None:
        make_scg(ref, a.scg or ["DW", "OU", "L63", "L96"])
    if a.l96_full:
        make_l96_full(ref)
    if a.rosenbrock:
        make_scg_rosenbrock(ref)
    if a.l96_mid:
        make_l96_mid(ref)
    if a.scg_full is not None:
        make_scg_full(ref, a.scg_full or ["L63", "L96"])
    print(json.dumps({"numpy": np.__version__}))
