#!/usr/bin/env python
"""
Golden fixtures for the hyper-parameter gradients the reference's hot path computes and
discards (SURVEY.md section 8 f3): dEsde_dtheta, dEsde_dsigma of model.energy
(double_well.py:251-257, ornstein_uhlenbeck.py:223-229, lorenz_63.py:327-343,
lorenz_96.py:420-434) and dEobs_dr of GaussianLikelihood.gradients (gaussian_like.py:194,226); plus PriorKL0.gradients
(prior_kl0.py:94-175).

Inputs are taken from the existing per-evaluation fixtures (eval_<MODEL>_rk2.npz: A, b from x,
the marginal moments mt, st, theta, sigma, obs_t, obs_y, R), so the two sets stay consistent.
Runs the UNMODIFIED reference (a checkout named by VGPA_REFERENCE, or baseline/_ref):

    python tests/golden/make_golden_hyper.py
"""
import contextlib
import io
import os
import sys
import types
from pathlib import Path

import numpy as np

REF = Path(os.environ.get("VGPA_REFERENCE", Path(__file__).resolve().parents[2] / "baseline" / "_ref"))
HERE = Path(__file__).resolve().parent


def main():
    if not REF.exists():
        raise SystemExit("the reference tree is missing: set VGPA_REFERENCE to a checkout of vrettasm/VGPA")
    sys.dont_write_bytecode = True
    sys.path.insert(0, str(REF))
    sys.modules.setdefault("h5py", types.ModuleType("h5py"))
    from src.var_bayes.simulation import dynamical_systems
    from src.var_bayes.gaussian_like import GaussianLikelihood
    from src.var_bayes.prior_kl0 import PriorKL0
    for model in ("DW", "OU", "L63", "L96"):
        g = np.load(HERE / f"eval_{model}_rk2.npz", allow_pickle=True)
        D, N, dt = int(g["D"]), int(g["N"]), float(g["dt"])
        x = g["x"]
        if D == 1:
            A, b = x[:N], x[N:]
            sigma, theta = float(g["sigma"][0]), float(g["theta"][0])
            R = float(g["R"][0])
            obs_y = g["obs_y"].reshape(-1)
        else:
            A, b = x[:N * D * D].reshape(N, D, D), x[N * D * D:].reshape(N, D)
            sigma, theta = list(g["sigma"]), (list(g["theta"]) if model == "L63" else float(g["theta"][0]))
            R = np.diag(g["R"])
            obs_y = g["obs_y"]
        with contextlib.redirect_stdout(io.StringIO()):
            proc = dynamical_systems[model](sigma, theta, 1234)
        proc.time_window = dt * np.arange(N)          # energy() only reads time_step
        obs_t = [np.int64(t) for t in g["obs_t"]]
        Esde, _, (_, _, dth, dsig) = proc.energy(A, b, g["mt"], g["st"], obs_t)
        lik = GaussianLikelihood(obs_y, obs_t, R, None, D == 1)
        _, _, dr = lik.gradients(g["mt"], g["st"])
        # PriorKL0.gradients (prior_kl0.py:94-175) at the t = 0 multipliers of the same evaluation
        if D == 1:
            kl0 = PriorKL0(float(np.ravel(g["mu0"])[0]), float(np.ravel(g["tau0"])[0]), True)
            dk_m, dk_s = kl0.gradients(float(np.ravel(g["m0"])[0]), float(np.ravel(g["s0"])[0]), g["lamt"][0], g["psit"][0])
        else:
            kl0 = PriorKL0(g["mu0"], g["tau0"], False)
            dk_m, dk_s = kl0.gradients(g["m0"], g["s0"], g["lamt"][0], g["psit"][0])
        assert abs(float(Esde) - float(g["Esde"])) <= 1e-12 * abs(float(g["Esde"])), (model, Esde, g["Esde"])
        np.savez_compressed(HERE / f"hyper_{model}.npz", model=model, dEsde_dtheta=np.asarray(dth, dtype=float),
                            dEsde_dsigma=np.asarray(dsig, dtype=float), dEobs_dr=np.asarray(dr, dtype=float),
                            dKL0_dm0=np.asarray(dk_m, dtype=float), dKL0_ds0=np.asarray(dk_s, dtype=float))
        print(model, "dEsde_dtheta", np.asarray(dth).shape, "dEsde_dsigma", np.asarray(dsig).shape,
              "dEobs_dr", np.asarray(dr).shape, float(np.abs(dr).max()))


if __name__ == "__main__":
    main()
