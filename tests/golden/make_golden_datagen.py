#!/usr/bin/env python
"""
Golden fixtures for data generation (SURVEY.md section 8 f4): sample paths and noisy
observations produced by the UNMODIFIED reference classes
(src/dynamics/{double_well,ornstein_uhlenbeck,lorenz_63,lorenz_96}.py: make_trajectory;
src/dynamics/stochastic_process.py:130-230: collect_obs), together with the random draws
they consumed.  The draws are recovered by replaying a second numpy Generator with the same
seed through the same sequence of calls, and are STORED, so the tests do not depend on the
numpy version's Generator stream.

Runs with the reference checkout (VGPA_REFERENCE, or baseline/_ref):

    python tests/golden/make_golden_datagen.py
"""
import contextlib
import io
import os
import sys
import types
from pathlib import Path

import numpy as np
from numpy.random import SeedSequence, default_rng

REF = Path(os.environ.get("VGPA_REFERENCE", Path(__file__).resolve().parents[2] / "baseline" / "_ref"))
HERE = Path(__file__).resolve().parent
SEED = 31415926535

CASES = {  # model: (sigma, theta, tf, dt, obs density, obs noise)
    "DW": (0.8, 1.0, 10.0, 0.01, 2, 0.04),
    "OU": (0.8, 2.0, 10.0, 0.01, 2, 0.04),
    "L63": ([10.0, 10.0, 10.0], [10.0, 28.0, 2.6667], 5.0, 0.01, 5, [2.0, 2.0, 2.0]),
    "L96": ([4.0] * 40, 8.0, 2.0, 0.01, 8, [1.0] * 40),
}


def main():
    if not REF.exists():
        raise SystemExit("the reference tree is missing: set VGPA_REFERENCE to a checkout of vrettasm/VGPA")
    sys.dont_write_bytecode = True
    sys.path.insert(0, str(REF))
    sys.modules.setdefault("h5py", types.ModuleType("h5py"))
    from src.var_bayes.simulation import dynamical_systems
    for model, (sigma, theta, tf, dt, density, r_obs) in CASES.items():
        with contextlib.redirect_stdout(io.StringIO()):
            proc = dynamical_systems[model](sigma, theta, SEED)
        proc.make_trajectory(0.0, tf, dt)
        path = np.array(proc.sample_path, dtype=float)
        obs_t, obs_y, obs_noise = proc.collect_obs(density, r_obs)
        N = proc.time_window.size
        M = len(obs_t)
        # replay the generator: stochastic_process.py:21-25 builds default_rng(SeedSequence(seed))
        rng = default_rng(SeedSequence(SEED))
        rec = {}
        if model == "DW":                                   # double_well.py:145-154
            rec["u_start"] = np.float64(rng.random())
            rec["n_start"] = np.float64(rng.standard_normal())
            z = rng.standard_normal(N)
        elif model == "OU":                                 # ornstein_uhlenbeck.py:151
            z = rng.standard_normal(N)
        else:                                               # lorenz_63.py:223 / lorenz_96.py:302
            z = rng.standard_normal((len(sigma), N))
        D = 1 if model in ("DW", "OU") else len(sigma)
        xi = rng.standard_normal(M) if D == 1 else rng.standard_normal((D, M))    # stochastic_process.py:196,225
        assert path[0] == proc.sample_path[0] if D == 1 else True
        rec.update(model=model, D=np.int64(D), N=np.int64(N), dt=np.float64(dt), tf=np.float64(tf),
                   theta=np.atleast_1d(np.asarray(theta, dtype=float)),
                   sigma=np.atleast_1d(np.asarray(sigma, dtype=float)),
                   R=np.atleast_1d(np.asarray(r_obs, dtype=float)),
                   z=z, xi=xi, x_start=np.atleast_1d(path[0]).astype(float),
                   path=path, obs_t=np.asarray(obs_t, dtype=np.int64), obs_y=np.asarray(obs_y, dtype=float))
        np.savez_compressed(HERE / f"datagen_{model}.npz", **rec)
        print(model, "N", N, "M", M, "path", path.shape, "obs_y", np.asarray(obs_y).shape, flush=True)


if __name__ == "__main__":
    main()
