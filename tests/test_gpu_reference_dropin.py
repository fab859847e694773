"""
The drop-in, performed literally (INTEGRATION.md section 1): the UNMODIFIED reference (a checkout named
by VGPA_REFERENCE, or baseline/_ref; these tests skip without one) builds its own Simulation, dynamics,
FwdOde, BwdOde, GaussianLikelihood and PriorKL0
(src/var_bayes/simulation.py:92-207), `vgpa_b200.variational.VarGP` takes the place of
src/var_bayes/variational.py:VarGP in the constructor call of simulation.py:209, and the
reference's own optimiser (src/numerics/optim_scg.py:75-285) drives free_energy / gradient on the
CUDA path.  The traces must match the ones the reference recorded with its own VarGP
(tests/golden/scg_*.npz) within 1e-6 (BASELINE.json), and a single evaluation must match the
reference's own VarGP, evaluated right here on the box's CPU, to 1e-9 per gradient block (and, without
the reference tree, the outputs it recorded in tests/golden/eval_*.npz).
"""
import contextlib
import io
import sys

import numpy as np
import pytest

from conftest import GOLDEN, rel_err

sys.path.insert(0, str(GOLDEN))
import make_golden as mg  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    try:
        from baseline.refload import import_reference
        return import_reference()
    except ImportError as e:     # numba / scipy / the tree itself absent on this box
        pytest.skip(f"the unmodified reference is not importable here: {e}")


def _swap(ref, params):
    from baseline.refload import reference_objects
    from vgpa_b200.variational import VarGP
    sim, args = reference_objects(ref, params)
    assert type(args[0]).__module__.startswith("src.dynamics")           # the reference's own model object
    assert type(args[3]).__module__ == "src.var_bayes.fwd_ode"
    return sim, args, VarGP(*args)


@pytest.mark.parametrize("model,method,tf", [("DW", "euler", None), ("L63", "heun", 2.0)])
def test_reference_scg_drives_cuda_vargp(ref, model, method, tf):
    g = np.load(GOLDEN / f"scg_{model}.npz")
    sim, args, vgpa = _swap(ref, mg.config(model, method, tf))
    x0 = vgpa.initialization()
    assert np.array_equal(x0, g["x"])
    scg = ref["SCG"](vgpa.free_energy, vgpa.gradient,
                     {"max_it": int(g["max_it"]), "x_tol": 1.0e-6, "f_tol": 1.0e-8, "display": False})
    with contextlib.redirect_stdout(io.StringIO()):
        x, fx = scg(x0.copy())
    n_ref, n_new = int(g["n_it"]), int(scg.stats["MaxIt"])
    n = min(n_ref, n_new)
    assert abs(n_ref - n_new) <= max(2, n_ref // 50), (n_ref, n_new)
    refs, new = g["trace_fx"][:n], scg.stats["fx"][:n]
    assert np.max(np.abs(new - refs) / np.maximum(np.abs(refs), 1.0)) < 1e-6
    assert abs(fx - float(g["fx_final"])) <= 1e-6 * max(abs(float(g["fx_final"])), 1.0)
    # arg_out feeds Simulation.run / save (simulation.py:266): same keys and shapes as the reference's
    out = vgpa.arg_out
    assert {"m0", "s0", "mt", "st", "Efx", "Edf", "lamt", "psit"} <= set(out)
    vgpa.close()


@pytest.mark.parametrize("model,method,tf", [("OU", "rk4", None), ("L63", "rk2", 2.0), ("L96", "rk2", 0.2)])
def test_single_evaluation_against_live_reference(ref, model, method, tf):
    """Same objects, two VarGP classes: the reference's (numpy / numba, on this box's CPU) and the
    CUDA one, at a dense perturbation of x0."""
    sim, args, vgpa = _swap(ref, mg.config(model, method, tf))
    ref_vgpa = ref["VarGP"](*args)
    x0 = ref_vgpa.initialization()
    assert np.array_equal(x0, vgpa.initialization())
    x = mg.perturb(x0, vgpa.dim_d, vgpa.dim_n, np.random.default_rng([mg.SEED, 11]))
    F_ref = ref_vgpa.free_energy(x)
    g_ref = ref_vgpa.gradient(x)
    F = vgpa.free_energy(x)
    gr = vgpa.gradient(x)
    assert abs(F - F_ref) <= 1e-9 * abs(F_ref)
    na = vgpa.dim_n * vgpa.dim_d * vgpa.dim_d
    assert rel_err(gr[:na], g_ref[:na]) < 1e-9 and rel_err(gr[na:], g_ref[na:]) < 1e-9
    for k in ("mt", "st", "lamt", "psit"):
        assert rel_err(vgpa.arg_out[k], ref_vgpa.arg_out[k]) < 1e-9, k
    vgpa.close()


@pytest.mark.parametrize("model,method,tf", [("OU", "rk4", None), ("L63", "rk2", 2.0), ("L96", "rk2", 0.2)])
def test_single_evaluation_against_recorded_reference(model, method, tf):
    """The check above where the reference tree is absent: the CUDA VarGP, set up by this package's own
    Simulation, at the evaluation point of tests/golden/eval_<model>_<method>.npz, against what the
    reference's VarGP returned there."""
    from vgpa_b200 import Simulation
    g = np.load(GOLDEN / f"eval_{model}_{method}.npz")
    sim = Simulation("t")
    sim.setup(mg.config(model, method, tf))
    vgpa = sim.build()
    assert np.array_equal(vgpa.initialization(), g["x0"])
    F = vgpa.free_energy(g["x"])
    gr = vgpa.gradient(g["x"])
    assert abs(F - float(g["F"])) <= 1e-9 * abs(float(g["F"]))
    na = vgpa.dim_n * vgpa.dim_d * vgpa.dim_d
    assert rel_err(gr[:na], g["grad"][:na]) < 1e-9 and rel_err(gr[na:], g["grad"][na:]) < 1e-9
    for k in ("mt", "st", "lamt", "psit"):
        assert rel_err(vgpa.arg_out[k], g[k]) < 1e-9, k
    vgpa.close()
