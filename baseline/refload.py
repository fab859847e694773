"""Import the unmodified reference (vrettasm/VGPA).  It is not part of this repository: it is found in the
checkout named by the environment variable VGPA_REFERENCE, else in baseline/_ref (git-ignored).  The
reference is pure Python (numpy / scipy / numba); h5py is only used by Simulation.save / load
(src/var_bayes/simulation.py:1,293,336) and is stubbed when absent."""
import contextlib
import io
import os
import sys
import types
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF_COPY = HERE / "_ref"


def reference_root():
    env = os.environ.get("VGPA_REFERENCE")
    for cand in ([Path(env)] if env else []) + [REF_COPY]:
        if (cand / "src" / "var_bayes" / "variational.py").exists():
            return cand
    return None


def import_reference():
    """dict of the reference's classes, or ImportError with the reason (missing tree, numba, scipy)."""
    root = reference_root()
    if root is None:
        raise ImportError("the reference tree is missing: set VGPA_REFERENCE to a checkout of vrettasm/VGPA")
    sys.dont_write_bytecode = True
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    try:
        import h5py  # noqa: F401
    except ImportError:
        sys.modules.setdefault("h5py", types.ModuleType("h5py"))
    import numba  # noqa: F401  (ImportError propagates with its own message)
    import scipy  # noqa: F401
    from src.var_bayes.simulation import Simulation
    from src.var_bayes.fwd_ode import FwdOde
    from src.var_bayes.bwd_ode import BwdOde
    from src.var_bayes.gaussian_like import GaussianLikelihood
    from src.var_bayes.prior_kl0 import PriorKL0
    from src.var_bayes.variational import VarGP
    from src.numerics.optim_scg import SCG
    return dict(Simulation=Simulation, FwdOde=FwdOde, BwdOde=BwdOde, GaussianLikelihood=GaussianLikelihood,
                PriorKL0=PriorKL0, VarGP=VarGP, SCG=SCG, root=str(root))


def reference_objects(ref, params, override=None):
    """Simulation.setup (simulation.py:92-176) and the constructor block of Simulation.run
    (simulation.py:189-207) with the reference's own classes: everything VarGP's constructor takes.
    `override`: entries of Simulation.m_data replaced after setup (e.g. obs_y, m0 of an ensemble member)."""
    with contextlib.redirect_stdout(io.StringIO()):
        sim = ref["Simulation"](params.get("Output_Name", "ref"))
        sim.setup(params, None)
    md = sim.m_data
    md.update(override or {})
    dt = md["time_window"]["dt"]
    fwd = ref["FwdOde"](dt, md["ode_solver"], md["single_dim"])
    bwd = ref["BwdOde"](dt, md["ode_solver"], md["single_dim"])
    lik = ref["GaussianLikelihood"](md["obs_y"], md["obs_t"], md["obs_noise"], md["obs_setup"]["operator"],
                                    md["single_dim"])
    kl0 = ref["PriorKL0"](md["mu0"], md["tau0"], md["single_dim"])
    args = (md["model"], md["m0"], md["s0"], fwd, bwd, lik, kl0, md["obs_y"], md["obs_t"])
    return sim, args
