"""CPU checks of Lorenz 96 at state dimensions other than 40: the library exports the run-time-D data-generation
calls and the header declares them; the Python layer checks the supported range 10 <= D <= 64 before any device
work; the numpy restatement of Lorenz96.make_trajectory that the GPU tests compare against at other D equals the
oracle's D = 40 data generation (pinned to the reference's goldens) bit for bit."""
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
LIB = ROOT / "vgpa_b200" / "libvgpa_b200.so"
NEW = ("vgpa_make_trajectory_dim", "vgpa_make_trajectory_device_dim")


def test_header_declares_the_dim_calls():
    h = (ROOT / "include" / "vgpa_b200.h").read_text()
    for name in NEW:
        assert re.search(rf"\bint {name}\(int device, int model, int D, int N,", h), name


def test_library_exports_the_dim_calls():
    if not LIB.exists():
        pytest.skip("library not built")
    out = subprocess.run(["nm", "-D", "--defined-only", str(LIB)], capture_output=True, text=True).stdout
    for name in NEW:
        assert re.search(rf"\bT {name}$", out, re.M), name


def test_model_dim_range():
    from vgpa_b200._lib import model_dim
    assert model_dim("L96") == 40 and model_dim("L96", 10) == 10 and model_dim("L96", 64) == 64
    with pytest.raises(ValueError, match="Insufficient"):
        model_dim("L96", 9)
    with pytest.raises(ValueError, match="10 <= dim_d <= 64"):
        model_dim("L96", 65)
    with pytest.raises(ValueError):
        model_dim("L63", 4)


@pytest.mark.parametrize("D", [9, 65])
def test_lorenz96_constructor_range(D):
    from vgpa_b200.dynamics import Lorenz96
    with pytest.raises(ValueError):
        Lorenz96([1.0] * D, 8.0, dim_d=D)


def test_lorenz96_constructor_accepts_d20():
    from vgpa_b200.dynamics import Lorenz96
    assert Lorenz96([1.0] * 20, 8.0, dim_d=20).dim_d == 20


def test_numpy_restatement_equals_oracle_at_d40(oracle):
    from test_gpu_l96_dims import l96_path
    D, N, dt = 40, 120, 0.01
    rng = np.random.default_rng(4)
    z = rng.standard_normal((D, N))
    sig = 0.5 + rng.random(D)
    ref = oracle.make_trajectory("L96", N, dt, [8.3], sig, z)
    got = l96_path(D, N, dt, 8.3, sig, z)
    assert np.array_equal(got.view(np.int64), ref.view(np.int64))
