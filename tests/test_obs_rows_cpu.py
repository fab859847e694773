"""
Per-problem observation schedules (vgpa_create_obs_rows, BatchEvaluator with a list of obs_t arrays) without a
device: the header declares the call, the library exports it, and every argument error is raised before CUDA is
touched, naming the problem it is about.
"""
import ctypes as C
import re

import numpy as np
import pytest

from conftest import ROOT


def _base(B=3, N=11, M=2):
    return dict(model="OU", method="rk4", N=N, dt=0.01, theta=[2.0], sigma=[0.8], R=[0.04], m0=[0.0], s0=[[0.2]],
                E0=0.0, B=B)


def test_header_declares_and_library_exports_create_obs_rows():
    header = (ROOT / "include" / "vgpa_b200.h").read_text()
    assert re.search(r"int vgpa_create_obs_rows\(const vgpa_desc \*desc, const int64_t \*obs_t, int64_t obs_t_stride,"
                     r"\s*const int32_t \*M, vgpa_handle \*\*out\);", header)
    lib = C.CDLL(str(ROOT / "vgpa_b200" / "libvgpa_b200.so"))
    assert hasattr(lib, "vgpa_create_obs_rows")


@pytest.mark.parametrize("obs_t,obs_y,match", [
    ([[3, 6], [2], [6, 3]], [np.zeros((2, 1)), np.zeros(1), np.zeros(2)], "problem 2"),
    ([[3, 6], [2, 2], [4]], [np.zeros((2, 1)), np.zeros(2), np.zeros(1)], "problem 1"),
    ([[3, 6], [2], [4, 11]], [np.zeros((2, 1)), np.zeros(1), np.zeros(2)], "problem 2"),
    ([[3, 6], [-1], [4]], [np.zeros((2, 1)), np.zeros(1), np.zeros(1)], "problem 1"),
    ([[3, 6], [2]], [np.zeros(2), np.zeros(1)], "3 per-problem"),
    ([[3, 6], [2], [4]], np.zeros((3, 2, 1)), "obs_y"),
    ([[3, 6], [2], [4]], [np.zeros(2), np.zeros(2), np.zeros(1)], "obs_y of problem 1"),
    ([[3, 6], [[2]], [4]], [np.zeros(2), np.zeros(1), np.zeros(1)], "obs_t of problem 1"),
    ([[3, 6], [2.5], [4]], [np.zeros(2), np.zeros(1), np.zeros(1)], "obs_t of problem 1"),
])
def test_batch_evaluator_rejects_bad_schedules(obs_t, obs_y, match):
    from vgpa_b200.engine import BatchEvaluator
    with pytest.raises(ValueError, match=match):
        BatchEvaluator(obs_t=obs_t, obs_y=obs_y, **_base())


def test_l96_observation_shapes_are_checked_per_problem():
    from vgpa_b200.engine import BatchEvaluator
    D = 12
    kw = dict(model="L96", method="rk2", N=11, dt=0.01, theta=[8.0], sigma=np.ones(D), R=np.ones(D), m0=np.zeros(D),
              s0=np.eye(D), E0=0.0, B=2, D=D)
    with pytest.raises(ValueError, match="obs_y of problem 1"):
        BatchEvaluator(obs_t=[[3], [4, 5]], obs_y=[np.zeros((1, D)), np.zeros(2 * D)], **kw)
    with pytest.raises(ValueError, match="obs_y of problem 0"):       # (M_p,) is accepted for D = 1 only
        BatchEvaluator(obs_t=[[3], [4, 5]], obs_y=[np.zeros(D), np.zeros((2, D))], **kw)


def _c_create(obs_t_desc, rows, stride, counts, B=3, M=2, N=11):
    """vgpa_create_obs_rows on an OU descriptor; returns (rc, message)."""
    from vgpa_b200._lib import VgpaDesc, lib
    keep = []

    def arr(a, t=np.float64):
        a = np.ascontiguousarray(a, dtype=t)
        keep.append(a)
        return a

    d = VgpaDesc()
    d.model, d.method, d.D, d.N, d.M, d.B, d.device = 1, 3, 1, N, M, B, 0
    d.dt = d.dt_model = 0.01
    for name, val in (("theta", [2.0]), ("sigma", [0.8]), ("R", [0.04]), ("m0", [0.0]), ("s0", [0.2]), ("E0", [0.0]),
                      ("obs_y", np.zeros(max(M, 1)))):
        setattr(d, name, arr(val).ctypes.data_as(C.POINTER(C.c_double)))
        setattr(d, name + "_stride", 0)
    if obs_t_desc is not None:
        d.obs_t = arr(obs_t_desc, np.int64).ctypes.data_as(C.POINTER(C.c_int64))
    r = None if rows is None else arr(rows, np.int64)
    c = None if counts is None else arr(counts, np.int32)
    h = C.c_void_p()
    rc = lib.vgpa_create_obs_rows(C.byref(d), None if r is None else r.ctypes.data, stride,
                                  None if c is None else c.ctypes.data, C.byref(h))
    lib.vgpa_last_error.restype = C.c_char_p
    msg = lib.vgpa_last_error(None).decode()
    if h.value:              # a device is present and the schedules were valid
        lib.vgpa_destroy(h)
    return rc, msg


@pytest.mark.parametrize("desc_t,rows,stride,counts,match", [
    ([3, 6], [3, 6, 2, 5, 4, 7], 2, None, "desc->obs_t must be NULL"),
    (None, [3, 6, 2, 5, 4, 7], 1, None, "obs_t_stride 1"),
    (None, [3, 6, 2, 5, 4, 7], -2, None, "obs_t_stride -2"),
    (None, [3, 6, 2, 5, 4, 7], 2, [2, -1, 1], "M of problem 1 is -1"),
    (None, [3, 6, 2, 5, 4, 7], 2, [2, 1, 3], "M of problem 2 is 3"),
    (None, [3, 6, 2, 5, 7, 4], 2, None, "obs_t of problem 2 must be sorted unique"),
    (None, [3, 6, 2, 5, 7, 4], 2, [2, 2, 1], None),          # problem 2 uses its first index only: valid
    (None, [3, 6, 2, 11, 4, 7], 2, [2, 1, 2], None),         # index 11 lies beyond problem 1's count
    (None, [3, 6, 2, 11, 4, 7], 2, None, "obs_t of problem 1 must be sorted unique indices in \\[0, N\\)"),
    (None, [6, 3], 0, [1, 2, 1], "obs_t of problem 1"),     # one shared row: problem 1 takes both entries
    (None, None, 2, None, "obs_t is NULL"),
])
def test_create_obs_rows_validates_before_touching_the_device(desc_t, rows, stride, counts, match):
    rc, msg = _c_create(desc_t, rows, stride, counts)
    if match is None:    # the schedules pass validation: what fails next is the device (none here) or nothing
        assert rc in (0, 3), (rc, msg)
        assert rc == 0 or "problem" not in msg
    else:
        assert rc == 1, (rc, msg)
        assert re.search(match, msg), msg
