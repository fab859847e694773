"""
Partially observed problems (vgpa_create_observed, vgpa_obs_energy_observed, BatchEvaluator(observed=...),
GaussianLikelihood(operator=...)) without a device: the header declares both calls and the library exports them, every
argument error is raised before CUDA is touched and names what it is about, and the masked CPU reference
(partial_obs_oracle.py) agrees with the pinned oracle: bit for bit with every component observed, and through the
large-R limit otherwise (an unobserved component is a component observed with infinite noise).
"""
import ctypes as C
import re

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, grad_err
from oracle import Problem
from partial_obs_oracle import PartialObsOracle


def test_header_declares_and_library_exports_the_observed_calls():
    header = (ROOT / "include" / "vgpa_b200.h").read_text()
    assert re.search(r"int vgpa_create_observed\(const vgpa_desc \*desc, const int64_t \*obs_t, int64_t obs_t_stride,"
                     r"\s*const int32_t \*M,\s*const uint64_t \*observed, int64_t observed_stride, vgpa_handle \*\*out\);",
                     header)
    assert re.search(r"int vgpa_obs_energy_observed\(int device, int D, int N, int M, const int64_t \*obs_t,"
                     r"\s*const double \*obs_y,\s*const double \*R, uint64_t observed, const double \*mt,"
                     r"\s*const double \*st,\s*double \*Eobs, double \*jm, double \*js\);", header)
    lib = C.CDLL(str(ROOT / "vgpa_b200" / "libvgpa_b200.so"))
    assert hasattr(lib, "vgpa_create_observed") and hasattr(lib, "vgpa_obs_energy_observed")


def _c_create(model, D, words, stride, B=3, N=11, obs_t=(3, 6)):
    """vgpa_create_observed on a small descriptor with one shared schedule; returns (rc, message)."""
    from vgpa_b200._lib import VgpaDesc, lib
    keep = []

    def arr(a, t=np.float64):
        a = np.ascontiguousarray(a, dtype=t)
        keep.append(a)
        return a

    M = len(obs_t)
    d = VgpaDesc()
    d.model, d.method, d.D, d.N, d.M, d.B, d.device = model, 3, D, N, M, B, 0
    d.dt = d.dt_model = 0.01
    nth = 3 if model == 2 else 1
    for name, val in (("theta", np.ones(nth)), ("sigma", np.ones(D)), ("R", np.ones(D)), ("m0", np.zeros(D)),
                      ("s0", np.eye(D)), ("E0", [0.0]), ("obs_y", np.zeros(M * D))):
        setattr(d, name, arr(val).ctypes.data_as(C.POINTER(C.c_double)))
        setattr(d, name + "_stride", 0)
    ot = arr(obs_t, np.int64)
    w = None if words is None else arr(words, np.uint64)
    h = C.c_void_p()
    rc = lib.vgpa_create_observed(C.byref(d), ot.ctypes.data, 0, None, None if w is None else w.ctypes.data, stride,
                                  C.byref(h))
    msg = lib.vgpa_last_error(None).decode()
    if h.value:              # a device is present and the arguments were valid
        lib.vgpa_destroy(h)
    return rc, msg


@pytest.mark.parametrize("model,D,words,stride,match", [
    (2, 3, [0b101, 0, 0b010], 1, "mask of problem 1 has no bit set"),
    (2, 3, [0b101, 0b011, 0b1000], 1, "mask of problem 2 has a bit at or above D = 3"),
    (2, 3, [0], 0, "mask of problem 0 has no bit set"),
    (1, 1, [0b10], 0, "mask of problem 0 has a bit at or above D = 1"),           # D = 1 with bit 0 clear
    (1, 1, [0b11, 0b1, 0b1], 1, "mask of problem 0 has a bit at or above D = 1"),
    (2, 3, [0b101], -1, "observed_stride -1"),
    (3, 12, [1 << 11, 1 << 12, 1], 1, "mask of problem 1 has a bit at or above D = 12"),
    (2, 3, [0b101, 0b011, 0b111], 1, None),
    (2, 3, [0b001], 0, None),
    (3, 64, [1 << 63, 1, 1], 1, None),                                          # bit 63 is a component at D = 64
])
def test_create_observed_validates_before_touching_the_device(model, D, words, stride, match):
    rc, msg = _c_create(model, D, words, stride)
    if match is None:        # valid masks: what fails next is the device (none here) or nothing
        assert rc in (0, 3), (rc, msg)
        assert rc == 0 or "mask" not in msg
    else:
        assert rc == 1, (rc, msg)
        assert re.search(match, msg), msg


@pytest.mark.parametrize("D,word,match", [(3, 0, "no bit set"), (3, 0b1000, "at or above D = 3"),
                                          (1, 0b10, "at or above D = 1")])
def test_obs_energy_observed_validates_the_mask(D, word, match):
    from vgpa_b200._lib import lib
    N, M = 5, 1
    ot = np.array([2], dtype=np.int64)
    oy, R, mt, st = np.zeros(M * D), np.ones(D), np.zeros(N * D), np.zeros(N * D * D)
    E, jm, js = np.zeros(1), np.zeros(N * D), np.zeros(N * D * D)
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    rc = lib.vgpa_obs_energy_observed(0, D, N, M, ot.ctypes.data_as(C.POINTER(C.c_int64)), p(oy), p(R), word, p(mt),
                                      p(st), p(E), p(jm), p(js))
    assert rc == 1
    assert re.search(match, lib.vgpa_last_error(None).decode())


def _l63_kw(B=2):
    return dict(model="L63", method="rk2", N=11, dt=0.01, theta=[10.0, 28.0, 8 / 3], sigma=np.ones(3), R=np.ones(3),
                obs_t=[3, 6], obs_y=np.zeros((2, 3)), m0=np.zeros(3), s0=np.eye(3), E0=0.0, B=B)


@pytest.mark.parametrize("observed,match", [
    ([0, 0], "duplicate component index"),
    ([0, 3], "out of range"),
    ([-1], "out of range"),
    ([], "no component is observed"),
    (np.array([True, False]), "bool mask needs 3 entries"),
    (np.zeros(3, dtype=bool), "no component is observed"),
    ([[0], [1], [2]], "expected 2 per-problem masks"),
    ([[0], [1, 1]], "observed of problem 1: duplicate"),
    ([[0], []], "observed of problem 1: no component"),
    (np.ones((2, 4), dtype=bool), "observed of problem 0: a bool mask needs 3"),
    ([0.0, 1.0], "must be integers"),
])
def test_batch_evaluator_rejects_bad_masks(observed, match):
    from vgpa_b200.engine import BatchEvaluator
    with pytest.raises(ValueError, match=match):
        BatchEvaluator(observed=observed, **_l63_kw())


def test_mask_forms_give_the_same_words():
    from vgpa_b200.engine import observed_words
    assert observed_words([2, 0], 4, 3)[1] == 0 and int(observed_words([2, 0], 4, 3)[0][0]) == 0b101
    assert int(observed_words(np.array([True, False, True]), 4, 3)[0][0]) == 0b101
    w, s = observed_words([[0], [1, 2], [2], [0, 1, 2]], 4, 3)
    assert s == 1 and w.tolist() == [1, 6, 4, 7]
    w2, _ = observed_words(np.array([[1, 0, 0], [0, 1, 1], [0, 0, 1], [1, 1, 1]], dtype=bool), 4, 3)
    assert w2.tolist() == w.tolist()
    assert int(observed_words([63], 1, 64)[0][0]) == 1 << 63


@pytest.mark.parametrize("kw,match", [
    (dict(values=np.zeros((4, 2)), noise=np.eye(2), operator=[0, 0]), "duplicate component"),
    (dict(values=np.zeros((4, 2)), noise=np.eye(2), operator=[0, -1]), "non-negative component indices"),
    (dict(values=np.zeros((4, 3)), noise=np.eye(2), operator=[0, 2]), "values of shape \\(4, 3\\)"),
    (dict(values=np.zeros((4, 2)), noise=np.eye(3), operator=[0, 2]), "noise of shape \\(3, 3\\)"),
    (dict(values=np.zeros((4, 2)), noise=np.ones(3), operator=[0, 2]), "noise of shape \\(3,\\)"),
    (dict(values=np.zeros((4, 2)), noise=np.eye(2), operator=[[1, 0, 0], [0, 0, 2]]), "rows of the identity"),
    (dict(values=np.zeros((4, 2)), noise=np.eye(2), operator=[[1, 0, 0], [1, 0, 0]]), "duplicate component"),
    (dict(values=np.zeros((4, 2)), noise=np.eye(2), operator=[[0.5, 0.5, 0], [0, 0, 1]]), "rows of the identity"),
    (dict(values=np.zeros((4, 2)), noise=np.eye(2), operator=np.zeros((2, 2, 2))), "unsupported observation operator"),
])
def test_likelihood_rejects_what_is_not_a_selection(kw, match):
    from vgpa_b200.likelihood import GaussianLikelihood
    with pytest.raises(ValueError, match=match):
        GaussianLikelihood(times=np.arange(4), single_dim=False, **kw)


def test_likelihood_places_the_observations_in_operator_order():
    from vgpa_b200.likelihood import GaussianLikelihood
    y = np.arange(8.0).reshape(4, 2)
    for op in ([2, 0], [[0, 0, 1], [1, 0, 0]]):
        lik = GaussianLikelihood(y, np.arange(4), np.diag([3.0, 5.0]), op, single_dim=False)
        yf, R, cols = lik.on_state(3)
        assert cols == [2, 0]
        assert np.array_equal(yf[:, 2], y[:, 0]) and np.array_equal(yf[:, 0], y[:, 1]) and not yf[:, 1].any()
        assert R[2] == 3.0 and R[0] == 5.0
    with pytest.raises(ValueError, match="selects component 4"):
        GaussianLikelihood(y, np.arange(4), np.diag([3.0, 5.0]), [4, 0], single_dim=False).on_state(3)
    ident = GaussianLikelihood(np.zeros((4, 3)), np.arange(4), np.eye(3), np.eye(3), single_dim=False)
    assert ident.on_state(3)[2] is None


# ---- the masked CPU reference against the pinned oracle ------------------------------------------------------------
@pytest.fixture(scope="module")
def masked(oracle):
    return PartialObsOracle(oracle)


def _golden_problem(name):
    g = np.load(GOLDEN / f"eval_{name}.npz")
    return Problem.from_golden(g), g["x"]


def _with(prob, **kw):
    d = {k: getattr(prob, k) for k in ("model", "method", "D", "N", "dt", "theta", "sigma", "R", "obs_t", "obs_y",
                                       "m0", "s0", "E0", "dt_model")}
    d.update(kw)
    return Problem(**d)


def _masks(D):
    rng = np.random.default_rng(D)
    return {"one": 1 << (D // 2), "all_but_one": ((1 << D) - 1) & ~(1 << 1), "alternating": sum(1 << i for i in range(0, D, 2)),
            "random": int(sum(1 << int(i) for i in rng.choice(D, D // 3, replace=False)))}


@pytest.mark.parametrize("name", ["L63_rk2", "L63_euler", "L96_rk4", "OU_rk4"])
def test_full_mask_is_the_oracle_bit_for_bit(oracle, masked, name):
    prob, x = _golden_problem(name)
    word = (1 << prob.D) - 1
    a, b = oracle.eval(prob, x, full=True), masked.eval(prob, word, x, full=True)
    for k in ("F", "Eobs", "grad", "lamt", "psit"):
        assert np.array_equal(np.asarray(a[k]).ravel(), np.asarray(b[k]).ravel()), k
    assert np.array_equal(oracle.initialization(prob), masked.initialization(prob, word))


@pytest.mark.parametrize("name", ["L63_rk2", "L63_rk4", "L96_rk2"])
@pytest.mark.parametrize("kind", ["one", "all_but_one", "alternating", "random"])
def test_mask_is_the_large_noise_limit_of_the_oracle(oracle, masked, name, kind):
    """The masked problem against the oracle's identity problem with R_i = 1e100 off the mask: every gradient block
    to 1e-12, and F once the count term of the unobserved components is added."""
    prob, x = _golden_problem(name)
    D, M = prob.D, len(prob.obs_t)
    word = _masks(D)[kind]
    hidden = np.array([i for i in range(D) if not (word >> i) & 1])
    R_big = np.array(prob.R, dtype=float).copy()
    R_big[hidden] = 1e100
    Fm, gm = masked.eval(prob, word, x)
    Fu, gu = oracle.eval(_with(prob, R=R_big), x)
    assert grad_err(gm, gu, prob.N, D) < 1e-12
    count = 0.5 * M * np.sum(np.log(2 * np.pi) + np.log(R_big[hidden]))
    assert abs(Fm + count - Fu) <= 1e-12 * abs(Fu)


def test_masked_reference_ignores_unobserved_inputs_and_initialises_them_with_m0(oracle, masked):
    prob, x = _golden_problem("L63_rk2")
    word = 0b101
    clean = _with(prob, obs_y=np.where([1, 0, 1], prob.obs_y, 0.0), R=np.where([1, 0, 1], prob.R, 0.0))
    nan = _with(prob, obs_y=np.where([1, 0, 1], prob.obs_y, np.nan), R=np.where([1, 0, 1], prob.R, np.nan))
    a, b = masked.eval(clean, word, x, full=True), masked.eval(nan, word, x, full=True)
    for k in ("F", "grad", "lamt", "psit"):
        assert np.array_equal(a[k], b[k]), k
    x0, x0_full = masked.initialization(nan, word), oracle.initialization(prob)
    N, D = prob.N, prob.D
    b0, b0_full = x0[N * D * D:].reshape(N, D), x0_full[N * D * D:].reshape(N, D)
    assert np.array_equal(x0[:N * D * D], x0_full[:N * D * D])
    assert np.array_equal(b0[:, [0, 2]], b0_full[:, [0, 2]])
    assert np.array_equal(b0[:, 1], 0.5 * (prob.sigma[1] / 0.25) * np.full(N, prob.m0[1]))
