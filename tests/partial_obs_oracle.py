"""
The CPU reference for partially observed problems (vgpa_create_observed): the oracle's evaluation with an observation
operator that selects the components set in a bit word.  TEST INFRASTRUCTURE ONLY.

The pinned oracle (oracle/vgpa_oracle.c) evaluates the identity operator.  This module composes its exported stages --
oracle_fwd, oracle_energy, oracle_bwd, oracle_gradient, oracle_initialization -- unchanged, and restates only what the
mask changes, in the oracle's own loop order and operations (it is built without FMA contraction, so a Python loop of
IEEE double operations reproduces its bits):

  Eobs  = 1/2 [ sum_n sum_{i in O} ((y_ni - m_i(t_n))^2 / R_i + S_ii[n] / R_i) + M (D_o log 2pi + sum_{i in O} log R_i) ]
  jumps   -(y_ni - m_i(t_n)) / R_i and 0.5 / R_i at t_n for i in O, 0 otherwise
  x0      the oracle's spline for observed components; b0(t)_i = a_ii m0_i for unobserved ones (A0 unchanged)

With every bit set the result is the oracle's, bit for bit (tests/test_partial_obs_cpu.py).  Unobserved columns of
obs_y and entries of R are never read.
"""
import ctypes as C
import math
from dataclasses import replace

import numpy as np

LOG2PI = 1.8378770664093453      # gaussian_like.py:12, as in the oracle
_dp = C.POINTER(C.c_double)


def _p(a):
    return a.ctypes.data_as(_dp)


def _seen(word, i):
    return (int(word) >> i) & 1


class PartialObsOracle:
    def __init__(self, oracle):
        self.o = oracle
        L = oracle.lib
        L.oracle_gradient.restype = None
        L.oracle_gradient.argtypes = L.oracle_bwd.argtypes[:1] + [_dp] * 8

    @staticmethod
    def _clean(prob, word):
        """The problem with every unobserved entry of obs_y and R replaced by a finite placeholder (never read)."""
        D = prob.D
        seen = np.array([_seen(word, i) for i in range(D)], dtype=bool)
        y = np.where(seen, np.asarray(prob.obs_y, dtype=float).reshape(-1, D), 0.0)
        R = np.where(seen, np.atleast_1d(np.asarray(prob.R, dtype=float)), 1.0)
        return replace(prob, obs_y=y, R=R, _keep=[])

    def eobs(self, prob, word, mt, st):
        D, M = prob.D, len(prob.obs_t)
        R = np.atleast_1d(np.asarray(prob.R, dtype=float)).tolist()
        y = np.asarray(prob.obs_y, dtype=float).reshape(-1, D)
        mt, st = np.asarray(mt, dtype=float).reshape(-1, D), np.asarray(st, dtype=float).reshape(-1, D, D)
        if D == 1:                                         # one component: always observed
            cp = prob.c_struct()
            m1, s1 = np.ascontiguousarray(mt.ravel()), np.ascontiguousarray(st.ravel())
            self.o.lib.oracle_eobs.restype = C.c_double
            return self.o.lib.oracle_eobs(C.byref(cp), _p(m1), _p(s1))
        obs = [i for i in range(D) if _seen(word, i)]
        logdet = 0.0
        for i in obs:
            logdet += math.log(math.sqrt(R[i]))
        logdet *= 2.0
        e = 0.0
        for n in range(M):
            t = int(prob.obs_t[n])
            zz, tr = 0.0, 0.0
            for i in obs:
                zi = (float(y[n, i]) - float(mt[t, i])) / math.sqrt(R[i])
                zz += zi * zi
                tr += (1.0 / R[i]) * float(st[n, i, i])     # S indexed by the ordinal n (F5)
            e += zz + tr
        return 0.5 * (e + M * (len(obs) * LOG2PI + logdet))

    def jumps(self, prob, word, mt):
        D, N = prob.D, prob.N
        R = np.atleast_1d(np.asarray(prob.R, dtype=float))
        y = np.asarray(prob.obs_y, dtype=float).reshape(-1, D)
        mt = np.asarray(mt, dtype=float).reshape(N, D)
        jm, js = np.zeros((N, D)), np.zeros((N, D, D))
        for n, t in enumerate(np.asarray(prob.obs_t, dtype=np.int64)):
            for i in range(D):
                if _seen(word, i):
                    jm[t, i] = -(y[n, i] - mt[t, i]) / R[i]
                    js[t, i, i] = 0.5 / R[i]
        return jm, js

    def eval(self, prob, word, x, want_grad=True, full=False):
        """F and the gradient (full=True: a dict with parts and every trajectory) of the masked problem."""
        L = self.o.lib
        D, N = prob.D, prob.N
        nv, nm = N * D, N * D * D
        x = np.ascontiguousarray(x, dtype=np.float64)
        cp = self._clean(prob, word).c_struct()
        mt, st = np.empty(nv), np.empty(nm)
        Ef, Edf, dEm, dEs, esde_t = np.empty(nv), np.empty(nm), np.empty(nv), np.empty(nm), np.empty(N)
        Esde = np.zeros(1)
        self.o._raise(L.oracle_fwd(C.byref(cp), _p(x), _p(mt), _p(st)))
        Eobs = self.eobs(prob, word, mt, st)
        self.o._raise(L.oracle_energy(C.byref(cp), _p(x), _p(mt), _p(st), _p(Esde), _p(esde_t), _p(Ef), _p(Edf),
                                      _p(dEm), _p(dEs)))
        jm, js = self.jumps(prob, word, mt)
        lam, psi = np.empty(nv), np.empty(nm)
        self.o._raise(L.oracle_bwd(C.byref(cp), _p(x), _p(dEm), _p(dEs), _p(jm), _p(js), _p(lam), _p(psi)))
        F = prob.E0 + float(Esde[0]) + Eobs
        grad = None
        if want_grad or full:
            grad = np.empty(x.size)
            L.oracle_gradient(C.byref(cp), _p(x), _p(mt), _p(st), _p(lam), _p(psi), _p(Ef), _p(Edf), _p(grad))
        if not full:
            return F, grad
        return {"F": F, "E0": prob.E0, "Esde": float(Esde[0]), "Eobs": Eobs, "grad": grad,
                "mt": mt.reshape(N, D), "st": st.reshape(N, D, D), "lamt": lam.reshape(N, D),
                "psit": psi.reshape(N, D, D)}

    def initialization(self, prob, word, t0=0.0):
        """VarGP.initialization with the unobserved components on the constant mean path m0."""
        D, N = prob.D, prob.N
        x0 = self.o.initialization(self._clean(prob, word), t0)
        b0 = x0[N * D * D:].reshape(N, D)
        m0 = np.atleast_1d(np.asarray(prob.m0, dtype=float))
        sigma = np.atleast_1d(np.asarray(prob.sigma, dtype=float))
        for i in range(D):
            if not _seen(word, i):
                b0[:, i] = 0.5 * (sigma[i] / 0.25) * m0[i]
        return x0
