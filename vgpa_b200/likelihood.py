"""
GaussianLikelihood (src/var_bayes/likelihood.py:13-100 + gaussian_like.py:14-243):
holds the observations and evaluates Eobs and its jump tables ON THE GPU
(vgpa_obs_energy, vgpa_obs_energy_observed).  Diagonal noise, and an observation
operator that selects state components -- the identity, or the sim_params JSON's
list of observed components (Observations.operator, the reference's h_mask) --
as the sim_params JSON schema produces them.
"""
import numpy as np

from . import engine


def _selected_columns(h):
    """The components a non-identity operator selects, in its row order: h is a 1-D list of distinct component
    indices, or a D_o x D matrix whose rows are distinct rows of the identity.  Anything else raises ValueError."""
    if h.ndim == 1:
        if h.size == 0 or not np.issubdtype(h.dtype, np.integer) or np.any(h < 0):
            raise ValueError(f" GaussianLikelihood: the operator list must hold non-negative component indices, got {h.tolist()}")
        cols = h.astype(np.int64)
    elif h.ndim == 2:
        cols = np.argmax(h, axis=1) if h.shape[1] else np.zeros(0, dtype=np.int64)
        sel = np.zeros(h.shape)
        sel[np.arange(h.shape[0]), cols] = 1.0
        if h.shape[0] == 0 or h.shape[0] > h.shape[1] or np.any(h != sel):
            raise ValueError(" GaussianLikelihood: the CUDA path supports an observation operator that selects state"
                             " components only (rows of the identity).")
    else:
        raise ValueError(f" GaussianLikelihood: unsupported observation operator of shape {h.shape}.")
    if np.unique(cols).size != cols.size:
        raise ValueError(f" GaussianLikelihood: duplicate component in the observation operator {cols.tolist()}")
    return cols


class GaussianLikelihood(object):
    __slots__ = ("obs_v", "obs_t", "obs_n", "obs_h", "obs_cols", "single_dim", "device")

    def __init__(self, values, times, noise, operator=None, single_dim=True, device=0):
        self.obs_t = np.asarray(times)
        self.obs_v = np.asarray(values)
        self.obs_n = np.asarray(noise)
        self.obs_cols = None                  # None: the identity; else the observed components, in operator order
        if operator is None:
            y0 = self.obs_v[0]
            self.obs_h = np.asarray(1) if y0.ndim == 0 else np.eye(y0.size)
        else:
            self.obs_h = np.asarray(operator)
            eye = np.asarray(1) if self.obs_h.ndim == 0 else np.eye(self.obs_h.shape[0])
            if self.obs_h.shape != eye.shape or np.any(self.obs_h != eye):
                self.obs_cols = _selected_columns(self.obs_h)
                Do, M = self.obs_cols.size, self.obs_t.size
                if self.obs_v.size != M * Do or (self.obs_v.ndim == 2 and self.obs_v.shape != (M, Do)):
                    raise ValueError(f" GaussianLikelihood: values of shape {self.obs_v.shape} do not match the"
                                     f" operator: expected ({M}, {Do})")
                if not (self.obs_n.size == Do or self.obs_n.shape == (Do, Do)):
                    raise ValueError(f" GaussianLikelihood: noise of shape {self.obs_n.shape} does not match the"
                                     f" operator: expected {Do} values or {Do} x {Do}")
        self.single_dim = single_dim
        self.device = device

    values = property(lambda self: self.obs_v)
    times = property(lambda self: self.obs_t)
    operator = property(lambda self: self.obs_h)

    @property
    def noise(self):
        return self.obs_n

    @noise.setter
    def noise(self, new_value):
        self.obs_n = new_value

    def noise_diag(self):
        r = np.asarray(self.obs_n, dtype=float)
        if r.ndim == 2:
            if np.count_nonzero(r - np.diag(np.diagonal(r))):
                raise ValueError(" GaussianLikelihood: the CUDA path supports a diagonal"
                                 " observation noise only.")
            return np.diagonal(r).copy()
        return np.atleast_1d(r)

    def on_state(self, D):
        """The observations in the state's D columns: (obs_y (M, D), R (D,), observed) where observed is None
        for the identity operator, else the list of observed components; the values of the other columns
        are placeholders that are never read (zeros, and ones for R).  ValueError when the operator selects a
        component outside [0, D)."""
        R = self.noise_diag()
        if self.obs_cols is None:
            return self.obs_v, R, None
        cols = self.obs_cols
        if cols.max() >= D:
            raise ValueError(f" GaussianLikelihood: the operator selects component {int(cols.max())}, the state has {D}")
        M = self.obs_t.size
        y = np.zeros((M, D))
        y[:, cols] = np.asarray(self.obs_v, dtype=float).reshape(M, cols.size)
        r = np.ones(D)
        r[cols] = np.broadcast_to(R, cols.shape)
        return (y.reshape(-1) if D == 1 else y), r, cols.tolist()

    def _energy(self, m, s, with_dr):
        m = np.asarray(m, dtype=float)
        y, R, cols = self.on_state(1 if m.ndim == 1 else m.shape[1])
        if cols is not None and m.ndim == 1:      # the one component of a 1-D state: the identity
            cols = None
        word = None if cols is None else sum(1 << c for c in cols)
        return engine.obs_energy(self.obs_t, y, R, m, s, self.device, with_dr=with_dr and word is None,
                                 observed=word)

    def __call__(self, m, s):
        """Eobs (gaussian_like.py:69-153)."""
        return self._energy(m, s, False)[0]

    def gradients(self, m, s=None):
        """dEobs_dm, dEobs_ds, dEobs_dr (gaussian_like.py:155-243), as (N, D) and (N, D, D) tables over the
        state's components (zero at unobserved ones).  As in the reference, the 1-D dEobs_dr needs the marginal
        variances s; the n-D one is all zeros of shape (N, M, M)."""
        m = np.asarray(m, dtype=float)
        if s is None:
            s = np.zeros(m.shape + (() if m.ndim == 1 else (m.shape[1],)))
        out = self._energy(m, s, True)
        if len(out) == 4:
            return out[1], out[2], out[3]
        M = self.obs_t.size
        return out[1], out[2], np.zeros((m.shape[0], M, M))
