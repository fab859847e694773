"""
Host-side mirror of the reference's StochasticProcess family
(src/dynamics/stochastic_process.py, double_well.py, ornstein_uhlenbeck.py,
lorenz_63.py, lorenz_96.py): same constructor signatures `(sigma, theta, r_seed)`,
same properties (`sigma`, `theta`, `inverse_sigma`, `single_dim`, `sample_path`,
`time_window`, `time_step`, `rng`), same `make_trajectory` / `collect_obs`
random streams, and `energy(A, b, m, S, obs_t)` with the reference's return
structure -- but `energy` runs on the GPU (vgpa_model_energy), never on the CPU.

The data-generation methods consume the numpy Generator exactly as the reference
does, so that the same seed gives the same trajectory, observations and initial
moments.  By default their arithmetic is plain numpy (set-up code must run without a
GPU); with `device=<int>` the Euler-Maruyama loop / the observation noise run on the
GPU (vgpa_make_trajectory, vgpa_collect_obs: the single-path view of the batched
generators ensembles use, engine.make_trajectories / collect_observations) and give
the same values (tests/test_gpu_datagen.py).
"""
import numpy as np
from numpy.random import SeedSequence, default_rng

from . import engine
from ._lib import L96_DIMS


class StochasticProcess(object):
    """stochastic_process.py:5-230"""

    model_key = None

    def __init__(self, r_seed=None, single_dim=True):
        # stochastic_process.py:21-25
        self.rand_g = default_rng(SeedSequence(r_seed)) if r_seed else default_rng()
        self.single_dimension = single_dim
        self.xt = None
        self.tk = None

    @property
    def single_dim(self):
        return self.single_dimension

    @property
    def sample_path(self):
        if self.xt is None:
            raise NotImplementedError(f" {self.__class__.__name__}: Sample path has not been created.")
        return self.xt

    @sample_path.setter
    def sample_path(self, new_value):
        self.xt = new_value

    @property
    def time_window(self):
        if self.tk is None:
            raise NotImplementedError(f" {self.__class__.__name__}: Time window has not been created yet.")
        return self.tk

    @time_window.setter
    def time_window(self, new_value):
        self.tk = new_value

    @property
    def time_step(self):
        if self.tk is None:
            raise NotImplementedError(f" {self.__class__.__name__}: Time window has not been created yet.")
        return np.abs(self.tk[1] - self.tk[0])

    @property
    def rng(self):
        return self.rand_g

    def collect_obs(self, n_obs, rn, h_mask=None, device=None):
        """stochastic_process.py:130-230: equidistant noisy observations."""
        if self.tk is None or self.xt is None:
            raise NotImplementedError(f" {self.__class__.__name__}:"
                                      f" Sample path (or time window) have not been created.")
        rn = np.asarray(rn)
        dt = np.diff(self.tk)[0]
        if n_obs > int(1.0 / dt):
            raise ValueError(f" {self.__class__.__name__}:"
                             f" Observation density exceeds the number of samples.")
        dim_m = int(np.floor(np.abs(self.tk[0] - self.tk[-1]) * n_obs))
        dim_t = self.tk.size
        idx = np.linspace(0, dim_t, dim_m + 2, dtype=int)
        obs_t = sorted(np.unique(idx[1:-1]))
        obs_y = np.take(self.xt, obs_t, axis=0)
        if h_mask:
            obs_y = obs_y[:, h_mask]
        dim_d = 1 if obs_y.ndim == 1 else obs_y.shape[-1]
        if dim_d == 1:
            obs_noise = rn
            xi = self.rand_g.standard_normal(dim_m)
            if device is not None and not h_mask:
                return obs_t, engine.collect_observations(self.xt, obs_t, [float(rn)], xi[None], device)[0], obs_noise
            # one observed component of an n-D path (h_mask of length 1): obs_y is (M, 1), one draw per observation
            obs_y += (np.sqrt(obs_noise) * xi).reshape(obs_y.shape)
        else:
            obs_noise = np.diag(rn) if rn.ndim == 1 else rn * np.eye(dim_d)
            sq_rn = np.sqrt(obs_noise)
            xi = self.rand_g.standard_normal((dim_d, dim_m))
            if device is not None and not h_mask:
                return obs_t, engine.collect_observations(self.xt, obs_t, np.diagonal(obs_noise), xi[None],
                                                          device)[0], obs_noise
            obs_y += sq_rn.dot(xi).T
        return obs_t, obs_y, obs_noise

    # -- the GPU stage ---------------------------------------------------------
    def _sigma_diag(self):
        s = np.asarray(self.sigma, dtype=float)
        if s.ndim == 2:
            if np.count_nonzero(s - np.diag(np.diagonal(s))):
                raise ValueError(f" {self.__class__.__name__}: the CUDA path supports a diagonal"
                                 f" system noise only (what the sim_params JSON can express).")
            return np.diagonal(s).copy()
        return np.atleast_1d(s)

    def energy(self, linear_a, offset_b, m, s, obs_t):
        """model.energy: returns Esde, (Ef, Edf), (dEsde_dm, dEsde_ds, dEsde_dtheta, dEsde_dsigma),
        all computed on the GPU.  (VarGP's hot path does not come through here: it never needs the
        two hyper-parameter gradients, which the reference computes and discards, variational.py:175.)"""
        Esde, Ef, Edf, dm, ds, dth, dsig = engine.model_energy(self.model_key, self.theta, self._sigma_diag(),
                                                               linear_a, offset_b, m, s, float(self.time_step),
                                                               hyper=True)
        return Esde, (Ef, Edf), (dm, ds, dth, dsig)


class _Scalar1D(StochasticProcess):
    """Shared constructor/property logic of the two 1-D models."""

    def __init__(self, sigma, theta, r_seed=None):
        super().__init__(r_seed, single_dim=True)
        if sigma <= 0.0:
            raise ValueError(f" {self.__class__.__name__}: The diffusion noise value: {sigma},"
                             f" should be strictly positive.")
        self._sigma = sigma
        self.sig_inv = 1.0 / sigma
        self._theta = theta

    @property
    def theta(self):
        return self._theta

    @theta.setter
    def theta(self, new_value):
        self._theta = new_value

    @property
    def sigma(self):
        return self._sigma

    @sigma.setter
    def sigma(self, new_value):
        if new_value <= 0.0:
            raise ValueError(f" {self.__class__.__name__}: The sigma value:"
                             f" {new_value}, should be strictly positive.")
        self._sigma = new_value
        self.sig_inv = 1.0 / self._sigma

    @property
    def inverse_sigma(self):
        return self.sig_inv


class DoubleWell(_Scalar1D):
    """double_well.py:8-262"""
    model_key = "DW"

    def make_trajectory(self, t0, tf, dt=0.01, device=None):
        tk = np.arange(t0, tf + dt, dt)
        dim_t = tk.size
        x = np.zeros(dim_t)
        x[0] = +self._theta if self.rng.random() > 0.5 else -self._theta
        x[0] += np.sqrt(0.5 * self._sigma * dt) * self.rng.standard_normal()
        z = self.rng.standard_normal(dim_t)
        if device is not None:
            x = engine.make_trajectories("DW", dim_t, dt, [self._theta], [self._sigma], z, [x[0]], device)[0]
        else:
            ek = np.sqrt(self._sigma * dt) * z
            for t in range(1, dim_t):
                x[t] = x[t - 1] + 4.0 * x[t - 1] * (self._theta - x[t - 1] ** 2) * dt + ek[t]
        self.sample_path = x
        self.time_window = tk


class OrnsteinUhlenbeck(_Scalar1D):
    """ornstein_uhlenbeck.py:8-234"""
    model_key = "OU"

    def make_trajectory(self, t0, tf, dt=0.01, mu=0.0, device=None):
        tk = np.arange(t0, tf + dt, dt)
        dim_t = tk.size
        x = np.zeros(dim_t)
        x[0] = mu
        z = self.rng.standard_normal(dim_t)
        if device is not None:
            x = engine.make_trajectories("OU", dim_t, dt, [self._theta, mu], [self._sigma], z, [mu], device)[0]
        else:
            ek = np.sqrt(self._sigma * dt) * z
            for t in range(1, dim_t):
                x[t] = x[t - 1] + self._theta * (mu - x[t - 1]) * dt + ek[t]
        self.sample_path = x
        self.time_window = tk


def _chol_inv(x):
    """utilities.py:203-217"""
    c_inv = np.linalg.solve(np.linalg.cholesky(x), np.eye(x.shape[0]))
    return c_inv.T.dot(c_inv), c_inv


class _VectorND(StochasticProcess):
    dim_d = None

    def _set_sigma(self, sigma):
        sigma = np.asarray(sigma, dtype=float)
        if sigma.ndim == 0:
            # the reference rejects a 0-d array here (SURVEY.md F6); a scalar is the
            # obvious intent of the shipped JSON files, so it is accepted.
            self._sigma = float(sigma) * np.eye(self.dim_d)
        elif sigma.ndim == 1:
            self._sigma = np.diag(sigma)
        elif sigma.ndim == 2:
            self._sigma = sigma
        else:
            raise ValueError(f" {self.__class__.__name__}: Wrong input dimensions: {sigma.ndim}")
        if self._sigma.shape != (self.dim_d, self.dim_d):
            raise ValueError(f" {self.__class__.__name__}: Wrong matrix dimensions: {self._sigma.shape}")
        if np.any(np.linalg.eigvals(self._sigma) <= 0.0):
            raise RuntimeError(f" {self.__class__.__name__}:"
                               f" Noise matrix {self._sigma} is not positive definite.")
        self.sig_inv, _ = _chol_inv(self._sigma)

    @property
    def theta(self):
        return self._theta

    @theta.setter
    def theta(self, new_value):
        self._theta = new_value

    @property
    def sigma(self):
        return self._sigma

    @sigma.setter
    def sigma(self, new_value):
        self._set_sigma(new_value)

    @property
    def inverse_sigma(self):
        return self.sig_inv

    def _noise_path(self, dt, dim_t, z=None):
        # lorenz_63.py:203-219 / lorenz_96.py:289-302 (scipy's upper Cholesky factor)
        from scipy.linalg import cholesky, LinAlgError
        try:
            ek = cholesky(self._sigma * dt)
        except LinAlgError:
            ek = np.sqrt(np.eye(self.dim_d) * self._sigma * dt)
        return ek.dot(self.rng.standard_normal((self.dim_d, dim_t)) if z is None else z).T

    def _gpu_path(self, dt, dim_t, device):
        """The reference's burn-in and Euler-Maruyama loop on the GPU, fed with this object's own draws."""
        z = self.rng.standard_normal((self.dim_d, dim_t))
        return engine.make_trajectories(self.model_key, dim_t, dt, np.atleast_1d(self._theta), self._sigma_diag(),
                                        z, None, device)[0]


def _l63(state, u):
    """lorenz_63.py:8-37"""
    x, y, z = state
    sigma, rho, beta = u
    return np.array([sigma * (y - x), (rho - z) * x - y, x * y - beta * z])


def _l96(x, u):
    """lorenz_96.py:85-101 on a 1-D state (ordinary cyclic shifts)."""
    return (np.roll(x, -1) - np.roll(x, +2)) * np.roll(x, +1) - x + u


class Lorenz63(_VectorND):
    """lorenz_63.py:40-635"""
    model_key = "L63"
    dim_d = 3

    def __init__(self, sigma, theta, r_seed=None):
        super().__init__(r_seed, single_dim=False)
        self._set_sigma(sigma)
        self._theta = np.asarray(theta, dtype=float)

    def make_trajectory(self, t0, tf, dt=0.01, device=None):
        tk = np.arange(t0, tf + dt, dt)
        dim_t = tk.size
        if device is not None:
            self.sample_path, self.time_window = self._gpu_path(dt, dim_t, device), tk
            return
        x0 = np.ones(3)
        delta_t = 1.0e-3
        for _ in range(5000):
            x0 = x0 + _l63(x0, self._theta) * delta_t
        x = np.zeros((dim_t, 3))
        x[0] = x0
        ek = self._noise_path(dt, dim_t)
        for t in range(1, dim_t):
            x[t] = x[t - 1] + _l63(x[t - 1], self._theta) * dt + ek[t]
        self.sample_path = x
        self.time_window = tk


class Lorenz96(_VectorND):
    """lorenz_96.py:104-464"""
    model_key = "L96"

    def __init__(self, sigma, theta, r_seed=None, dim_d=40):
        StochasticProcess.__init__(self, r_seed, single_dim=False)
        if dim_d < 10:
            raise ValueError(f" {self.__class__.__name__}: Insufficient state vector dimensions: {dim_d}")
        if dim_d > L96_DIMS[1]:
            raise ValueError(f" {self.__class__.__name__}: dim_d = {dim_d} is outside the range the CUDA path"
                             f" supports ({L96_DIMS[0]} <= dim_d <= {L96_DIMS[1]}).")
        self.dim_d = int(dim_d)
        self._set_sigma(sigma)
        self._theta = np.asarray(theta, dtype=float)

    def make_trajectory(self, t0, tf, dt=0.01, device=None):
        tk = np.arange(t0, tf + dt, dt)
        dim_t = tk.size
        if device is not None:
            self.sample_path, self.time_window = self._gpu_path(dt, dim_t, device), tk
            return
        x0 = self._theta * np.ones(self.dim_d)
        delta_t = 1.0e-3
        x0[int(self.dim_d / 2.0)] += delta_t
        for _ in range(5000):
            x0 = x0 + _l96(x0, self._theta) * delta_t
        x = np.zeros((dim_t, self.dim_d))
        x[0] = x0
        ek = self._noise_path(dt, dim_t)
        for t in range(1, dim_t):
            x[t] = x[t - 1] + _l96(x[t - 1], self._theta) * dt + ek[t]
        self.sample_path = x
        self.time_window = tk


# simulation.py:20
dynamical_systems = {"DW": DoubleWell, "OU": OrnsteinUhlenbeck, "L63": Lorenz63, "L96": Lorenz96}
