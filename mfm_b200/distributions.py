"""Targets of the MFM hot path — device-resident mirror of the reference's distributions.py.

Same class names, constructor arguments and methods (logprob / loglik / logprior /
initialize_model / sample_model) as distributions.py:42-97,114-165,231-314, but every method works
on a batch of positions [N, d] (CUDA tensors) and is backed by the C-ABI target descriptor
(include/mfm_b200.h::mfm_target_t).  `dist.tempered(beta)` is the device replacement for the
closure `lambda x: beta * dist.loglik(x) + dist.logprior(x)` (exe_flow_matching.py:301,316).
"""
from __future__ import annotations

import itertools
import os

import numpy as np
import torch

from . import _lib, random as mrandom

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


class DeviceLogDensity:
    """Callable device log-density `x -> beta*loglik(x) + logprior(x)` with a CUDA value_and_grad."""

    def __init__(self, dist: "Distribution", beta: float = 1.0):
        self.dist = dist
        self.beta = float(beta)

    def desc(self) -> _lib.TargetDesc:
        return self.dist._desc(self.beta)

    def value_and_grad(self, x: torch.Tensor, want_loglik: bool = False):
        lib = _lib.load()
        x = x.contiguous()
        n, d = x.shape
        assert d == self.dist.dim
        logp = torch.empty(n, dtype=torch.float32, device=x.device)
        grad = torch.empty_like(x)
        ll = torch.empty(n, dtype=torch.float32, device=x.device) if want_loglik else None
        desc = self.desc()
        ws = _lib.workspace(lib.mfm_target_workspace_bytes(desc, n), x.device, "target")
        _lib.check(lib.mfm_logdensity_and_grad(desc, n, _lib.ptr(x), _lib.ptr(logp), _lib.ptr(grad), _lib.ptr(ll),
                                               _lib.ptr(ws), ws.numel(), _lib.stream()))
        return (logp, grad, ll) if want_loglik else (logp, grad)

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        single = x.dim() == 1
        v, _ = self.value_and_grad(x[None] if single else x)
        return v[0] if single else v


class Distribution:
    dim: int
    _kind: int

    def __init__(self, device=None):
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.log_Z = 0.0
        self.n_plots = 0
        self.can_sample = False

    # -- descriptor --------------------------------------------------------------------------
    def _fill(self, d: _lib.TargetDesc):
        raise NotImplementedError

    def _desc(self, beta: float) -> _lib.TargetDesc:
        d = _lib.TargetDesc()
        d.kind, d.dim, d.beta = self._kind, self.dim, float(beta)
        self._fill(d)
        return d

    def tempered(self, beta: float = 1.0) -> DeviceLogDensity:
        return DeviceLogDensity(self, beta)

    # -- reference method names ----------------------------------------------------------------
    def logprob(self, x):
        return self.tempered(1.0)(x)

    def loglik(self, x):
        single = x.dim() == 1
        _, _, ll = self.tempered(1.0).value_and_grad(x[None] if single else x, want_loglik=True)
        return ll[0] if single else ll

    def logprior(self, x):
        return self.logprob(x) - self.loglik(x)

    def log_prob(self, x):
        return self.logprob(x)

    def _tensor(self, a):
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(self.device)


class GaussianMixture(Distribution):
    """distributions.py:42-77 (dim is fixed to 2 there, :54)."""
    _kind = _lib.TARGET_GMM

    def __init__(self, modes, covs, weights, device=None):
        super().__init__(device)
        modes = np.asarray(modes, np.float32)
        covs = np.asarray(covs, np.float32)
        if covs.ndim == 3:                      # full diagonal matrices as in the default args
            covs = np.stack([np.diag(c) for c in covs])
        self.dim = 2
        assert modes.shape[1] == 2, "GaussianMixture is two-dimensional in the reference"
        self.modes = self._tensor(modes)
        self.covs = self._tensor(covs)
        self.chol_covs = self._tensor(np.sqrt(covs))          # distributions.py:51
        self.weights = self._tensor(np.asarray(weights, np.float32))

    def _fill(self, d):
        d.n_modes = self.modes.shape[0]
        d.modes, d.stds, d.weights = self.modes.data_ptr(), self.chol_covs.data_ptr(), self.weights.data_ptr()

    def initialize_model(self, rng_key, n_chain):
        keys = mrandom.split(rng_key, n_chain)
        self.init_params = mrandom.normal(keys, (self.dim,))


class IndepGaussian(Distribution):
    """distributions.py:80-97."""
    _kind = _lib.TARGET_GAUSS

    def __init__(self, dim, mean=0.0, var=1.0, device=None):
        super().__init__(device)
        self.dim, self.mean, self.std = dim, float(mean), float(np.sqrt(var))

    def _fill(self, d):
        d.gauss_mean, d.gauss_std = self.mean, self.std

    def initialize_model(self, rng_key, n_chain):
        self.init_params = mrandom.normal(mrandom.split(rng_key, n_chain), (self.dim,))

    def sample_model(self, rng_key):
        """rng_key uint32[2] -> [d]; uint32[N,2] -> [N,d] (the vmapped form, exe_flow_matching.py:155)."""
        return self.mean + self.std * mrandom.normal(rng_key, (self.dim,))

    def _fill_ref(self, d: _lib.FieldDesc):
        """As the reference distribution of a flow (mfm_field_t::ref_*)."""
        d.ref_kind, d.ref_mean, d.ref_std = _lib.REF_INDEP_GAUSS, self.mean, self.std


def phi_four_base_band(dim, alpha=0.1, beta=20.0):
    """Band Cholesky factor of PhiFourBase's tridiagonal precision P = beta (diag(2c + 1/c) - c (sub + super diagonal)),
    c = alpha dim, in float64: P = L L^T with L lower bidiagonal, diagonal l[d] and sub-diagonal s[d] (s[i] = L[i][i-1],
    s[0] = 0).  Returns (l, s, log_norm) with log_norm = -d/2 log 2 pi + sum log l_i = -(d log 2 pi + log det P^-1) / 2, the
    constant of logprob (distributions.py:168-226)."""
    c = alpha * dim
    p, q = beta * (2.0 * c + 1.0 / c), -beta * c
    l, s = np.empty(dim), np.zeros(dim)
    l[0] = np.sqrt(p)
    for i in range(1, dim):
        s[i] = q / l[i - 1]
        l[i] = np.sqrt(p - s[i] * s[i])
    log_norm = float(-0.5 * dim * np.log(2.0 * np.pi) + np.log(l).sum())
    return l, s, log_norm


class PhiFourBase(Distribution):
    """distributions.py:168-226: the Gaussian part of the phi-four action, N(0, P^-1) with the tridiagonal precision P above;
    ref_dists['phifour'] (exe_flow_matching.py:53).  A reference distribution only: sample_model = L^-T normal(key, (d,)) and
    logprob run as CUDA kernels (mfm_ref_sample / mfm_ref_logprob, one band solve / one sum of squares per row, never a dense
    d x d factor).  The band factor is formed in float64 here and handed to the device as float32."""

    def __init__(self, dim, alpha=0.1, beta=20.0, prior_type="coupled", device=None):
        if prior_type == "coupled_pbc":
            raise NotImplementedError("prior_type='coupled_pbc' cannot be constructed in the reference: it assigns into jnp arrays "
                                      "and divides dim to a float (distributions.py:168-226)")
        if prior_type != "coupled":
            raise ValueError(f"unknown prior_type {prior_type!r}: 'coupled'")
        super().__init__(device)
        self.dim, self.alpha, self.beta, self.prior_type = int(dim), float(alpha), float(beta), prior_type
        c = self.alpha * self.dim
        self.l, self.s, self.log_norm = phi_four_base_band(self.dim, self.alpha, self.beta)
        # a[d] = -s_{i+1} / l_i, 1 / l[d], beta c, beta / c: the layout of mfm_field_t::ref_band (back-substitution coefficients
        # x_i = a_i x_{i+1} + z_i / l_i, rounded to float32 once from float64)
        a = np.zeros(self.dim)
        a[:-1] = -self.s[1:] / self.l[:-1]
        self.band = self._tensor(np.concatenate([a, 1.0 / self.l, [self.beta * c, self.beta / c]]))
        self.can_sample = True

    def _fill_ref(self, d: _lib.FieldDesc):
        """As the reference distribution of a flow (mfm_field_t::ref_*).  ref_mean / ref_std stay (0, 1)."""
        d.ref_mean, d.ref_std = 0.0, 1.0
        d.ref_kind, d.ref_band, d.ref_log_norm = _lib.REF_PHI4_BASE, self.band.data_ptr(), self.log_norm

    def _ref_desc(self) -> _lib.FieldDesc:
        d = _lib.FieldDesc()
        d.dim = self.dim
        self._fill_ref(d)
        return d

    def _desc(self, beta: float):
        raise NotImplementedError("PhiFourBase is a reference distribution only: it has no target descriptor (no MALA, no field "
                                  "score term)")

    def tempered(self, beta: float = 1.0):
        raise NotImplementedError("PhiFourBase is a reference distribution only: it cannot be tempered or used as a MALA target")

    def initialize_model(self, rng_key, n_chain):
        raise NotImplementedError("PhiFourBase is a reference distribution only: it is not a target to initialise chains for")

    def sample_model(self, rng_key):
        """rng_key uint32[2] -> [d]; uint32[N,2] -> [N,d] (vmap(sample_model), exe_flow_matching.py:156,453)."""
        lib = _lib.load()
        single = rng_key.dim() == 1
        keys = (rng_key[None] if single else rng_key).contiguous()
        out = torch.empty((keys.shape[0], self.dim), dtype=torch.float32, device=keys.device)
        _lib.check(lib.mfm_ref_sample(self._ref_desc(), _lib.ptr(keys), keys.shape[0], _lib.ptr(out), _lib.stream()))
        return out[0] if single else out

    def logprob(self, x):
        """x [d] -> scalar; [N,d] -> [N]:  -x^T P x / 2 + log_norm."""
        lib = _lib.load()
        single = x.dim() == 1
        xx = (x[None] if single else x).to(torch.float32).contiguous()
        out = torch.empty(xx.shape[0], dtype=torch.float32, device=xx.device)
        _lib.check(lib.mfm_ref_logprob(self._ref_desc(), xx.shape[0], _lib.ptr(xx), _lib.ptr(out), _lib.stream()))
        return out[0] if single else out

    def loglik(self, x):
        return self.logprob(x)

    def logprior(self, x):
        return torch.zeros(x.shape[:-1], dtype=torch.float32, device=x.device)          # logprior is 0 (distributions.py:168-226)


class PhiFour(Distribution):
    """distributions.py:114-165 (Dirichlet(0) boundary, no tilt)."""
    _kind = _lib.TARGET_PHI4

    def __init__(self, dim, a=0.1, beta=20.0, bc=("dirichlet", 0), tilt=None, device=None):
        super().__init__(device)
        if bc[0] != "dirichlet" or bc[1] != 0 or tilt is not None:
            raise NotImplementedError("only the configuration the reference runs: Dirichlet(0), no tilt")
        self.dim, self.a, self.beta, self.bc, self.tilt = dim, a, beta, bc, tilt

    def _fill(self, d):
        d.phi_a, d.phi_beta = self.a, self.beta

    def initialize_model(self, rng_key, n_chain):
        keys = mrandom.split(rng_key, n_chain)
        self.init_params = mrandom.uniform(keys, (self.dim,)) * 2 - 1     # distributions.py:162-164


def get_bin_counts(points: np.ndarray, n_bins: int) -> np.ndarray:
    """Histogram of [0,1]^2 points on an n_bins x n_bins grid; points on the upper edge fall in
    the last bin (same rule as cox_process_utils.py:28-55)."""
    idx = np.minimum(np.floor(np.asarray(points, np.float64) * n_bins).astype(np.int64), n_bins - 1)
    counts = np.zeros((n_bins, n_bins))
    np.add.at(counts, (idx[:, 0], idx[:, 1]), 1.0)
    return counts


class LogGaussianCoxPines(Distribution):
    """distributions.py:231-314.  Unwhitened parameterisation (what multi_modal.py constructs): the dense Gaussian prior is
    applied as x K^-1 (one GEMM) instead of two triangular solves against chol(K); K^-1 is formed once in float64 on the host
    (cond(K) = 27.6).  use_whitened=True (:276-297): the state is the white noise e, latents f = L e + mu - value and gradient
    are two GEMMs against the Cholesky factor, the field's Hessian terms two more."""
    _kind = _lib.TARGET_PINES

    def __init__(self, dim, file_path=None, use_whitened=False, device=None):
        super().__init__(device)
        self.use_whitened = bool(use_whitened)
        if self.use_whitened:
            self._kind = _lib.TARGET_PINES_WHITE
        self.dim = dim
        n = int(np.sqrt(dim))
        self._num_grid_per_dim = n
        if file_path is not None:
            counts = get_bin_counts(np.genfromtxt(file_path, delimiter=","), n)
        else:
            if n != 40:
                raise ValueError("bundled bin counts are for the 40x40 grid; pass file_path=finpines.csv")
            counts = np.loadtxt(os.path.join(_DATA, "pines_counts_40x40.txt"))
        self._poisson_a = 1.0 / dim
        self._signal_variance, self._beta = 1.91, 1.0 / 33
        pts = np.array(list(itertools.product(range(n), range(n))), np.float64)
        dist = np.sqrt(((pts[:, None, :] - pts[None]) ** 2).sum(-1))
        K = self._signal_variance * np.exp(-dist / (n * self._beta))
        L = np.linalg.cholesky(K)
        self._half_log_det = float(np.log(np.abs(np.diag(L))).sum())
        self._log_norm = float(-0.5 * dim * np.log(2 * np.pi) - self._half_log_det)
        self._mu_zero = float(np.log(126.0) - 0.5 * self._signal_variance)
        Linv = np.linalg.solve(L, np.eye(dim))
        Kinv = Linv.T @ Linv
        Kinv = 0.5 * (Kinv + Kinv.T)
        self._flat_bin_counts = self._tensor(counts.reshape(dim))
        self._kinv = self._tensor(Kinv)
        self._kinv_mu = self._tensor(self._mu_zero * Kinv.sum(0))
        self._kinv_diag = self._tensor(np.diag(Kinv))
        self._cholesky_gram = self._tensor(L)
        if self.use_whitened:
            self._log_norm = float(-0.5 * dim * np.log(2 * np.pi))              # _white_gaussian_log_normalizer (:267)
            self._chol_t = self._tensor(L.T)
            self._chol_sq_t = self._tensor((L * L).T)
            self._mu_vec = self._tensor(np.full(dim, self._mu_zero))
        # K^-1 is the constant B operand of every pines GEMM: its scaled-fp16 split (include/mfm_b200.h, mfm_gemm_presplit) is
        # made once here instead of in shared memory by every CTA of every call
        self._kinv_split = None
        if self.device.type == "cuda" and dim % 16 == 0:
            lib = _lib.load()
            if lib.mfm_gemm_h16_enabled():
                m = torch.empty(dim * dim + 16, dtype=torch.float32, device=self.device)
                with torch.cuda.device(self.device):
                    _lib.check(lib.mfm_gemm_presplit(self._kinv.data_ptr(), m.data_ptr(), dim * dim, _lib.stream()))
                self._kinv_split = m

    def _fill(self, d):
        d.counts, d.kinv = self._flat_bin_counts.data_ptr(), self._kinv.data_ptr()
        d.kinv_mu, d.kinv_diag = self._kinv_mu.data_ptr(), self._kinv_diag.data_ptr()
        d.kinv_split = self._kinv_split.data_ptr() if self._kinv_split is not None else None
        if self.use_whitened:
            d.chol, d.chol_t = self._cholesky_gram.data_ptr(), self._chol_t.data_ptr()
            d.chol_sq_t, d.mu_vec = self._chol_sq_t.data_ptr(), self._mu_vec.data_ptr()
        d.mu, d.log_norm, d.poisson_a = self._mu_zero, self._log_norm, self._poisson_a

    def initialize_model(self, rng_key, n_chain):
        eps = mrandom.normal(mrandom.split(rng_key, n_chain), (self.dim,))
        # initialisation only: mu + L @ eps (distributions.py:312-314)
        self.init_params = (self._mu_zero + eps @ self._cholesky_gram.T).contiguous()
