"""Thin object wrapper over the C-ABI handle: one ``Engine`` = one GPU + one stream.

Every method is a single call into ``libcgpcm_b200.so``; numpy arrays / torch tensors are only
containers for the bytes that cross the boundary.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import (GRAD_ALL, GRAD_ALPHA, GRAD_GAMMA, GRAD_MU_U, GRAD_OMEGA, GRAD_S2, GRAD_S2F, GRAD_VAR_U,
                   MODE_FROZEN, MODE_FULL)

TERM_NAMES = ['s2 complexity', 'p(z) complexity', 'q*(z) complexity', 'q*(z) fit',
              'general conditioning penalty', 'q(u) conditioning penalty', '-KL[q(u)||p(u)]']


def n_params(nh):
    return 5 + nh + nh * (nh + 1) // 2


class Engine(object):
    def __init__(self, nh, nx, causal=True, causal_id=False, device=0):
        self.nh, self.nx = int(nh), int(nx)
        self.device = int(device)
        self._h = ctypes.c_void_p()
        L = _lib.lib()
        rc = L.cgpcm_create(ctypes.byref(self._h), self.device, self.nh, self.nx, int(bool(causal)),
                            int(bool(causal_id)), None)
        if rc != 0:
            self._h = ctypes.c_void_p()
            if rc == -2:
                raise _lib.CgpcmError(rc, 'no usable CUDA device %d (cgpcm_b200 has no CPU fallback)' % self.device)
            _lib.check(rc)
        self.n_local = 0
        self.rank, self.world = 0, 1

    # -- lifetime
    def close(self):
        if getattr(self, '_h', None) and self._h.value:
            _lib.lib().cgpcm_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        _lib.check(rc, self._h)

    # -- configuration
    def set_option(self, key, value):
        self._ck(_lib.lib().cgpcm_set_option(self._h, key.encode(), float(value)))

    def comm_init(self, unique_id, rank, world):
        """Join the NCCL communicator described by the 128-byte ``unique_id`` (see ``unique_id()``)."""
        buf = (ctypes.c_char * 128).from_buffer_copy(bytes(unique_id)) if unique_id is not None else None
        self._ck(_lib.lib().cgpcm_comm_init(self._h, buf, int(rank), int(world)))
        self.rank, self.world = int(rank), int(world)

    @staticmethod
    def unique_id():
        buf = (ctypes.c_char * 128)()
        _lib.check(_lib.lib().cgpcm_comm_unique_id(buf))
        return bytes(buf)

    def set_data(self, t, y, th, tx):
        """This rank's observations and the inducing inputs (host or device float64 buffers)."""
        n = int(t.shape[0])
        if int(y.shape[0]) != n or int(th.shape[0]) != self.nh or int(tx.shape[0]) != self.nx:
            raise ValueError('shape mismatch in set_data')
        self._ck(_lib.lib().cgpcm_set_data(self._h, _lib.ptr(t) if n else None, _lib.ptr(y) if n else None, n,
                                            _lib.ptr(th), _lib.ptr(tx)))
        self.n_local = n

    # -- compute
    def psi(self, alpha, gamma, omega, per_observation=False):
        """Psi statistics (``mats[...]`` of ``src/core/cgpcm.py:235-243``) as numpy arrays."""
        hyp = np.array([alpha, gamma, omega], dtype=np.float64)
        out = {'sum_Axx': np.empty((self.nx, self.nx)), 'Ahh': np.empty((self.nh, self.nh)),
               'a': np.empty(1), 'sum_Ahx_y': np.empty((self.nh, self.nx))}
        ahx = axx = None
        if per_observation:
            ahx = np.empty((self.n_local, self.nh, self.nx))
            axx = np.empty((self.n_local, self.nx, self.nx))
        self._ck(_lib.lib().cgpcm_psi(self._h, _lib.ptr(hyp), _lib.ptr(out['sum_Axx']), _lib.ptr(out['Ahh']),
                                       _lib.ptr(out['a']), _lib.ptr(out['sum_Ahx_y']), _lib.ptr(ahx), _lib.ptr(axx)))
        out['a'] = float(out['a'][0])
        if per_observation:
            out['Ahx'], out['Axx'] = ahx, axx
        return out

    def precompute(self, alpha, gamma, omega, reg):
        hyp = np.array([alpha, gamma, omega], dtype=np.float64)
        self._ck(_lib.lib().cgpcm_precompute(self._h, _lib.ptr(hyp), float(reg)))

    def frozen_mats(self):
        """``sum_Bxx``, ``sum_Bhh``, ``sum_b``, ``sum_Ahx_y`` of the precomputed regime (``src/core/cgpcm.py:255-267``)."""
        out = {'sum_Bxx': np.empty((self.nx, self.nx)), 'sum_Bhh': np.empty((self.nh, self.nh)),
               'sum_b': np.empty(1), 'sum_Ahx_y': np.empty((self.nh, self.nx))}
        self._ck(_lib.lib().cgpcm_frozen_mats(self._h, _lib.ptr(out['sum_Bxx']), _lib.ptr(out['sum_Bhh']),
                                               _lib.ptr(out['sum_b']), _lib.ptr(out['sum_Ahx_y'])))
        out['sum_b'] = float(out['sum_b'][0])
        return out

    def elbo_grad(self, params, mode=MODE_FULL, grad_mask=GRAD_ALL, reg=1e-8, want_grad=True, out_grad=None):
        """(elbo, terms[7], grad or None).  ``params``: host numpy (pinned torch also fine) or CUDA tensor."""
        if int(params.shape[0]) != n_params(self.nh):
            raise ValueError('params must have length %d' % n_params(self.nh))
        elbo = np.empty(1)
        terms = np.empty(7)
        grad = None
        if want_grad:
            grad = out_grad if out_grad is not None else np.empty(n_params(self.nh))
        self._ck(_lib.lib().cgpcm_elbo_grad(self._h, _lib.ptr(params), int(mode), int(grad_mask), float(reg),
                                             _lib.ptr(elbo), _lib.ptr(terms), _lib.ptr(grad)))
        return float(elbo[0]), terms, grad

    def elbo_smf(self, params, sample, mode=MODE_FULL, reg=1e-8):
        """``elbo(smf=True, sample=sample)`` and the pseudo-log-likelihood of ``sample`` for the slice sampler:
        ``(elbo, terms[7], log_lik)`` (``src/core/cgpcm.py:527-531,848-872``)."""
        sample = np.ascontiguousarray(np.asarray(sample, dtype=np.float64).ravel())
        if sample.shape[0] != self.nh or int(params.shape[0]) != n_params(self.nh):
            raise ValueError('shape mismatch in elbo_smf')
        elbo, terms, ll = np.empty(1), np.empty(7), np.empty(1)
        self._ck(_lib.lib().cgpcm_elbo_smf(self._h, _lib.ptr(params), int(mode), float(reg), _lib.ptr(sample),
                                            _lib.ptr(elbo), _lib.ptr(terms), _lib.ptr(ll)))
        return float(elbo[0]), terms, float(ll[0])

    def elbo_smf_batch(self, params, samples, reg=1e-8, want_elbo=True):
        """``elbo_smf`` in the precomputed regime for every row of ``samples`` ([B, nh]) in one call:
        ``(elbo[B], terms[B, 7], log_lik[B])``.  ``want_elbo=False`` skips the jittered factorisation and returns
        ``(None, None, log_lik)`` (what the slice sampler needs).  A sample's values do not depend on the batch."""
        samples = np.ascontiguousarray(np.asarray(samples, dtype=np.float64))
        if samples.ndim != 2 or samples.shape[1] != self.nh or samples.shape[0] < 1 or \
                int(params.shape[0]) != n_params(self.nh):
            raise ValueError('shape mismatch in elbo_smf_batch')
        B = samples.shape[0]
        elbo, terms = (np.empty(B), np.empty((B, 7))) if want_elbo else (None, None)
        ll = np.empty(B)
        self._ck(_lib.lib().cgpcm_elbo_smf_batch(self._h, _lib.ptr(params), float(reg), _lib.ptr(samples), B,
                                                  _lib.ptr(elbo), _lib.ptr(terms), _lib.ptr(ll)))
        return elbo, terms, ll

    def predict_f(self, params, t_star, samples, smf=False, reg=1e-8):
        """Posterior ``(mean, var)`` of the function at ``t_star`` averaged over the filter ``samples`` ([B, nh])
        (``src/core/cgpcm.py:781-846``); needs the frozen statistics."""
        t_star = np.ascontiguousarray(np.asarray(t_star, dtype=np.float64).ravel())
        samples = np.ascontiguousarray(np.asarray(samples, dtype=np.float64).reshape(-1, self.nh))
        if int(params.shape[0]) != n_params(self.nh) or samples.shape[0] < 1:
            raise ValueError('shape mismatch in predict_f')
        mean, var = np.empty(t_star.shape[0]), np.empty(t_star.shape[0])
        self._ck(_lib.lib().cgpcm_predict_f(self._h, _lib.ptr(params), float(reg), _lib.ptr(t_star) if t_star.size else None,
                                             int(t_star.shape[0]), _lib.ptr(samples), int(samples.shape[0]),
                                             int(bool(smf)), _lib.ptr(mean), _lib.ptr(var)))
        return mean, var

    def predict_f_batch(self, params, t_star, samples, smf=True, reg=1e-8, per_sample=True):
        """Predictive moments of the function at ``t_star`` for every filter sample ([B, nh]) in one call:
        ``(mean[n], var[n], mean_s[n, B], var_s[n, B])``.  ``mean_s[:, b]`` and ``var_s[:, b]`` are the mean and
        variance under sample b's q(z) (``smf=True``: q(z | h_b); ``smf=False``: the one q(z) of q(u)); ``mean`` and
        ``var`` are their sample averages, what :meth:`predict_f` returns.  ``per_sample=False`` returns ``None`` for
        the last two.  A sample's moments do not depend on the other samples of the call; needs the frozen statistics."""
        t_star = np.ascontiguousarray(np.asarray(t_star, dtype=np.float64).ravel())
        samples = np.ascontiguousarray(np.asarray(samples, dtype=np.float64))
        if samples.ndim == 1:
            samples = samples.reshape(1, -1)
        if samples.ndim != 2 or samples.shape[1] != self.nh or samples.shape[0] < 1 or \
                int(params.shape[0]) != n_params(self.nh):
            raise ValueError('shape mismatch in predict_f_batch')
        n, B = t_star.shape[0], samples.shape[0]
        mean, var = np.empty(n), np.empty(n)
        mean_s, var_s = (np.empty((n, B)), np.empty((n, B))) if per_sample else (None, None)
        if n:
            self._ck(_lib.lib().cgpcm_predict_f_batch(self._h, _lib.ptr(params), float(reg), _lib.ptr(t_star), n,
                                                       _lib.ptr(samples), B, int(bool(smf)), _lib.ptr(mean),
                                                       _lib.ptr(var), _lib.ptr(mean_s), _lib.ptr(var_s)))
        return mean, var, mean_s, var_s

    def predict_f_cov(self, params, t_star, samples, smf=True, reg=1e-8, per_sample=False, noise=None):
        """Joint predictive covariance of the function at ``t_star`` (at most 4096 inputs) for every filter sample
        ([B, nh]) in one call: ``(mean[n], cov[n, n], mean_s[n, B], cov_s[B, n, n], draws[n, B])``.  ``cov_s[b]`` is the
        covariance of f under sample b's q(z) (``smf`` as in :meth:`predict_f_batch`; its diagonal is that method's
        ``var_s[:, b]``); ``mean`` and ``cov`` are the sample averages (``diag(cov)`` is :meth:`predict_f`'s variance).
        The mixture covariance of the samples is ``cov + np.cov(mean_s, bias=True)``.  ``per_sample=False`` returns
        ``None`` for ``cov_s``.  With standard normal ``noise`` ([n, B]), ``draws[:, b] = mean_s[:, b] +
        chol(cov_s[b] + reg I) noise[:, b]``, else ``None``.  A sample's outputs do not depend on the other samples of
        the call; needs the frozen statistics."""
        t_star = np.ascontiguousarray(np.asarray(t_star, dtype=np.float64).ravel())
        samples = np.ascontiguousarray(np.asarray(samples, dtype=np.float64))
        if samples.ndim == 1:
            samples = samples.reshape(1, -1)
        if samples.ndim != 2 or samples.shape[1] != self.nh or samples.shape[0] < 1 or \
                int(params.shape[0]) != n_params(self.nh):
            raise ValueError('shape mismatch in predict_f_cov')
        n, B = t_star.shape[0], samples.shape[0]
        draws = None
        if noise is not None:
            noise = np.ascontiguousarray(np.asarray(noise, dtype=np.float64))
            if noise.shape != (n, B):
                raise ValueError('noise must have shape (n_star, B)')
            draws = np.empty((n, B))
        mean_s, cov = np.empty((n, B)), np.empty((n, n))
        cov_s = np.empty((B, n, n)) if per_sample else None
        if n:
            self._ck(_lib.lib().cgpcm_predict_f_cov(self._h, _lib.ptr(params), float(reg), _lib.ptr(t_star), n,
                                                     _lib.ptr(samples), B, int(bool(smf)), _lib.ptr(mean_s),
                                                     _lib.ptr(cov_s), _lib.ptr(cov), _lib.ptr(noise), _lib.ptr(draws)))
        return mean_s.mean(1), cov, mean_s, cov_s, draws

    def predict_logpdf(self, params, t_star, y_star, samples, smf=True, reg=1e-8, noise=True, white=False):
        """Joint log predictive density of the block ``y_star`` at ``t_star`` (at most 4096 inputs) for every filter
        sample ([B, nh]) in one call: ``(lp, lp_s[B], white_s[n, B] or None)``.  ``lp_s[b] = log N(y_star; m_b, C_b +
        d I)`` with ``m_b``, ``C_b`` the mean and covariance of :meth:`predict_f_cov` (``smf`` as there) and ``d`` the
        noise variance ``s2`` (``noise=True``: ``y_star`` are observations) or ``reg`` (``noise=False``: ``y_star`` is
        f itself); ``lp`` is the log density under the mixture of the samples, ``log mean_b exp(lp_s[b])``.
        ``white=True`` also returns the whitened residuals ``L_b^-1 (y_star - m_b)``, ``L_b L_b^T = C_b + d I``.  A
        sample's ``lp_s`` and residuals do not depend on the other samples of the call; needs the frozen statistics."""
        t_star = np.ascontiguousarray(np.asarray(t_star, dtype=np.float64).ravel())
        y_star = np.ascontiguousarray(np.asarray(y_star, dtype=np.float64).ravel())
        samples = np.ascontiguousarray(np.asarray(samples, dtype=np.float64))
        if samples.ndim == 1:
            samples = samples.reshape(1, -1)
        if samples.ndim != 2 or samples.shape[1] != self.nh or samples.shape[0] < 1 or \
                int(params.shape[0]) != n_params(self.nh) or y_star.shape != t_star.shape:
            raise ValueError('shape mismatch in predict_logpdf')
        n, B = t_star.shape[0], samples.shape[0]
        lp, lp_s = np.empty(1), np.empty(B)
        white_s = np.empty((n, B)) if white else None
        self._ck(_lib.lib().cgpcm_predict_logpdf(self._h, _lib.ptr(params), float(reg), _lib.ptr(t_star),
                                                  _lib.ptr(y_star), n, _lib.ptr(samples), B, int(bool(smf)),
                                                  int(bool(noise)), _lib.ptr(lp), _lib.ptr(lp_s), _lib.ptr(white_s)))
        return float(lp[0]), lp_s, white_s

    def kernel_samples(self, params, t, samples, reg=1e-8):
        """Kernel samples ``k[n, b]`` of ``predict_k`` at lags ``t`` for filter ``samples`` ([B, nh])
        (``src/core/cgpcm.py:610-634``), before normalisation."""
        t = np.ascontiguousarray(np.asarray(t, dtype=np.float64).ravel())
        samples = np.ascontiguousarray(np.asarray(samples, dtype=np.float64).reshape(-1, self.nh))
        out = np.empty((t.shape[0], samples.shape[0]))
        if t.shape[0]:
            self._ck(_lib.lib().cgpcm_kernel_samples(self._h, _lib.ptr(np.ascontiguousarray(params[:5])), float(reg),
                                                      _lib.ptr(t), int(t.shape[0]), _lib.ptr(samples),
                                                      int(samples.shape[0]), _lib.ptr(out)))
        return out

    def filter_samples(self, params, t, samples, noise, reg=1e-8):
        """Posterior draws ``[n, B]`` of the filter at ``t`` for filter ``samples`` ([B, nh]) and standard normal
        ``noise`` ([n, B]) (``src/core/cgpcm.py:663-779``)."""
        t = np.ascontiguousarray(np.asarray(t, dtype=np.float64).ravel())
        samples = np.ascontiguousarray(np.asarray(samples, dtype=np.float64).reshape(-1, self.nh))
        noise = np.ascontiguousarray(np.asarray(noise, dtype=np.float64).reshape(t.shape[0], samples.shape[0]))
        out = np.empty((t.shape[0], samples.shape[0]))
        if t.shape[0]:
            self._ck(_lib.lib().cgpcm_filter_samples(self._h, _lib.ptr(np.ascontiguousarray(params[:5])), float(reg),
                                                      _lib.ptr(t), int(t.shape[0]), _lib.ptr(samples),
                                                      int(samples.shape[0]), _lib.ptr(noise), _lib.ptr(out)))
        return out

    def akm_sample(self, params, t, sample_h, e, reg=1e-8, want_cov=False):
        """One draw ``f = sqrt(s2_f) chol(reg(K)) e`` of the Approximate Kernel Model at inputs ``t`` for the filter
        draw ``sample_h`` [nh] and the standard normal draw ``e`` [n] (``AKM.f``, ``src/core/cgpcm.py:382-392``).
        Returns ``f`` [n], and the covariance ``reg(K)`` [n, n] when ``want_cov``."""
        t = np.ascontiguousarray(np.asarray(t, dtype=np.float64).ravel())
        sample_h = np.ascontiguousarray(np.asarray(sample_h, dtype=np.float64).ravel())
        e = np.ascontiguousarray(np.asarray(e, dtype=np.float64).ravel())
        if sample_h.shape[0] != self.nh or e.shape[0] != t.shape[0]:
            raise ValueError('sample_h must have nh entries and e one entry per input')
        f = np.empty(t.shape[0])
        K = np.empty((t.shape[0], t.shape[0])) if want_cov else None
        self._ck(_lib.lib().cgpcm_akm_sample(self._h, _lib.ptr(np.ascontiguousarray(params[:5])), float(reg),
                                              _lib.ptr(t), int(t.shape[0]), _lib.ptr(sample_h), _lib.ptr(e),
                                              _lib.ptr(f), _lib.ptr(K) if want_cov else None))
        return (f, K) if want_cov else f

    def fpi(self, params, num, high_reg=False, reg=1e-8):
        """``num`` rounds of the fixed-point iteration on the frozen Psi statistics, then the optimal q(z):
        ``(mu_u[nh], var_u[nh(nh+1)/2], mu_z[nx], var_z[nx(nx+1)/2])`` (``src/core/cgpcm.py:479-516,577-592``)."""
        if int(params.shape[0]) != n_params(self.nh):
            raise ValueError('params must have length %d' % n_params(self.nh))
        mu_u, var_u = np.empty(self.nh), np.empty(self.nh * (self.nh + 1) // 2)
        mu_z, var_z = np.empty(self.nx), np.empty(self.nx * (self.nx + 1) // 2)
        self._ck(_lib.lib().cgpcm_fpi(self._h, _lib.ptr(params), int(num), int(bool(high_reg)), float(reg),
                                       _lib.ptr(mu_u), _lib.ptr(var_u), _lib.ptr(mu_z), _lib.ptr(var_z)))
        return mu_u, var_u, mu_z, var_z

    def fpi_qz(self, params, mu_z, var_z, num, high_reg=False, reg=1e-8):
        """``fpi(num, z=False)`` + ``convert(z=False)`` from the explicit q(z) = N(mu_z, reg(Lz Lz^T)):
        ``(mu_u, var_u, mu_z, var_z)`` (``src/core/cgpcm.py:479-516,577-592`` with ``z=False``)."""
        mu_z = np.ascontiguousarray(np.asarray(mu_z, dtype=np.float64).ravel())
        var_z = np.ascontiguousarray(np.asarray(var_z, dtype=np.float64).ravel())
        if mu_z.shape[0] != self.nx or var_z.shape[0] != self.nx * (self.nx + 1) // 2:
            raise ValueError('shape mismatch in fpi_qz')
        mu_u, var_u = np.empty(self.nh), np.empty(self.nh * (self.nh + 1) // 2)
        mz, vz = np.empty(self.nx), np.empty(self.nx * (self.nx + 1) // 2)
        self._ck(_lib.lib().cgpcm_fpi_qz(self._h, _lib.ptr(params), _lib.ptr(mu_z), _lib.ptr(var_z), int(num),
                                          int(bool(high_reg)), float(reg), _lib.ptr(mu_u), _lib.ptr(var_u),
                                          _lib.ptr(mz), _lib.ptr(vz)))
        return mu_u, var_u, mz, vz

    def elbo_qz(self, params, mu_z, var_z, reg=1e-8):
        """``elbo(z=False)``: ``(elbo, terms[7])`` of the bound saturated for q(u) (``src/core/cgpcm.py:518-575``)."""
        mu_z = np.ascontiguousarray(np.asarray(mu_z, dtype=np.float64).ravel())
        var_z = np.ascontiguousarray(np.asarray(var_z, dtype=np.float64).ravel())
        if mu_z.shape[0] != self.nx or var_z.shape[0] != self.nx * (self.nx + 1) // 2:
            raise ValueError('shape mismatch in elbo_qz')
        elbo, terms = np.empty(1), np.empty(7)
        self._ck(_lib.lib().cgpcm_elbo_qz(self._h, _lib.ptr(np.ascontiguousarray(params[:5])), _lib.ptr(mu_z),
                                           _lib.ptr(var_z), float(reg), _lib.ptr(elbo), _lib.ptr(terms)))
        return float(elbo[0]), terms

    def last_timing(self):
        t = np.zeros(12)
        self._ck(_lib.lib().cgpcm_last_timing(self._h, _lib.ptr(t)))
        return dict(total_ms=float(t[0]), forward_ms=float(t[1]), backward_ms=float(t[2]), algebra_ms=float(t[3]),
                    axx_ms=float(t[4]), gemm_ms=float(t[5]), launches=int(t[6]), gemm_flops=float(t[7]),
                    gemm_launches=int(t[8]), gemm_flops_executed=float(t[9]), ahx_gen_ms=float(t[10]),
                    own_sweeps_ms=float(t[11]))


def bvn_cdf(x1, x2, rho):
    """The reference's native op ``bvn_cdf(x1, x2, rho)`` (``src/core/exponentiated_quadratic.py:552``):
    element-wise on three equal-length float64 vectors (numpy -> numpy, CUDA tensor -> CUDA tensor)."""
    if isinstance(x1, np.ndarray):
        x1, x2, rho = [np.ascontiguousarray(v, dtype=np.float64).ravel() for v in (x1, x2, rho)]
        if not (x1.shape == x2.shape == rho.shape):
            raise ValueError('x1, x2, rho must have equal length')
        out = np.empty_like(x1)
    else:
        import torch
        if not (x1.shape == x2.shape == rho.shape) or x1.dim() != 1:
            raise ValueError('x1, x2, rho must be rank-1 and of equal length')
        out = torch.empty_like(x1)
    _lib.check(_lib.lib().cgpcm_bvn_cdf(_lib.ptr(x1), _lib.ptr(x2), _lib.ptr(rho), _lib.ptr(out), int(x1.shape[0]),
                                         None))
    return out
