"""Pair statistics of the joint predictive covariance of f (cgpcm_predict_f_cov), for the tests: the reference's
``expq_Axx`` integrand at two distinct inputs through the restated ``integrate_box`` (``psi_axx_pairs_generic``), its
closed form (``psi_axx_pairs``), and ``oracle.model.predict_f`` with pair statistics (``predict_f_cov``).  Built on the
oracle's own pieces; TEST INFRASTRUCTURE ONLY."""
import math

import numpy as np
import torch

from oracle import expq
from oracle.bvn_torch import bvn_cdf as _bvn_cdf_torch
from oracle.model import (DT, T, from_natural, model_matrices, optimal_q, prior_kernels, psi_Ahx, psi_center_closed,
                          psi_closed, reg, unpack, vec_to_tril)


def psi_axx_pairs_generic(t1, t2, tx, alpha, gamma, omega, causal=True, causal_id=False):
    """The reference's own ``expq_Axx`` integrand (``kh(t1 - tau1, t2 - tau2) kxs(tau1, tx1) kxs(tx2, tau2)``,
    ``cgpcm.py:111-121``) at DISTINCT inputs ``t1`` (axis 0) and ``t2`` (axis 1), through the restated ``integrate_box``:
    upper limits ``t1``, ``t2`` (causal), ``min(t1, tx1)``, ``min(t2, tx2)`` (``causal_id``) or ``inf`` (acausal).
    ``psi_generic`` only evaluates it at ``t2 = t1``.  Returns [n1, n2, nx, nx].  Small sizes only."""
    t1v, t2v, tx = T(t1), T(t2), T(tx)
    v = expq.var
    tau1, tau2, t1, t2, tx1, tx2 = v('tau1'), v('tau2'), v('t1'), v('t2'), v('tx1'), v('tx2')
    kh = lambda x, y: expq.kh(alpha, gamma, x, y)
    kxs = lambda x, y: expq.kxs(omega, x, y)
    expq_Axx = kh(t1 - tau1, t2 - tau2) * kxs(tau1, tx1) * kxs(tx2, tau2)
    n1, n2, nx = t1v.shape[0], t2v.shape[0], tx.shape[0]
    vm = {'t1': t1v.reshape(-1, 1, 1, 1), 't2': t2v.reshape(1, -1, 1, 1), 'tx1': tx.reshape(1, 1, -1, 1),
          'tx2': tx.reshape(1, 1, 1, -1)}
    vm['min_t1_tx1'] = torch.minimum(vm['t1'], vm['tx1'])
    vm['min_t2_tx2'] = torch.minimum(vm['t2'], vm['tx2'])
    if causal:
        up1, up2 = (v('min_t1_tx1'), v('min_t2_tx2')) if causal_id else (t1, t2)
    else:
        up1 = up2 = expq.inf
    Axx = torch.as_tensor(expq_Axx.integrate_box(('tau1', -expq.inf, up1), ('tau2', -expq.inf, up2), **vm))
    return (Axx * torch.ones(n1, n2, nx, nx, dtype=DT)).reshape(n1, n2, nx, nx)


def psi_axx_pairs(t1, t2, tx, alpha, gamma, omega, causal=True, causal_id=False):
    """Closed form of the same: ``psi_Axx`` with ``dk = t1 - tx_k`` and ``dl = t2 - tx_l``.  With ``s1 = t1 - tau1``,
    ``s2 = t2 - tau2`` the quadratic form of the double integral does not change and only its linear terms move, so the
    envelope ``exp(G)``, the BVN arguments and the ``causal_id`` shifts take ``dk`` from ``t1`` and ``dl`` from ``t2``.
    Returns [n1, n2, nx, nx]."""
    t1, t2, tx = T(t1), T(t2), T(tx)
    alpha, gamma, omega = T(alpha), T(gamma), T(omega)
    A = alpha + gamma + omega
    det = 4 * (A * A - gamma * gamma)
    S11, S12 = 2 * A / det, 2 * gamma / det
    dk = (t1[:, None] - tx[None, :])[:, None, :, None]
    dl = (t2[:, None] - tx[None, :])[None, :, None, :]
    g1 = omega * (1 - 2 * omega * S11)
    g2 = 4 * omega ** 2 * S12
    G = -g1 * (dk ** 2 + dl ** 2) + g2 * dk * dl
    pref = 2 * math.pi / torch.sqrt(det) * torch.exp(G)
    if not causal:
        return pref
    p = 2 * omega * torch.sqrt(S11)
    q = 2 * omega * S12 / torch.sqrt(S11)
    x1 = p * dk + q * dl
    x2 = q * dk + p * dl
    if causal_id:
        x1 = x1 - torch.clamp(dk, min=0.) / torch.sqrt(S11)
        x2 = x2 - torch.clamp(dl, min=0.) / torch.sqrt(S11)
    rho = (gamma / A) * torch.ones_like(x1)
    return pref * _bvn_cdf_torch(x1, x2, rho)


def predict_f_cov(params, t, y, th, tx, r, t_star, samples_h, smf=False, causal=True, causal_id=False):
    """``predict_f`` with pair statistics: per filter sample ``h_b`` the predictive mean ``[n*]`` and the covariance
    ``C_b[p, q] = E[f_p f_q | h_b] - mu_p mu_q`` ``[n*, n*]`` of the function at ``t_star``, with
        ``E[f_p f_q | h] = s2_f (a_c(t_p - t_q) + <Ahh_c(t_p - t_q), mh> + <Axx(t_p, t_q), mx> + <mh Ahx_q mx, Ahx_p>)``
    (``psi_center_closed`` at the lags, ``psi_axx_pairs``, ``psi_Ahx``).  At ``p = q`` this is ``predict_f``'s second
    moment.  Returns ``(mean_s [n*, B], cov_s [B, n*, n*])``."""
    with torch.no_grad():
        nh = len(th)
        s2, s2_f, alpha, gamma, omega, mu_u, var_u = unpack(T(np.asarray(params, np.float64)), nh)
        k = prior_kernels(th, tx, alpha, gamma, omega, r)
        a, Ahh, Axx, Ahx = psi_closed(t, th, tx, alpha, gamma, omega, causal, causal_id)
        m = model_matrices(y, a, Ahh, Axx, Ahx, k['iKh'], k['iKx'])
        ts = T(t_star)
        n = ts.shape[0]
        Ahx_s = psi_Ahx(ts, th, tx, alpha, gamma, omega, causal, causal_id)                  # [n, nh, nx]
        Axx_p = psi_axx_pairs(ts, ts, tx, alpha, gamma, omega, causal, causal_id)            # [n, n, nx, nx]
        a_c, Ahh_c = psi_center_closed((ts[:, None] - ts[None, :]).reshape(-1), th, alpha, gamma, causal)
        a_c, Ahh_c = a_c.reshape(n, n), Ahh_c.reshape(n, n, nh, nh)
        Lq = vec_to_tril(var_u)
        h_var = reg(Lq @ Lq.T, r)
        mus, covs = [], []
        for hs in samples_h:
            h = T(np.asarray(hs, np.float64)).reshape(-1, 1)
            if smf:
                lam, P = optimal_q(m, k, s2, s2_f, h, h @ h.T, True)
            else:
                lam, P = optimal_q(m, k, s2, s2_f, mu_u, h_var + mu_u @ mu_u.T, True)
            xm, xv = from_natural(P, lam, r)
            mu = s2_f ** .5 * (h.T @ Ahx_s @ xm).reshape(-1)
            mh = h @ h.T - k['iKh']
            mx = xv + xm @ xm.T - k['iKx']
            Tq = mh @ Ahx_s @ mx                                                               # [n, nh, nx]
            E = s2_f * (a_c + torch.einsum('pqij,ij->pq', Ahh_c, mh) + torch.einsum('pqkl,kl->pq', Axx_p, mx)
                        + torch.einsum('pik,qik->pq', Ahx_s, Tq))
            mus.append(mu)
            covs.append(E - mu[:, None] * mu[None, :])
    return torch.stack(mus, 1).numpy().copy(), torch.stack(covs, 0).numpy().copy()
