"""Host-side mirror of the reference's model API for the VCGPCM ELBO path.

Same names, argument meaning and error behaviour as ``src/core/cgpcm.py`` for
``VCGPCM.from_recipe`` (``:32-109``), ``precompute`` / ``undo_precompute`` (``:270-292``), ``elbo``
(``:518-575``) and the ``vars`` dictionary of trainable variables, so that
``experiment.train``'s schedule (``src/core/experiment.py:209-250``) runs unchanged.  Nothing is
computed here: the TF graph of the reference is replaced by one call into ``libcgpcm_b200.so`` per
``sess.run`` (see ``engine.Engine``).  Tensors of the reference become small lazy handles
(``Var``, ``Positive``, ``Objective``, ``Term``) that ``Session.run`` evaluates.
"""
import os

import numpy as np

from . import config
from .engine import (Engine, TERM_NAMES, GRAD_S2, GRAD_S2F, GRAD_ALPHA, GRAD_GAMMA, GRAD_OMEGA, GRAD_MU_U,
                     GRAD_VAR_U, MODE_FROZEN, MODE_FULL)
from .util import length_scale, to_float, tril_to_vec, vec_to_tril

_HEAD = ['s2', 's2_f', 'alpha', 'gamma', 'omega']
_MASK = {'s2': GRAD_S2, 's2_f': GRAD_S2F, 'alpha': GRAD_ALPHA, 'gamma': GRAD_GAMMA, 'omega': GRAD_OMEGA,
         'mu_u': GRAD_MU_U, 'var_u': GRAD_VAR_U}


# ----------------------------------------------------------------------------- lazy handles
class Var(object):
    """A trainable variable (the reference: ``tf.Variable``).  Positive quantities are stored as
    logs, exactly like ``var_pos`` (``src/core/tf_util.py:323-332``)."""

    def __init__(self, name, value):
        self.name = name
        self.value = np.array(value, dtype=np.float64)

    def assign(self, value):
        value = np.asarray(value, dtype=np.float64)
        if value.size != self.value.size:
            raise ValueError('cannot assign value of size %d to variable %r of size %d'
                             % (value.size, self.name, self.value.size))
        return _Assign(self, value.reshape(self.value.shape))

    def eval(self):
        return self.value.copy()

    @property
    def size(self):
        return self.value.size


class _Assign(object):
    def __init__(self, var, value):
        self.var, self.value = var, value

    def run(self):
        self.var.value = self.value.copy()
        return self.var.value


class Positive(object):
    """``tf.exp(var)`` of a log-variable: ``mod.s2``, ``mod.alpha`` ..."""

    def __init__(self, var):
        self.var = var

    def eval(self):
        return float(np.exp(self.var.value))

    def __float__(self):
        return self.eval()


class Term(object):
    """One of the 7 ELBO terms (``src/core/cgpcm.py:543-566``)."""

    def __init__(self, objective, index):
        self.objective, self.index = objective, index

    def eval(self):
        if hasattr(self.objective, '_run'):
            return self.objective._run()[1][self.index]
        return self.objective.mod._evaluate(want_grad=False)[1][self.index]


class Objective(object):
    """The ELBO as a lazy scalar supporting unary minus (callers minimise ``-elbo``)."""

    def __init__(self, mod, sign=1.0):
        self.mod, self.sign = mod, sign
        self.smf = False

    def __neg__(self):
        return Objective(self.mod, -self.sign)

    def eval(self):
        return self.sign * self.mod._evaluate(want_grad=False)[0]

    def value_and_grad(self, var_list):
        """Value and gradient w.r.t. the concatenation of ``var_list`` (what ``ScipyOptimizerInterface``
        fetches with one ``sess.run([loss, packed_grad])``)."""
        names = [v.name for v in var_list]
        e, _, g = self.mod._evaluate(want_grad=True, names=names)
        return self.sign * e, self.sign * self.mod._slice_grad(g, names)


class QzObjective(object):
    """``elbo(z=False)`` (``src/core/cgpcm.py:518-575``): the bound saturated for q(u) as a lazy scalar.  Value and
    terms; no task of the reference optimises q(z) directly, and no gradient is provided."""

    def __init__(self, mod, sign=1.0):
        self.mod, self.sign = mod, sign

    def __neg__(self):
        return QzObjective(self.mod, -self.sign)

    def _run(self):
        return self.mod._evaluate_qz()

    def eval(self):
        return self.sign * self._run()[0]

    def value_and_grad(self, var_list):
        raise NotImplementedError('the gradient of elbo(z=False) is not available: train q(u) with z=True '
                                  '(experiment.train does), or iterate fpi(z=False)')


class SmfObjective(object):
    """``elbo(smf=True, sample=...)`` (``src/core/cgpcm.py:527-531``) as a lazy scalar; no gradient."""

    def __init__(self, mod, sample=None, sign=1.0):
        self.mod, self.sample, self.sign = mod, sample, sign

    def __neg__(self):
        return SmfObjective(self.mod, self.sample, -self.sign)

    def _run(self):
        s = self.sample if self.sample is not None else self.mod.sample_q()
        return self.mod._evaluate_smf(s)

    def eval(self):
        return self.sign * self._run()[0]


class Session(object):
    """No-op stand-in for ``tf_util.Session`` (``src/core/tf_util.py:335-400``): owns the device choice
    and the process-group facts, and evaluates lazy handles."""

    def __init__(self, device=None, rank=None, world=None):
        self.rank, self.world = 0, 1
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                self.rank, self.world = dist.get_rank(), dist.get_world_size()
        except ImportError:
            pass
        if rank is not None:
            self.rank = rank
        if world is not None:
            self.world = world
        if device is None:
            device = int(os.environ.get('LOCAL_RANK', '0')) if self.world > 1 else 0
        self.device = device

    def run(self, fetches, feed_dict=None, **kw_args):
        if isinstance(fetches, (list, tuple)):
            return [self.run(f) for f in fetches]
        if isinstance(fetches, _Assign):
            return fetches.run()
        if hasattr(fetches, 'eval'):
            return fetches.eval()
        return fetches

    def close(self):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *args):
        return False


# ----------------------------------------------------------------------------- model
class CGPCM(object):
    """Causal Gaussian Process Convolution Model: hyper-parameters and inducing inputs."""

    _required_pars = ['sess', 'e', 'th', 'tx', 's2', 's2_f', 'alpha', 'gamma', 'omega', 'vars', 'causal',
                      'causal_id']

    def __init__(self, **kw_args):
        # same contract as Parametrisable (src/core/parametrisable.py:9-21)
        for par in self._required_pars:
            if par not in kw_args:
                raise RuntimeError('must specify "{}"'.format(par))
        for k, v in kw_args.items():
            setattr(self, k, v)
        self._precomputed = False

    @classmethod
    def from_recipe(cls, sess, e, nx, nh, tau_w, tau_f, causal, causal_id=False, noise_init=1e-4,
                    tx_range=None):
        """Generate parameters for the CGPCM and construct afterwards (``src/core/cgpcm.py:32-109``).

        :param sess: ``Session``
        :param e: observations (``.x`` inputs, ``.y`` outputs); every rank passes the *whole* series,
                  the model keeps this rank's contiguous slice
        :param nx: number of inducing points for noise
        :param nh: number of inducing points for filter
        :param tau_w: length of kernel window
        :param tau_f: length scale of function prior
        :param causal: causal model
        :param causal_id: causal interdomain transformation
        :param noise_init: initialisation of noise
        :param tx_range: range of the inducing points for x, taken from ``e`` by default
        """
        vars = {}
        tau_ws = 1
        causal_extra_points = 2

        def var_pos(name, init):
            vars[name] = Var(name, np.log(init))
            return Positive(vars[name])

        alpha = 2 * length_scale(tau_w)
        gamma = length_scale(tau_f) - .5 * alpha
        s2_f = var_pos('s2_f', to_float((2 * alpha / np.pi) ** .5))
        if causal:
            gamma += 3. * alpha / 8.
            alpha /= 4.
        alpha = var_pos('alpha', to_float(alpha))
        gamma = var_pos('gamma', to_float(gamma))
        if nx > 0:
            tx_range = (min(e.x), max(e.x)) if tx_range is None else tx_range
            dtx = (tx_range[1] - tx_range[0]) / nx
            omega = .5 * length_scale(dtx)
            tx = np.linspace(tx_range[0], tx_range[1], nx)
        else:
            # the AKM has no noise-side inducing inputs (src/core/cgpcm.py:77-79): omega = nan, tx = []
            omega = np.nan
            tx = np.zeros(0)
        omega = var_pos('omega', to_float(omega))
        if not causal and nh % 2 == 0:
            nh += 1
        if causal:
            th = np.linspace(0, 2 * tau_ws * tau_w, nh)
            dth = th[1] - th[0]
            th = th - dth * causal_extra_points
        else:
            th = np.linspace(-tau_ws * tau_w, tau_ws * tau_w, nh)
        s2 = var_pos('s2', to_float(noise_init))
        return cls(sess=sess, th=th, tx=tx, s2=s2, s2_f=s2_f, alpha=alpha, gamma=gamma, omega=omega, vars=vars,
                   e=e, causal=causal, causal_id=causal_id, tau_w=tau_w, tau_f=tau_f, nh=nh, nx=nx,
                   noise_init=noise_init, tx_range=tx_range)


def shard_bounds(n, rank, world, cost=None):
    """Contiguous slice ``[lo, hi)`` of ``n`` observations owned by ``rank``.  Without ``cost`` the sizes differ by
    <= 1; with ``cost`` (``n`` non-negative per-observation costs, see ``window_costs``) the slices carry equal shares
    of the total cost: observations near the ends of a series see fewer inducing inputs of the noise process inside
    their window and are cheaper, so equal counts would leave the inner ranks with ~35 % more work."""
    if cost is not None and world > 1 and n >= world:
        cum = np.cumsum(np.asarray(cost, dtype=np.float64))
        if cum.shape[0] != n:
            raise ValueError('cost must have one entry per observation')
        if cum[-1] > 0:
            cuts = [0]
            for r in range(1, world):
                c = int(np.searchsorted(cum, cum[-1] * r / world))
                cuts.append(min(max(c, cuts[-1] + 1), n - (world - r)))      # every rank keeps >= 1 observation
            cuts.append(n)
            return cuts[rank], cuts[rank + 1]
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def rebalance_costs(cost, bounds, times):
    """Per-observation costs corrected by measured shard times: ``bounds[r] = (lo, hi)`` of rank ``r`` under ``cost`` and
    ``times[r]`` the device time its sweeps took.  Every observation of shard ``r`` is rescaled by the ratio of the
    shard's measured share to its modelled share, so that ``shard_bounds`` on the result moves the cuts towards equal
    *measured* time (the model of ``window_costs`` is per observation; chunk windows are unions rounded to multiples
    of eight and the GEMM kernels are less efficient on the narrow windows at the ends of a series: the end shards of
    an 8-way split of the bench series ran 3 % and 10 % longer than the inner ones).  Pure host logic, no
    communication: the caller gathers ``times``."""
    cost = np.array(cost, dtype=np.float64)
    times = np.asarray(times, dtype=np.float64)
    if len(bounds) != times.shape[0] or np.any(times <= 0):
        raise ValueError('one positive time per shard')
    model = np.array([cost[lo:hi].sum() for lo, hi in bounds])
    if np.any(model <= 0):
        return cost
    scale = (times / times.sum()) / (model / model.sum())
    for (lo, hi), f in zip(bounds, scale):
        cost[lo:hi] *= f
    return cost


def window_radius(alpha, gamma, omega, cull):
    """``|t - tx|`` beyond which every ``Ahx`` element has a Gaussian envelope below ``exp(-cull)``: the radius
    ``plan_chunks`` (csrc/cgpcm.cu) gives the windows of inducing inputs (``cull = 746``: exactly 0 in IEEE double)."""
    A = alpha + gamma + omega
    e_hh = ((alpha + gamma) * A - gamma * gamma) / A
    e_dd = omega * (alpha + gamma) / A
    e_hd = 2.0 * gamma * omega / A
    lam = e_dd - e_hd * e_hd / (4.0 * e_hh)
    return float(np.sqrt(cull / lam)) if (cull > 0 and lam > 0) else float('inf')


def window_costs(t, tx, nh, radius):
    """Per-observation cost proxy for ``shard_bounds``: with ``kw`` inducing inputs of the noise process inside the
    window of observation ``n``, the contractions cost ``nh kw (4 nh + 7 kw)`` flop (T1, Q, Hbar: ``nh^2 kw``-type;
    right-multiplies and C1: ``nh kw^2``-type), the Ahx kernels ``~ nh kw`` and the Axx kernel ``~ kw^2`` elements
    (weights from the bench shape's per-kernel times, profiles/r01_launches_exact746_N1e5_M200.csv), plus a
    per-observation term for what does not shrink with the window."""
    t = np.asarray(t, dtype=np.float64)
    txs = np.sort(np.asarray(tx, dtype=np.float64))
    if not np.isfinite(radius):
        return np.ones(t.shape[0])
    kw = (np.searchsorted(txs, t + radius, side='right') - np.searchsorted(txs, t - radius, side='left')).astype(np.float64)
    kw = np.maximum(kw, 8.0)
    return nh * kw * (4.0 * nh + 7.0 * kw + 430.0) + 480.0 * kw * kw + 100.0 * nh * txs.shape[0]


class AKM(CGPCM):
    """Approximate Kernel Model (``src/core/cgpcm.py:295-422``): the generative model the toy experiment's series are
    drawn from (``data.load_akm``).  Filter draw ``h ~ N(0, reg(iKh))`` in the reference's parametrisation, function
    draw ``f = sqrt(s2_f) chol(reg(K)) e`` with ``K = a + tr((h h^T - iKh) Ahh)`` at all pairs of inputs
    (``cgpcm_akm_sample``), kernel ``k`` at lags (``cgpcm_kernel_samples``)."""

    _required_pars = ['sess', 'th', 's2', 's2_f', 'alpha', 'gamma', 'causal', 'causal_id']

    def __init__(self, **kw_args):
        CGPCM.__init__(self, **kw_args)
        self.th = np.ascontiguousarray(self.th, dtype=np.float64)
        self.nh = self.th.shape[0]
        # the engine wants a noise side: eight dummy inducing inputs and omega = 1, none of which the AKM's
        # statistics (functions of th, alpha, gamma only) read
        self.engine = Engine(self.nh, 8, causal=self.causal, causal_id=False, device=getattr(self.sess, 'device', 0))
        self.engine.set_data(np.zeros(1), np.zeros(1), self.th, np.linspace(0., 1., 8))
        self.h_draw = self.e_draw = self.t = None
        self._rng = getattr(self.sess, 'rng', None) or np.random

    def _pack5(self):
        return np.array([float(self.vars['s2'].value), float(self.vars['s2_f'].value), float(self.vars['alpha'].value),
                         float(self.vars['gamma'].value), 0.0])

    def _prior_factor(self):
        """Cholesky factor of ``reg(iKh)``, the covariance of ``h_prior`` (``cgpcm.py:216-220``)."""
        r = config.reg
        alpha, gamma, th = self.alpha.eval(), self.gamma.eval(), self.th
        Kh = np.exp(-alpha * (th[:, None] ** 2 + th[None, :] ** 2) - gamma * (th[:, None] - th[None, :]) ** 2)
        Lh = np.linalg.cholesky(Kh + r * np.eye(self.nh))
        iLh = np.linalg.solve(Lh, np.eye(self.nh))
        return np.linalg.cholesky(iLh.T @ iLh + r * np.eye(self.nh))

    def sample_h(self, h=None):
        """Sample filter (``cgpcm.py:353-362``); ``h``: a draw in the parametrisation of the filter."""
        if h is None:
            self.h_draw = self._prior_factor() @ self._rng.randn(self.nh, 1)
        else:
            self.h_draw = np.asarray(h, dtype=np.float64).reshape(self.nh, 1)

    def sample_f(self, t):
        """Sample function (``cgpcm.py:364-371``)."""
        self.t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        self.e_draw = self._rng.randn(self.t.shape[0], 1)

    def sample(self, t, h=None):
        """Sample filter and function (``cgpcm.py:373-380``)."""
        self.sample_h(h)
        self.sample_f(t)

    def f(self):
        """Construct function (``cgpcm.py:382-392``)."""
        from .data import Data
        return Data(self.t, self.engine.akm_sample(self._pack5(), self.t, self.h_draw, self.e_draw, reg=config.reg))

    def h(self, t):
        """Construct filter (``cgpcm.py:394-408``): ``k_h(t, th) h``, positive times only for the causal model."""
        from .data import Data
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        alpha, gamma, th = self.alpha.eval(), self.gamma.eval(), self.th
        Kfu = np.exp(-alpha * (t[:, None] ** 2 + th[None, :] ** 2) - gamma * (t[:, None] - th[None, :]) ** 2)
        d = Data(t, (Kfu @ self.h_draw).ravel())
        return d.positive_part() if self.causal else d

    def k(self, t):
        """Construct the kernel (``cgpcm.py:410-421``)."""
        from .data import Data
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        return Data(t, self.engine.kernel_samples(self._pack5(), t, self.h_draw.reshape(1, -1), reg=config.reg)[:, 0])

    def k_prior(self, t, iters=1000, psd=False, granularity=1):
        """Prior distribution over kernels or PSDs (``cgpcm.py:304-351``): mean, lists of lower and upper bounds."""
        from .data import Data
        from .util import fft_spectrum
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        hs = (self._prior_factor() @ self._rng.randn(self.nh, int(iters))).T
        samples = self.engine.kernel_samples(self._pack5(), t, hs, reg=config.reg)                # [n, iters]
        x = t
        if psd:
            x, spec = fft_spectrum(t, samples)
            samples = np.abs(spec)
        mu = samples.mean(axis=1)
        qs = np.arange(granularity, 50 - granularity, granularity)
        lowers = [Data(x, np.percentile(samples, q, axis=1)) for q in qs]
        uppers = [Data(x, np.percentile(samples, 100 - q, axis=1)) for q in qs]
        return Data(x, mu), lowers, uppers


class VCGPCM(CGPCM):
    """Variational inference in the CGPCM (``src/core/cgpcm.py:425-872``), ELBO path."""

    def __init__(self, **kw_args):
        CGPCM.__init__(self, **kw_args)
        if np.size(self.tx) == 0:
            raise ValueError('nx must be positive')
        self.th = np.ascontiguousarray(self.th, dtype=np.float64)
        self.tx = np.ascontiguousarray(self.tx, dtype=np.float64)
        self.nh, self.nx = self.th.shape[0], self.tx.shape[0]
        self.n = self.e.x.shape[0]
        self.sum_y2 = float(np.sum(self.e.y ** 2))
        sess = self.sess
        self.engine = Engine(self.nh, self.nx, causal=self.causal, causal_id=self.causal_id,
                             device=getattr(sess, 'device', 0))
        rank, world = getattr(sess, 'rank', 0), getattr(sess, 'world', 1)
        # Every host-side random draw (mu_u, q(u) / prior samples, prediction noise, the slice sampler's angles) must
        # be the SAME on every rank: the ranks contract their shards with these values and NCCL sums the partials.
        # One process: numpy's global generator, as in the reference (np.random.seed controls it).  Several ranks: a
        # private generator seeded with a value rank 0 draws from ITS global generator and broadcasts.
        self._rng = getattr(sess, 'rng', None) or np.random       # batch.run gives every task a private generator
        if world > 1:
            self._init_comm(rank, world)
            self._rng = np.random.RandomState(self._shared_seed(rank))
        cost = None
        if world > 1:
            # balance the shards at the recipe's hyper-parameters and the library's default cull (80)
            cost = window_costs(self.e.x, self.tx, self.nh,
                                window_radius(self.alpha.eval(), self.gamma.eval(), self.omega.eval(), 80.0))
        lo, hi = shard_bounds(self.n, rank, world, cost)
        self.engine.set_data(self.e.x[lo:hi], self.e.y[lo:hi], self.th, self.tx)
        self._init_inducing_points()
        if world > 1:
            # host LAPACK is not guaranteed to be bit-identical across ranks (thread counts differ): rank 0's q(u) wins
            import torch.distributed as dist
            names = ('mu_u', 'var_u', 'mu_z', 'var_z')
            box = [tuple(self.vars[k].value for k in names) if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            for k, v in zip(names, box[0]):
                self.vars[k].value = v.copy()
        self._cache = None
        self._frozen_hyp = None

    def _init_comm(self, rank, world):
        import torch.distributed as dist
        box = [Engine.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        self.engine.comm_init(box[0], rank, world)

    @staticmethod
    def _shared_seed(rank):
        import torch.distributed as dist
        box = [int(np.random.randint(0, 2 ** 31 - 1)) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    def _init_inducing_points(self):
        """``src/core/cgpcm.py:435-445``: ``mu_u ~ N(0, reg(iKh))``, ``var_u = tril_to_vec(chol(reg(iKh)))``.
        Host numpy on an nh x nh matrix, once per model; the reference draws with the TF RNG."""
        r = config.reg
        alpha, gamma = self.alpha.eval(), self.gamma.eval()
        th = self.th
        Kh = np.exp(-alpha * (th[:, None] ** 2 + th[None, :] ** 2) - gamma * (th[:, None] - th[None, :]) ** 2)
        Kh = Kh + r * np.eye(self.nh)
        Lh = np.linalg.cholesky(Kh)
        iLh = np.linalg.solve(Lh, np.eye(self.nh))
        iKh = iLh.T @ iLh
        Lp = np.linalg.cholesky(iKh + r * np.eye(self.nh))
        self.vars['mu_u'] = Var('mu_u', Lp @ self._rng.randn(self.nh, 1))
        self._prior_factor_cache = ((alpha, gamma, r), Lp)
        self.vars['var_u'] = Var('var_u', tril_to_vec(Lp))
        # q(z) (cgpcm.py:447-456): mu_z ~ N(0, reg(iKx)), var_z = tril_to_vec(chol(reg(iKx))); only the z = False
        # variants read it before convert() assigns it
        omega, tx = self.omega.eval(), self.tx
        Kx = (.5 * np.pi / omega) ** .5 * np.exp(-.5 * omega * (tx[:, None] - tx[None, :]) ** 2) + r * np.eye(self.nx)
        iLx = np.linalg.solve(np.linalg.cholesky(Kx), np.eye(self.nx))
        Lz = np.linalg.cholesky(iLx.T @ iLx + r * np.eye(self.nx))
        self.vars['mu_z'] = Var('mu_z', Lz @ self._rng.randn(self.nx, 1))
        self.vars['var_z'] = Var('var_z', tril_to_vec(Lz))

    # -- parameter vector of the C-ABI
    def _pack(self):
        return np.concatenate([np.array([float(self.vars[k].value) for k in _HEAD]),
                               self.vars['mu_u'].value.ravel(), self.vars['var_u'].value.ravel()])

    def _slice_grad(self, g, names):
        parts = []
        for nm in names:
            if nm in _HEAD:
                parts.append(g[_HEAD.index(nm):_HEAD.index(nm) + 1])
            elif nm == 'mu_u':
                parts.append(g[5:5 + self.nh])
            elif nm == 'var_u':
                parts.append(g[5 + self.nh:])
            else:
                raise KeyError('variable %r is not on the ELBO path' % nm)
        return np.concatenate(parts)

    def _evaluate(self, want_grad, names=None):
        p = self._pack()
        mode = MODE_FROZEN if self._precomputed else MODE_FULL
        mask = 0
        for nm in (names or []):
            mask |= _MASK[nm]
        key = (p.tobytes(), mode, config.reg, mask if want_grad else -1)
        if self._cache is not None and self._cache[0][:3] == key[:3] and (
                not want_grad or self._cache[0][3] == key[3]):
            return self._cache[1]
        out = self.engine.elbo_grad(p, mode=mode, grad_mask=mask, reg=config.reg, want_grad=want_grad)
        self._cache = (key, out)
        return out

    # -- reference API
    def precompute(self, recompute=False):
        """Freeze the Psi statistics at the current hyper-parameters (``src/core/cgpcm.py:270-284``)."""
        if recompute and self._precomputed:
            self.undo_precompute()
        if not self._precomputed:
            hyp = (self.alpha.eval(), self.gamma.eval(), self.omega.eval())
            self.engine.precompute(hyp[0], hyp[1], hyp[2], config.reg)
            self._frozen_hyp = hyp
            self._precomputed = True
            self._cache = None

    def undo_precompute(self):
        """Revert precomputation (``src/core/cgpcm.py:286-292``)."""
        if self._precomputed:
            self._precomputed = False
            self._cache = None

    def elbo(self, smf=False, sample=None, z=True):
        """Construct the ELBO: ``(elbo, terms)`` with ``terms`` the 7 named fetches
        (``src/core/cgpcm.py:518-575``).  ``smf=True``: the stochastic SMF bound at ``sample`` (a fresh draw from
        q(u) per evaluation if ``None``); value only."""
        if not z:
            if smf:
                raise NotImplementedError('the SMF bound is only available saturated for q(z) (z=True)')
            obj = QzObjective(self)
            names = ['s2 complexity', 'p(u) complexity', 'q*(u) complexity', 'q*(u) fit',
                     'general conditioning penalty', 'q(z conditioning penalty', '-KL[q(u)||p(u)]']   # sic: cgpcm.py:559-564
            terms = [{'name': nm, 'tensor': Term(obj, i), 'modifier': '.2e'} for i, nm in enumerate(names)]
            return obj, terms
        if smf:
            obj = SmfObjective(self, sample)
            terms = [{'name': nm, 'tensor': Term(obj, i), 'modifier': '.2e'} for i, nm in enumerate(TERM_NAMES)]
            return obj, terms
        obj = Objective(self)
        terms = [{'name': nm, 'tensor': Term(obj, i), 'modifier': '.2e'} for i, nm in enumerate(TERM_NAMES)]
        return obj, terms

    def _with_frozen_stats(self, fn):
        temporary = not self._precomputed
        if temporary:                      # symbolic mats in the reference = statistics at the current hyper-parameters
            self.precompute()
        try:
            return fn()
        finally:
            if temporary:
                self.undo_precompute()

    def _fpi(self, num, high_reg, z=True):
        if z:
            return self._with_frozen_stats(lambda: self.engine.fpi(self._pack(), num, high_reg=high_reg, reg=config.reg))
        return self._with_frozen_stats(lambda: self.engine.fpi_qz(
            self._pack(), self.vars['mu_z'].value, self.vars['var_z'].value, num, high_reg=high_reg, reg=config.reg))

    def _evaluate_qz(self):
        return self._with_frozen_stats(lambda: self.engine.elbo_qz(
            self._pack(), self.vars['mu_z'].value, self.vars['var_z'].value, reg=config.reg))

    def fpi(self, num=50, z=True, high_reg=False):
        """Fixed-point iteration on q(u) (``src/core/cgpcm.py:479-516``): ``num`` rounds of optimal q(z) given q(u),
        optimal q(u) given q(z); assigns ``mu_u`` and ``var_u``."""
        if not z:
            # fixed-point iteration on q(z): q(z) -> optimal q(u) -> optimal q(z); assigns mu_z and var_z
            _, _, mu_z, var_z = self._fpi(num, high_reg, z=False)
            self.vars['mu_z'].value = mu_z.reshape(self.vars['mu_z'].value.shape)
            self.vars['var_z'].value = var_z
            return
        mu_u, var_u, _, _ = self._fpi(num, high_reg)
        self.vars['mu_u'].value = mu_u.reshape(self.vars['mu_u'].value.shape)
        self.vars['var_u'].value = var_u
        self._cache = None

    def convert(self, z=True):
        """Assign q(z) after optimising q(u) (``src/core/cgpcm.py:577-592``): ``vars['mu_z']``, ``vars['var_z']``."""
        if not z:
            # assign q(u) after optimising q(z)
            mu_u, var_u, _, _ = self._fpi(0, False, z=False)
            self.vars['mu_u'].value = mu_u.reshape(self.vars['mu_u'].value.shape)
            self.vars['var_u'].value = var_u
            self._cache = None
            return
        _, _, mu_z, var_z = self._fpi(0, False)
        self.vars['mu_z'] = Var('mu_z', mu_z.reshape(-1, 1))
        self.vars['var_z'] = Var('var_z', var_z)

    # -- SMF bound and posterior samples of the filter (src/core/cgpcm.py:527-531,594-608,848-872)
    def _evaluate_smf(self, sample):
        mode = MODE_FROZEN if self._precomputed else MODE_FULL
        return self.engine.elbo_smf(self._pack(), sample, mode=mode, reg=config.reg)

    def _q_cov_factor(self):
        L = vec_to_tril(self.vars['var_u'].value)
        return np.linalg.cholesky(L @ L.T + config.reg * np.eye(self.nh))

    def sample_q(self):
        """A draw from q(u) = N(mu_u, reg(L L^T)) (``Normal.sample``, ``src/core/distribution.py:44-58``)."""
        return self.vars['mu_u'].value.reshape(-1, 1) + self._q_cov_factor() @ self._rng.randn(self.nh, 1)

    def _prior_factor(self):
        """Cholesky factor of ``reg(iKh)`` (``src/core/cgpcm.py:216-220``), cached per (alpha, gamma, reg): the slice
        sampler asks for one prior draw per step and the factor only changes with the hyper-parameters."""
        alpha, gamma, r = self.alpha.eval(), self.gamma.eval(), config.reg
        cache = getattr(self, '_prior_factor_cache', None)
        if cache is not None and cache[0] == (alpha, gamma, r):
            return cache[1]
        th = self.th
        Kh = np.exp(-alpha * (th[:, None] ** 2 + th[None, :] ** 2) - gamma * (th[:, None] - th[None, :]) ** 2)
        Lh = np.linalg.cholesky(Kh + r * np.eye(self.nh))
        iLh = np.linalg.solve(Lh, np.eye(self.nh))
        Lp = np.linalg.cholesky(iLh.T @ iLh + r * np.eye(self.nh))
        self._prior_factor_cache = ((alpha, gamma, r), Lp)
        return Lp

    def sample_prior(self):
        """A draw from the prior of ``K_u^-1 u``: ``N(0, reg(iKh))`` (``src/core/cgpcm.py:219-220``)."""
        return self._prior_factor() @ self._rng.randn(self.nh, 1)

    def elbo_smf(self, samples_h):
        """Monte-Carlo estimate of the SMF bound: ``(mean, standard error)`` (``src/core/cgpcm.py:594-608``)."""
        elbos = [self._evaluate_smf(x)[0] for x in samples_h]
        return np.mean(elbos), np.std(elbos) / len(samples_h) ** .5

    def sample(self, iters=200, burn=None, chains=1):
        """Samples from the posterior over filters by elliptical slice sampling (``src/core/cgpcm.py:848-872``).
        ``chains > 1``: that many chains from the mean of q(u), each with a generator seeded from the model's, whose
        proposals are scored together (``Engine.elbo_smf_batch``, precomputed regime); returns one list of ``iters``
        states per chain."""
        from .sample import ESS, MultiESS
        if burn is None:
            burn = iters
        if chains == 1:
            ess = ESS(lambda x: self._evaluate_smf(x)[2], self.sample_prior, rng=self._rng)
            ess.move(self.vars['mu_u'].value.reshape(-1, 1))
            if burn > 0:
                ess.sample(burn)
            return ess.sample(iters)
        if chains < 1:
            raise ValueError('chains must be >= 1')
        rngs = [np.random.RandomState(int(s)) for s in self._rng.randint(0, 2 ** 31 - 1, size=int(chains))]
        mu = self.vars['mu_u'].value.reshape(-1, 1)

        def run():
            p = self._pack()
            mess = MultiESS(lambda xs: self.engine.elbo_smf_batch(p, np.stack([x.ravel() for x in xs]), reg=config.reg,
                                                                  want_elbo=False)[2],
                            [lambda r=r: self._prior_factor() @ r.randn(self.nh, 1) for r in rngs],
                            x_inits=[mu.copy() for _ in rngs], rngs=rngs)
            if burn > 0:
                mess.sample(burn)
            return mess.sample(iters)
        return self._with_frozen_stats(run)

    def predict_f(self, t, samples_h=50, precompute=True):
        """Predict the function at ``t`` (``src/core/cgpcm.py:781-846``).  ``samples_h`` numeric: that many draws
        from q(u) with the optimal q(z) of q(u); a list of filter samples (e.g. from :meth:`sample`): the SMF
        approximation, q(z | h) per sample.  Returns ``UncertainData(mean, lower, upper, std)`` of ``Data``."""
        from .data import Data, UncertainData
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        if np.isscalar(samples_h) or isinstance(samples_h, (int, np.integer)):
            samples, smf = [self.sample_q() for _ in range(int(samples_h))], False
        else:
            samples, smf = list(samples_h), True
        samples = np.stack([np.asarray(x, dtype=np.float64).ravel() for x in samples])
        temporary = not self._precomputed
        if temporary:
            self.precompute()
        try:
            mu, var = self.engine.predict_f(self._pack(), t, samples, smf=smf, reg=config.reg)
        finally:
            if temporary:
                self.undo_precompute()
        std = np.maximum(var, 0) ** .5
        return UncertainData(mean=Data(t, mu), lower=Data(t, mu - 2 * std), upper=Data(t, mu + 2 * std),
                             std=Data(t, std))

    def predict_f_samples(self, t, samples_h=50):
        """Predictive mean and variance of the function at ``t`` for each filter sample: ``(mean[n, B], var[n, B])``.
        ``samples_h`` as in :meth:`predict_f`: a number draws that many samples from q(u), all under the optimal q(z)
        of q(u); a list of filter samples (e.g. the states of :meth:`sample`, flattened over chains) gives each its
        own q(z | h_b).  :meth:`predict_f`'s mean and variance are the row means ``mean.mean(1)`` and ``var.mean(1)``;
        the variance of the mixture of the samples' predictive distributions is ``var.mean(1) + mean.var(1)``."""
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        if np.isscalar(samples_h) or isinstance(samples_h, (int, np.integer)):
            samples, smf = [self.sample_q() for _ in range(int(samples_h))], False
        else:
            samples, smf = list(samples_h), True
        samples = np.stack([np.asarray(x, dtype=np.float64).ravel() for x in samples])
        _, _, mean, var = self._with_frozen_stats(
            lambda: self.engine.predict_f_batch(self._pack(), t, samples, smf=smf, reg=config.reg))
        return mean, var

    def _filter_batch(self, samples_h):
        if np.isscalar(samples_h) or isinstance(samples_h, (int, np.integer)):
            samples, smf = [self.sample_q() for _ in range(int(samples_h))], False
        else:
            samples, smf = list(samples_h), True
        return np.stack([np.asarray(x, dtype=np.float64).ravel() for x in samples]), smf

    def predict_f_cov(self, t, samples_h=50, per_sample=False):
        """Joint predictive distribution of the function at ``t`` (at most 4096 inputs): ``(mean[n], cov[n, n])`` with
        ``cov`` the covariance of the mixture of the samples' predictive distributions, ``cov_avg + Cov_b(mean_s)``;
        ``cov_avg``, the sample average of the per-sample covariances, has :meth:`predict_f`'s variance on its
        diagonal.  ``samples_h`` as in :meth:`predict_f_samples`.  ``per_sample=True`` also returns
        ``(mean_s[n, B], cov_s[B, n, n])``, each sample's mean and covariance."""
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        samples, smf = self._filter_batch(samples_h)
        mean, cov, mean_s, cov_s, _ = self._with_frozen_stats(lambda: self.engine.predict_f_cov(
            self._pack(), t, samples, smf=smf, reg=config.reg, per_sample=per_sample))
        mix = cov + np.atleast_2d(np.cov(mean_s, bias=True))
        return (mean, mix, mean_s, cov_s) if per_sample else (mean, mix)

    def sample_f(self, t, samples_h=50):
        """Posterior sample paths of the function at ``t`` (at most 4096 inputs), one per filter sample: ``[n, B]``,
        column b a draw from the joint predictive distribution under sample b's q(z) (``samples_h`` as in
        :meth:`predict_f_samples`).  The standard normal noise comes from the model's generator, so every rank draws
        the same paths."""
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        samples, smf = self._filter_batch(samples_h)
        noise = self._rng.randn(t.shape[0], samples.shape[0])
        return self._with_frozen_stats(lambda: self.engine.predict_f_cov(
            self._pack(), t, samples, smf=smf, reg=config.reg, noise=noise))[4]

    def log_predictive_density(self, t, y, samples_h=50, joint=True, noise=True, per_sample=False):
        """Log density of held-out values ``y`` at ``t`` under the mixture of the samples' predictive distributions
        (``samples_h`` as in :meth:`predict_f_samples`).  ``noise=True``: ``y`` are observations, each sample's
        predictive covariance plus ``s2 I``; ``noise=False``: ``y`` is the function itself, plus ``reg I``.

        ``joint=True`` (at most 4096 inputs): the joint log density of the block, ``log mean_b N(y; m_b, C_b + d I)``
        (:meth:`Engine.predict_logpdf`); ``per_sample=True`` returns ``(lp, lp_s[B], white[n, B])``, each sample's
        joint log density and whitened residuals.  ``joint=False``: the log density of each point under the mixture of
        the samples' marginals, ``log mean_b N(y_p; m_bp, v_bp + d)``, an array ``[n]`` (no limit on n);
        ``per_sample=True`` returns ``(lp[n], lp_s[n, B])``."""
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        y = np.asarray(getattr(y, 'y', y), dtype=np.float64).ravel()
        if y.shape != t.shape:
            raise ValueError('y must have one value per input')
        samples, smf = self._filter_batch(samples_h)
        if joint:
            lp, lp_s, white = self._with_frozen_stats(lambda: self.engine.predict_logpdf(
                self._pack(), t, y, samples, smf=smf, reg=config.reg, noise=noise, white=per_sample))
            return (lp, lp_s, white) if per_sample else lp
        p = self._pack()
        _, _, mean, var = self._with_frozen_stats(
            lambda: self.engine.predict_f_batch(p, t, samples, smf=smf, reg=config.reg))
        v = var + (np.exp(p[0]) if noise else config.reg)
        bad = np.argwhere(~(v > 0))
        if bad.size:
            i, b = bad[0]
            raise ValueError('predictive variance %g of sample %d at point %d is not positive' % (v[i, b], b, i))
        lp_s = -.5 * (np.log(2 * np.pi * v) + (y[:, None] - mean) ** 2 / v)
        # log mean_b exp(lp_s[:, b]), shifted by the largest term and added in ascending b
        top = lp_s.max(1)
        acc = np.zeros(t.shape[0])
        for b in range(lp_s.shape[1]):
            acc += np.exp(lp_s[:, b] - top)
        lp = top + np.log(acc) - np.log(lp_s.shape[1])
        return (lp, lp_s) if per_sample else lp

    def predict_k(self, t, samples_h=200, psd=False, normalise=True):
        """Predict the kernel, or the PSD via the kernel approximation, at lags ``t``
        (``src/core/cgpcm.py:610-661``): Monte-Carlo over filter samples (numeric ``samples_h``: draws from q(u)).
        The kernel samples come from the GPU (``cgpcm_kernel_samples``); normalisation, the FFT and the percentile
        band are post-processing of those samples.  Returns ``UncertainData(mean, lower, upper, std)``."""
        from .data import Data, UncertainData
        from .util import fft_spectrum, lower_perc, upper_perc
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        if np.isscalar(samples_h) or isinstance(samples_h, (int, np.integer)):
            samples = [self.sample_q() for _ in range(int(samples_h))]
        else:
            samples = list(samples_h)
        samples = np.stack([np.asarray(x, dtype=np.float64).ravel() for x in samples])
        k = self.engine.kernel_samples(self._pack(), t, samples, reg=config.reg)          # [n, B]
        if normalise:
            k = k / k.max(axis=0, keepdims=True)
        x = t
        if psd:
            x, spec = fft_spectrum(t, k)
            k = np.abs(spec)
        return UncertainData(mean=Data(x, k.mean(axis=1)), lower=Data(x, np.percentile(k, lower_perc, axis=1)),
                             upper=Data(x, np.percentile(k, upper_perc, axis=1)), std=Data(x, k.std(axis=1)))

    def _filter_draws(self, t, samples_h):
        if np.isscalar(samples_h) or isinstance(samples_h, (int, np.integer)):
            samples = [self.sample_q() for _ in range(int(samples_h))]
        else:
            samples = list(samples_h)
        samples = np.stack([np.asarray(x, dtype=np.float64).ravel() for x in samples])
        noise = self._rng.randn(t.shape[0], samples.shape[0])
        return self.engine.filter_samples(self._pack(), t, samples, noise, reg=config.reg)       # [n, B]

    @staticmethod
    def _mc_stats(x, samples):
        from .data import Data, UncertainData
        from .util import lower_perc, upper_perc
        return UncertainData(mean=Data(x, samples.mean(axis=1)), lower=Data(x, np.percentile(samples, lower_perc, axis=1)),
                             upper=Data(x, np.percentile(samples, upper_perc, axis=1)), std=Data(x, samples.std(axis=1)))

    def predict_h(self, t, samples_h=500, normalise=True, phase_transform='minimum_phase'):
        """Predict the filter at ``t`` (``src/core/cgpcm.py:714-779``).  The posterior draws of the filter come from the
        GPU (``cgpcm_filter_samples``); the positive part, the phase transform (``None``, ``'minimum_phase'`` or
        ``'zero_phase'``, the three ``experiment.predict`` asks for, ``src/core/experiment.py:316-321``), the energy
        normalisation and the percentile band are post-processing of those draws."""
        from .util import minimum_phase, zero_phase, energy
        if phase_transform not in (None, 'minimum_phase', 'zero_phase'):
            raise NotImplementedError('phase_transform must be None, "minimum_phase" or "zero_phase"')
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        draws = self._filter_draws(t, samples_h)
        keep = t >= 0 if self.causal else np.ones(t.shape[0], dtype=bool)
        x = t[keep]
        x_out = zero_phase(x, np.zeros_like(x))[0] if phase_transform == 'zero_phase' else x
        cols = []
        for b in range(draws.shape[1]):
            y = draws[keep, b]
            if phase_transform == 'minimum_phase':
                y = minimum_phase(y)
            elif phase_transform == 'zero_phase':
                y = zero_phase(x, y)[1]
            if normalise:
                y = y / energy(x_out, y) ** .5
            cols.append(y)
        return self._mc_stats(x_out, np.stack(cols, 1))

    def predict_psd(self, t, samples_h=500, normalise=True):
        """Predict the PSD from posterior draws of the filter (``src/core/cgpcm.py:663-712``): autocorrelation of
        every draw, then the reference's FFT convention."""
        from .util import autocorrelation, fft_spectrum
        t = np.asarray(getattr(t, 'x', t), dtype=np.float64).ravel()
        draws = self._filter_draws(t, samples_h)
        cols, freq = [], None
        for b in range(draws.shape[1]):
            lags, ac = autocorrelation(t, draws[:, b], normalise=normalise)
            freq, spec = fft_spectrum(lags, ac)
            cols.append(np.abs(spec))
        return self._mc_stats(freq, np.stack(cols, 1))

    @property
    def mats(self):
        """The sums of ``mats`` the ELBO reads (``src/core/cgpcm.py:235-267``) at the current (or frozen)
        hyper-parameters as numpy arrays: ``a, Ahh, sum_a, sum_Ahh, sum_Axx, sum_Ahx_y, sum_b, sum_Bxx, sum_Bhh``.
        (The per-observation tensors ``Axx, Ahx, b, Bxx, Bhh`` that the reference also keeps are never materialised;
        ``engine.psi(..., per_observation=True)`` returns ``Axx`` / ``Ahx`` on request.)"""
        hyp = self._frozen_hyp if self._precomputed else (self.alpha.eval(), self.gamma.eval(), self.omega.eval())
        out = self.engine.psi(*hyp)
        out.update(self._with_frozen_stats(self.engine.frozen_mats))
        out['sum_a'] = self.n * out['a']
        out['sum_Ahh'] = self.n * out['Ahh']
        return out
