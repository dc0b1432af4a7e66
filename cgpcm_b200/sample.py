"""Elliptical slice sampling (Murray, Adams & MacKay 2010) with the interface of the reference's ``ESS``
(``src/core/sample.py:8-130``): ``ESS(log_lik, sample_prior, x_init)``, ``move``, ``update``, ``sample(num)``.

``log_lik`` returns the log of a quantity proportional to the likelihood of the target; ``sample_prior`` draws from
the zero-mean Gaussian prior.  Every state is a point on the ellipse through the current state and a fresh prior
draw; the bracket of the angle shrinks towards 0 until the proposal lies above the slice.

``MultiESS`` runs several such chains in lock-step so that one call of a batched log-likelihood scores the pending
proposals of all chains."""
import numpy as np


class ESS(object):
    _min_theta = 1e-10

    def __init__(self, log_lik, sample_prior, x_init=None, rng=None):
        self._log_lik = log_lik
        self._sample_prior = sample_prior
        self._rng = rng if rng is not None else np.random
        self._x = sample_prior() if x_init is None else x_init
        self._log_lik_x = log_lik(self._x)
        self.attempts = []

    def move(self, x, log_lik=None):
        """Move the sampler to a new state."""
        self._x = x
        self._log_lik_x = self._log_lik(x) if log_lik is None else log_lik

    def update(self, log_lik):
        """Replace the log-likelihood function."""
        self._log_lik = log_lik

    def _step(self):
        u = self._log_lik_x - self._rng.exponential(1.0)          # slice height
        nu = self._sample_prior()                                  # the ellipse
        theta = self._rng.uniform(0, 2 * np.pi)
        lo, hi = theta - 2 * np.pi, theta
        attempts = 0
        while True:
            attempts += 1
            theta = self._rng.uniform(lo, hi)
            x = np.cos(theta) * self._x + np.sin(theta) * nu
            ll = self._log_lik(x)
            if ll > u or abs(theta) < self._min_theta:
                self._x, self._log_lik_x = x, ll
                return attempts
            if theta > 0:
                hi = theta
            else:
                lo = theta

    def sample(self, num=1):
        """``num`` successive states (a list; a single state if ``num == 1``)."""
        out = []
        for _ in range(num):
            self.attempts.append(self._step())
            out.append(self._x)
        return out if len(out) > 1 else out[0]


class MultiESS(object):
    """C elliptical-slice chains advanced together.  ``log_lik_batch(xs)`` scores a list of states at once;
    ``sample_priors[c]()`` and ``rngs[c]`` are chain c's prior draw and generator.  Every chain consumes its own
    generator in the order ``ESS`` does, so with the same generator and the same log-likelihood values chain c's
    states equal those of ``ESS(log_lik, sample_priors[c], x_inits[c], rngs[c])`` draw for draw.  Each round scores
    the current proposal of every chain that still needs states; a chain that accepts starts its next step at once."""
    _min_theta = ESS._min_theta

    def __init__(self, log_lik_batch, sample_priors, x_inits=None, rngs=None):
        self._log_lik_batch = log_lik_batch
        self._sample_priors = list(sample_priors)
        C = len(self._sample_priors)
        self._rngs = list(rngs) if rngs is not None else [np.random] * C
        if x_inits is None:
            x_inits = [None] * C
        if len(self._rngs) != C or len(x_inits) != C:
            raise ValueError('one generator and one initial state per chain')
        self._x = [sp() if x0 is None else x0 for sp, x0 in zip(self._sample_priors, x_inits)]
        self._log_lik_x = [float(v) for v in self._log_lik_batch(self._x)]
        self.attempts = [[] for _ in range(C)]

    @property
    def chains(self):
        return len(self._x)

    def _start(self, c):
        """Slice height, ellipse and first angle of chain c's next step (the draws of ``ESS._step``, in its order)."""
        rng = self._rngs[c]
        u = self._log_lik_x[c] - rng.exponential(1.0)
        nu = self._sample_priors[c]()
        theta = rng.uniform(0, 2 * np.pi)
        return [u, nu, theta - 2 * np.pi, theta, 0, None]        # u, nu, lo, hi, attempts, proposal angle

    def _propose(self, c, st):
        st[5] = self._rngs[c].uniform(st[2], st[3])
        st[4] += 1
        return np.cos(st[5]) * self._x[c] + np.sin(st[5]) * st[1]

    def sample(self, num=1):
        """``num`` successive states of every chain: a list of C lists."""
        C = len(self._x)
        out = [[] for _ in range(C)]
        if num < 1:
            return out
        steps = [self._start(c) for c in range(C)]
        props = [self._propose(c, steps[c]) for c in range(C)]
        active = list(range(C))
        while active:
            lls = self._log_lik_batch([props[c] for c in active])
            still = []
            for c, ll in zip(active, lls):
                ll, st = float(ll), steps[c]
                if ll > st[0] or abs(st[5]) < self._min_theta:
                    self._x[c], self._log_lik_x[c] = props[c], ll
                    self.attempts[c].append(st[4])
                    out[c].append(props[c])
                    if len(out[c]) == num:
                        continue
                    steps[c] = st = self._start(c)
                elif st[5] > 0:
                    st[3] = st[5]
                else:
                    st[2] = st[5]
                props[c] = self._propose(c, st)
                still.append(c)
            active = still
        return out
