"""cgpcm_b200.sample.MultiESS: C elliptical-slice chains in lock-step with one batched log-likelihood call per round
reproduce C independent ESS chains draw for draw, and sample the right distribution."""
import numpy as np

from cgpcm_b200.sample import ESS, MultiESS


def _target(m, s2):
    return lambda x: float(-.5 * np.sum((x - m) ** 2) / s2)


def test_multi_ess_reproduces_independent_chains():
    m, s2, C = np.array([[1.5], [-0.5], [0.3]]), 0.2, 5
    ll = _target(m, s2)
    x0s = [np.full((3, 1), 0.1 * c) for c in range(C)]
    # reference: C separate ESS runs, each with its own generator
    want = []
    for c in range(C):
        rng = np.random.RandomState(100 + c)
        ess = ESS(ll, lambda rng=rng: rng.randn(3, 1), x_init=x0s[c].copy(), rng=rng)
        ess.sample(7)
        want.append((ess.sample(25), ess.attempts))
    rngs = [np.random.RandomState(100 + c) for c in range(C)]
    sizes = []

    def batch(xs):
        sizes.append(len(xs))
        return np.array([ll(x) for x in xs])
    mess = MultiESS(batch, [lambda rng=rng: rng.randn(3, 1) for rng in rngs], x_inits=[x.copy() for x in x0s],
                    rngs=rngs)
    mess.sample(7)
    got = mess.sample(25)
    assert len(got) == C and all(len(g) == 25 for g in got)
    for c in range(C):
        assert all(np.array_equal(a, b) for a, b in zip(got[c], want[c][0]))
        assert mess.attempts[c] == want[c][1]
    # proposals of several chains were scored together, never more than one per chain
    assert max(sizes) == C and min(sizes) >= 1
    assert len(sizes) < sum(len(a) for _, a in want)


def test_multi_ess_pooled_moments_on_a_gaussian_target():
    """Prior N(0, I_2), likelihood N(x; m, s^2 I) -> posterior N(m / (1 + s^2), s^2 / (1 + s^2) I)."""
    m, s2, C = np.array([[1.5], [-0.5]]), 0.5, 8
    rngs = [np.random.RandomState(c) for c in range(C)]
    ll = _target(m, s2)
    mess = MultiESS(lambda xs: [ll(x) for x in xs], [lambda rng=rng: rng.randn(2, 1) for rng in rngs],
                    x_inits=[np.zeros((2, 1)) for _ in rngs], rngs=rngs)
    mess.sample(100)
    xs = np.concatenate([np.concatenate(ch, 1) for ch in mess.sample(600)], 1)
    want_mean, want_var = m.ravel() / (1 + s2), s2 / (1 + s2)
    assert np.abs(xs.mean(1) - want_mean).max() < 0.06
    assert np.abs(xs.var(1) - want_var).max() < 0.05
    assert all(min(a) >= 1 for a in mess.attempts)


def test_multi_ess_draws_initial_states_from_the_prior():
    rngs = [np.random.RandomState(c) for c in range(3)]
    mess = MultiESS(lambda xs: [0.0] * len(xs), [lambda rng=rng: rng.randn(2, 1) for rng in rngs], rngs=rngs)
    assert mess.chains == 3 and mess.sample(0) == [[], [], []]
    out = mess.sample(2)
    assert [len(o) for o in out] == [2, 2, 2]
