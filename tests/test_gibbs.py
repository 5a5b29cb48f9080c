"""CPU: the Gibbs sampler's definition (DESIGN.md "Gibbs posterior samples"), through its restatement tests/gibbs_ref.py.

Our log / exp against numpy's, the gamma draws' moments, posterior moments of pi on small loci against quadrature of the exact
posterior, and determinism: the same inputs give the same bits, while the seed, the round and the locus position all change them."""
import numpy as np
import pytest
from scipy import integrate

import gibbs_ref as gr
from strawberry_b200.synth import _sm64


def _ulps(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)))


def test_log_is_within_2_ulp_of_numpy():
    rng = np.random.default_rng(1)
    x = np.concatenate([
        np.array([5e-324, 1e-320, 2.2250738585072014e-308 / 3, 2.2250738585072014e-308, 1.0, 2.0, 0.5, np.sqrt(0.5), 1.7976931348623157e308]),
        np.nextafter(np.sqrt(0.5), [0, 1]), np.nextafter(1.0, [0, 2]), 1.0 + np.arange(-1000, 1000) * 2.0 ** -52,
        10.0 ** rng.uniform(-320, 308, 200_000), rng.uniform(0.5, 2.0, 200_000),
        2.0 ** np.arange(-1074, 1024, dtype=np.float64),
    ])
    got, ref = gr.g_log(x), np.log(x)
    one = x == 1.0
    assert (got[one] == 0.0).all()
    assert _ulps(got[~one], ref[~one]).max() <= 2.0


def test_exp_is_within_2_ulp_of_numpy():
    rng = np.random.default_rng(2)
    ln2 = np.log(2.0)
    x = np.concatenate([
        rng.uniform(-745, 709.7, 200_000), rng.uniform(-1, 1, 100_000), rng.uniform(-1e-8, 1e-8, 1000),
        np.arange(-1074, 1024) * ln2, (np.arange(-1074, 1024) + 0.5) * ln2, np.array([0.0, -0.0, 709.78, -708.4, -720.0, -744.0]),
    ])
    got, ref = gr.g_exp(x), np.exp(x)
    nz = ref > 2.2250738585072014e-308                         # normal results: relative ulps
    assert _ulps(got[nz], ref[nz]).max() <= 2.0
    sub = ~nz                                                  # subnormal results: within 2 units of the smallest subnormal
    assert (np.abs(got[sub] - ref[sub]) <= 2 * 5e-324).all()
    assert gr.g_exp(np.array([800.0]))[0] == np.inf and gr.g_exp(np.array([-800.0]))[0] == 0.0


@pytest.mark.parametrize("a", [0.01, 0.5, 1.0, 3.7, 1e4])
def test_gamma_moments(a):
    N = 40_000
    with np.errstate(over="ignore"):
        keys = _sm64(np.arange(N, dtype=np.uint64) + np.uint64(int(a * 1000) + 7))
    g = gr.gamma(np.full(N, a), keys)
    assert (g >= 0).all() and np.isfinite(g).all()
    se_mean = np.sqrt(a / N)
    se_var = np.sqrt((2 * a * a + 6 * a) / N)
    assert abs(g.mean() - a) < 4 * se_mean, (g.mean(), a)
    assert abs(g.var() - a) < 4 * se_var, (g.var(), a)


def _replicated_batch(alpha, n, L):
    """L copies of one locus (rows of dense alpha, counts n) as a flat batch"""
    alpha = np.asarray(alpha, np.float64)
    R, T = alpha.shape
    col = np.tile(np.arange(T), R)
    rp1 = np.arange(R + 1) * T
    return dict(loc_row_off=np.arange(L + 1, dtype=np.int64) * R, loc_iso_off=np.arange(L + 1, dtype=np.int64) * T,
                row_ptr=np.concatenate([[0], (rp1[1:][None, :] + (np.arange(L) * R * T)[:, None]).ravel()]).astype(np.int64),
                col=np.tile(col, L).astype(np.int32), alpha=np.tile(alpha.ravel(), L), count=np.tile(np.asarray(n, np.int32), L),
                iso_len=np.full(L * T, 1000, np.int32))


def _posterior_moments(alpha, n, prior):
    """E[pi] and Var[pi] of the exact posterior prod_i (sum_j F_ij pi_j)^n_i Dir(pi; prior), F = alpha / column sums"""
    F = np.asarray(alpha) / np.asarray(alpha).sum(0)
    T = F.shape[1]

    def dens(pi):
        return np.exp(np.sum(np.asarray(n) * np.log(F @ pi)) + (prior - 1) * np.sum(np.log(pi)))

    if T == 2:
        def q(f):
            return integrate.quad(lambda p: f(np.array([p, 1 - p])), 0, 1, epsabs=0, epsrel=1e-10, limit=200)[0]
    else:
        def q(f):
            return integrate.dblquad(lambda p2, p1: f(np.array([p1, p2, 1 - p1 - p2])), 0, 1, 0, lambda p1: 1 - p1, epsabs=0, epsrel=1e-9)[0]
    Z = q(dens)
    mean = np.array([q(lambda pi, j=j: pi[j] * dens(pi)) for j in range(T)]) / Z
    m2 = np.array([q(lambda pi, j=j: pi[j] ** 2 * dens(pi)) for j in range(T)]) / Z
    return mean, m2 - mean ** 2


@pytest.mark.parametrize("alpha,n", [
    ([[0.5, 0.2], [0.1, 0.7], [0.3, 0.3]], [6, 3, 5]),
    ([[0.4, 0.3, 0.0], [0.0, 0.5, 0.2], [0.2, 0.0, 0.6], [0.1, 0.1, 0.1]], [4, 7, 3, 5]),
])
def test_posterior_moments_match_quadrature(alpha, n):
    prior, L, per = 1.0, 2000, 2                   # L independent chains (one per locus position), `per` thinned samples each
    b = _replicated_batch(alpha, n, L)
    T = len(alpha[0])
    th0 = np.full(L * T, sum(n) / T)
    ch = gr.Chain(b, th0, np.zeros(L, np.int32), seed=11, prior=prior)
    draws = []
    for s in range(per):
        while ch.r < 30 + (s + 1) * 5:
            ch.step()
        draws.append(ch.pi.reshape(L, T).copy())
    x = np.stack(draws, 1)                          # [chain, sample, isoform]
    mean, var = _posterior_moments(alpha, n, prior)
    for j in range(T):
        m_chain = x[:, :, j].mean(1)
        assert abs(m_chain.mean() - mean[j]) < 4 * m_chain.std(ddof=1) / np.sqrt(L), (j, m_chain.mean(), mean[j])
        dev = ((x[:, :, j] - mean[j]) ** 2).mean(1)
        assert abs(dev.mean() - var[j]) < 4 * dev.std(ddof=1) / np.sqrt(L), (j, dev.mean(), var[j])


def _small_batch():
    return _replicated_batch([[0.5, 0.2, 0.1], [0.1, 0.7, 0.0], [0.3, 0.3, 0.3]], [9, 4, 20], 3)


def test_determinism_and_dependence_on_seed_round_and_locus():
    b = _small_batch()
    th0 = np.full(9, 11.0)
    st = np.zeros(3, np.int32)
    a = gr.samples(b, th0, st, seed=5, n=3, thin=2, burn_in=3, prior=0.01, total_mapped_reads=1e6)
    again = gr.samples(b, th0, st, seed=5, n=3, thin=2, burn_in=3, prior=0.01, total_mapped_reads=1e6)
    assert np.array_equal(a["theta"], again["theta"])
    other = gr.samples(b, th0, st, seed=6, n=3, thin=2, burn_in=3, prior=0.01, total_mapped_reads=1e6)
    assert not np.array_equal(a["theta"], other["theta"])
    # identical loci at different positions follow different chains; the same position gives the same chain
    t = a["theta"][0].reshape(3, 3)
    assert not np.array_equal(t[0], t[1]) and not np.array_equal(t[1], t[2])
    moved = gr.samples(b, th0, st, seed=5, n=3, thin=2, burn_in=3, prior=0.01, total_mapped_reads=1e6, locus_ids=[2, 0, 1])
    mt = moved["theta"][0].reshape(3, 3)
    assert np.array_equal(mt[0], t[2]) and np.array_equal(mt[1], t[0])
    # every round draws afresh, and a sample's theta sums to the locus' kept fragments
    assert gr.round_key(5, 1) != gr.round_key(5, 2)
    assert not np.array_equal(a["theta"][0], a["theta"][1])
    assert np.allclose(a["theta"].reshape(3, 3, 3).sum(2), 33.0, rtol=1e-12)


def test_unsampled_loci_repeat_the_point_estimate():
    b = _small_batch()
    th0 = np.array([11.0, 11, 11, 5, 5, 5, 11, 11, 11])
    st = np.array([0, 2, 0], np.int32)               # ZERO_DENOM: not sampled
    a = gr.samples(b, th0, st, seed=5, n=2, thin=1, burn_in=0, prior=0.5, total_mapped_reads=1e6)
    assert (a["theta"][:, 3:6] == 5.0).all()
    assert not (a["theta"][:, :3] == 11.0).all()


def test_block_sum_emulation_order():
    """block_sum<256> adds strided partials, butterflies within warps, then the warp totals in order: not np.sum's order"""
    rng = np.random.default_rng(3)
    v = rng.standard_normal(5000) * 10.0 ** rng.uniform(-8, 8, 5000)
    off = np.array([0, 1, 300, 5000])
    got = gr.block_sum(v, off)
    assert got[0] == v[0]
    part = np.zeros(256)
    for j in range(4700):
        part[j % 256] += v[300 + j]
    w = part.reshape(8, 32)
    for o in (16, 8, 4, 2, 1):
        w = w + w[:, np.arange(32) ^ o]
    t = 0.0
    for k in range(8):
        t += w[k, 0]
    assert got[2] == t
