"""The numpy reference of the multi-chain diagnostics (tests/chain_diag_ref.py) on cases whose answer is known by hand:
i.i.d. draws, antithetic draws, chains with shifted means, constant rows and too few draws."""
import math

import numpy as np

import chain_diag_ref as ref


def _ar1(rng, K, S, rho):
    x = np.empty((K, S))
    x[:, 0] = rng.standard_normal(K) / math.sqrt(1 - rho * rho)
    for s in range(1, S):
        x[:, s] = rho * x[:, s - 1] + rng.standard_normal(K)
    return x


def test_iid_draws_give_ess_near_the_number_of_draws():
    rng = np.random.default_rng(1)
    K, S = 4, 1000
    d = [ref.diagnostics(rng.standard_normal((K, S))) for _ in range(40)]
    for key in ("ess_bulk", "ess_tail"):
        r = np.array([x[key] for x in d]) / (K * S)
        assert 0.9 < r.mean() < 1.1, (key, r.mean())
        assert np.all((r > 0.6) & (r < 1.6)), (key, r.min(), r.max())
    rh = np.array([x["rhat"] for x in d])
    assert np.all(rh < 1.01) and np.all(rh > 0.99)


def test_antithetic_draws_give_ess_above_the_number_of_draws():
    rng = np.random.default_rng(2)
    K, S = 4, 1000
    for _ in range(10):
        d = ref.diagnostics(_ar1(rng, K, S, -0.5))
        assert d["ess_bulk"] > 1.5 * K * S  # tau = (1 + rho) / (1 - rho) = 1/3
    # positive autocorrelation: far fewer
    d = ref.diagnostics(_ar1(rng, K, S, 0.9))
    assert d["ess_bulk"] < 0.2 * K * S


def test_shifted_chain_means_give_a_large_rhat():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((4, 500)) + np.arange(4)[:, None] * 3.0
    d = ref.diagnostics(x)
    assert d["rhat"] > 2
    # a chain that drifts within itself: the split halves disagree even with one chain
    y = np.linspace(0, 10, 400)[None, :] + rng.standard_normal((1, 400)) * 0.1
    assert ref.diagnostics(y)["rhat"] > 2


def test_constant_rows_and_short_chains_give_nan():
    d = ref.diagnostics(np.full((3, 50), 2.5))
    assert all(math.isnan(d[k]) for k in ("rhat", "ess_bulk", "ess_tail"))
    for S in (1, 2, 3):
        d = ref.diagnostics(np.random.default_rng(S).standard_normal((4, S)))
        assert all(math.isnan(d[k]) for k in ("rhat", "ess_bulk", "ess_tail"))
    assert not math.isnan(ref.diagnostics(np.random.default_rng(4).standard_normal((4, 4)))["rhat"])


def test_split_drops_the_middle_draw_of_odd_chains():
    x = np.arange(14.0).reshape(2, 7)
    y = ref.split(x)
    assert y.shape == (4, 3)
    assert np.array_equal(y, [[0, 1, 2], [7, 8, 9], [4, 5, 6], [11, 12, 13]])
    # ties are ranked on average: z-scale of (0, 0, 1, 1) is symmetric
    z = ref.z_scale(np.array([[0.0, 0.0], [1.0, 1.0]]))
    assert z[0, 0] == z[0, 1] and math.isclose(z[0, 0], -z[1, 0], rel_tol=1e-14)


def test_pooled_summary_matches_numpy():
    rng = np.random.default_rng(5)
    d = rng.standard_normal((3, 17, 6))
    s = ref.summarize(d, (0.1, 0.5))
    pooled = d.transpose(2, 0, 1).reshape(6, -1)
    assert np.array_equal(s["quantiles"], np.quantile(pooled, (0.1, 0.5), axis=1).T)
    assert np.allclose(s["sd"], pooled.std(axis=1, ddof=1))
