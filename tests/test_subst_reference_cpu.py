"""The complex-step reference of tests/subst_reference.py pinned on the CPU: against a
50-digit pruning differentiated by central differences (mpmath), where fp64 shortcuts
would go wrong -- a branch with (lambda_k - lambda_l) tau ~ 1000, exactly repeated
eigenvalues, nearly repeated ones, extreme frequencies, zero and 1e-12 branches -- and
against the oracle's log likelihoods and central differences on DS1.
"""
import mpmath
import numpy as np
import pytest

from conftest import load_fixture
from libsbn_b200 import trees
import subst_reference as ref

DIGITS = 50
DIFFERENCE_STEP = mpmath.mpf("1e-20")


def mp_stick_breaking(y):
    stick, x = mpmath.mpf(1), []
    for k, value in enumerate(y):
        z = 1 / (1 + mpmath.exp(-(value - mpmath.log(len(y) - k))))
        x.append(stick * z)
        stick -= stick * z
    return x + [stick]


def mp_log_likelihood(substitution, site, tips, weights, parent_ids, lengths, shape, y, category_rates=None):
    """logL at the coordinates y, every step at DIGITS digits (lengths may be mpf; Weibull
    category rates from the shape unless category_rates gives them)."""
    if substitution == "GTR":
        exchangeabilities, freqs = mp_stick_breaking(y[:5]), mp_stick_breaking(y[5:8])
    else:
        exchangeabilities, freqs = [1, y[0], 1, 1, y[0], 1], mp_stick_breaking(y[1:4])
    q = mpmath.zeros(4, 4)
    index = 0
    for i in range(4):
        for j in range(i + 1, 4):
            q[i, j] = exchangeabilities[index] * freqs[j]
            q[j, i] = exchangeabilities[index] * freqs[i]
            index += 1
    for i in range(4):
        q[i, i] = -sum(q[i, j] for j in range(4) if j != i)
    q /= -sum(freqs[i] * q[i, i] for i in range(4))
    if category_rates is not None:
        rates = list(category_rates)
    elif site == "constant":
        rates = [mpmath.mpf(1)]
    else:
        count = int(site.split("+")[1])
        rates = [(-mpmath.log(1 - mpmath.mpf(2 * c + 1) / (2 * count))) ** (1 / mpmath.mpf(shape))
                 for c in range(count)]
        mean = sum(rates) / count
        rates = [r / mean for r in rates]
    node_count = len(parent_ids) + 1
    taxa = len(tips)
    children = [[] for _ in range(node_count)]
    for child, parent in enumerate(parent_ids):
        children[parent].append(child)
    total = mpmath.mpf(0)
    matrices = [[mpmath.expm(q * (mpmath.mpf(lengths[e]) * r)) for r in rates] for e in range(node_count - 1)]
    for p in range(len(weights)):
        site_likelihood = mpmath.mpf(0)
        for c in range(len(rates)):
            partial = {}
            for leaf in range(taxa):
                s = int(tips[leaf][p])
                partial[leaf] = [mpmath.mpf(1) if s >= 4 or s == i else mpmath.mpf(0) for i in range(4)]
            for node in range(taxa, node_count):
                vector = [mpmath.mpf(1)] * 4
                for child in children[node]:
                    P = matrices[child][c]
                    vector = [vector[i] * sum(P[i, s] * partial[child][s] for s in range(4)) for i in range(4)]
                partial[node] = vector
            site_likelihood += sum(freqs[i] * partial[node_count - 1][i] for i in range(4)) / len(rates)
        total += mpmath.mpf(float(weights[p])) * mpmath.log(site_likelihood)
    return total


def mp_gradient(substitution, site, tips, weights, parent_ids, lengths, params):
    base, _ = ref.coordinates(substitution, params)
    shape = params[10 if substitution == "GTR" else 5] if site != "constant" else None
    args = (substitution, site, tips, weights, parent_ids, lengths, shape)
    with mpmath.workdps(DIGITS):
        y = [mpmath.mpf(float(v)) for v in base]
        logl = mp_log_likelihood(*args, y)
        gradient = []
        for j in range(len(y)):
            plus, minus = list(y), list(y)
            plus[j] += DIFFERENCE_STEP
            minus[j] -= DIFFERENCE_STEP
            difference = mp_log_likelihood(*args, plus) - mp_log_likelihood(*args, minus)
            gradient.append(float(difference / (2 * DIFFERENCE_STEP)))
        return float(logl), np.array(gradient)


def eigenvalue_spread(substitution, params):
    """lambda_max - lambda_min of the normalised rate matrix of a parameter row."""
    base, model = ref.coordinates(substitution, params)
    eigenvalues = np.linalg.eigvals(ref.rate_matrix(*model(base)).real).real
    return eigenvalues.max() - eigenvalues.min()


def small_case(taxa, seed):
    rng = np.random.default_rng(seed)
    tips, _ = trees.random_alignment(taxa, 15, seed, gap_fraction=0.05)
    weights = rng.integers(1, 4, size=15).astype(np.float64)
    parent_ids = trees.random_unrooted_topology(taxa, rng)
    lengths = rng.uniform(0.02, 0.4, size=len(parent_ids) + 1)
    return tips, weights, parent_ids, lengths


GTR_RANDOM = [0.1, 0.3, 0.05, 0.15, 0.25, 0.15, 0.3, 0.2, 0.15, 0.35]
CASES = {
    # one branch where (lambda_k - lambda_l) tau ~ 1000 in the fastest category
    "gtr_weibull4_long_branch": ("GTR", "weibull+4", 5, GTR_RANDOM + [0.6], "long"),
    "gtr_constant_zero_branches": ("GTR", "constant", 4, GTR_RANDOM, "degenerate"),
    # kappa = 1 with uniform frequencies: JC69, exactly repeated eigenvalues
    "hky_kappa1_uniform": ("HKY", "constant", 4, [0.25, 0.25, 0.25, 0.25, 1.0], "degenerate"),
    "hky_kappa1_uniform_weibull4": ("HKY", "weibull+4", 3, [0.25, 0.25, 0.25, 0.25, 1.0, 0.8], None),
    "hky_kappa_near_1": ("HKY", "weibull+4", 4, [0.25, 0.25, 0.25, 0.25, 1.0 + 1e-9, 1.3], None),
    "gtr_extreme_frequencies": ("GTR", "constant", 5, GTR_RANDOM[:6] + [0.94, 0.02, 0.02, 0.02], "long"),
    "hky_extreme_frequencies": ("HKY", "weibull+4", 4, [0.94, 0.02, 0.02, 0.02, 3.0, 0.5], "degenerate"),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_complex_step_matches_fifty_digit_central_differences(name):
    substitution, site, taxa, params, branches = CASES[name]
    params = np.array(params)
    tips, weights, parent_ids, lengths = small_case(taxa, seed=len(name))
    if branches == "long":
        fastest = ref.site_rates(site, params[-1] if site != "constant" else None)[0].max()
        lengths[1] = 1000.0 / (eigenvalue_spread(substitution, params) * fastest)
    elif branches == "degenerate":
        lengths[0], lengths[2] = 0.0, 1e-12
    logl, gradient = ref.log_likelihood_and_gradient(substitution, site, tips, weights, parent_ids, lengths, params)
    want_logl, want = mp_gradient(substitution, site, tips, weights, parent_ids, lengths, params)
    assert abs(logl - want_logl) <= 1e-13 * abs(want_logl)
    assert np.all(np.isfinite(gradient))
    assert np.max(np.abs(gradient - want)) <= 1e-12 * np.max(np.abs(want))


def test_matches_the_oracle_on_ds1():
    """The oracle's central differences (the reference's delta 1e-6 on the same coordinates)
    agree within their noise floor, the log likelihoods to rounding."""
    from oracle import phylo

    fx = load_fixture("ds1_gtr_weibull4")
    count = 3
    want = phylo.gradients("GTR", "weibull+4", fx["patterns"], fx["weights"], fx["parent_ids"][:count],
                           fx["branch_lengths"][:count], fx["params"][:count])
    for t in range(count):
        logl, gradient = ref.log_likelihood_and_gradient("GTR", "weibull+4", fx["patterns"], fx["weights"],
                                                         fx["parent_ids"][t], fx["branch_lengths"][t], fx["params"][t])
        assert abs(logl - want["log_likelihood"][t]) <= 1e-12 * abs(logl)
        fd_noise = abs(logl) * 1e-12 / 1e-6
        assert np.max(np.abs(gradient - want["substitution_model"][t])) < fd_noise


def test_masks_are_the_sum_over_their_states():
    """An ambiguous tip is the sum of its states' tip vectors: with masks that are all single
    states or missing, the result is the state result; an R (A or G) in one tip gives the
    sum of the A and G likelihoods of that one-pattern alignment."""
    tips, weights, parent_ids, lengths = small_case(5, seed=3)
    params = np.array(GTR_RANDOM + [0.7])
    masks = trees.states_to_masks(tips)
    by_states = ref.log_likelihood_and_gradient("GTR", "weibull+4", tips, weights, parent_ids, lengths, params)
    by_masks = ref.log_likelihood_and_gradient("GTR", "weibull+4", masks, weights, parent_ids, lengths, params,
                                               masks=True)
    assert by_masks[0] == pytest.approx(by_states[0], rel=1e-14)
    np.testing.assert_allclose(by_masks[1], by_states[1], rtol=1e-12, atol=1e-12 * np.max(np.abs(by_states[1])))
    column = tips[:, :1].copy()
    likelihoods = []
    for state in (0, 2):
        column[1, 0] = state
        likelihoods.append(np.exp(ref.log_likelihood_and_gradient("GTR", "weibull+4", column, [1.0], parent_ids,
                                                                  lengths, params)[0]))
    ambiguous = trees.states_to_masks(column)
    ambiguous[1, 0] = 0b0101
    got = np.exp(ref.log_likelihood_and_gradient("GTR", "weibull+4", ambiguous, [1.0], parent_ids, lengths, params,
                                                 masks=True)[0])
    assert got == pytest.approx(sum(likelihoods), rel=1e-13)


def test_thousand_taxon_ladder_does_not_underflow():
    """Per-node rescaling: 1000 taxa on a ladder (deeper than Python's recursion limit) give a
    finite logL and gradient where the unscaled site likelihoods are far below fp64's range."""
    taxa = 1000
    tips, weights = trees.random_alignment(taxa, 8, seed=2)
    parent_ids = trees.ladder_topology(taxa)
    lengths = np.random.default_rng(3).uniform(0.01, 0.2, size=len(parent_ids) + 1)
    logl, gradient = ref.log_likelihood_and_gradient("HKY", "constant", tips, weights, parent_ids, lengths,
                                                     [0.1, 0.2, 0.3, 0.4, 2.0])
    assert np.isfinite(logl) and logl < -1000
    assert np.all(np.isfinite(gradient)) and gradient.shape == (4,)
