"""The per-site reference of tests/site_reference.py pinned on the CPU: its weighted sum is the
existing references' logL (subst_reference.prune, invariant_reference.log_likelihood and the
time-tree reference) to 1e-12, and its BEAGLE form (site_reference.beagle_case) is the
per-pattern split of beagle_reference's logL.  The device libraries are held to it in
tests/test_site_log_likelihoods_gpu.py.
"""
import numpy as np
import pytest

import beagle_reference as br
import invariant_reference as inv
import site_reference as sr
import subst_reference as ref
import time_tree_reference as tt
from libsbn_b200 import trees
from libsbn_b200.beagle import gtr_eigensystem
from test_invariant_cpu import invariant_alignment

RTOL = 1e-12


def random_row(substitution, site, rng, p=None, clock=False):
    row = {"JC69": [], "GTR": list(rng.dirichlet(np.ones(6) * 2)) + list(rng.dirichlet(np.ones(4) * 4)),
           "HKY": list(rng.dirichlet(np.ones(4) * 4)) + [rng.uniform(0.5, 4.0)]}[substitution]
    if not site.startswith("constant"):
        row.append(rng.uniform(0.3, 2.0))
    if p is not None:
        row.append(p)
    if clock:
        row.append(0.0)
    return np.array(row)


PLAIN = [("JC69", "constant", False), ("GTR", "weibull+4", False), ("HKY", "gamma+4", True),
         ("GTR", "gamma+3", True), ("HKY", "weibull+20", False)]


@pytest.mark.parametrize("substitution,site,masks", PLAIN)
def test_weighted_sum_is_the_pruning(substitution, site, masks):
    tips, weights = invariant_alignment(12, 97, seed=len(site), masks=masks)
    parent_ids, lengths = trees.random_tree_batch(12, 2, seed=3)
    rng = np.random.default_rng(4)
    for t in range(2):
        params = random_row(substitution, site, rng)
        sites = sr.site_log_likelihoods(substitution, site, tips, parent_ids[t], lengths[t], params, masks)
        assert sites.shape == (97,) and np.all(np.isfinite(sites))
        qs, freqs, rates, category_weights, _ = sr.model_of(substitution, site, params)
        want = ref.prune(qs, freqs, rates, category_weights, tips, weights, parent_ids[t], lengths[t], masks)[0].real
        assert abs(sites @ weights - want) <= RTOL * abs(want)


@pytest.mark.parametrize("substitution,site", [("JC69", "constant+I"), ("GTR", "weibull+4+I"), ("HKY", "gamma+4+I")])
@pytest.mark.parametrize("p", [0.0, 0.5, 0.95])
@pytest.mark.parametrize("masks", [False, True])
def test_weighted_sum_is_the_invariant_reference(substitution, site, p, masks):
    tips, weights = invariant_alignment(10, 83, seed=5, masks=masks)
    parent_ids, lengths = trees.random_tree_batch(10, 1, seed=6)
    params = random_row(substitution, site, np.random.default_rng(7), p)
    sites = sr.site_log_likelihoods(substitution, site, tips, parent_ids[0], lengths[0], params, masks)
    base = inv.base_site(site)
    category, category_weights = tt.category_rates(base, tt.shape_of(substitution, base, params), np.zeros(1))
    qs, freqs = tt.substitution_model(substitution, params, np.zeros((1, 0)))
    want = inv.log_likelihood(qs, freqs, category.real, category_weights, [p], tips, weights, parent_ids[0],
                              lengths[0][None, :], masks)[0].real
    assert abs(sites @ weights - want) <= RTOL * abs(want)
    if p == 0.0:  # the mixture at p = 0 is the plain model
        plain = sr.site_log_likelihoods(substitution, base, tips, parent_ids[0], lengths[0], params[:-1], masks)
        np.testing.assert_allclose(sites, plain, rtol=1e-14)


@pytest.mark.parametrize("relaxed", [False, True])
def test_time_tree_sums_and_lengths(relaxed):
    """Effective lengths are the engine's branch lengths x rates; the weighted sum is the time-tree
    reference's logL (its Jacobian apart)."""
    tips, weights = invariant_alignment(9, 61, seed=8)
    batch = trees.random_time_trees(9, 2, seed=9, relaxed=relaxed)
    rng = np.random.default_rng(10)
    for t in range(2):
        lengths = sr.time_tree_lengths(batch, t)
        np.testing.assert_allclose(lengths[:-1], batch["branch_lengths"][t][:-1] * batch["rates"][t], rtol=1e-13)
        params = random_row("GTR", "weibull+4", rng, clock=True)
        tree = tt.TimeTree("GTR", "weibull+4", tips, weights, batch, t, params)
        logl, _, _ = tree.evaluate(np.zeros((1, tree.size)))
        sites = sr.time_tree_matrix("GTR", "weibull+4", tips, {k: v[t:t + 1] if k != "rate_count" else v
                                                                for k, v in batch.items()}, params[None, :])[0]
        assert abs(sites @ weights - logl) <= RTOL * abs(logl)


def test_deep_ladder_stays_finite():
    """A 600-taxon ladder: the per-node factors keep every site finite, far below the fp64 range."""
    taxa = 600
    tips, _ = trees.random_alignment(taxa, 7, seed=11)
    weights = np.arange(1.0, 8.0)
    parent_ids = trees.ladder_topology(taxa)
    lengths = np.full(len(parent_ids) + 1, 0.4)
    sites = sr.site_log_likelihoods("JC69", "constant", tips, parent_ids, lengths, np.zeros(0))
    assert np.all(np.isfinite(sites)) and np.all(sites < -708)
    qs, freqs, rates, category_weights, _ = sr.model_of("JC69", "constant", np.zeros(0))
    want = ref.prune(qs, freqs, rates, category_weights, tips, weights, parent_ids, lengths)[0].real
    assert abs(sites @ weights - want) <= RTOL * abs(want)


@pytest.mark.parametrize("categories,masks", [(1, False), (3, True), (4, False), (20, False)])
def test_beagle_form_sums_to_the_beagle_reference(categories, masks):
    """site_reference.beagle_case, the reference the device library's beagleGetSiteLogLikelihoods is
    held to, weighted by the case's pattern weights is beagle_reference's logL of the same case."""
    case = br.random_case(30, 53, categories, 120 + categories, "libsbn", masks=masks)
    _, _, _, freqs, q = gtr_eigensystem()
    sites = sr.beagle_case(case, q, freqs)
    logl = br.reference(case, edges=[])[0]
    assert np.all(np.isfinite(sites))
    assert abs(sites @ case["weights"] - logl) <= RTOL * abs(logl)
