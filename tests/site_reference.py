"""TEST INFRASTRUCTURE: an exact reference for the [tree][pattern] matrix of log site
likelihoods (sbnb_site_log_likelihoods_*, beagleGetSiteLogLikelihoods).

s[k] is what the walk adds into logL with the pattern weight w_k, before the weight:
log L_k of the mixture over the rate categories, or with +I log((1 - p) L_k + p I_k), so that
sum_k w_k s[k] = logL.  Everything is built from the existing references:
invariant_reference.per_site_log_variable (a plain complex128 pruning, scipy.linalg.expm per
edge and category, a real rescaling factor per node so that 1000 taxa do not underflow),
invariant_reference.mixture_log_likelihood for +I, subst_reference.tip_vectors through both,
and time_tree_reference's heights for the effective lengths of a time tree (clock rate x
height difference).  Nothing is formed in the walk's scaled domain.
"""
import numpy as np

import invariant_reference as inv
import time_tree_reference as tt


def model_of(substitution, site, params):
    """(Q [1][4][4], pi [1][4], category rates [C] (divided by 1 - p with +I), weights [C], p)."""
    params = np.asarray(params, dtype=np.float64)
    invariant = site.endswith("+I")
    base = inv.base_site(site) if invariant else site
    rates, weights = tt.category_rates(base, tt.shape_of(substitution, base, params), np.zeros(1))
    qs, freqs = tt.substitution_model(substitution, params, np.zeros((1, 0)))
    p = float(params[inv.pinv_index(substitution, site)]) if invariant else 0.0
    return qs, freqs, rates[0].real / (1.0 - p), np.asarray(weights, dtype=np.float64), p


def site_log_likelihoods(substitution, site, tips, parent_ids, lengths, params, masks=False):
    """[pattern] log site likelihoods of one tree (parent ids and one length per node, used as is)."""
    qs, freqs, rates, weights, p = model_of(substitution, site, params)
    log_l = inv.per_site_log_variable(qs, freqs, rates[None, :], weights[None, :], tips, parent_ids,
                                      np.asarray(lengths, dtype=np.float64), masks)
    if site.endswith("+I"):
        log_l = inv.mixture_log_likelihood(log_l, p, inv.invariant_terms(freqs, tips, masks))
    return log_l[0].real


def time_tree_lengths(batch, t):
    """[nodes] effective lengths of tree t of a random_time_trees batch: rate x (h_parent - h)."""
    parent_ids = np.asarray(batch["parent_ids"][t])
    ratios = np.asarray(batch["height_ratios"][t], dtype=np.float64)
    n = len(ratios) + 1
    h = tt.heights(parent_ids, np.asarray(batch["node_bounds"][t], dtype=np.float64), ratios[None, :n - 2],
                   ratios[n - 2])[0]
    lengths = np.zeros(2 * n - 1)
    lengths[:-1] = np.asarray(batch["rates"][t], dtype=np.float64) * (h[parent_ids] - h[:-1])
    return lengths


def matrix(substitution, site, tips, parent_ids, lengths, params, masks=False):
    """[T][pattern] of a batch of unrooted (or already effective-length) trees."""
    return np.array([site_log_likelihoods(substitution, site, tips, parent_ids[t], lengths[t], params[t], masks)
                     for t in range(len(params))])


def time_tree_matrix(substitution, site, tips, batch, params, masks=False):
    """[T][pattern] of a random_time_trees batch, on the rate-scaled lengths (no Jacobian)."""
    return np.array([site_log_likelihoods(substitution, site, tips, batch["parent_ids"][t], time_tree_lengths(batch, t),
                                          params[t], masks) for t in range(len(params))])


def beagle_case(case, q, freqs):
    """[pattern] log site likelihoods of a beagle_reference.random_case (GTR of gtr_eigensystem)."""
    import beagle_reference as br
    parents = br.parent_ids(case["post"], case["n"])
    log_l = inv.per_site_log_variable(np.asarray(q, dtype=np.complex128)[None], np.asarray(freqs)[None],
                                      np.asarray(case["rates"])[None, :], np.asarray(case["category_weights"])[None, :],
                                      case["states"], parents, np.asarray(case["lengths"])[:2 * case["n"] - 1],
                                      case["masks"])
    return log_l[0].real
