"""TEST INFRASTRUCTURE: likelihoods and gradients of an alignment of nucleotide masks from
the unchanged CPU oracle, by linearity.

A site's likelihood is linear in each tip's partial vector, and the partial of an ambiguous
tip is the sum of the indicator vectors of its states.  So the likelihood of a pattern with
ambiguous tips is the sum of the likelihoods of the state patterns it expands to (one state
per ambiguous tip, every combination), and its gradient of log L is their gradients of
log L weighted by L_i / sum L_i.  Patterns without an ambiguous tip go to the oracle as they
are, in one call.  Every term is an ordinary state-mode oracle evaluation.
"""
import itertools

import numpy as np

# the per-tree results that are sums over patterns of d log L_p (and log L_p itself)
KEYS = ("log_likelihood", "branch", "substitution_model", "site_model", "ratios_root_height", "clock_model")
SINGLE = {1: 0, 2: 1, 4: 2, 8: 3, 15: 4}


def states_of(mask):
    return [s for s in range(4) if mask >> s & 1]


def expand(column):
    """The state columns a mask column expands to (15 stays the gap state 4)."""
    choices = [[SINGLE[m]] if m in SINGLE else states_of(m) for m in column]
    return np.array(list(itertools.product(*choices)), dtype=np.uint8)


def gradients(oracle, substitution, site, masks, weights, parent_ids, branch_lengths, params, rescaling=False,
              rooted=False, batch_unambiguous=True, **rooted_kwargs):
    """oracle.gradients for an alignment of masks: {key: [T]...} as the oracle returns them."""
    def call(states, w):
        return oracle.gradients(substitution, site, states, w, parent_ids, branch_lengths, params,
                                rescaling=rescaling, rooted=rooted, **rooted_kwargs)
    return _by_linearity(call, KEYS, masks, weights, batch_unambiguous)


def log_likelihoods(oracle, substitution, site, masks, weights, parent_ids, branch_lengths, params, rescaling=False,
                    rooted=False, **rooted_kwargs):
    """oracle.log_likelihoods for an alignment of masks (rooted: with the log-det Jacobian)."""
    def call(states, w):
        return {"log_likelihood": oracle.log_likelihoods(substitution, site, states, w, parent_ids, branch_lengths,
                                                         params, rescaling=rescaling, rooted=rooted, **rooted_kwargs)}
    return _by_linearity(call, KEYS[:1], masks, weights, True)["log_likelihood"]


def _by_linearity(call, keys, masks, weights, batch_unambiguous):
    masks = np.asarray(masks, dtype=np.uint8)
    weights = np.asarray(weights, dtype=np.float64)
    ambiguous = ~np.isin(masks, list(SINGLE)).all(axis=0)
    to_states = np.vectorize(lambda m: SINGLE[m], otypes=[np.uint8])
    # the terms every call carries whatever the patterns (the rooted log-det Jacobian)
    base = call(np.full((masks.shape[0], 1), 4, dtype=np.uint8), np.zeros(1))
    total = {k: base[k].copy() for k in keys}
    plain = ~ambiguous if batch_unambiguous else np.zeros_like(ambiguous)
    if plain.any():
        got = call(to_states(masks[:, plain]), weights[plain])
        for k in keys:
            total[k] += got[k] - base[k]
    for p in np.flatnonzero(~plain):
        terms = [call(column[:, None], np.ones(1)) for column in expand(masks[:, p])]
        logs = np.array([t["log_likelihood"] - base["log_likelihood"] for t in terms])  # [terms][T]
        top = logs.max(axis=0)
        share = np.exp(logs - top)
        total["log_likelihood"] += weights[p] * (top + np.log(share.sum(axis=0)))
        share /= share.sum(axis=0)
        for k in keys[1:]:
            mixed = sum(s.reshape((-1,) + (1,) * (t[k].ndim - 1)) * (t[k] - base[k]) for s, t in zip(share, terms))
            total[k] += weights[p] * mixed
    return total

