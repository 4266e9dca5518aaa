"""TEST INFRASTRUCTURE: an exact reference for the GP engine on a generated subsplit DAG.

Every tree tau the DAG holds (tests/gp_dag.py) is pruned on its own with
subst_reference.prune -- complex128, every transition matrix scipy.linalg.expm(Q r_c t), a real
rescaling factor per pattern -- and the trees are summed with their SBN probabilities
P(tau) = q(rootsplit) * prod q(child | parent).  Nothing of the engine's formulas is shared: no
PLVs, no eigensystem, no rescaling counts, no LogAdd fold.  With identity pattern weights prune
returns one log likelihood per pattern:

- marginal, pattern k:   log sum_tau P(tau) L_k(tau);
- per-GPCSP value of e:  sum_k w_k log( sum_{tau containing e} P(tau) L_k(tau) / q(e) ),
  the normalisation of the LIKELIHOOD and INCREMENT_MARGINAL records (oracle/gp.py);
- its derivative in e's branch length by the complex step (h = 1e-30) on that length;
- the exact optimum of the per-GPCSP value in log t on the engine's interval;
- the SBN update q'(e) ~ q(e) exp(per-GPCSP value of e) within e's group (hybrid marginals,
  when given, in place of the per-GPCSP values).

The enumeration is capped at 5 000 trees (SubsplitDAG.trees): the DAGs of the tests hold at
most a few hundred.
"""
import math

import numpy as np
import scipy.optimize
import scipy.special

import subst_reference

STEP = 1e-30
MIN_LOG_BRANCH_LENGTH, MAX_LOG_BRANCH_LENGTH = -13.9, 1.1  # gp_engine.hpp:88-89


def rate_matrix(substitution, params):
    """(Q, pi) of the engine's "entire substitution" parameter block."""
    params = np.asarray(params, dtype=np.float64)
    if substitution == "JC69":
        rates, freqs = np.ones(6), np.full(4, 0.25)
    elif substitution == "HKY":
        freqs, kappa = params[:4], params[4]
        rates = np.array([1.0, kappa, 1.0, 1.0, kappa, 1.0])
    elif substitution == "GTR":
        rates, freqs = params[:6], params[6:10]
    else:
        raise ValueError(substitution)
    return subst_reference.rate_matrix(rates, freqs), np.asarray(freqs, dtype=np.complex128)


class Model:
    def __init__(self, substitution="JC69", params=(), site="constant", shape=None):
        self.q_matrix, self.freqs = rate_matrix(substitution, params)
        self.rates, self.proportions = subst_reference.site_rates(site, shape)


def _tree_log_likelihoods(dag, model, tips, branch_lengths, tree, masks, stepped=()):
    """[1 + len(stepped)][P] complex per-pattern log likelihoods of one tree: at the given lengths,
    then once per GPCSP of `stepped` with that GPCSP's length moved by i * STEP."""
    parent_ids, lengths, child_of = dag.tree_shape(tree, branch_lengths)
    J = 1 + len(stepped)
    lengths = np.tile(lengths.astype(np.complex128), (J, 1))
    for j, g in enumerate(stepped):
        lengths[j + 1, child_of[g]] += 1j * STEP
    P = np.asarray(tips).shape[1]
    return subst_reference.prune(np.repeat(model.q_matrix[None], J, axis=0), np.repeat(model.freqs[None], J, axis=0),
                                 model.rates, model.proportions, tips, np.eye(P), parent_ids, lengths, masks)


def _log_sum(values, axis=0):
    """log sum exp over `axis` of complex logs (real maximum subtracted: the imaginary parts ride along)."""
    peak = np.max(values.real, axis=axis, keepdims=True)
    return np.squeeze(peak, axis=axis) + np.log(np.sum(np.exp(values - peak), axis=axis))


class Reference:
    """Everything about one DAG, one model, one alignment and one set of branch lengths."""

    def __init__(self, dag, model, tips, weights, branch_lengths, q=None, masks=False, derivatives=True):
        self.dag, self.model, self.tips, self.masks = dag, model, tips, masks
        self.weights = np.asarray(weights, dtype=np.float64)
        self.branch_lengths = np.asarray(branch_lengths, dtype=np.float64)
        self.q = dag.q if q is None else np.asarray(q, dtype=np.float64)
        self.trees = dag.trees()
        self.log_prior = np.array([np.sum(np.log(self.q[list(t)])) for t in self.trees])
        # per tree: [1 + edges][P] -- at the lengths, then stepped on each non-rootsplit GPCSP
        self.stepped = [tuple(g for g in t if dag.edges[g][0] is not None) if derivatives else () for t in self.trees]
        self.per_tree = [_tree_log_likelihoods(dag, model, tips, self.branch_lengths, t, masks, s)
                         for t, s in zip(self.trees, self.stepped)]
        base = np.array([x[0].real for x in self.per_tree])  # [tree][P]
        self.per_pattern_marginal = _log_sum(base + self.log_prior[:, None])
        self.containing = [[] for _ in range(dag.gpcsp_count)]
        for i, t in enumerate(self.trees):
            for g in t:
                self.containing[g].append(i)

    def log_marginal_likelihood(self):
        return float(self.per_pattern_marginal @ self.weights)

    def per_pattern_gpcsp(self, g):
        """log( sum_{tau containing g} P(tau) L_k(tau) / q(g) ) per pattern k."""
        rows = self.containing[g]
        base = np.array([self.per_tree[i][0].real for i in rows]) + self.log_prior[rows, None]
        return _log_sum(base) - math.log(self.q[g])

    def per_gpcsp_log_likelihoods(self):
        return np.array([self.per_pattern_gpcsp(g) @ self.weights for g in range(self.dag.gpcsp_count)])

    def log_likelihood_matrix(self):
        return np.array([self.per_pattern_gpcsp(g) for g in range(self.dag.gpcsp_count)])

    def per_gpcsp_components_of_full_log_marginal(self, site_count):
        return self.per_gpcsp_log_likelihoods() + float(site_count) * np.log(self.q)

    def derivative(self, g):
        """(value, d value / d t_g, sum_k w_k |d log l_k / d t_g|) of the per-GPCSP value of g."""
        rows = self.containing[g]
        stepped = np.array([self.per_tree[i][1 + self.stepped[i].index(g)] for i in rows]) + self.log_prior[rows, None]
        per_pattern = _log_sum(stepped)
        slopes = per_pattern.imag / STEP
        return (float((per_pattern.real - math.log(self.q[g])) @ self.weights), float(slopes @ self.weights),
                float(np.abs(slopes) @ self.weights))

    def value_at(self, g, branch_length):
        """The per-GPCSP value of g with its length set to branch_length (the others unchanged)."""
        lengths = self.branch_lengths.copy()
        lengths[g] = branch_length
        rows = self.containing[g]
        base = np.array([_tree_log_likelihoods(self.dag, self.model, self.tips, lengths, self.trees[i], self.masks)[0].real
                         for i in rows]) + self.log_prior[rows, None]
        return float((_log_sum(base) - math.log(self.q[g])) @ self.weights)

    def optimum(self, g):
        """(log t, value) maximising the per-GPCSP value of g on the engine's interval (bounded Brent)."""
        result = scipy.optimize.minimize_scalar(lambda x: -self.value_at(g, math.exp(x)), method="bounded",
                                                bounds=(MIN_LOG_BRANCH_LENGTH, MAX_LOG_BRANCH_LENGTH),
                                                options={"xatol": 1e-10, "maxiter": 500})
        return float(result.x), -float(result.fun)

    def updated_sbn_parameters(self, hybrid=None):
        """UpdateSBNProbabilities over every group of more than one GPCSP."""
        values = self.per_gpcsp_log_likelihoods() if hybrid is None else np.asarray(hybrid, dtype=np.float64)
        q = self.q.copy()
        for start, stop in self.dag.groups:
            if stop - start > 1:
                unnormalised = values[start:stop] + np.log(self.q[start:stop])
                q[start:stop] = np.exp(unnormalised - scipy.special.logsumexp(unnormalised))
        return q
