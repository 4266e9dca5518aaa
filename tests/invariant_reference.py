"""TEST INFRASTRUCTURE: an exact reference for site models with a proportion p of invariable
sites (+I), the log-likelihood and every gradient, p included.

Per site pattern k, with L_k the mixture over the rate categories (the rates divided by
1 - p) and I_k the summed frequencies of the states every tip of the pattern allows,

    lik_k = (1 - p) L_k + p I_k.

L_k comes from a plain post-order pruning in complex128 (the one of tests/subst_reference.py:
scipy.linalg.expm per edge and category, a real rescaling factor per node), I_k from the tip
vectors; nothing is formed in the walk's scaled domain.  Derivatives are taken by the complex
step (h = 1e-30) in every input at once, batched on a leading axis: edge lengths (or the
height ratios, root height and clock rates of a time tree), the shape, p and the
substitution coordinates.

`mixture_as_category` is the independent check of the mixture formula: +I as one more rate
category of rate 0 and weight p (every other weight times 1 - p), pruned by
subst_reference.prune, whose zero-rate transition matrices are the identity.
"""
import numpy as np
import scipy.linalg

import subst_reference as ref
import time_tree_reference as tt

STEP = ref.STEP


def base_site(site):
    assert site.endswith("+I"), site
    return site[:-2]


def pinv_index(substitution, site):
    """Column of the proportion invariant in a parameter row: the end of the site block."""
    return {"JC69": 0, "GTR": 10, "HKY": 5}[substitution] + (base_site(site) != "constant")


def invariant_terms(freqs, tips, masks):
    """[J][pattern] I_k: sum over the states every tip allows of pi_s."""
    allowed = np.prod(ref.tip_vectors(tips, masks), axis=0)  # [pattern][4], 0/1
    return np.einsum("ps,js->jp", allowed, np.asarray(freqs, dtype=np.complex128))


def per_site_log_variable(qs, freqs, category_rates, category_weights, tips, parent_ids, lengths, masks):
    """[J][pattern] log L_k: subst_reference.prune without the pattern sum."""
    J = len(qs)
    parent_ids = np.asarray(parent_ids)
    node_count = len(parent_ids) + 1
    taxa, pattern_count = np.asarray(tips).shape
    lengths = np.broadcast_to(np.asarray(lengths)[..., :node_count - 1], (J, node_count - 1))
    tau = lengths[:, :, None] * np.asarray(category_rates)[:, None, :]  # [J][edge][C]
    transition = scipy.linalg.expm(qs[:, None, None] * tau[:, :, :, None, None])
    C = tau.shape[2]
    leaves = ref.tip_vectors(tips, masks)
    children = [[] for _ in range(node_count)]
    for child, parent in enumerate(parent_ids):
        children[parent].append(child)
    partial, log_scale = {}, np.zeros((J, pattern_count))
    for node in range(taxa, node_count):
        product = None
        for child in children[node]:
            below = partial.pop(child) if child >= taxa else leaves[child][None, None]
            evolved = np.matmul(np.broadcast_to(below, (J, C) + below.shape[2:]), transition[:, child].swapaxes(-1, -2))
            product = evolved if product is None else product * evolved
        scale = np.max(product.real, axis=(1, 3))
        scale = np.where(scale > 0, scale, 1.0)
        partial[node] = product / scale[:, None, :, None]
        log_scale += np.log(scale)
    root = partial.pop(node_count - 1)
    site_likelihood = np.einsum("jc,jcps,js->jp", np.asarray(category_weights, dtype=np.complex128), root,
                                np.asarray(freqs, dtype=np.complex128))
    return np.log(site_likelihood) + log_scale


def log_likelihood(qs, freqs, category_rates, category_weights, pinv, tips, weights, parent_ids, lengths, masks):
    """[J] logL of J complex evaluations: category_rates [J][C] before the 1 / (1 - p) factor,
    pinv [J]."""
    pinv = np.asarray(pinv, dtype=np.complex128)
    J = len(qs)
    rates = np.asarray(category_rates) / (1.0 - pinv)[:, None]
    cw = np.broadcast_to(np.asarray(category_weights, dtype=np.complex128), (J, len(category_weights)))
    log_l = per_site_log_variable(qs, freqs, rates, cw, tips, parent_ids, lengths, masks)
    invariant = invariant_terms(freqs, tips, masks)
    return mixture_log_likelihood(log_l, pinv[:, None], invariant) @ np.asarray(weights, dtype=np.float64)


def mixture_log_likelihood(log_l, pinv, invariant):
    """log((1 - p) L + p I) from log L, factored by its larger term, so that neither exp(-log L)
    (1000 taxa: L below the fp64 range) nor exp(log L) overflows.  Both forms are evaluated and
    the one whose factor is the larger term is kept."""
    weighted = pinv * invariant
    with np.errstate(over="ignore", invalid="ignore", divide="ignore", under="ignore"):
        # L ((1 - p) + p I / L): the variable term is the larger one (or p I = 0)
        variable = log_l + np.log((1.0 - pinv) + np.where(weighted == 0, 0.0, weighted * np.exp(-log_l)))
        # p I (1 + (1 - p) L / (p I)): the invariant term is the larger one
        invariant_first = np.log(weighted) + np.log1p((1.0 - pinv) * np.exp(log_l) / weighted)
        larger_variable = (weighted == 0) | (log_l.real + np.log(np.abs(1.0 - pinv)) >= np.log(np.abs(weighted)))
    return np.where(larger_variable, variable, invariant_first)


def mixture_as_category(substitution, site, tips, weights, parent_ids, lengths, params, masks=False):
    """logL with +I as one more rate category (rate 0, weight p): subst_reference.prune."""
    params = np.asarray(params, dtype=np.float64)
    p = params[pinv_index(substitution, site)]
    shape = tt.shape_of(substitution, base_site(site), params)
    category, category_weights = tt.category_rates(base_site(site), shape, np.zeros(1))
    qs, freqs = tt.substitution_model(substitution, params, np.zeros((1, 0)))
    rates = np.append(category[0].real / (1.0 - p), 0.0)
    cw = np.append(category_weights * (1.0 - p), p)
    return float(ref.prune(qs, freqs, rates, cw, tips, weights, parent_ids, np.asarray(lengths, dtype=np.float64),
                           masks)[0].real)


class Model:
    """Site, shape, p and substitution model of one parameter row, complex-steppable."""

    def __init__(self, substitution, site, params):
        self.substitution, self.site = substitution, site
        self.params = np.asarray(params, dtype=np.float64)
        self.shape = tt.shape_of(substitution, base_site(site), self.params)
        self.pinv = float(self.params[pinv_index(substitution, site)])
        self.site_width = (self.shape is not None) + 1
        self.subst_width = tt.substitution_size(substitution)

    def evaluate(self, tips, weights, parent_ids, lengths, site_steps, subst_steps, masks):
        """[J] complex logL; site_steps [J][site_width] (shape, p), subst_steps [J][subst_width]."""
        J = len(lengths)
        site_steps = np.asarray(site_steps, dtype=np.float64)
        shape_steps = site_steps[:, 0] if self.shape is not None else np.zeros(J)
        category, category_weights = tt.category_rates(base_site(self.site), self.shape, shape_steps)
        category = np.broadcast_to(category, (J, category.shape[1]))
        pinv = self.pinv + 1j * STEP * site_steps[:, -1]
        qs, freqs = tt.substitution_model(self.substitution, self.params, np.asarray(subst_steps).reshape(J, -1))
        return log_likelihood(qs, freqs, category, category_weights, pinv, tips, weights, parent_ids, lengths, masks)


def unrooted_gradient(substitution, site, tips, weights, parent_ids, lengths, params, masks=False):
    """(logL, {"branch_lengths": [edges] d/d every edge as given, "site_model": [shape | p],
    "substitution_model": coordinates}) of one tree."""
    model = Model(substitution, site, params)
    parent_ids = np.asarray(parent_ids)
    edges = len(parent_ids)
    J = edges + model.site_width + model.subst_width
    direction = np.eye(J)
    stepped = np.broadcast_to(np.asarray(lengths, dtype=np.float64), (J, edges + 1)).astype(np.complex128)
    stepped[:, :edges] += 1j * STEP * direction[:, :edges]
    total = model.evaluate(tips, weights, parent_ids, stepped, direction[:, edges:edges + model.site_width],
                           direction[:, edges + model.site_width:], masks)
    g = total.imag / STEP
    out = {"branch_lengths": g[:edges], "site_model": g[edges:edges + model.site_width]}
    if model.subst_width:
        out["substitution_model"] = g[edges + model.site_width:]
    return float(total[0].real), out


class InvariantTimeTree(tt.TimeTree):
    """time_tree_reference.TimeTree with the +I mixture: the site-model block is [shape | p]."""

    def __init__(self, substitution, site, tips, weights, batch, t, params, masks=False):
        self.model = Model(substitution, site, params)
        super().__init__(substitution, base_site(site), tips, weights, batch, t, params, masks)
        self.site = site
        self.blocks = [(k, w) for k, w in self.blocks if k != "site_model"]
        self.blocks.insert(2, ("site_model", self.model.site_width))
        self.size = sum(w for _, w in self.blocks)

    def evaluate(self, directions):
        d = np.atleast_2d(np.asarray(directions, dtype=np.float64))
        n, N = self.n, 2 * self.n - 1
        at = np.cumsum([0] + [w for _, w in self.blocks])
        block = {key: d[:, at[i]:at[i + 1]] for i, (key, _) in enumerate(self.blocks)}
        position = block["ratios_root_height"]
        ratios = self.ratios[None, :n - 2] + 1j * STEP * position[:, :n - 2]
        h = tt.heights(self.parent_ids, self.bounds, ratios, self.ratios[n - 2] + 1j * STEP * position[:, n - 2])
        rates = self.rates[None, :] + 1j * STEP * block["clock_model"]
        lengths = np.zeros((len(d), N), dtype=np.complex128)
        lengths[:, :N - 1] = rates * (h[:, self.parent_ids] - h[:, :N - 1])
        logl = self.model.evaluate(self.tips, self.weights, self.parent_ids, lengths, block["site_model"],
                                   block.get("substitution_model", np.zeros((len(d), 0))), self.masks)
        jacobian = tt.log_det_jacobian(self.parent_ids, self.bounds, h)
        total = logl + jacobian
        return float(logl[0].real), float(jacobian[0].real), total.imag / STEP
