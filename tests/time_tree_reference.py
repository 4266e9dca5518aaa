"""TEST INFRASTRUCTURE: an exact reference for the time-tree gradient (height ratios, root
height, clock rates, site shape, substitution coordinates) and for the unrooted
branch-length and site-shape gradients.

One function of all real inputs, evaluated in complex128,

    F(ratios, root height, clock rates, shape, substitution coordinates) = logL + log det J,

differentiated by the complex step (h = 1e-30) along directions batched on a leading axis:
the unit vectors give the whole gradient, a few seeded random vectors give directional
derivatives g . v of trees too large for one evaluation per coordinate.  logL is
tests/subst_reference.py's pruning (scipy.linalg.expm per edge and category), which shares
no formula with the walk or the CPU oracle: no pre-order pass, no chain rule through the
heights, no closed-form d rate / d shape.

- Heights, top-down: h_i = b_i + r_i (h_parent - b_i), the root at the root height -- the
  float64 expression of trees.random_time_trees, so the real parts are the engine's heights.
- Lengths: edge e evolves for rate_e (h_parent(e) - h_e).
- log det J = sum over non-root internal i of log(h_parent(i) - b_i)
  (LogDetJacobianHeightRatios).
- Clock: the engine's convention, the rates of the tree batch (the parameter row's clock
  column is unused).  Strict clock (rate_count 1): d/dc of rates + c (1, ..., 1); relaxed:
  d/d rate_e per edge.
- Weibull shape: complex-stepped directly (the closed-form quantiles are analytic).  Gamma
  shape: scipy's inverse incomplete gamma takes no complex argument, so the category rates
  are stepped along d rate / d shape, which is taken from 40-digit mpmath (findroot on the
  regularised incomplete gamma, central difference with h = 1e-15).

The coordinate vector is the engine's block order: ratios (n - 2) and the root height (one
"ratios_root_height" block of n - 1), clock (rate_count), shape (0 or 1), substitution
coordinates (0, 4 or 8).
"""
import functools

import mpmath
import numpy as np
import scipy.special

import subst_reference as ref

STEP = ref.STEP
GAMMA_DIGITS = 40
GAMMA_STEP = mpmath.mpf("1e-15")


def gamma_rate_derivative(shape, count):
    """d (normalised median category rate) / d shape of discrete Gamma(shape, rate = shape)."""
    return np.array(_gamma_rate_derivative(float(shape), int(count)))


@functools.lru_cache(maxsize=None)
def _gamma_rate_derivative(shape, count):
    with mpmath.workdps(GAMMA_DIGITS):
        quantiles = [mpmath.mpf(2 * c + 1) / (2 * count) for c in range(count)]
        start = scipy.special.gammaincinv(shape, (2.0 * np.arange(count) + 1.0) / (2.0 * count))

        def rates(a):
            x = [mpmath.findroot(lambda v, q=q: mpmath.gammainc(a, 0, v, regularized=True) - q, mpmath.mpf(s))
                 for q, s in zip(quantiles, start)]
            mean = sum(x) / count
            return [v / mean for v in x]
        a = mpmath.mpf(shape)
        plus, minus = rates(a + GAMMA_STEP), rates(a - GAMMA_STEP)
        return tuple(float((p - m) / (2 * GAMMA_STEP)) for p, m in zip(plus, minus))


def category_rates(site, shape, shape_steps):
    """[J][C] category rates with the shape stepped by i * STEP * shape_steps[j], and the weights."""
    if site == "constant":
        return np.ones((len(shape_steps), 1)), np.ones(1)
    rates, weights = ref.site_rates(site, shape)
    if site.startswith("gamma"):
        derivative = gamma_rate_derivative(shape, len(rates))
        return rates[None, :] + 1j * STEP * np.asarray(shape_steps)[:, None] * derivative[None, :], weights
    return np.array([ref.site_rates(site, shape + 1j * STEP * s)[0] for s in shape_steps]), weights


def substitution_model(substitution, params, steps):
    """(Q [J][4][4], pi [J][4]) with the coordinates stepped by i * STEP * steps[j] (J x 0: unstepped)."""
    if substitution == "JC69":
        q = ref.rate_matrix([1.0] * 6, [0.25] * 4)
        return np.broadcast_to(q, (len(steps), 4, 4)), np.full((len(steps), 4), 0.25, dtype=np.complex128)
    base, model = ref.coordinates(substitution, np.asarray(params, dtype=np.float64))
    qs, freqs = [], []
    for step in steps:
        exchangeabilities, pi = model(list(np.asarray(base, dtype=np.complex128) + (1j * STEP * step if len(step) else 0)))
        qs.append(ref.rate_matrix(exchangeabilities, pi))
        freqs.append(pi)
    return np.array(qs), np.array(freqs, dtype=np.complex128)


def substitution_size(substitution):
    return {"JC69": 0, "GTR": 8, "HKY": 4}[substitution]


def shape_of(substitution, site, params):
    return None if site == "constant" else float(params[{"JC69": 0, "GTR": 10, "HKY": 5}[substitution]])


def heights(parent_ids, bounds, ratios, root_height):
    """[J][nodes] heights, top-down, from [J][n - 2] ratios and [J] root heights."""
    parent_ids = np.asarray(parent_ids)
    N = len(parent_ids) + 1
    n = (N + 1) // 2
    ratios = np.asarray(ratios)
    h = np.broadcast_to(np.asarray(bounds, dtype=ratios.dtype), (len(ratios), N)).copy()
    h[:, N - 1] = root_height
    for node in range(N - 2, n - 1, -1):
        h[:, node] = bounds[node] + ratios[:, node - n] * (h[:, parent_ids[node]] - bounds[node])
    return h


def log_det_jacobian(parent_ids, bounds, h):
    N = len(parent_ids) + 1
    n = (N + 1) // 2
    nodes = np.arange(n, N - 1)
    return np.sum(np.log(h[:, np.asarray(parent_ids)[nodes]] - np.asarray(bounds)[nodes]), axis=1)


class TimeTree:
    """One dated tree of a random_time_trees batch with its model: F and its derivatives."""

    def __init__(self, substitution, site, tips, weights, batch, t, params, masks=False):
        self.substitution, self.site, self.tips, self.weights, self.masks = substitution, site, tips, weights, masks
        self.parent_ids = np.asarray(batch["parent_ids"][t])
        self.bounds = np.asarray(batch["node_bounds"][t], dtype=np.float64)
        self.ratios = np.asarray(batch["height_ratios"][t], dtype=np.float64)
        self.rates = np.asarray(batch["rates"][t], dtype=np.float64)
        self.rate_count = int(batch["rate_count"])
        self.params = np.asarray(params, dtype=np.float64)
        self.shape = shape_of(substitution, site, self.params)
        self.n = len(self.ratios) + 1
        self.blocks = [("ratios_root_height", self.n - 1), ("clock_model", self.rate_count)]
        if self.shape is not None:
            self.blocks.append(("site_model", 1))
        if substitution_size(substitution):
            self.blocks.append(("substitution_model", substitution_size(substitution)))
        self.size = sum(w for _, w in self.blocks)

    def evaluate(self, directions):
        """(logL, log det J, [J] d F / d direction) at the tree's inputs."""
        d = np.atleast_2d(np.asarray(directions, dtype=np.float64))
        n, N = self.n, 2 * self.n - 1
        at = np.cumsum([0] + [w for _, w in self.blocks])
        block = {key: d[:, at[i]:at[i + 1]] for i, (key, _) in enumerate(self.blocks)}
        position = block["ratios_root_height"]
        ratios = self.ratios[None, :n - 2] + 1j * STEP * position[:, :n - 2]
        h = heights(self.parent_ids, self.bounds, ratios, self.ratios[n - 2] + 1j * STEP * position[:, n - 2])
        rates = self.rates[None, :] + 1j * STEP * block["clock_model"]  # (a strict step broadcasts)
        lengths = np.zeros((len(d), N), dtype=np.complex128)
        lengths[:, :N - 1] = rates * (h[:, self.parent_ids] - h[:, :N - 1])
        shape_steps = block["site_model"][:, 0] if "site_model" in block else np.zeros(len(d))
        category, category_weights = category_rates(self.site, self.shape, shape_steps)
        qs, freqs = substitution_model(self.substitution, self.params,
                                       block.get("substitution_model", np.zeros((len(d), 0))))
        logl = ref.prune(qs, freqs, category, category_weights, self.tips, self.weights, self.parent_ids, lengths,
                         self.masks)
        jacobian = log_det_jacobian(self.parent_ids, self.bounds, h)
        total = logl + jacobian
        return float(logl[0].real), float(jacobian[0].real), total.imag / STEP

    def gradient(self):
        """(logL, log det J, {block: d F / d block})."""
        logl, jacobian, g = self.evaluate(np.eye(self.size))
        return logl, jacobian, self.split(g)

    def split(self, g):
        out, at = {}, 0
        for key, width in self.blocks:
            out[key] = g[at:at + width]
            at += width
        return out

    def edge_derivatives(self):
        """The raw sums a walk hands to the host finishing: d logL / d s_e (s_e the effective
        length of edge e) and, with rate categories, d logL / d (shape used on edge e only) / s_e."""
        N = 2 * self.n - 1
        h = heights(self.parent_ids, self.bounds, self.ratios[None, :self.n - 2], self.ratios[self.n - 2])[0]
        s = self.rates * (h[self.parent_ids] - h[:N - 1])
        qs, freqs = substitution_model(self.substitution, self.params, np.zeros((N - 1, 0)))
        eye = np.eye(N - 1)
        category, category_weights = category_rates(self.site, self.shape, np.zeros(1))
        grad = np.zeros(N)
        grad[:N - 1] = ref.prune(qs, freqs, category[0], category_weights, self.tips, self.weights, self.parent_ids,
                                 s[None, :] + 1j * STEP * eye, self.masks).imag / STEP
        rgrad = np.zeros(N)
        if self.shape is not None:
            stepped, _ = category_rates(self.site, self.shape, np.ones(1))
            per_edge = np.where(eye[:, :, None] > 0, stepped[0][None, None, :], category[0][None, None, :])
            rgrad[:N - 1] = ref.prune(qs, freqs, per_edge, category_weights, self.tips, self.weights, self.parent_ids,
                                      np.broadcast_to(s, (N - 1, N - 1)), self.masks).imag / STEP / s
        return grad, rgrad


def unrooted_gradient(substitution, site, tips, weights, parent_ids, lengths, params, masks=False):
    """(logL, d logL / d (length of every edge of the tree as given), d logL / d shape or None)."""
    parent_ids = np.asarray(parent_ids)
    edges = len(parent_ids)
    shape = shape_of(substitution, site, params)
    J = edges + (shape is not None)
    steps = np.zeros(J)
    if shape is not None:
        steps[edges] = 1.0
    category, category_weights = category_rates(site, shape, steps)
    qs, freqs = substitution_model(substitution, params, np.zeros((J, 0)))
    stepped = np.broadcast_to(np.asarray(lengths, dtype=np.float64), (J, edges + 1)).astype(np.complex128)
    stepped[np.arange(edges), np.arange(edges)] += 1j * STEP
    total = ref.prune(qs, freqs, category, category_weights, tips, weights, parent_ids, stepped, masks)
    g = total.imag / STEP
    return float(total[0].real), g[:edges], (g[edges] if shape is not None else None)
