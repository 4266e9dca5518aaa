"""TEST INFRASTRUCTURE: an exact reference for d logL / d (substitution-model coordinates).

A plain post-order pruning in complex128, differentiated by the complex step:
g_j = Im logL(theta + i h e_j) / h with h = 1e-30.  Nothing is subtracted, so the
derivative is exact to fp64 rounding, like the log likelihood itself.  It shares no
formula with the fused walk's analytic gradient: no eigendecomposition, no Phi, no
V^-1 dQ V, no pre-order pass -- every transition matrix is scipy.linalg.expm(Q r_c t).

Coordinates are the engine's (libsbn_b200/csrc/model.cpp, engine.cu):
- GTR: the 5 stick-breaking coordinates of the six exchangeabilities, then the 3 of the
  four frequencies, y_k = logit(z_k) + log(K - k - 1).
- HKY: kappa itself, then the 3 frequency coordinates.
Parameter rows are in the engine's block order: GTR rates, frequencies, [shape];
HKY frequencies, kappa, [shape].

The tree is given as parent ids in the reference's convention (children have smaller
ids than their parents, the root is the last node), with one length per node that
the pruning uses as is: a trifurcating unrooted root, a bifurcating root, or the
effective lengths of a time tree (clock rate x height difference).  Every model here
is reversible with the root at stationarity, so where on the root edge pair the root
sits does not change logL or its gradient (the pulley principle): the engine's root
slide need not be repeated.
"""
import numpy as np
import scipy.linalg
import scipy.special

STEP = 1e-30


def stick_breaking(y):
    """Coordinates (K - 1) -> simplex (K), model.cpp StickBreaking; complex-safe."""
    count = len(y) + 1
    stick, x = 1.0, []
    for k, value in enumerate(y):
        z = 1.0 / (1.0 + np.exp(-(value - np.log(count - k - 1.0))))
        x.append(stick * z)
        stick = stick - stick * z
    return x + [stick]


def stick_breaking_inverse(x):
    """Simplex (K) -> coordinates (K - 1), model.cpp StickBreakingInverse."""
    y, used = [], 0.0
    for k in range(len(x) - 1):
        z = x[k] / (1.0 - used)
        y.append(np.log(z / (1.0 - z)) + np.log(len(x) - k - 1.0))
        used += x[k]
    return y


def rate_matrix(rates, freqs):
    """GTR Q (exchangeabilities AC AG AT CG CT GT) scaled to one expected substitution
    per unit time, as model.cpp GeneralTimeReversible builds it; complex-safe."""
    q = np.zeros((4, 4), dtype=np.complex128)
    index = 0
    for i in range(4):
        for j in range(i + 1, 4):
            q[i, j] = rates[index] * freqs[j]
            q[j, i] = rates[index] * freqs[i]
            index += 1
    row_sums = q.sum(axis=1)
    q[np.diag_indices(4)] = -row_sums
    return q / np.sum(row_sums * np.asarray(freqs, dtype=np.complex128))


def site_rates(site, shape):
    """Category rates (mean 1) and weights: the median discretisation of Weibull (closed
    form) or Gamma(shape, rate = shape) (scipy's inverse incomplete gamma)."""
    if site == "constant":
        return np.ones(1), np.ones(1)
    kind, _, count = site.partition("+")
    count = int(count) if count else 4
    quantiles = (2.0 * np.arange(count) + 1.0) / (2.0 * count)
    if kind == "weibull":
        rates = (-np.log(1.0 - quantiles)) ** (1.0 / shape)
    elif kind == "gamma":
        rates = scipy.special.gammaincinv(shape, quantiles)
    else:
        raise ValueError(f"site model {site!r}")
    return rates / rates.mean(), np.full(count, 1.0 / count)


def coordinates(substitution, params):
    """(base coordinates, their count, coordinates -> (rates, freqs)) of a parameter row."""
    if substitution == "GTR":
        base = stick_breaking_inverse(list(params[:6])) + stick_breaking_inverse(list(params[6:10]))
        return base, lambda y: (stick_breaking(y[:5]), stick_breaking(y[5:8]))
    if substitution == "HKY":
        base = [params[4]] + stick_breaking_inverse(list(params[:4]))
        return base, lambda y: ([1.0, y[0], 1.0, 1.0, y[0], 1.0], stick_breaking(y[1:4]))
    raise ValueError(f"substitution model {substitution!r}")


def tip_vectors(tips, masks):
    """[taxon][pattern] states (0..3, >= 4 missing) or nucleotide masks -> [taxon][pattern][4]."""
    tips = np.asarray(tips).astype(np.int64)
    if masks:
        return ((tips[..., None] >> np.arange(4)) & 1).astype(np.float64)
    return np.where(tips[..., None] >= 4, 1.0, (tips[..., None] == np.arange(4)).astype(np.float64))


def prune(qs, freqs, category_rates, category_weights, tips, weights, parent_ids, lengths, masks=False):
    """Per-evaluation logL of J complex evaluations of one tree, batched on a leading axis.

    qs: [J][4][4] rate matrices; freqs: [J][4]; category_rates: [C] or [J][C], or
    [J][edge][C] for rates that differ per edge; category_weights: [C]; lengths: [nodes]
    or [J][nodes] (the root's entry is unused)."""
    J = len(qs)
    parent_ids = np.asarray(parent_ids)
    node_count = len(parent_ids) + 1
    taxa, pattern_count = np.asarray(tips).shape
    lengths = np.broadcast_to(np.asarray(lengths)[..., :node_count - 1], (J, node_count - 1))
    category_rates = np.asarray(category_rates)
    if category_rates.ndim < 3:
        category_rates = np.broadcast_to(category_rates, (J, len(category_weights)))[:, None, :]
    tau = lengths[:, :, None] * category_rates  # [J][edge][C]
    transition = scipy.linalg.expm(qs[:, None, None] * tau[:, :, :, None, None])  # [J][edge][C][4][4]
    C = tau.shape[2]
    leaves = tip_vectors(tips, masks)
    children = [[] for _ in range(node_count)]
    for child, parent in enumerate(parent_ids):
        children[parent].append(child)
    partial, log_scale = {}, np.zeros((J, pattern_count))
    for node in range(taxa, node_count):  # every child id is smaller than its parent's
        product = None
        for child in children[node]:
            below = partial.pop(child) if child >= taxa else leaves[child][None, None]
            # (P L)[j, c, p, i] = sum_s P[j, c, i, s] L[j, c, p, s]
            evolved = np.matmul(np.broadcast_to(below, (J, C) + below.shape[2:]),
                                transition[:, child].swapaxes(-1, -2))
            product = evolved if product is None else product * evolved
        # a real factor per pattern: the complex step is untouched and 1000 taxa do not underflow
        scale = np.max(product.real, axis=(1, 3))
        scale = np.where(scale > 0, scale, 1.0)
        partial[node] = product / scale[:, None, :, None]
        log_scale += np.log(scale)
    root = partial.pop(node_count - 1)
    site_likelihood = np.einsum("c,jcps,js->jp", category_weights, root, np.asarray(freqs, dtype=np.complex128))
    per_site = np.log(site_likelihood) + log_scale
    return per_site @ np.asarray(weights, dtype=np.float64)


def model_at(substitution, params, base, step):
    """(Q [J][4][4], pi [J][4]): one evaluation per coordinate, that coordinate stepped by i * step."""
    _, model = coordinates(substitution, params)
    qs, freqs = [], []
    for j in range(len(base)):
        y = np.array(base, dtype=np.complex128)
        y[j] += 1j * step
        exchangeabilities, pi = model(list(y))
        qs.append(rate_matrix(exchangeabilities, pi))
        freqs.append(pi)
    return np.array(qs), np.array(freqs, dtype=np.complex128)


def log_likelihood_and_gradient(substitution, site, tips, weights, parent_ids, lengths, params, masks=False):
    """(logL, d logL / d coordinates in the engine's order) of one tree.

    tips: [taxon][pattern]; parent_ids: [nodes - 1]; lengths: [nodes] (the root's entry is
    unused); params: the substitution and site blocks of an engine parameter row."""
    params = np.asarray(params, dtype=np.float64)
    base, _ = coordinates(substitution, params)
    shape = params[10 if substitution == "GTR" else 5] if site != "constant" else None
    rates, category_weights = site_rates(site, shape)
    # one complex evaluation per coordinate, batched on a leading axis
    qs, freqs = model_at(substitution, params, base, STEP)
    total = prune(qs, freqs, rates, category_weights, tips, weights, parent_ids,
                  np.asarray(lengths, dtype=np.float64), masks)
    return float(total[0].real), total.imag / STEP
