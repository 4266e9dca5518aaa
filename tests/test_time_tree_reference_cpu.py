"""The time-tree reference of tests/time_tree_reference.py pinned on the CPU:

- against central differences of a 50-digit mpmath F on small dated trees (the same pruning
  as test_subst_reference_cpu.py's, the heights, lengths and Jacobian in mpmath too);
- against the CPU oracle on the four influenza fixtures, which says that the reference means
  what libsbn means: the Jacobian, its sign, the clock convention, the site-model derivative;
- as the input and the answer of the host finishing of rooted gradients (csrc/rooted.cpp,
  sbnb_finish_gradients): the reference's exact per-edge derivatives go in, its coordinate
  gradient must come out;
- and the invariants of trees.random_time_trees.
"""
import mpmath
import numpy as np
import pytest
import scipy.special

from conftest import load_fixture
import libsbn_b200 as sbn
from libsbn_b200 import sharding, trees
import subst_reference as ref
import time_tree_reference as tt
from test_subst_reference_cpu import DIGITS, DIFFERENCE_STEP, mp_log_likelihood

GTR_ROW = [0.1, 0.3, 0.05, 0.15, 0.25, 0.15, 0.3, 0.2, 0.15, 0.35]
HKY_ROW = [0.3, 0.2, 0.15, 0.35, 2.5]


def row(substitution, site, shape=0.7):
    head = {"JC69": [], "GTR": GTR_ROW, "HKY": HKY_ROW}[substitution]
    return np.array(head + ([shape] if site != "constant" else []) + [0.0])  # (+ the unused clock column)


def mp_gamma_rates(shape, count):
    quantiles = [mpmath.mpf(2 * c + 1) / (2 * count) for c in range(count)]
    start = scipy.special.gammaincinv(float(shape), [float(q) for q in quantiles])
    x = [mpmath.findroot(lambda v, q=q: mpmath.gammainc(shape, 0, v, regularized=True) - q, mpmath.mpf(s))
         for q, s in zip(quantiles, start)]
    mean = sum(x) / count
    return [v / mean for v in x]


def mp_objective(tree, x):
    """F = logL + log det J at the coordinate vector x (mpf), every step at DIGITS digits."""
    n, N = tree.n, 2 * tree.n - 1
    at, block = 0, {}
    for key, width in tree.blocks:
        block[key] = x[at:at + width]
        at += width
    ratios, root_height = block["ratios_root_height"][:n - 2], block["ratios_root_height"][n - 2]
    bounds = [mpmath.mpf(b) for b in tree.bounds]
    h = list(bounds)
    h[N - 1] = root_height
    for node in range(N - 2, n - 1, -1):
        h[node] = bounds[node] + ratios[node - n] * (h[tree.parent_ids[node]] - bounds[node])
    clock = block["clock_model"]
    rates = [mpmath.mpf(r) + clock[0] for r in tree.rates] if tree.rate_count == 1 else list(clock)
    lengths = [rates[e] * (h[tree.parent_ids[e]] - h[e]) for e in range(N - 1)] + [mpmath.mpf(0)]
    jacobian = sum(mpmath.log(h[tree.parent_ids[i]] - bounds[i]) for i in range(n, N - 1))
    shape = block["site_model"][0] if "site_model" in block else None
    category = mp_gamma_rates(shape, int(tree.site.split("+")[1])) if tree.site.startswith("gamma") else None
    if tree.substitution == "JC69":
        substitution, y = "HKY", [mpmath.mpf(1)] + [mpmath.mpf(v) for v in ref.stick_breaking_inverse([0.25] * 4)]
    else:
        substitution, y = tree.substitution, list(block["substitution_model"])
    return mp_log_likelihood(substitution, tree.site, tree.tips, tree.weights,
                             tree.parent_ids, lengths, shape, y, category_rates=category) + jacobian


def mp_gradient(tree):
    """Central differences of mp_objective at DIGITS digits; the clock of a strict tree is a
    step added to every rate, so its base value is 0."""
    with mpmath.workdps(DIGITS):
        base = [mpmath.mpf(float(v)) for v in tree.ratios]
        base += [mpmath.mpf(0)] if tree.rate_count == 1 else [mpmath.mpf(float(r)) for r in tree.rates]
        if tree.shape is not None:
            base.append(mpmath.mpf(tree.shape))
        if tt.substitution_size(tree.substitution):
            base += [mpmath.mpf(float(v)) for v in ref.coordinates(tree.substitution, tree.params)[0]]
        value = mp_objective(tree, base)
        gradient = []
        for j in range(len(base)):
            plus, minus = list(base), list(base)
            plus[j] += DIFFERENCE_STEP
            minus[j] -= DIFFERENCE_STEP
            gradient.append(float((mp_objective(tree, plus) - mp_objective(tree, minus)) / (2 * DIFFERENCE_STEP)))
        return float(value), np.array(gradient)


SMALL_CASES = [("JC69", "weibull+4", False), ("JC69", "gamma+3", True), ("GTR", "weibull+4", True),
               ("GTR", "gamma+3", False), ("HKY", "weibull+4", False), ("HKY", "gamma+3", True)]


@pytest.mark.parametrize("substitution,site,relaxed", SMALL_CASES,
                         ids=[f"{s}-{m}-{'relaxed' if r else 'strict'}" for s, m, r in SMALL_CASES])
def test_complex_step_matches_fifty_digit_central_differences(substitution, site, relaxed):
    """6 taxa, tips at 3 dates, 8 patterns: every coordinate of F, to 1e-12 of the largest."""
    batch = trees.random_time_trees(6, 1, seed=len(site) + 3 * relaxed, epochs=3, relaxed=relaxed)
    tips, weights = trees.random_alignment(6, 8, seed=5, gap_fraction=0.05)
    tree = tt.TimeTree(substitution, site, tips, weights, batch, 0, row(substitution, site))
    logl, jacobian, gradient = tree.gradient()
    want_value, want = mp_gradient(tree)
    got = np.concatenate([gradient[key] for key, _ in tree.blocks])
    assert abs(logl + jacobian - want_value) <= 1e-13 * abs(want_value)
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want)), f"\n{got}\n{want}"


def test_gamma_rate_derivative_is_the_slope_of_scipy_rates():
    """The 40-digit d rate / d shape against a plain fp64 central difference of scipy's rates,
    which it must match to that difference's own noise (~1e-8)."""
    for shape, count in ((0.2, 8), (0.7, 3), (2.5, 16)):
        h = 1e-5 * shape
        difference = (ref.site_rates(f"gamma+{count}", shape + h)[0] -
                      ref.site_rates(f"gamma+{count}", shape - h)[0]) / (2 * h)
        got = tt.gamma_rate_derivative(shape, count)
        assert np.max(np.abs(got - difference)) <= 1e-6 * np.max(np.abs(difference))


FLUA = ["flua_jc69_strict", "flua_gtr_strict", "flua_jc69_varied_rates", "flua_jc69_weibull4_strict"]


@pytest.mark.parametrize("name", FLUA)
def test_matches_the_oracle_on_the_influenza_fixtures(name):
    """The oracle's rooted blocks (reference_quirks=False) are the derivatives of F: ratios and
    root height with the log-det-Jacobian gradient, the clock as the sum over edges of
    d F / d rate_e (a step added to every rate; the varied-rates fixture tells it from
    d/dc of c x rates), the site shape.  logL and the Jacobian to rounding."""
    from oracle import phylo

    fx = load_fixture(name)
    batch = dict(parent_ids=fx["parent_ids"], node_bounds=fx["node_bounds"], height_ratios=fx["height_ratios"],
                 rates=fx["rates"], rate_count=1)
    params = fx["params"][0] if fx["substitution"] != "JC69" or fx["site"] != "constant" else np.zeros(1)
    tree = tt.TimeTree(fx["substitution"], fx["site"], fx["patterns"], fx["weights"], batch, 0, params)
    logl, jacobian, gradient = tree.gradient()
    want = phylo.gradients(fx["substitution"], fx["site"], fx["patterns"], fx["weights"], fx["parent_ids"],
                           fx["branch_lengths"], fx["params"], rooted=True, rates=fx["rates"],
                           node_heights=fx["node_heights"], node_bounds=fx["node_bounds"],
                           height_ratios=fx["height_ratios"], rate_count=1, reference_quirks=False)
    assert abs(logl - want["log_likelihood"][0]) <= 1e-12 * abs(logl)
    assert jacobian == pytest.approx(fx["golden_jacobian"] if "golden_jacobian" in fx else jacobian, abs=1e-8)
    n = fx["patterns"].shape[0]
    on_host = sharding.finish_log_likelihoods_rooted(n, sbn.TreeBatch(
        fx["parent_ids"], fx["branch_lengths"], fx["rates"], fx["node_heights"], fx["node_bounds"],
        fx["height_ratios"], 1), np.zeros(1))
    assert on_host[0] == pytest.approx(jacobian, rel=1e-13)
    blocks = [("ratios_root_height", want["ratios_root_height"][0]), ("clock_model", want["clock_model"][0])]
    if fx["site"] != "constant":
        blocks.append(("site_model", want["site_model"][:1]))
    for key, oracle_value in blocks:
        error = np.max(np.abs(gradient[key] - oracle_value)) / np.max(np.abs(gradient[key]))
        assert error <= 1e-9, f"{key}: {error:.2e}"


def finish_on_host(substitution, site, taxa, tree_count, seed, relaxed, patterns=12):
    """The reference's raw per-edge sums through sbnb_finish_gradients, and the reference's
    own coordinate gradients."""
    batch = trees.random_time_trees(taxa, tree_count, seed=seed, relaxed=relaxed)
    tips, weights = trees.random_alignment(taxa, patterns, seed=seed + 1, gap_fraction=0.05)
    rng = np.random.default_rng(seed)
    params = np.array([row(substitution, site, shape=rng.uniform(0.3, 2.0)) for _ in range(tree_count)])
    spec = sbn.PhyloModelSpecification(substitution, site, "strict")  # (relaxed: rate_count 2n - 2)
    references, grads, rgrads = [], [], []
    for t in range(tree_count):
        tree = tt.TimeTree(substitution, site, tips, weights, batch, t, params[t])
        references.append(tree.gradient())
        grad, rgrad = tree.edge_derivatives()
        grads.append(grad)
        rgrads.append(rgrad)
    tree_batch = sbn.TreeBatch(**batch)
    categories = len(ref.site_rates(site, 1.0)[0])
    finished = sharding.finish_gradients(spec, taxa, tree_batch, True, False, np.array([r[0] for r in references]),
                                         np.array(grads), np.array(rgrads), categories)
    return references, finished


@pytest.mark.parametrize("substitution,site,taxa,relaxed", [
    ("GTR", "weibull+4", 9, False), ("HKY", "gamma+3", 9, True), ("JC69", "weibull+2", 12, True),
    ("JC69", "weibull+2", 200, False), ("HKY", "constant", 200, True)])
def test_host_finishing_of_rooted_gradients(substitution, site, taxa, relaxed):
    """csrc/rooted.cpp and the site-model sum, fed d logL / d s_e and d logL / d(shape on edge
    e) / s_e of several trees, give the reference's d F / d (ratios, root height, clock, shape)."""
    references, finished = finish_on_host(substitution, site, taxa, 3 if taxa < 100 else 2, seed=taxa + 7 * relaxed,
                                          relaxed=relaxed,
                                          patterns=12 if taxa < 100 else 4)
    for t, ((logl, _, want), got) in enumerate(zip(references, finished)):
        assert got.log_likelihood == logl
        for key in ("ratios_root_height", "clock_model") + (("site_model",) if site != "constant" else ()):
            error = np.max(np.abs(got.gradient[key] - want[key])) / np.max(np.abs(want[key]))
            assert error <= 1e-9, f"tree {t} {key}: {error:.2e}"


@pytest.mark.parametrize("relaxed", [False, True])
@pytest.mark.parametrize("ladder", [False, True])
def test_time_tree_generator_invariants(relaxed, ladder):
    taxa, count = 30, 5
    batch = trees.random_time_trees(taxa, count, seed=3, relaxed=relaxed, ladder=ladder, topology_count=2)
    n, N = taxa, 2 * taxa - 1
    assert batch["rate_count"] == (N - 1 if relaxed else 1)
    tree_batch = sbn.TreeBatch(**batch)
    assert tree_batch.tree_count == count and tree_batch.node_count == N
    assert np.array_equal(batch["parent_ids"][0], batch["parent_ids"][2])  # topologies reused cyclically
    assert not np.array_equal(batch["node_bounds"][0], batch["node_bounds"][2])  # with their own dates
    for t in range(count):
        parent = batch["parent_ids"][t]
        heights, bounds, ratios = batch["node_heights"][t], batch["node_bounds"][t], batch["height_ratios"][t]
        assert np.all(parent > np.arange(N - 1)) and parent.max() == N - 1
        assert np.array_equal(heights[:n], bounds[:n]) and len(np.unique(bounds[:n])) > 1
        for node in range(n, N):
            assert bounds[node] == max(bounds[c] for c in np.flatnonzero(parent == node))
        assert np.all((ratios[:n - 2] >= 1e-3) & (ratios[:n - 2] <= 0.999))
        assert ratios[n - 2] == heights[N - 1] > bounds[N - 1]
        # the heights are the reference's, bit for bit
        assert np.array_equal(tt.heights(parent, bounds, ratios[None, :n - 2], ratios[n - 2])[0], heights)
        assert np.array_equal(batch["branch_lengths"][t, :N - 1], heights[parent] - heights[:N - 1])
        assert batch["branch_lengths"][t, N - 1] == 0.0 and np.all(batch["branch_lengths"][t, :N - 1] > 0)
        rates = batch["rates"][t]
        assert np.all(rates > 0)
        assert len(np.unique(rates)) > 1 if relaxed else (np.all(rates == rates[0]) and rates[0] != 1.0)
        pairs = [bounds[node] == bounds[c] for node in range(n, N - 1) for c in np.flatnonzero(parent == node) if c >= n]
        assert any(pairs) and not all(pairs)  # both sides of the epoch test
