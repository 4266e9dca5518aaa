"""Invariable sites (+I) on the host: the "<site>+I" specifications, the normalised model
tables, the finishing entry sbnb_finish_gradients_invariant against NumPy on synthetic
sums, and a self-check of the exact reference of tests/invariant_reference.py."""
import ctypes

import numpy as np
import pytest

import libsbn_b200 as sbn
from libsbn_b200 import _capi, sharding, trees
import invariant_reference as inv
import subst_reference as ref

SBNB_ERR_INVALID_ARGUMENT, SBNB_ERR_MODEL = -1, -5


def tables(site, row, substitution="JC69"):
    """(code, rates, weights, rate derivatives) of sbnb_debug_model_tables."""
    lib = _capi.load()
    row = np.ascontiguousarray(row, dtype=np.float64)
    rates, weights, drates = (np.full(32, np.nan) for _ in range(3))
    code = lib.sbnb_debug_model_tables(substitution.encode(), site.encode(), b"none", _capi.as_double_ptr(row),
                                       None, None, None, None, None, _capi.as_double_ptr(rates),
                                       _capi.as_double_ptr(weights), _capi.as_double_ptr(drates))
    count = int(np.sum(~np.isnan(rates)))
    return code, rates[:count], weights[:count], drates[:count]


@pytest.mark.parametrize("site", ["constant+I", "weibull+I", "weibull+4+I", "gamma+I", "gamma+8+I", "weibull+32+I"])
def test_invariant_specs_are_accepted(site):
    row = [0.7, 0.2] if site != "constant+I" else [0.2]
    assert tables(site, row)[0] == 0


@pytest.mark.parametrize("site", ["weibull+4+J", "weibull+4+I+I", "constant+I+I", "gamma+I4", "weibull+4I",
                                  "weibull+", "weibull+I+4", "constant+J", "weibull+x"])
def test_malformed_suffixes_are_refused(site):
    lib = _capi.load()
    code, *_ = tables(site, [0.7, 0.2, 0.1])
    assert code == SBNB_ERR_INVALID_ARGUMENT
    assert "Site model not known" in lib.sbnb_last_error().decode()


def test_weibull_4_plus_i_is_not_weibull_4():
    """"weibull+4+I" reads p after the shape (weibull+4 has no such entry) and 4 categories."""
    code, plain, _, _ = tables("weibull+4", [0.7])
    code_i, rates, weights, _ = tables("weibull+4+I", [0.7, 0.25])
    assert code == 0 and code_i == 0 and len(rates) == 4 and np.all(weights == 0.25)
    np.testing.assert_allclose(rates, plain / 0.75, rtol=1e-15)


@pytest.mark.parametrize("site,row", [("weibull+4", [0.7]), ("gamma+4", [0.7]), ("weibull+20", [1.3]),
                                      ("constant", [])])
@pytest.mark.parametrize("p", [0.0, 0.05, 0.5, 0.95])
def test_rates_are_normalised(site, row, p):
    _, rates, weights, drates = tables(site, row)
    _, rates_i, weights_i, drates_i = tables(site + "+I", row + [p])
    assert np.array_equal(weights, weights_i)
    if p == 0.0:  # bitwise the tables without +I
        assert np.array_equal(rates, rates_i) and np.array_equal(drates, drates_i)
    np.testing.assert_allclose(rates_i, rates / (1 - p), rtol=1e-15)
    np.testing.assert_allclose(drates_i, drates / (1 - p), rtol=1e-15, atol=0)
    # the mean rate over all sites stays 1
    assert abs((1 - p) * np.dot(weights_i, rates_i) - 1.0) < 1e-14


@pytest.mark.parametrize("p", [1.0, -0.01, float("nan"), float("inf"), 1.5])
def test_p_outside_0_1_is_a_model_error(p):
    code, *_ = tables("weibull+4+I", [0.7, p])
    assert code == SBNB_ERR_MODEL
    assert "Proportion invariant" in _capi.load().sbnb_last_error().decode()


def synthetic_sums(rng, T, N, coords):
    return (rng.normal(size=T), rng.normal(size=(T, N)), rng.normal(size=(T, N)), rng.normal(size=(T, 20)),
            rng.normal(size=(T, 5)))


def reference_finish(substitution, site, batch, params, logl, grad, rgrad, subst, invs):
    """NumPy restatement: fixed-node zeroing, [shape | p] site row, R + p E in the contraction."""
    lib = _capi.load()
    n = (batch.node_count + 2) // 2 if batch.node_count % 2 == 0 else (batch.node_count + 1) // 2
    out = []
    shape_column = site != "constant+I"
    p_column = inv.pinv_index(substitution, site)
    for t in range(batch.tree_count):
        lengths = batch.branch_lengths[t].copy()
        parents = batch.parent_ids[t]
        assert batch.node_count == 2 * n - 1
        root = 2 * n - 2
        root_children = [c for c, parent in enumerate(parents) if parent == root]
        # slide the root onto child 0 (the host's child order: the lower id is child 0 here)
        fixed, kept = max(root_children), min(root_children)
        lengths[kept] += lengths[fixed]
        lengths[fixed] = 0.0
        g = grad[t].copy()
        p = params[t, p_column]
        site_row = ([np.dot(rgrad[t, :-1], lengths[:-1])] if shape_column else []) + \
            [invs[t, 0] + np.dot(g[:-1], lengths[:-1]) / (1 - p)]
        b = np.zeros((8, 16))
        dfreqs = np.zeros((8, 4))
        count = ctypes.c_int32()
        row = np.ascontiguousarray(params[t])
        lib.sbnb_debug_substitution_derivatives(substitution.encode(), site.encode(), b"none",
                                                _capi.as_double_ptr(row), _capi.as_double_ptr(b),
                                                _capi.as_double_ptr(dfreqs), ctypes.byref(count))
        r = subst[t, 16:] + p * invs[t, 1:]
        substitution_row = b[:count.value] @ subst[t, :16] + dfreqs[:count.value] @ r
        out.append((logl[t], g, fixed, np.array(site_row), substitution_row))
    return out


@pytest.mark.parametrize("substitution,site", [("GTR", "weibull+4+I"), ("HKY", "constant+I"), ("GTR", "gamma+8+I")])
@pytest.mark.parametrize("p", [0.0, 0.3])
def test_finishing_entry_against_numpy(substitution, site, p):
    rng = np.random.default_rng(5)
    n, T = 9, 4
    parent_ids, lengths = trees.random_tree_batch(n, T, seed=6, rooted=True)
    batch = sbn.TreeBatch(parent_ids, lengths)
    width = {"GTR": 10, "HKY": 5}[substitution] + (site != "constant+I") + 1
    params = np.empty((T, width))
    for t in range(T):
        freqs = list(rng.dirichlet(np.ones(4) * 4))
        row = (list(rng.dirichlet(np.ones(6) * 2)) + freqs) if substitution == "GTR" else freqs + [2.0]
        if site != "constant+I":
            row.append(0.8)
        params[t] = row + [p]
    logl, grad, rgrad, subst, invs = synthetic_sums(rng, T, 2 * n - 1, 8)
    categories = 1 if site == "constant+I" else int(site.split("+")[1])
    spec = sbn.PhyloModelSpecification(substitution, site, "none")
    got = sharding.finish_gradients_invariant(spec, n, batch, False, params, logl, grad, rgrad, subst, invs,
                                              categories, 1 + (site != "constant+I"))
    want = reference_finish(substitution, site, batch, params, logl, grad, rgrad, subst, invs)
    for g, (logl_t, edges, fixed, site_row, substitution_row) in zip(got, want):
        assert g.log_likelihood == logl_t
        branch = g.gradient["branch_lengths"]
        assert branch[fixed] == 0.0
        edges[fixed] = 0.0
        np.testing.assert_array_equal(branch, edges)
        np.testing.assert_allclose(g.gradient["site_model"], site_row, rtol=1e-13)
        np.testing.assert_allclose(g.gradient["substitution_model"], substitution_row, rtol=1e-12, atol=1e-12)


def test_old_finishing_entries_refuse_invariant_specs():
    lib = _capi.load()
    parent_ids, lengths = trees.random_tree_batch(5, 1, seed=1)
    struct = sbn.TreeBatch(parent_ids, lengths).as_struct()
    N = 9
    logl, grad, rgrad = np.zeros(1), np.zeros(N), np.zeros(N)
    out = _capi.GradientOutStruct()
    site_model = np.zeros(2)
    out.site_model = _capi.as_double_ptr(site_model)
    code = lib.sbnb_finish_gradients(b"JC69", b"weibull+4+I", b"none", 5, ctypes.byref(struct), 0, 0,
                                     _capi.as_double_ptr(logl), _capi.as_double_ptr(grad), _capi.as_double_ptr(rgrad),
                                     ctypes.byref(out))
    assert code == SBNB_ERR_INVALID_ARGUMENT
    assert "sbnb_finish_gradients_invariant" in lib.sbnb_last_error().decode()
    params = np.array([0.7, 0.1])
    code = lib.sbnb_finish_gradients_analytic(b"JC69", b"weibull+4+I", b"none", 5, ctypes.byref(struct), 0,
                                              _capi.as_double_ptr(params), _capi.as_double_ptr(logl),
                                              _capi.as_double_ptr(grad), _capi.as_double_ptr(rgrad), None,
                                              ctypes.byref(out))
    assert code == SBNB_ERR_INVALID_ARGUMENT
    assert "sbnb_finish_gradients_invariant" in lib.sbnb_last_error().decode()
    # and the new entry refuses a model without +I
    code = lib.sbnb_finish_gradients_invariant(b"JC69", b"weibull+4", b"none", 5, ctypes.byref(struct), 0,
                                               _capi.as_double_ptr(params), _capi.as_double_ptr(logl),
                                               _capi.as_double_ptr(grad), _capi.as_double_ptr(rgrad), None,
                                               _capi.as_double_ptr(np.zeros(5)), ctypes.byref(out))
    assert code == SBNB_ERR_INVALID_ARGUMENT


def invariant_alignment(taxa, patterns, seed, constant_fraction=0.3, masks=False):
    """Random columns, a fraction of them constant (one state, a few gaps / ambiguities)."""
    rng = np.random.default_rng(seed)
    if masks:
        tips, _ = trees.random_masked_alignment(taxa, patterns, seed, ambiguous_fraction=0.05, gap_fraction=0.02)
    else:
        tips, _ = trees.random_alignment(taxa, patterns, seed, gap_fraction=0.03)
    tips = tips.copy()
    constant = rng.random(patterns) < constant_fraction
    state = rng.integers(0, 4, size=patterns)
    code = (1 << state) if masks else state
    tips[:, constant] = code[constant]
    gaps = (rng.random(tips.shape) < 0.05) & constant[None, :]
    tips[gaps] = 15 if masks else 4
    weights = rng.integers(1, 4, size=patterns).astype(np.float64)
    return tips, weights


@pytest.mark.parametrize("substitution,site", [("JC69", "constant+I"), ("GTR", "weibull+4+I"),
                                               ("HKY", "gamma+4+I")])
@pytest.mark.parametrize("p", [0.0, 0.05, 0.5, 0.95])
@pytest.mark.parametrize("masks", [False, True])
def test_reference_mixture_equals_zero_rate_category(substitution, site, p, masks):
    """The reference's mixture formula equals +I pruned as an extra category of rate 0."""
    rng = np.random.default_rng(11)
    tips, weights = invariant_alignment(8, 60, seed=3, masks=masks)
    parent_ids, lengths = trees.random_tree_batch(8, 1, seed=4)
    row = {"JC69": [], "GTR": list(rng.dirichlet(np.ones(6) * 2)) + list(rng.dirichlet(np.ones(4) * 4)),
           "HKY": list(rng.dirichlet(np.ones(4) * 4)) + [2.5]}[substitution]
    row += ([] if site == "constant+I" else [0.6]) + [p]
    logl, gradient = inv.unrooted_gradient(substitution, site, tips, weights, parent_ids[0], lengths[0], row, masks)
    other = inv.mixture_as_category(substitution, site, tips, weights, parent_ids[0], lengths[0], row, masks)
    assert abs(logl - other) <= 1e-13 * abs(other)
    # at p = 0 the mixture is the plain model
    if p == 0.0:
        plain = site[:-2]
        base = ref.log_likelihood_and_gradient(substitution, plain, tips, weights, parent_ids[0], lengths[0],
                                               row[:-1], masks)[0] if substitution != "JC69" else None
        if base is not None:
            assert abs(logl - base) <= 1e-13 * abs(base)
    # d logL / dp by the complex step against a central difference
    if 0.0 < p < 0.9:
        h = 1e-6
        up, down = list(row), list(row)
        up[-1] += h
        down[-1] -= h
        fd = (inv.mixture_as_category(substitution, site, tips, weights, parent_ids[0], lengths[0], up, masks) -
              inv.mixture_as_category(substitution, site, tips, weights, parent_ids[0], lengths[0], down, masks)) / (2 * h)
        assert abs(gradient["site_model"][-1] - fd) <= 1e-6 * max(1.0, abs(fd))


def test_reference_mixture_on_a_thousand_taxa():
    """L far below the fp64 range (1000 taxa): the reference's mixture stays finite and equals the
    zero-rate category pruning, and its complex step gives finite derivatives."""
    taxa = 1000
    tips, weights = invariant_alignment(taxa, 64, seed=31, constant_fraction=0.5)
    parent_ids, lengths = trees.random_tree_batch(taxa, 1, seed=32)
    rng = np.random.default_rng(33)
    row = list(rng.dirichlet(np.ones(6) * 2)) + list(rng.dirichlet(np.ones(4) * 4)) + [0.8, 0.3]
    model = inv.Model("GTR", "weibull+4+I", row)
    directions = rng.normal(size=(2, 10))
    stepped = np.broadcast_to(lengths[0], (2, lengths.shape[1])).astype(np.complex128)
    total = model.evaluate(tips, weights, parent_ids[0], stepped, directions[:, :2], directions[:, 2:], False)
    other = inv.mixture_as_category("GTR", "weibull+4+I", tips, weights, parent_ids[0], lengths[0], row)
    assert np.all(np.isfinite(total.real)) and np.all(np.isfinite(total.imag))
    assert abs(total[0].real - other) <= 1e-13 * abs(other)
