"""The CUDA GP engine, through the C ABI, against the exact reference of tests/gp_reference.py on
generated subsplit DAGs (tests/gp_dag.py): every launch regime and shared-memory fallback of the
interpreter -- each test asserts the regime it covers through GPEngine.launch_plan -- 1-8 rate
categories (Weibull and gamma), JC69 / GTR / HKY, state and mask tips, deep rescaling, a root
group longer than the UpdateSBNProbabilities scratch, and Brent's search.  The numpy oracle is
used only where the reference has no counterpart: PLVs and rescaling counts, and a Brent sweep.

Bars: marginal and per-GPCSP values 1e-9 relative; LogLikelihoodAndDerivative's derivative
1e-8 x sum_k w_k |d log l_k / dt| (scale-aware: an edge near its optimum does not cancel the bar
away); SBN parameters 1e-9 relative."""
import math

import numpy as np
import pytest

import gp_dag
import gp_reference
import libsbn_b200 as sbn
from oracle import gp

pytestmark = pytest.mark.gpu

GTR = [0.10, 0.24, 0.07, 0.15, 0.33, 0.11, 0.15, 0.35, 0.3, 0.2]  # (the engine asks rates summing to 1)
HKY = [0.35, 0.15, 0.2, 0.3, 2.7]
PARAMS = {"JC69": (), "GTR": GTR, "HKY": HKY}
TOLERANCE = math.ldexp(1.0, 1 - gp.GPEngineOracle.SIGNIFICANT_DIGITS)  # Brent's, gp_engine.hpp:91


def close(got, want, rtol=1e-9):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    assert np.all(err <= rtol), f"worst rel err {err.max():.3e} at {np.argmax(err)}"


def alignment(dag, patterns, seed, gap_fraction=0.05, tree=None):
    rng = np.random.default_rng(seed)
    lengths = rng.uniform(0.02, 0.4, dag.gpcsp_count)
    tree = dag.trees()[0] if tree is None else tree
    tips = gp_dag.simulate_states(dag, tree, lengths, patterns, rng, gap_fraction)
    weights = rng.integers(1, 5, patterns).astype(np.float64)
    return tips, weights, lengths


def engine_for(dag, tips, weights, lengths, substitution="JC69", site="constant", shape=None, threshold=1e-40,
               factory=None, **kwargs):
    factory = factory or (lambda *a, **k: sbn.GPEngine(*a, device=0, **k))
    engine = factory(tips, weights, int(weights.sum()), dag.plv_count, dag.gpcsp_count, rescaling_threshold=threshold,
                     sbn_prior=dag.q, unconditional_node_probabilities=dag.unconditional_node_probabilities,
                     inverted_sbn_prior=dag.inverted_sbn_prior, **kwargs)
    engine.set_substitution_model(substitution, PARAMS[substitution])
    if site != "constant":
        engine.set_site_model(site, [shape])
    engine.set_branch_lengths(lengths)
    engine.process_operations(dag.programs["populate_plvs"])
    engine.process_operations(dag.programs["compute_likelihoods"])
    return engine


def check_against_reference(engine, dag, tips, weights, lengths, substitution="JC69", site="constant", shape=None,
                            masks=False, edges=4, seed=0):
    want = gp_reference.Reference(dag, gp_reference.Model(substitution, PARAMS[substitution], site, shape), tips,
                                  weights, lengths, masks=masks)
    close(engine.get_log_marginal_likelihood(), want.log_marginal_likelihood())
    close(engine.get_per_gpcsp_log_likelihoods(), want.per_gpcsp_log_likelihoods())
    rng = np.random.default_rng(seed)
    for g in rng.choice(np.arange(dag.rootsplit_count, dag.gpcsp_count), size=min(edges, dag.gpcsp_count - dag.rootsplit_count),
                        replace=False):
        value, slope, scale = want.derivative(g)
        got = engine.log_likelihood_and_derivative(*dag.edge_plvs(g), int(g))
        close(got[0], value)
        assert abs(got[1] - slope) <= 1e-8 * scale, (g, got[1], slope)
    return want


SMALL = gp_dag.hybrid_dag(7, 12, seed=4)


@pytest.mark.parametrize("patterns,categories,regime", [(100, 1, "one CTA"), (600, 1, "cluster"),
                                                        (1500, 4, "mailbox"), (10000, 4, "strided")])
def test_launch_regimes(patterns, categories, regime):
    """E = patterns x categories: one CTA (E <= 128), a 2-8-CTA cluster, the cooperative mailbox (more
    than 8 CTAs, E <= 148 x 128), and the strided path (256 threads, several pairs per thread)."""
    site = "constant" if categories == 1 else f"weibull+{categories}"
    tips, weights, lengths = alignment(SMALL, patterns, seed=patterns)
    engine = engine_for(SMALL, tips, weights, lengths, "GTR", site, 0.6)
    plan = engine.launch_plan
    if regime == "one CTA":
        assert plan["blocks"] == 1
    elif regime == "cluster":
        assert 2 <= plan["blocks"] <= 8 and plan["cluster"]
    elif regime == "mailbox":
        assert plan["blocks"] > 8 and plan["threads"] == 128
    else:
        assert plan["threads"] == 256 and plan["blocks"] * plan["threads"] < patterns * categories
    check_against_reference(engine, SMALL, tips, weights, lengths, "GTR", site, 0.6)
    engine.process_operations(SMALL.programs["optimize_sbn_parameters"])
    want = gp_reference.Reference(SMALL, gp_reference.Model("GTR", GTR, site, 0.6), tips, weights, lengths,
                                  derivatives=False)
    close(engine.get_sbn_parameters(), want.updated_sbn_parameters())


def test_cluster_and_mailbox_give_the_same_bits(monkeypatch):
    tips, weights, lengths = alignment(SMALL, 300, seed=300)  # E = 600: five CTAs
    results = []
    for no_cluster in ("0", "1"):
        monkeypatch.setenv("SBNB_GP_NO_CLUSTER", no_cluster)
        engine = engine_for(SMALL, tips, weights, lengths, "HKY", "gamma+2", 0.8)
        assert engine.launch_plan["cluster"] == (no_cluster == "0") and engine.launch_plan["blocks"] > 1
        for name in ("branch_length_optimization", "populate_plvs", "compute_likelihoods", "optimize_sbn_parameters"):
            engine.process_operations(SMALL.programs[name])
        results.append([engine.get_branch_lengths(), engine.get_per_gpcsp_log_likelihoods(),
                        engine.get_sbn_parameters(), engine.get_plv(SMALL.plv_count - 1)])
    for a, b in zip(*results):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("kind", ["weibull", "gamma"])
@pytest.mark.parametrize("categories", [1, 2, 4, 8])
@pytest.mark.parametrize("shape", [0.3, 1.0, 3.0])
def test_rate_categories(kind, categories, shape):
    tips, weights, lengths = alignment(SMALL, 40, seed=categories)
    site = f"{kind}+{categories}"
    engine = engine_for(SMALL, tips, weights, lengths, "HKY", site, shape)
    assert engine.category_count == categories
    check_against_reference(engine, SMALL, tips, weights, lengths, "HKY", site, shape)


@pytest.mark.parametrize("substitution", ["JC69", "GTR", "HKY"])
def test_substitution_models_with_random_parameters(substitution):
    rng = np.random.default_rng(len(substitution))
    freqs = rng.dirichlet(np.full(4, 2.0))
    rates = rng.uniform(0.2, 3.0, 6)
    PARAMS_RANDOM = {"JC69": (), "GTR": list(rates / rates.sum()) + list(freqs), "HKY": list(freqs) + [rng.uniform(1, 5)]}
    tips, weights, lengths = alignment(SMALL, 64, seed=3)
    saved = PARAMS[substitution]
    PARAMS[substitution] = PARAMS_RANDOM[substitution]
    try:
        engine = engine_for(SMALL, tips, weights, lengths, substitution, "weibull+4", 0.5)
        check_against_reference(engine, SMALL, tips, weights, lengths, substitution, "weibull+4", 0.5)
    finally:
        PARAMS[substitution] = saved


def test_mask_tips_with_ambiguous_codes():
    rng = np.random.default_rng(17)
    tips, weights, lengths = alignment(SMALL, 80, seed=17, gap_fraction=0.0)
    masks = (1 << tips).astype(np.uint8)
    ambiguous = rng.random(masks.shape) < 0.15
    masks[ambiguous] = rng.integers(1, 16, int(ambiguous.sum()))
    masks[rng.random(masks.shape) < 0.05] = 15
    engine = engine_for(SMALL, masks, weights, lengths, "GTR", "gamma+4", 1.2, tip_encoding="masks")
    check_against_reference(engine, SMALL, masks, weights, lengths, "GTR", "gamma+4", 1.2, masks=True)


def test_global_matrix_cache_at_eight_categories():
    dag = gp_dag.hybrid_dag(9, 30, seed=5)
    assert dag.gpcsp_count > 100
    tips, weights, lengths = alignment(dag, 16, seed=5)
    engine = engine_for(dag, tips, weights, lengths, "GTR", "weibull+8", 0.7)
    assert not engine.launch_plan["shared_matrices"]
    check_against_reference(engine, dag, tips, weights, lengths, "GTR", "weibull+8", 0.7, edges=6)
    # a Brent sweep writes the cache; the oracle runs the same sweep
    want = engine_for(dag, tips, weights, lengths, "GTR", "weibull+8", 0.7, factory=gp.GPEngineOracle)
    for e in (engine, want):
        e.process_operations(dag.programs["branch_length_optimization"])
    close(engine.get_branch_lengths(), want.get_branch_lengths(), rtol=1e-3)


def test_global_matrix_cache_on_a_400_taxon_tree():
    dag = gp_dag.one_tree_dag(400, "random", seed=9)
    tips, weights, lengths = alignment(dag, 96, seed=9)
    engine = engine_for(dag, tips, weights, lengths, "HKY")
    assert not engine.launch_plan["shared_matrices"]
    check_against_reference(engine, dag, tips, weights, lengths, "HKY", edges=6)


@pytest.mark.parametrize("threshold", [1e-40, 1e-3, 0.5])
def test_global_rescaling_counts_on_a_1000_taxon_ladder(threshold):
    dag = gp_dag.one_tree_dag(1000, "ladder", seed=10)
    tips, weights, lengths = alignment(dag, 128, seed=10)
    lengths = lengths * 3.0  # long branches: small PLV entries at depth
    engine = engine_for(dag, tips, weights, lengths, "JC69", threshold=threshold)
    plan = engine.launch_plan
    assert not plan["shared_counts"]
    want = gp_reference.Reference(dag, gp_reference.Model("JC69"), tips, weights, lengths, derivatives=False)
    close(engine.get_log_marginal_likelihood(), want.log_marginal_likelihood())
    close(engine.get_per_gpcsp_log_likelihoods(), want.per_gpcsp_log_likelihoods())
    oracle = engine_for(dag, tips, weights, lengths, "JC69", threshold=threshold, factory=gp.GPEngineOracle)
    counts = engine.get_rescaling_counts()
    assert np.array_equal(counts, oracle.rescaling_counts)
    assert counts.max() >= (1 if threshold < 0.5 else 100)
    for index in (dag.plv(gp_dag.P_PLV, dag.node_count - 1), dag.plv(gp_dag.RHAT, 0), dag.plv(gp_dag.R_PLV, 1500)):
        close(engine.get_plv(index), oracle.plvs[index], rtol=1e-9 if threshold != 0.5 else 1e-8)


WIDE = gp_dag.wide_root_dag(10, 300, seed=8)


@pytest.mark.parametrize("source", ["per_gpcsp", "hybrid"])
def test_wide_root_group_sbn_update(source):
    """A root group of 300 GPCSPs: longer than the 256-double scratch, so the second pass recomputes."""
    tips, weights, lengths = alignment(WIDE, 48, seed=8)
    engine = engine_for(WIDE, tips, weights, lengths, "GTR", "weibull+2", 0.9)
    assert WIDE.groups[0][1] > engine.launch_plan["scratch"]
    want = gp_reference.Reference(WIDE, gp_reference.Model("GTR", GTR, "weibull+2", 0.9), tips, weights, lengths,
                                  derivatives=False)
    hybrid = None
    if source == "hybrid":
        hybrid = np.random.default_rng(1).normal(-300.0, 20.0, WIDE.gpcsp_count)
        engine.set_hybrid_marginals(hybrid)
        close(engine.get_hybrid_marginals(), hybrid, rtol=0)
    engine.process_operations(WIDE.programs["optimize_sbn_parameters"])
    close(engine.get_sbn_parameters(), want.updated_sbn_parameters(hybrid))


BRENT = gp_dag.one_tree_dag(8, "random", seed=21)


def _brent_case(kind):
    tips, weights, lengths = alignment(BRENT, 200, seed=21, gap_fraction=0.0)
    cherry = next(v for v in range(BRENT.taxon_count, BRENT.node_count)
                  if all(BRENT.is_leaf(c) for s in (0, 1) for _, c in BRENT.children[(v, s)]))
    (g0, a), (g1, b) = BRENT.children[(cherry, 0)][0], BRENT.children[(cherry, 1)][0]
    if kind == "zero":
        tips[b] = tips[a]
        return tips, weights, lengths, g1
    if kind == "saturated":
        tips[a] = np.random.default_rng(5).integers(0, 4, tips.shape[1])
        return tips, weights, lengths, g0
    return tips, weights, lengths, BRENT.parents[cherry][0][0]


@pytest.mark.parametrize("kind", ["interior", "zero", "saturated"])
def test_single_brent_search_finds_the_exact_optimum(kind):
    tips, weights, lengths, g = _brent_case(kind)
    engine = engine_for(BRENT, tips, weights, lengths, "HKY", "gamma+4", 0.8)
    want = gp_reference.Reference(BRENT, gp_reference.Model("HKY", HKY, "gamma+4", 0.8), tips, weights, lengths,
                                  derivatives=False)
    x_opt, f_opt = want.optimum(g)
    start = want.value_at(g, lengths[g])
    engine.process_operations(np.array([5, *BRENT.edge_plvs(g), g], dtype=np.int32))
    accepted = engine.get_branch_lengths()[g]
    x = math.log(accepted)
    assert abs(x - x_opt) <= 2 * (TOLERANCE * abs(x_opt) + TOLERANCE / 4), (kind, x, x_opt)
    assert want.value_at(g, accepted) >= start - 1e-9 * abs(start)
    if kind == "zero":
        assert x < -10
    if kind == "saturated":
        assert x > 0


def test_brent_sweep_against_the_oracle():
    tips, weights, lengths = alignment(SMALL, 300, seed=30)
    ours = engine_for(SMALL, tips, weights, lengths, "GTR", "gamma+2", 0.5)
    want = engine_for(SMALL, tips, weights, lengths, "GTR", "gamma+2", 0.5, factory=gp.GPEngineOracle)
    for e in (ours, want):
        e.process_operations(SMALL.programs["branch_length_optimization"])
    close(ours.get_branch_lengths(), want.get_branch_lengths(), rtol=1e-3)


def test_every_getter():
    tips, weights, lengths = alignment(SMALL, 50, seed=50)
    engine = engine_for(SMALL, tips, weights, lengths, "HKY", "weibull+2", 1.1)
    oracle = engine_for(SMALL, tips, weights, lengths, "HKY", "weibull+2", 1.1, factory=gp.GPEngineOracle)
    want = check_against_reference(engine, SMALL, tips, weights, lengths, "HKY", "weibull+2", 1.1, edges=2)
    site_count = int(weights.sum())
    close(engine.get_per_gpcsp_components_of_full_log_marginal(), want.per_gpcsp_components_of_full_log_marginal(site_count))
    close(engine.get_log_likelihood_matrix(), want.log_likelihood_matrix())
    close(engine.get_per_gpcsp_log_likelihoods(3, 5), want.per_gpcsp_log_likelihoods()[3:8])
    assert np.array_equal(engine.get_branch_lengths(), lengths)
    close(engine.get_sbn_parameters(), SMALL.q, rtol=0)
    assert np.array_equal(engine.get_rescaling_counts(), oracle.rescaling_counts)
    for index in range(SMALL.plv_count):
        close(engine.get_plv(index) + 1e-300, oracle.plvs[index] + 1e-300)
