"""The subsplit-DAG generator (tests/gp_dag.py) and the exact GP reference (tests/gp_reference.py),
pinned without a GPU: the reference's derivative against 50-digit central differences, the numpy
oracle running the generated programs against the reference (which pins the generator and the
per-GPCSP normalisation), and the generator's invariants."""
import math

import mpmath
import numpy as np
import pytest

import gp_dag
import gp_reference
from oracle import gp

GTR = [0.10, 0.24, 0.07, 0.15, 0.33, 0.11, 0.15, 0.35, 0.3, 0.2]  # (the engine asks rates summing to 1)
HKY = [0.35, 0.15, 0.2, 0.3, 2.7]
MODELS = {"JC69": (), "GTR": GTR, "HKY": HKY}
SITES = [("constant", None), ("weibull+2", 0.4), ("weibull+4", 1.0), ("weibull+8", 2.5), ("gamma+4", 0.7)]


def case(dag, patterns, seed, gap_fraction=0.05):
    """(tips, weights, branch lengths): an alignment evolved down the DAG's first tree, with gaps."""
    rng = np.random.default_rng(seed)
    lengths = rng.uniform(0.02, 0.4, dag.gpcsp_count)
    tips = gp_dag.simulate_states(dag, dag.trees()[0], lengths, patterns, rng, gap_fraction)
    weights = rng.integers(1, 5, patterns).astype(np.float64)
    return tips, weights, lengths


def run_oracle(dag, tips, weights, lengths, substitution, params, site, shape, threshold=1e-40):
    engine = gp.GPEngineOracle(tips, weights, int(weights.sum()), dag.plv_count, dag.gpcsp_count,
                               rescaling_threshold=threshold, sbn_prior=dag.q)
    engine.set_substitution_model(substitution, params)
    if site != "constant":
        engine.set_site_model(site, [shape])
    engine.set_branch_lengths(lengths)
    engine.process_operations(dag.programs["populate_plvs"])
    engine.process_operations(dag.programs["compute_likelihoods"])
    return engine


def close(got, want, rtol=1e-9):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    assert np.all(np.abs(got - want) <= rtol * np.abs(want)), np.max(np.abs(got - want) / np.abs(want))


DAGS = {
    "hybrid6x5": lambda: gp_dag.hybrid_dag(6, 5, seed=3),
    "hybrid7x12": lambda: gp_dag.hybrid_dag(7, 12, seed=4),
    "hybrid9x30": lambda: gp_dag.hybrid_dag(9, 30, seed=5),
    "random100": lambda: gp_dag.one_tree_dag(100, "random", seed=6),
    "ladder100": lambda: gp_dag.one_tree_dag(100, "ladder", seed=7),
    "wide_root": lambda: gp_dag.wide_root_dag(10, 300, seed=8),
}


# every site model on the small DAGs, constant and weibull+4 on the large ones
CASES = [(d, m, site, shape) for d in DAGS for m in MODELS for site, shape in SITES
         if d.startswith("hybrid") or site in ("constant", "weibull+4")]


@pytest.mark.parametrize("dag_name,substitution,site,shape", CASES)
def test_oracle_on_generated_programs_is_the_exact_marginal(dag_name, substitution, site, shape):
    """The oracle's marginal, per-GPCSP values, LogLikelihoodAndDerivative and SBN update, running the
    generated programs, against the sum over every tree the DAG holds."""
    dag = DAGS[dag_name]()
    tips, weights, lengths = case(dag, 12, seed=len(dag_name) + len(site))
    params = MODELS[substitution]
    want = gp_reference.Reference(dag, gp_reference.Model(substitution, params, site, shape), tips, weights, lengths)
    engine = run_oracle(dag, tips, weights, lengths, substitution, params, site, shape, threshold=1e-8)
    close(engine.get_log_marginal_likelihood(), want.log_marginal_likelihood())
    close(engine.get_per_gpcsp_log_likelihoods(), want.per_gpcsp_log_likelihoods())
    rng = np.random.default_rng(0)
    for g in rng.choice(np.arange(dag.rootsplit_count, dag.gpcsp_count), size=4, replace=False):
        value, slope, scale = want.derivative(g)
        got = engine.log_likelihood_and_derivative(*dag.edge_plvs(g), g)
        close(got[0], value)
        assert abs(got[1] - slope) <= 1e-8 * scale
    engine.process_operations(dag.programs["optimize_sbn_parameters"])
    close(engine.get_sbn_parameters(), want.updated_sbn_parameters())


def _mp_per_gpcsp(dag, model_args, tips, weights, lengths, g, t):
    """The per-GPCSP value of g at length t in mpmath (50 digits): every tree holding g pruned with
    mpmath.expm, no rescaling."""
    substitution, params, site, shape = model_args
    q_matrix, freqs = gp_reference.rate_matrix(substitution, params)
    Q = mpmath.matrix([[mpmath.mpf(float(x.real)) for x in row] for row in q_matrix])
    pi = [mpmath.mpf(float(x.real)) for x in freqs]
    rates, proportions = gp_reference.subst_reference.site_rates(site, shape)
    lengths = np.array(lengths, dtype=object)
    lengths[g] = t
    per_pattern = [mpmath.mpf(0)] * tips.shape[1]
    for tree in dag.trees():
        if g not in tree:
            continue
        parent_ids, _, child_of = dag.tree_shape(tree, np.zeros(dag.gpcsp_count))
        length_of = {child_of[e]: lengths[e] for e in child_of}
        prior = mpmath.fprod([mpmath.mpf(float(dag.q[e])) for e in tree])
        nodes = len(parent_ids) + 1
        for k in range(tips.shape[1]):
            site_likelihood = mpmath.mpf(0)
            for rate, proportion in zip(rates, proportions):
                partial = {}
                for leaf in range(dag.taxon_count):
                    s = int(tips[leaf, k])
                    partial[leaf] = [mpmath.mpf(1 if s >= 4 or s == i else 0) for i in range(4)]
                for node in range(dag.taxon_count, nodes):
                    vector = [mpmath.mpf(1)] * 4
                    for child in [c for c in range(nodes - 1) if parent_ids[c] == node]:
                        P = mpmath.expm(Q * (mpmath.mpf(float(rate)) * length_of[child]))
                        vector = [vector[i] * mpmath.fsum(P[i, j] * partial[child][j] for j in range(4)) for i in range(4)]
                    partial[node] = vector
                site_likelihood += mpmath.mpf(float(proportion)) * mpmath.fsum(pi[i] * partial[nodes - 1][i] for i in range(4))
            per_pattern[k] += prior * site_likelihood
    return mpmath.fsum(mpmath.mpf(float(w)) * mpmath.log(x / mpmath.mpf(float(dag.q[g])))
                       for w, x in zip(weights, per_pattern))


@pytest.mark.parametrize("substitution,site,shape", [("JC69", "constant", None), ("HKY", "weibull+2", 0.5),
                                                     ("GTR", "gamma+2", 1.5)])
def test_reference_derivative_against_50_digit_central_differences(substitution, site, shape):
    dag = gp_dag.hybrid_dag(4, 3, seed=11)
    tips, weights, lengths = case(dag, 3, seed=12)
    model_args = (substitution, MODELS[substitution], site, shape)
    want = gp_reference.Reference(dag, gp_reference.Model(*model_args), tips, weights, lengths)
    mpmath.mp.dps = 50
    try:
        for g in range(dag.rootsplit_count, dag.gpcsp_count):
            value, slope, _ = want.derivative(g)
            t, h = mpmath.mpf(float(lengths[g])), mpmath.mpf(10) ** -20
            assert abs(value - float(_mp_per_gpcsp(dag, model_args, tips, weights, lengths, g, t))) <= 1e-12 * abs(value)
            central = (_mp_per_gpcsp(dag, model_args, tips, weights, lengths, g, t + h) -
                       _mp_per_gpcsp(dag, model_args, tips, weights, lengths, g, t - h)) / (2 * h)
            assert abs(slope - float(central)) <= 1e-12 * max(abs(float(central)), 1.0)
    finally:
        mpmath.mp.dps = 15


@pytest.mark.parametrize("dag_name", list(DAGS))
def test_generator_invariants(dag_name):
    """Groups contiguous and q normalised within each; rootsplits first; children before parents; the
    DAG's tree count is the enumeration's; every program passes the device's scheduler."""
    from libsbn_b200.gp_engine import schedule_program
    dag = DAGS[dag_name]()
    bounds = [g for group in dag.groups for g in group]
    assert bounds[0] == 0 and bounds[-1] == dag.gpcsp_count and bounds == sorted(bounds)
    assert dag.groups[0] == (0, dag.rootsplit_count)
    for start, stop in dag.groups:
        assert stop > start and abs(dag.q[start:stop].sum() - 1.0) < 1e-12
        parents = {dag.edges[g][:2] for g in range(start, stop)}
        assert len(parents) == 1
    for v, side, child in dag.edges:
        assert v is None or child < v
    assert dag.plv_count == 6 * dag.node_count
    assert dag.tree_count() == len(dag.trees()) == len(set(dag.trees()))
    for name, program in dag.programs.items():
        assert schedule_program(dag.plv_count, dag.gpcsp_count, program).size <= program.size, name


def test_small_dags_hold_hybrids_and_the_wide_root_does_not():
    assert gp_dag.hybrid_dag(7, 12, seed=4).tree_count() > 12
    wide = gp_dag.wide_root_dag(10, 300, seed=8)
    assert wide.tree_count() == 300 and wide.groups[0] == (0, 300)
    assert gp_dag.one_tree_dag(400, "random", seed=9).gpcsp_count > 753  # C = 1 matrices leave shared memory
    assert gp_dag.one_tree_dag(1000, "ladder", seed=10).plv_count > 11000


@pytest.mark.parametrize("dag_name", ["hybrid7x12", "wide_root"])
def test_scheduled_generated_programs_compute_the_same_bits(dag_name):
    from libsbn_b200.gp_engine import schedule_program
    dag = DAGS[dag_name]()
    tips, weights, lengths = case(dag, 6, seed=1)
    engines = [run_oracle(dag, tips, weights, lengths, "GTR", GTR, "weibull+2", 0.8) for _ in range(2)]
    for name in ("populate_plvs", "compute_likelihoods", "branch_length_optimization", "populate_plvs",
                 "compute_likelihoods", "optimize_sbn_parameters"):
        program = dag.programs[name]
        engines[0].process_operations(program)
        engines[1].process_operations(schedule_program(dag.plv_count, dag.gpcsp_count, program))
        assert np.array_equal(engines[0].plvs, engines[1].plvs)
        assert np.array_equal(engines[0].branch_lengths, engines[1].branch_lengths)
        assert np.array_equal(engines[0].q, engines[1].q)
        assert np.array_equal(engines[0].rescaling_counts, engines[1].rescaling_counts)
        assert np.array_equal(engines[0].log_likelihoods, engines[1].log_likelihoods, equal_nan=True)


def test_schedule_marks_exactly_the_rootward_sources():
    """The device learns a source's direction from bit 16 (+ u) of the scheduled record's word 0: set
    exactly for increments out of r-hat / r / r-tilde PLVs, never for leafward ones."""
    from libsbn_b200.gp_engine import schedule_program
    dag = DAGS["hybrid7x12"]()
    words = [int(w) for w in schedule_program(dag.plv_count, dag.gpcsp_count, dag.programs["populate_plvs"])]
    pc, seen = 0, 0
    while pc < len(words):
        kind = words[pc] & 0xff
        size = {0: 2, 1: 3, 2: 4, 3: 4, 4: 4, 5: 4, 6: 3, 7: 1, 8: 4}.get(kind)
        if kind == 9:
            size = 3 + words[pc + 2]
        elif kind == 10:
            size = 3 + 2 * words[pc + 2]
        sources = [words[pc + 3]] if kind == 2 else words[pc + 4:pc + size:2] if kind == 10 else []
        for u, src in enumerate(sources):
            assert bool(words[pc] & (1 << (16 + u))) == (src >= gp_dag.RHAT * dag.node_count), (pc, src)
            seen += src >= gp_dag.RHAT * dag.node_count
        pc += size
    assert seen > 0


def test_rootward_plvs_evolve_by_the_transposed_matrix():
    """With unequal frequencies P(t) is not symmetric: a rootward PLV (one carrying the stationary
    distribution) evolves as P(t)^T r.  Evolving it by P(t) leaves the marginal right (it only uses
    leafward PLVs) but every per-GPCSP value below the rootsplits wrong by percents."""
    dag = gp_dag.hybrid_dag(6, 5, seed=3)
    tips, weights, lengths = case(dag, 30, seed=1)
    want = gp_reference.Reference(dag, gp_reference.Model("GTR", GTR), tips, weights, lengths, derivatives=False)
    engine = run_oracle(dag, tips, weights, lengths, "GTR", GTR, "constant", None)
    close(engine.get_per_gpcsp_log_likelihoods(), want.per_gpcsp_log_likelihoods())
    assert engine.rootward[dag.plv(gp_dag.RHAT, 0)] and not engine.rootward[dag.plv(gp_dag.P_PLV, dag.node_count - 1)]
