"""17 to 32 rate categories on the fused tree walk, where every category of a site pattern
has its own lane of a warp (counts above 16 run padded to 32 lanes): the CUDA path against
the CPU oracle, against itself across the engine's modes (CUDA-graph replay, device groups,
staged runs finished on the host, the analytic and finite-difference substitution gradients),
and against the BEAGLE-compatible device library, which shares no kernel with the walk.

Tolerances as in test_engine_gpu.py: logL 1e-10 relative, gradients 1e-8 relative to the
largest entry of the tree.
"""
import numpy as np
import pytest

from conftest import load_fixture
import libsbn_b200 as sbn
from libsbn_b200 import _capi, sharding, trees

pytestmark = pytest.mark.gpu

LOGL_RTOL = 1e-10
GRAD_RTOL = 1e-8
SITES = ["weibull+17", "weibull+20", "weibull+24", "weibull+32", "gamma+20"]
SUBSTITUTIONS = ["JC69", "GTR", "HKY"]
GTR_ROW = [0.05, 0.1, 0.15, 0.20, 0.25, 0.25, 0.1, 0.2, 0.3, 0.4]


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def grad_rel(a, b):
    a, b = np.atleast_2d(a), np.atleast_2d(b)
    return np.max(np.max(np.abs(a - b), axis=1) / np.maximum(np.max(np.abs(b), axis=1), 1e-300))


def stack(gradients, key):
    return np.array([g.gradient[key] for g in gradients])


def fd_noise(log_likelihoods):
    """Noise floor of central differences with delta 1e-6 on logL values that carry
    ~1e-12 relative rounding (see tests/test_oracle.py)."""
    return np.abs(log_likelihoods).max() * 1e-12 / 1e-6


def model_rows(substitution, site, tree_count, rng, clock=False):
    """A random model per tree: the engine's parameter rows, the oracle's rows (HKY handed to
    the oracle as GTR with kappa on the transitions) and the oracle's substitution model."""
    rows, oracle_rows = [], []
    for _ in range(tree_count):
        freqs = rng.dirichlet(np.ones(4) * 4)
        if substitution == "GTR":
            sub = list(rng.dirichlet(np.ones(6) * 2)) + list(freqs)
            oracle_sub = sub
        elif substitution == "HKY":
            kappa = rng.uniform(0.5, 4)
            sub = list(freqs) + [kappa]
            raw = np.array([1, kappa, 1, 1, kappa, 1.0])
            oracle_sub = list(raw / raw.sum()) + list(freqs)
        else:
            sub, oracle_sub = [], []
        tail = [rng.uniform(0.3, 2)] + ([0.0] if clock else [])  # (the clock rate rides in the tree batch)
        rows.append(sub + tail)
        oracle_rows.append(oracle_sub + tail)
    return np.array(rows), np.array(oracle_rows), "JC69" if substitution == "JC69" else "GTR"


def synthetic(taxa, patterns, seed, gap_fraction=0.03):
    states, _ = trees.random_alignment(taxa, patterns, seed, gap_fraction=gap_fraction)
    weights = np.random.default_rng(seed).integers(1, 4, size=patterns).astype(np.float64)
    return states, weights


@pytest.mark.parametrize("site", SITES)
@pytest.mark.parametrize("substitution", SUBSTITUTIONS)
@pytest.mark.parametrize("rescaling", [False, True], ids=["plain", "rescaled"])
def test_unrooted_against_oracle(oracle, substitution, site, rescaling):
    taxa, patterns, tree_count = 21, 509, 3  # (509: the last 16-pattern tile is ragged)
    seed = len(site) * 100 + SUBSTITUTIONS.index(substitution)
    states, weights = synthetic(taxa, patterns, seed)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed)
    rng = np.random.default_rng(seed)
    params, oracle_params, oracle_sub = model_rows(substitution, site, tree_count, rng)
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "none"), states, weights)
    assert engine.category_count == int(site.split("+")[1])
    batch = sbn.TreeBatch(parent_ids, lengths)
    got = engine.log_likelihoods(batch, params, rescaling)
    want = oracle.gradients(oracle_sub, site, states, weights, parent_ids, lengths, oracle_params,
                            rescaling=rescaling)
    assert rel(got, want["log_likelihood"]) < LOGL_RTOL
    grads = engine.gradients(batch, params, rescaling, substitution_gradient=False)
    assert rel([g.log_likelihood for g in grads], want["log_likelihood"]) < LOGL_RTOL
    assert grad_rel(stack(grads, "branch_lengths"), want["branch"]) < GRAD_RTOL
    assert grad_rel(stack(grads, "site_model").T, want["site_model"][None, :]) < GRAD_RTOL


@pytest.mark.parametrize("site", SITES)
@pytest.mark.parametrize("substitution", SUBSTITUTIONS)
@pytest.mark.parametrize("rescaling", [False, True], ids=["plain", "rescaled"])
def test_rooted_against_oracle(oracle, substitution, site, rescaling):
    """Time trees (the influenza fixture's topology, heights and strict clock): log likelihoods
    with the log-det Jacobian, height-ratio, clock and site-model gradients."""
    fx = load_fixture("flua_jc69_strict")
    rng = np.random.default_rng(len(site) * 10 + SUBSTITUTIONS.index(substitution))
    params, oracle_params, oracle_sub = model_rows(substitution, site, 1, rng, clock=True)
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "strict"), fx["patterns"], fx["weights"])
    batch = sbn.TreeBatch(fx["parent_ids"], fx["branch_lengths"], fx["rates"], fx["node_heights"],
                          fx["node_bounds"], fx["height_ratios"], 1)
    args = (oracle_sub, site, fx["patterns"], fx["weights"], fx["parent_ids"], fx["branch_lengths"], oracle_params)
    kwargs = dict(rooted=True, rescaling=rescaling, rates=fx["rates"], node_heights=fx["node_heights"],
                  node_bounds=fx["node_bounds"])
    got = engine.log_likelihoods(batch, params, rescaling, rooted=True)
    assert rel(got, oracle.log_likelihoods(*args, **kwargs)) < LOGL_RTOL
    grads = engine.gradients(batch, params, rescaling, rooted=True, substitution_gradient=False)
    want = oracle.gradients(*args, height_ratios=fx["height_ratios"], **kwargs)
    assert rel([g.log_likelihood for g in grads], want["log_likelihood"]) < LOGL_RTOL
    for key in ("ratios_root_height", "clock_model"):
        assert grad_rel(stack(grads, key), want[key]) < GRAD_RTOL, key
    assert rel(stack(grads, "site_model")[:, 0], want["site_model"]) < GRAD_RTOL


@pytest.mark.parametrize("shape", ["ladder", "random"])
def test_thousand_taxa_at_32_categories_need_rescaling(oracle, shape):
    """Per-site likelihoods of 1000 taxa underflow fp64; the rescaling takes the maximum over
    all 32 lanes of a pattern."""
    taxa, patterns = 1000, 96
    states, weights = trees.random_alignment(taxa, patterns, 11, gap_fraction=0.01)
    rng = np.random.default_rng(13)
    if shape == "ladder":
        parent_ids = trees.ladder_topology(taxa)[None, :]
    else:
        parent_ids = trees.random_unrooted_topology(taxa, rng)[None, :]
    lengths = np.maximum(rng.exponential(0.1, size=(1, 2 * taxa - 2)), 1e-6)
    engine = sbn.Engine(sbn.PhyloModelSpecification("HKY", "weibull+32", "none"), states, weights)
    params = np.array([[0.1, 0.2, 0.3, 0.4, 2.0, 0.5]])
    raw = np.array([1, 2, 1, 1, 2, 1.0])
    oracle_params = np.array([list(raw / raw.sum()) + [0.1, 0.2, 0.3, 0.4, 0.5]])
    batch = sbn.TreeBatch(parent_ids, lengths)
    assert not np.isfinite(engine.log_likelihoods(batch, params, False)[0])
    grads = engine.gradients(batch, params, True, substitution_gradient=False)
    want = oracle.gradients("GTR", "weibull+32", states, weights, parent_ids, lengths, oracle_params, rescaling=True)
    assert np.isfinite(grads[0].log_likelihood)
    assert rel(grads[0].log_likelihood, want["log_likelihood"][0]) < LOGL_RTOL
    assert grad_rel(grads[0].gradient["branch_lengths"], want["branch"][0]) < GRAD_RTOL
    assert rel(grads[0].gradient["site_model"], want["site_model"]) < GRAD_RTOL


@pytest.mark.parametrize("substitution,site", [("GTR", "weibull+20"), ("HKY", "gamma+20"), ("GTR", "weibull+32")])
@pytest.mark.parametrize("rescaling", [False, True], ids=["plain", "rescaled"])
def test_analytic_substitution_gradient(oracle, substitution, site, rescaling):
    """The exact substitution gradient accumulated in the gradient sweep against the reference's
    16 central-difference sweeps, run by the same engine (their extra logL walks at 32 lanes) and
    by the oracle."""
    fx = load_fixture("ds1_gtr_weibull4")
    rng = np.random.default_rng(5)
    tree_count = fx["parent_ids"].shape[0]
    params, oracle_params, oracle_sub = model_rows(substitution, site, tree_count, rng)
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "none"), fx["patterns"], fx["weights"])
    batch = sbn.TreeBatch(fx["parent_ids"], fx["branch_lengths"])
    engine.set_substitution_gradient("fd")
    by_differences = engine.gradients(batch, params, rescaling)
    engine.set_substitution_gradient("analytic")
    analytic = engine.gradients(batch, params, rescaling)
    logl = np.array([g.log_likelihood for g in analytic])
    assert np.array_equal(logl, [g.log_likelihood for g in by_differences])
    assert np.array_equal(stack(analytic, "branch_lengths"), stack(by_differences, "branch_lengths"))
    a, d = stack(analytic, "substitution_model"), stack(by_differences, "substitution_model")
    assert a.shape == (tree_count, 8 if substitution == "GTR" else 4)
    assert np.max(np.abs(a - d)) < 2 * fd_noise(logl)
    want = oracle.gradients(oracle_sub, site, fx["patterns"], fx["weights"], fx["parent_ids"], fx["branch_lengths"],
                            oracle_params, rescaling=rescaling)
    assert rel(logl, want["log_likelihood"]) < LOGL_RTOL
    assert grad_rel(stack(analytic, "branch_lengths"), want["branch"]) < GRAD_RTOL
    if substitution == "GTR":  # (the oracle's HKY is a GTR: other coordinates)
        assert np.max(np.abs(a - want["substitution_model"])) < 2 * fd_noise(logl)


@pytest.mark.parametrize("site", ["weibull+20", "weibull+32"])
def test_graph_replay_is_bitwise_the_eager_call(site):
    """Repeated calls on an unchanged topology set replay the launch sequence as a CUDA graph
    (no timed walk launch); a replay with the inputs of an eager call returns the same bits."""
    fx = load_fixture("ds1_gtr_weibull4")
    params = fx["params"].copy()
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", site, "none"), fx["patterns"], fx["weights"])
    batch = sbn.TreeBatch(fx["parent_ids"], fx["branch_lengths"])
    eager = engine.gradients(batch, params, True)
    rng = np.random.default_rng(9)
    for _ in range(2):
        other = sbn.TreeBatch(fx["parent_ids"], fx["branch_lengths"] * rng.uniform(0.5, 1.5, fx["branch_lengths"].shape))
        engine.gradients(other, params, True)
    _, walks_before = engine.walk_timing()
    replayed = engine.gradients(batch, params, True)
    _, walks_after = engine.walk_timing()
    assert walks_after == walks_before  # the graph's walk launch is not one of the timed ones
    assert [g.log_likelihood for g in replayed] == [g.log_likelihood for g in eager]
    for key in eager[0].gradient:
        assert np.array_equal(stack(replayed, key), stack(eager, key)), key


@pytest.mark.parametrize("axis", ["trees", "patterns"])
def test_device_group_is_the_single_engine(axis):
    """A group with a repeated ordinal: tree slices are the single-device result bit for bit;
    pattern ranges add up to it up to the order of the additions."""
    fx = load_fixture("ds1_gtr_weibull4")
    spec = sbn.PhyloModelSpecification("GTR", "weibull+24", "none")
    params = fx["params"].copy()
    batch = sbn.TreeBatch(fx["parent_ids"], fx["branch_lengths"])
    single = sbn.Engine(spec, fx["patterns"], fx["weights"], 0)
    group = sbn.Engine(spec, fx["patterns"], fx["weights"], devices=[0, 0], shard_axis=axis)
    want = single.gradients(batch, params, True)
    got = group.gradients(batch, params, True)
    exact = axis == "trees"
    for g, w in zip(got, want):
        assert g.log_likelihood == w.log_likelihood if exact else rel(g.log_likelihood, w.log_likelihood) < 1e-12
        for key in w.gradient:
            a, b = np.asarray(g.gradient[key]), np.asarray(w.gradient[key])
            tol = 0.0 if exact else (1e-4 if key == "substitution_model" else 1e-11)
            assert np.max(np.abs(a - b)) <= tol * np.max(np.abs(b)), key


@pytest.mark.parametrize("analytic", [False, True], ids=["fd", "analytic"])
def test_staged_pattern_ranges_finished_on_the_host(analytic):
    """stage / run / fetch over pattern ranges (set_pattern_range), the raw sums added as ranks
    would all-reduce them, and sbnb_finish_gradients* on the host: the one-call result."""
    taxa, patterns, tree_count, world = 14, 3000, 4, 3
    states, weights = synthetic(taxa, patterns, 3)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=4)
    params = np.tile(np.array(GTR_ROW + [0.7]), (tree_count, 1))
    spec = sbn.PhyloModelSpecification("GTR", "gamma+20", "none")
    engine = sbn.Engine(spec, states, weights, 0)
    batch = sbn.TreeBatch(parent_ids, lengths)
    engine.set_substitution_gradient("analytic" if analytic else "fd")
    want = engine.gradients(batch, params, rescaling=True)
    total = None
    for rank in range(world):
        engine.set_pattern_range(*sharding.pattern_range(rank, world, patterns))
        staged = engine.stage(batch, params, substitution_fd=not analytic, substitution_analytic=analytic)
        staged.run(_capi.MODE_BRANCH_GRADIENT, True)
        parts = list(staged.fetch(gradients=True)) + ([staged.fetch_substitution_sums()] if analytic else [])
        staged.close()
        total = parts if total is None else [t + p for t, p in zip(total, parts)]
    engine.set_pattern_range(0, patterns)
    if analytic:
        got = sharding.finish_gradients_analytic(spec, taxa, batch, False, params, *total, engine.category_count)
    else:
        got = sharding.finish_gradients(spec, taxa, batch, False, True, *total, engine.category_count)
    np.testing.assert_allclose([g.log_likelihood for g in got], [g.log_likelihood for g in want], rtol=1e-12)
    for key in ("branch_lengths", "site_model"):
        a, b = stack(got, key), stack(want, key)
        assert np.max(np.abs(a - b)) <= 1e-10 * np.max(np.abs(b)), key
    a, b = stack(got, "substitution_model"), stack(want, "substitution_model")
    tol = 1e-10 * np.max(np.abs(b)) if analytic else fd_noise(total[0])
    assert np.max(np.abs(a - b)) <= tol


@pytest.mark.parametrize("categories", [20, 32])
def test_the_fused_walk_and_the_beagle_compatible_library_agree(categories):
    """Two device implementations that share no kernel, on one 100-taxon tree x 20k patterns:
    the fused walk behind the C ABI and BEAGLE's op-at-a-time schedule through
    libhmsbeagle_b200.so driven by FatBeagle's call sequence (fat_beagle.cpp:119-175).  (The
    unrooted gradient of a bifurcating tree slides the root, tree.cpp:72-78: the first root child
    carries the derivative of the merged edge.)"""
    from libsbn_b200 import beagle
    taxa, patterns, shape = 100, 20000, 0.5
    N = 2 * taxa - 1
    rng = np.random.default_rng(20261020 + categories)
    states = rng.integers(0, 4, size=(taxa, patterns), dtype=np.uint8)
    states[rng.random(states.shape) < 0.01] = 4
    weights = rng.integers(1, 4, size=patterns).astype(np.float64)
    post, pre = beagle.random_tree_operations(taxa, rng, True)
    parent_ids = np.full(N - 1, -1, dtype=np.int32)
    for op in post:
        parent_ids[op[3]] = parent_ids[op[5]] = op[0]
    lengths = np.maximum(rng.exponential(0.1, size=N), 1e-6)
    lengths[N - 1] = 0.0
    evec, ivec, evals, freqs, q = beagle.gtr_eigensystem()
    quantiles = (2.0 * np.arange(categories) + 1.0) / (2.0 * categories)
    rates = (-np.log(1.0 - quantiles)) ** (1.0 / shape)  # site_model.cpp:37-62
    rates /= rates.mean()
    library = beagle.Beagle(None, taxa, patterns, categories, True)
    library.set_tips(states.astype(np.int32), weights, True)
    library.set_model(evec, ivec, evals, freqs, rates, np.full(categories, 1.0 / categories))
    logl, sums, _, _ = library.log_likelihood_and_gradient(post, pre, lengths, q, rates, freqs, True, per_site=False)
    library.close()
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", f"weibull+{categories}", "none"), states, weights)
    params = np.array([GTR_ROW + [shape]])
    walk = engine.gradients(sbn.TreeBatch(parent_ids[None, :], lengths[None, :]), params, True,
                            substitution_gradient=False)[0]
    assert abs(walk.log_likelihood - logl) <= 1e-10 * abs(logl)
    gradient = walk.gradient["branch_lengths"]
    root_children = [int(post[-1][3]), int(post[-1][5])]
    others = np.array([e for e in range(N - 1) if e not in root_children])
    scale = np.max(np.abs(sums))
    assert np.max(np.abs(gradient[others] - sums[others])) <= 1e-8 * scale
    slid = gradient[root_children]
    carried = slid[np.argmax(np.abs(slid))]
    assert np.min(np.abs(slid)) == 0.0
    assert abs(carried - sums[root_children[0]]) <= 1e-8 * scale
    assert abs(carried - sums[root_children[1]]) <= 1e-8 * scale


def test_parameter_blocks_at_32_categories():
    """One shape parameter whatever the count; the engine reports the count it was given."""
    states, weights = synthetic(5, 40, 1)
    for substitution, site, clock, key, start, count in [("GTR", "weibull+32", "none", "Weibull shape", 10, 11),
                                                          ("HKY", "gamma+32", "strict", "Gamma shape", 5, 7),
                                                          ("JC69", "weibull+20", "none", "Weibull shape", 0, 1)]:
        engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, clock), states, weights)
        assert engine.category_count == int(site.split("+")[1]) and engine.param_count == count
        assert engine.param_block(key) == (start, 1) and engine.param_block("entire site") == (start, 1)


@pytest.mark.parametrize("site", ["weibull+33", "gamma+33", "weibull+64"])
def test_more_than_32_categories_are_refused(site):
    fx = load_fixture("hello_jc69")
    with pytest.raises(RuntimeError, match=r"\[1,32\].*libhmsbeagle_b200\.so"):
        sbn.Engine(sbn.PhyloModelSpecification("JC69", site, "none"), fx["patterns"], fx["weights"])
