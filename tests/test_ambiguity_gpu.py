"""Ambiguous nucleotides as partial tip states on the device: the fused tree walk over an
alignment of nucleotide masks against itself (masks without ambiguity are the state walk,
bit for bit), against the CPU oracle by linearity (tests/ambiguity_oracle.py), across the
engine's modes, and against the BEAGLE-compatible library driven by tip partials; the masked
site-pattern compression; and the GP engine's mask leaves.

Tolerances as in test_engine_gpu.py: logL 1e-10 relative, gradients 1e-8 relative to the
largest entry of the tree.
"""
import numpy as np
import pytest

import ambiguity_oracle
import gp_cases
from conftest import load_fixture
import libsbn_b200 as sbn
from libsbn_b200 import _capi, alignment, sharding, trees
from oracle import gp

pytestmark = pytest.mark.gpu

LOGL_RTOL = 1e-10
GRAD_RTOL = 1e-8
SUBSTITUTIONS = ["JC69", "GTR", "HKY"]
SITES = ["constant", "weibull+4", "gamma+8", "weibull+20"]
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
    """Noise floor of central differences with delta 1e-6 (see tests/test_oracle.py)."""
    return np.abs(log_likelihoods).max() * 1e-12 / 1e-6


def model_rows(substitution, site, tree_count, rng, clock=False):
    """Engine rows, oracle rows (HKY as a GTR with kappa on the transitions), oracle model."""
    rows, oracle_rows = [], []
    for _ in range(tree_count):
        freqs = rng.dirichlet(np.ones(4) * 4)
        if substitution == "GTR":
            sub = oracle_sub = list(rng.dirichlet(np.ones(6) * 2)) + list(freqs)
        elif substitution == "HKY":
            kappa = rng.uniform(0.5, 4)
            sub = list(freqs) + [kappa]
            raw = np.array([1, kappa, 1, 1, kappa, 1.0])
            oracle_sub = list(raw / raw.sum()) + list(freqs)
        else:
            sub, oracle_sub = [], []
        tail = ([] if site == "constant" else [rng.uniform(0.3, 2)]) + ([0.0] if clock else [])
        rows.append(sub + tail)
        oracle_rows.append(oracle_sub + tail)
    return np.array(rows), np.array(oracle_rows), "JC69" if substitution == "JC69" else "GTR"


def masked(taxa, patterns, seed, ambiguous_fraction=0.05):
    masks, _ = trees.random_masked_alignment(taxa, patterns, seed, ambiguous_fraction, gap_fraction=0.02)
    weights = np.random.default_rng(seed).integers(1, 4, size=patterns).astype(np.float64)
    return masks, weights


@pytest.mark.parametrize("site", ["constant", "weibull+4", "weibull+8", "weibull+32"])
@pytest.mark.parametrize("rescaling", [False, True], ids=["plain", "rescaled"])
def test_masks_without_ambiguity_are_the_states_bitwise(site, rescaling):
    """Single-state and missing masks run the state walk: every result block bit for bit."""
    taxa, patterns, tree_count = 17, 700, 3
    states, weights = trees.random_alignment(taxa, patterns, 5, gap_fraction=0.05)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, 6)
    spec = sbn.PhyloModelSpecification("GTR", site, "none")
    params = np.tile(np.array(GTR_ROW + ([] if site == "constant" else [0.6])), (tree_count, 1))
    batch = sbn.TreeBatch(parent_ids, lengths)
    by_states = sbn.Engine(spec, states, weights)
    by_masks = sbn.Engine(spec, trees.states_to_masks(states), weights, tip_encoding="masks")
    assert np.array_equal(by_masks.log_likelihoods(batch, params, rescaling),
                          by_states.log_likelihoods(batch, params, rescaling))
    for mode in ("analytic", "fd"):
        by_states.set_substitution_gradient(mode)
        by_masks.set_substitution_gradient(mode)
        want, got = by_states.gradients(batch, params, rescaling), by_masks.gradients(batch, params, rescaling)
        assert [g.log_likelihood for g in got] == [g.log_likelihood for g in want]
        for key in want[0].gradient:
            assert np.array_equal(stack(got, key), stack(want, key)), (mode, key)


@pytest.mark.parametrize("site", SITES)
@pytest.mark.parametrize("substitution", SUBSTITUTIONS)
@pytest.mark.parametrize("rescaling", [False, True], ids=["plain", "rescaled"])
def test_unrooted_against_oracle(oracle, substitution, site, rescaling):
    taxa, patterns, tree_count = 12, 181, 2
    seed = len(site) * 100 + SUBSTITUTIONS.index(substitution)
    masks, weights = masked(taxa, patterns, seed)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed)
    params, oracle_params, oracle_sub = model_rows(substitution, site, tree_count, np.random.default_rng(seed))
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "none"), masks, weights, tip_encoding="masks")
    batch = sbn.TreeBatch(parent_ids, lengths)
    want = ambiguity_oracle.gradients(oracle, oracle_sub, site, masks, weights, parent_ids, lengths, oracle_params,
                                      rescaling=rescaling)
    assert rel(engine.log_likelihoods(batch, params, rescaling), want["log_likelihood"]) < LOGL_RTOL
    grads = engine.gradients(batch, params, rescaling)
    logl = [g.log_likelihood for g in grads]
    assert rel(logl, want["log_likelihood"]) < LOGL_RTOL
    assert grad_rel(stack(grads, "branch_lengths"), want["branch"]) < GRAD_RTOL
    if site != "constant":
        assert grad_rel(stack(grads, "site_model").T, want["site_model"][None, :]) < GRAD_RTOL
    if substitution == "GTR":  # analytic against the oracle's central differences
        assert np.max(np.abs(stack(grads, "substitution_model") - want["substitution_model"])) < 4 * fd_noise(logl)


@pytest.mark.parametrize("site", ["weibull+4", "weibull+20"])
@pytest.mark.parametrize("substitution", SUBSTITUTIONS)
@pytest.mark.parametrize("rescaling", [False, True], ids=["plain", "rescaled"])
def test_rooted_against_oracle(oracle, substitution, site, rescaling):
    """Time trees with a strict clock (the influenza fixture's tree) over masked columns."""
    fx = load_fixture("flua_jc69_strict")
    taxa = fx["patterns"].shape[0]
    masks, weights = masked(taxa, 60, 17 + len(site), ambiguous_fraction=0.02)
    rng = np.random.default_rng(len(site) * 10 + SUBSTITUTIONS.index(substitution))
    params, oracle_params, oracle_sub = model_rows(substitution, site, 1, rng, clock=True)
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "strict"), masks, weights,
                        tip_encoding="masks")
    batch = sbn.TreeBatch(fx["parent_ids"], fx["branch_lengths"], fx["rates"], fx["node_heights"],
                          fx["node_bounds"], fx["height_ratios"], 1)
    want = ambiguity_oracle.gradients(oracle, oracle_sub, site, masks, weights, fx["parent_ids"], fx["branch_lengths"],
                                      oracle_params, rescaling=rescaling, rooted=True, rates=fx["rates"],
                                      node_heights=fx["node_heights"], node_bounds=fx["node_bounds"],
                                      height_ratios=fx["height_ratios"])
    kwargs = dict(rescaling=rescaling, rooted=True, rates=fx["rates"], node_heights=fx["node_heights"],
                  node_bounds=fx["node_bounds"])
    with_jacobian = ambiguity_oracle.log_likelihoods(oracle, oracle_sub, site, masks, weights, fx["parent_ids"],
                                                     fx["branch_lengths"], oracle_params, **kwargs)
    assert rel(engine.log_likelihoods(batch, params, rescaling, rooted=True), with_jacobian) < LOGL_RTOL
    grads = engine.gradients(batch, params, rescaling, rooted=True, substitution_gradient=False)
    assert rel([g.log_likelihood for g in grads], want["log_likelihood"]) < LOGL_RTOL
    for key in ("ratios_root_height", "clock_model"):
        assert grad_rel(stack(grads, key), want[key]) < GRAD_RTOL, key
    assert rel(stack(grads, "site_model")[:, 0], want["site_model"]) < GRAD_RTOL


@pytest.mark.parametrize("site", ["weibull+4", "weibull+32"])
def test_analytic_and_difference_substitution_gradients(oracle, site):
    taxa, patterns, tree_count = 10, 120, 2
    masks, weights = masked(taxa, patterns, 21, ambiguous_fraction=0.08)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, 22)
    params, oracle_params, _ = model_rows("GTR", site, tree_count, np.random.default_rng(23))
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", site, "none"), masks, weights, tip_encoding="masks")
    batch = sbn.TreeBatch(parent_ids, lengths)
    engine.set_substitution_gradient("fd")
    by_differences = engine.gradients(batch, params, True)
    engine.set_substitution_gradient("analytic")
    analytic = engine.gradients(batch, params, True)
    logl = np.array([g.log_likelihood for g in analytic])
    assert np.array_equal(logl, [g.log_likelihood for g in by_differences])
    a, d = stack(analytic, "substitution_model"), stack(by_differences, "substitution_model")
    assert np.max(np.abs(a - d)) < 2 * fd_noise(logl)
    want = ambiguity_oracle.gradients(oracle, "GTR", site, masks, weights, parent_ids, lengths, oracle_params,
                                      rescaling=True)
    assert np.max(np.abs(a - want["substitution_model"])) < 4 * fd_noise(logl)


def test_linearity_on_the_device():
    """One pattern: L with R at a tip = L with A + L with G, and the gradient identity."""
    taxa = 9
    parent_ids, lengths = trees.random_tree_batch(taxa, 4, seed=31)
    spec = sbn.PhyloModelSpecification("GTR", "weibull+4", "none")
    params = np.tile(np.array(GTR_ROW + [0.8]), (4, 1))
    batch = sbn.TreeBatch(parent_ids, lengths)
    column = np.array([[1], [2], [4], [8], [15], [2], [4], [1], [8]], dtype=np.uint8)
    results = {}
    for mask in (5, 1, 4):  # R, A, G at tip 3
        column[3, 0] = mask
        results[mask] = sbn.Engine(spec, column, np.ones(1), tip_encoding="masks").gradients(batch, params, True)
    l = {m: np.exp([g.log_likelihood for g in r]) for m, r in results.items()}
    assert rel(l[5], l[1] + l[4]) < 1e-12
    for key in ("branch_lengths", "site_model", "substitution_model"):
        g = {m: stack(r, key) for m, r in results.items()}
        identity = (l[1][:, None] * g[1] + l[4][:, None] * g[4]) / (l[1] + l[4])[:, None]
        assert grad_rel(g[5], identity) < 1e-10, key


def test_thousand_taxa_need_rescaling(oracle):
    """1000 taxa, ambiguity at a few taxa (so that the oracle's expansion stays small)."""
    taxa, patterns = 1000, 64
    states, weights = trees.random_alignment(taxa, patterns, 11, gap_fraction=0.01)
    masks = trees.states_to_masks(states)
    rng = np.random.default_rng(12)
    masks[:3][rng.random((3, patterns)) < 0.5] = 5  # R
    masks[10][rng.random(patterns) < 0.5] = 14  # B
    parent_ids = trees.random_unrooted_topology(taxa, rng)[None, :]
    lengths = np.maximum(rng.exponential(0.1, size=(1, 2 * taxa - 2)), 1e-6)
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+4", "none"), masks, weights, tip_encoding="masks")
    params = np.array([GTR_ROW + [0.5]])
    batch = sbn.TreeBatch(parent_ids, lengths)
    assert not np.isfinite(engine.log_likelihoods(batch, params, False)[0])
    grads = engine.gradients(batch, params, True, substitution_gradient=False)
    want = ambiguity_oracle.gradients(oracle, "GTR", "weibull+4", masks, weights, parent_ids, lengths, params,
                                      rescaling=True)
    assert rel(grads[0].log_likelihood, want["log_likelihood"][0]) < LOGL_RTOL
    assert grad_rel(grads[0].gradient["branch_lengths"], want["branch"][0]) < GRAD_RTOL
    assert rel(grads[0].gradient["site_model"], want["site_model"]) < GRAD_RTOL


@pytest.mark.parametrize("site", ["weibull+4", "weibull+32"])
def test_graph_replay_is_bitwise_the_eager_call(site):
    masks, weights = masked(20, 900, 41)
    parent_ids, lengths = trees.random_tree_batch(20, 6, 42)
    params = np.tile(np.array(GTR_ROW + [0.7]), (6, 1))
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", site, "none"), masks, weights, tip_encoding="masks")
    batch = sbn.TreeBatch(parent_ids, lengths)
    eager = engine.gradients(batch, params, True)
    rng = np.random.default_rng(9)
    for _ in range(2):
        engine.gradients(sbn.TreeBatch(parent_ids, lengths * rng.uniform(0.5, 1.5, lengths.shape)), params, True)
    _, walks_before = engine.walk_timing()
    replayed = engine.gradients(batch, params, True)
    _, walks_after = engine.walk_timing()
    assert walks_after == walks_before
    assert [g.log_likelihood for g in replayed] == [g.log_likelihood for g in eager]
    for key in eager[0].gradient:
        assert np.array_equal(stack(replayed, key), stack(eager, key)), key


@pytest.mark.parametrize("axis", ["trees", "patterns"])
def test_device_group_is_the_single_engine(axis):
    masks, weights = masked(15, 1200, 51)
    parent_ids, lengths = trees.random_tree_batch(15, 5, 52)
    params = np.tile(np.array(GTR_ROW + [0.7]), (5, 1))
    spec = sbn.PhyloModelSpecification("GTR", "weibull+8", "none")
    batch = sbn.TreeBatch(parent_ids, lengths)
    want = sbn.Engine(spec, masks, weights, 0, tip_encoding="masks").gradients(batch, params, True)
    got = sbn.Engine(spec, masks, weights, devices=[0, 0], shard_axis=axis, tip_encoding="masks").gradients(
        batch, params, True)
    exact = axis == "trees"
    for g, w in zip(got, want):
        assert g.log_likelihood == w.log_likelihood if exact else rel(g.log_likelihood, w.log_likelihood) < 1e-12
        for key in w.gradient:
            a, b = np.asarray(g.gradient[key]), np.asarray(w.gradient[key])
            tol = 0.0 if exact else (1e-4 if key == "substitution_model" else 1e-11)
            assert np.max(np.abs(a - b)) <= tol * np.max(np.abs(b)), key


@pytest.mark.parametrize("analytic", [False, True], ids=["fd", "analytic"])
def test_staged_pattern_ranges_finished_on_the_host(analytic):
    """Ranges of a masked alignment (some without an ambiguous tip: the engine still runs the
    ambiguous walk) staged, run, summed as ranks would, and finished by sbnb_finish_gradients*."""
    taxa, patterns, tree_count, world = 14, 3000, 4, 3
    masks, weights = masked(taxa, patterns, 3)
    masks[:, :1000] = trees.states_to_masks(trees.masks_to_states(masks[:, :1000]))
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=4)
    params = np.tile(np.array(GTR_ROW + [0.7]), (tree_count, 1))
    spec = sbn.PhyloModelSpecification("GTR", "gamma+8", "none")
    engine = sbn.Engine(spec, masks, weights, 0, tip_encoding="masks")
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


def test_pattern_sharded_engine_passes_the_encoding():
    masks, weights = masked(8, 200, 61)
    engine = sharding.PatternShardedEngine(sbn.PhyloModelSpecification("JC69", "constant", "none"), masks, weights,
                                           tip_encoding="masks")
    assert engine.engine.tip_encoding == "masks"
    parent_ids, lengths = trees.random_tree_batch(8, 2, 62)
    single = sbn.Engine(sbn.PhyloModelSpecification("JC69", "constant", "none"), masks, weights, tip_encoding="masks")
    batch = sbn.TreeBatch(parent_ids, lengths)
    assert np.array_equal(engine.log_likelihoods(batch), single.log_likelihoods(batch))


@pytest.mark.parametrize("taxa,patterns,categories,fraction", [(100, 100000, 4, 0.01), (1000, 2000, 32, 0.05)])
def test_the_fused_walk_and_the_beagle_compatible_library_agree(taxa, patterns, categories, fraction):
    """The walk over masks against libhmsbeagle_b200.so driven by tip partials (the bits of each
    mask), which shares no kernel with it.  (The unrooted gradient of a bifurcating tree slides
    the root: the first root child carries the derivative of the merged edge.)"""
    from libsbn_b200 import beagle
    shape = 0.5
    N = 2 * taxa - 1
    rng = np.random.default_rng(20261020 + taxa)
    masks, _ = trees.random_masked_alignment(taxa, patterns, 20261021 + taxa, fraction, gap_fraction=0.01)
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
    library = beagle.Beagle(None, taxa, patterns, categories, False)
    library.set_tips(masks, weights, False, masks=True)
    library.set_model(evec, ivec, evals, freqs, rates, np.full(categories, 1.0 / categories))
    logl, sums, _, _ = library.log_likelihood_and_gradient(post, pre, lengths, q, rates, freqs, True, per_site=False)
    library.close()
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", f"weibull+{categories}", "none"), masks, weights,
                        tip_encoding="masks")
    walk = engine.gradients(sbn.TreeBatch(parent_ids[None, :], lengths[None, :]), np.array([GTR_ROW + [shape]]), True,
                            substitution_gradient=False)[0]
    assert abs(walk.log_likelihood - logl) <= 1e-10 * abs(logl)
    gradient = walk.gradient["branch_lengths"]
    root_children = [int(post[-1][3]), int(post[-1][5])]
    others = np.array([e for e in range(N - 1) if e not in root_children])
    scale = np.max(np.abs(sums))
    assert np.max(np.abs(gradient[others] - sums[others])) <= 1e-8 * scale
    carried = gradient[root_children][np.argmax(np.abs(gradient[root_children]))]
    assert abs(carried - sums[root_children[0]]) <= 1e-8 * scale


@pytest.mark.parametrize("mask", [0, 16, 255])
def test_invalid_masks_are_refused(mask):
    masks, weights = masked(6, 50, 71)
    masks[4, 37] = mask
    spec = sbn.PhyloModelSpecification("JC69", "constant", "none")
    for make in (lambda: sbn.Engine(spec, masks, weights, tip_encoding="masks"),
                 lambda: sbn.Engine(spec, masks, weights, devices=[0, 0], tip_encoding="masks"),
                 lambda: sbn.GPEngine(masks, weights, 50, 6 * 11, 10, tip_encoding="masks")):
        with pytest.raises(_capi.SbnbError, match=rf"mask {mask} at taxon 4, pattern 37") as failure:
            make()
        assert failure.value.code == -1
    with pytest.raises(RuntimeError, match="tip_encoding"):
        sbn.Engine(spec, masks, weights, tip_encoding="iupac")


# ---- site-pattern compression -----------------------------------------------------------

def numpy_compression(sequences, table):
    """Patterns in order of first appearance and their multiplicities."""
    lut = np.full(256, 255, dtype=np.uint8)
    for symbol, value in table.items():
        lut[ord(symbol)] = value
    symbols = lut[np.frombuffer(b"".join(s.encode() for s in sequences), dtype=np.uint8).reshape(len(sequences), -1)]
    _, first, inverse, counts = np.unique(symbols.T, axis=0, return_index=True, return_inverse=True,
                                          return_counts=True)
    order = np.argsort(first)
    return symbols[:, first[order]], counts[order].astype(np.float64)


def test_masked_compression_against_numpy():
    rng = np.random.default_rng(81)
    alphabet = np.array(list("ACGTUacgtuRYSWKMBDHVNX?-ryswkmbdhvnx"))
    taxa, sites = 23, 20000
    columns = rng.choice(alphabet, size=(taxa, 700), p=None)
    picks = rng.integers(0, 700, size=sites)
    sequences = ["".join(row) for row in columns[:, picks]]
    got = sbn.SitePattern(sequences, ambiguity=True)
    patterns, weights = numpy_compression(sequences, alignment.iupac_mask_table())
    assert np.array_equal(got.patterns, patterns) and np.array_equal(got.weights, weights)
    # the state table of the same alphabet (no lower-case degenerate codes there)
    upper = ["".join(c if c in "acgt" else c.upper() for c in s) for s in sequences]
    state = sbn.SitePattern(upper)
    patterns, weights = numpy_compression(upper, alignment.symbol_table())
    assert np.array_equal(state.patterns, patterns) and np.array_equal(state.weights, weights)


def test_columns_that_differ_only_in_degenerate_codes_stay_distinct():
    sequences = ["AAAAA", "RYRNN", "CCCCC"]
    masked_patterns = sbn.SitePattern(sequences, ambiguity=True)
    assert masked_patterns.patterns.tolist() == [[1, 1, 1], [5, 10, 15], [2, 2, 2]]
    assert masked_patterns.weights.tolist() == [2.0, 1.0, 2.0]
    by_states = sbn.SitePattern(sequences)
    assert by_states.patterns.tolist() == [[0], [4], [1]] and by_states.weights.tolist() == [5.0]
    with pytest.raises(RuntimeError, match=r"^Symbol 'J' not known\.$"):
        sbn.SitePattern(["ACGT", "ACJT"], ambiguity=True)


# ---- GP engine ----------------------------------------------------------------------------

class MaskedGPOracle(gp.GPEngineOracle):
    """The NumPy GP oracle with leaf PLV entry s = bit s of the tip's mask."""

    def _initialize_plvs(self):
        C = len(self.rates)
        self.plvs = np.zeros((self.plv_count, self.pattern_count, 4 * C))
        for taxon in range(self.taxon_count):
            bits = ((self.tip_states[taxon].astype(np.int64)[:, None] >> np.arange(4)) & 1).astype(np.float64)
            self.plvs[taxon] = np.tile(bits, (1, C))
        self.rescaling_counts = np.zeros(self.plv_count, dtype=np.int64)


def gp_run(factory, fx, tips, **kwargs):
    engine = gp_cases.make_engine(factory, dict(fx, tip_states=tips), **kwargs)
    engine.process_operations(fx["program_populate_plvs"])
    engine.process_operations(fx["program_compute_likelihoods"])
    return engine


def test_gp_masked_leaves():
    fx = load_fixture("gp_five_taxon")
    gpu = lambda *args, **kwargs: sbn.GPEngine(*args, device=0, **kwargs)
    states = fx["tip_states"]
    plain = gp_run(gpu, fx, states)
    as_masks = gp_run(gpu, fx, trees.states_to_masks(states), tip_encoding="masks")
    assert as_masks.get_log_marginal_likelihood() == plain.get_log_marginal_likelihood()
    for index in range(fx["plv_count"]):
        assert np.array_equal(as_masks.get_plv(index), plain.get_plv(index)), index
    masks = trees.states_to_masks(states)
    rng = np.random.default_rng(91)
    masks[rng.random(masks.shape) < 0.2] = rng.choice([5, 10, 7, 12])
    engine = gp_run(gpu, fx, masks, tip_encoding="masks")
    oracle = gp_run(MaskedGPOracle, fx, masks)
    gp_cases.close(engine.get_log_marginal_likelihood(), oracle.get_log_marginal_likelihood())
    gp_cases.close(engine.get_per_gpcsp_log_likelihoods(), oracle.get_per_gpcsp_log_likelihoods())
    for index in range(fx["plv_count"]):
        gp_cases.close(engine.get_plv(index), oracle.plvs[index], atol=1e-300)
    for e in (engine, oracle):  # one Brent sweep over every branch length
        e.process_operations(fx["program_branch_length_optimization"])
    gp_cases.close(engine.get_branch_lengths(), oracle.get_branch_lengths(), rtol=1e-7)
