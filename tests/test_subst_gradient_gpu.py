"""The analytic substitution-model gradient of the fused walk (the SUBST instantiations of
TreeWalkOeKernel, K1's Phi, the host's <W, B_theta> + dpi/dtheta . R) against an exact
reference: tests/subst_reference.py differentiates a complex128 pruning by the complex step,
so it is exact to fp64 rounding and shares no formula with the walk.

The bar is max |a - ref| <= 1e-9 max |ref| per tree, logL to 1e-10 relative.  The walk sums
at most ~1e5 fp64 terms per entry, so its own error is ~1e-13 of the largest entry.  The
central differences of the other checks of this block resolve only ~1e-6 of |logL|, about
1 % of DS1's smallest coordinates.

Cases: every SUBST instantiation (1 to 32 lanes, GTR and HKY, plain and rescaled, a ragged
last tile); DS1 topologies; time trees; 1000 taxa with rescaling (the ladder takes the
pre-order 2^-384 boost); ambiguous tips; long, zero-length and degenerate branches; CUDA-graph
replay; staged pattern ranges finished on the host; a pattern-sharded device group.
"""
import numpy as np
import pytest

from conftest import load_fixture
import libsbn_b200 as sbn
from libsbn_b200 import _capi, sharding, trees
import subst_reference as ref
import time_tree_reference as tt

pytestmark = pytest.mark.gpu

LOGL_RTOL = 1e-10
SUBST_RTOL = 1e-9
EXTREME_FREQS = [0.94, 0.02, 0.02, 0.02]


def random_row(substitution, site, rng, freqs=None, clock=False):
    """An engine parameter row: the substitution block, the site shape, the clock rate."""
    freqs = list(rng.dirichlet(np.ones(4) * 4) if freqs is None else freqs)
    if substitution == "GTR":
        row = list(rng.dirichlet(np.ones(6) * 2)) + freqs
    else:
        row = freqs + [rng.uniform(0.5, 4.0)]
    if site != "constant":
        row.append(rng.uniform(0.3, 2.0))
    if clock:
        row.append(0.0)  # (the clock rate rides in the tree batch)
    return row


def synthetic(taxa=21, patterns=509, seed=3, masks=False):
    """509 patterns: the last tile of every lane count is ragged.  Gaps, weights 1..3."""
    if masks:
        tips, _ = trees.random_masked_alignment(taxa, patterns, seed, ambiguous_fraction=0.05, gap_fraction=0.02)
    else:
        tips, _ = trees.random_alignment(taxa, patterns, seed, gap_fraction=0.03)
    weights = np.random.default_rng(seed).integers(1, 4, size=patterns).astype(np.float64)
    return tips, weights


def check(got, substitution, site, tips, weights, parent_ids, lengths, params, masks=False, references=None,
          branches=True):
    """Every tree of `got` against the reference; returns the references for reuse.  With
    `branches`, also the branch-length and site-model blocks against
    time_tree_reference.unrooted_gradient (the complex step on every edge and the shape)."""
    references = references or [
        ref.log_likelihood_and_gradient(substitution, site, tips, weights, parent_ids[t], lengths[t], params[t],
                                        masks=masks) +
        (tt.unrooted_gradient(substitution, site, tips, weights, parent_ids[t], lengths[t], params[t], masks)[1:]
         if branches else (None, None)) for t in range(len(got))]
    for t, (g, (logl, want, branch, shape)) in enumerate(zip(got, references)):
        a = g.gradient["substitution_model"]
        assert a.shape == want.shape
        assert np.all(np.isfinite(a)), f"tree {t}: {a}"
        assert abs(g.log_likelihood - logl) <= LOGL_RTOL * abs(logl), f"tree {t}"
        error = np.max(np.abs(a - want)) / np.max(np.abs(want))
        assert error <= SUBST_RTOL, f"tree {t}: relative error {error:.3e}\n{a}\n{want}"
        if branch is not None:
            check_branches(g.gradient["branch_lengths"], branch, parent_ids[t], t)
        if shape is not None:
            assert abs(g.gradient["site_model"][0] - shape) <= SUBST_RTOL * abs(shape), f"tree {t}: site model"
    return references


def check_branches(a, want, parent_ids, t):
    """The engine's [2n-1] branch-length block against d logL / d (each edge of the tree as
    given).  A trifurcating tree keeps its edge ids, the two edges detrifurcation adds get 0;
    a bifurcating tree's root slide puts the root edge's derivative on the first child of the
    root and 0 on the second, so the two are compared as a sum (each side of the root edge
    has that derivative: the pulley principle)."""
    edges = len(parent_ids)
    root_children = np.flatnonzero(np.asarray(parent_ids) == edges)
    scale = np.max(np.abs(want))
    if len(root_children) == 3:
        assert np.all(a[edges:] == 0.0)
        error = np.max(np.abs(a[:edges] - want)) / scale
    else:
        first, second = root_children
        rest = np.setdiff1d(np.arange(edges), root_children)
        error = max(np.max(np.abs(a[rest] - want[rest])), abs(a[first] + a[second] - want[first]),
                    abs(a[first] + a[second] - want[second])) / scale
    assert error <= SUBST_RTOL, f"tree {t}: branch lengths, relative error {error:.3e}"


def run_both_modes(engine, batch, params, rooted=False):
    return [engine.gradients(batch, params, rescaling, rooted=rooted) for rescaling in (False, True)]


SITES = ["constant", "weibull+2", "gamma+3", "weibull+4", "weibull+8", "weibull+16", "weibull+20", "weibull+32"]


@pytest.mark.parametrize("site", SITES)
@pytest.mark.parametrize("substitution", ["GTR", "HKY"])
def test_every_walk_variant(substitution, site):
    """1, 2, 4 (gamma+3 padded), 4, 8, 16 lanes and 20, 32 (one pattern per warp), plain and
    rescaled, on 21 taxa x 509 patterns."""
    tips, weights = synthetic()
    rng = np.random.default_rng(SITES.index(site) * 2 + (substitution == "HKY"))
    parent_ids, lengths = trees.random_tree_batch(21, 2, seed=SITES.index(site) + 7)
    params = np.array([random_row(substitution, site, rng) for _ in range(2)])
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "none"), tips, weights)
    references = None
    for got in run_both_modes(engine, sbn.TreeBatch(parent_ids, lengths), params):
        references = check(got, substitution, site, tips, weights, parent_ids, lengths, params, references=references)


@pytest.mark.parametrize("substitution", ["GTR", "HKY"])
def test_ds1_topologies(substitution):
    fx = load_fixture("ds1_gtr_weibull4")
    count = 3
    rng = np.random.default_rng(21)
    params = np.array([random_row(substitution, "weibull+4", rng) for _ in range(count)])
    parent_ids, lengths = fx["parent_ids"][:count], fx["branch_lengths"][:count]
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, "weibull+4", "none"), fx["patterns"], fx["weights"])
    references = None
    for got in run_both_modes(engine, sbn.TreeBatch(parent_ids, lengths), params):
        references = check(got, substitution, "weibull+4", fx["patterns"], fx["weights"], parent_ids, lengths, params,
                           references=references)


@pytest.mark.parametrize("site", ["weibull+4", "weibull+20"])
@pytest.mark.parametrize("substitution", ["GTR", "HKY"])
def test_time_trees(substitution, site):
    """The influenza fixture's topology, heights and strict clock: the walk runs on the
    effective lengths, branch length x rate."""
    fx = load_fixture("flua_jc69_strict")
    rng = np.random.default_rng(len(site) + (substitution == "HKY"))
    params = np.array([random_row(substitution, site, rng, clock=True)])
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "strict"), fx["patterns"], fx["weights"])
    batch = sbn.TreeBatch(fx["parent_ids"], fx["branch_lengths"], fx["rates"], fx["node_heights"],
                          fx["node_bounds"], fx["height_ratios"], 1)
    effective = fx["branch_lengths"].copy()
    effective[:, :-1] *= fx["rates"]
    references = None
    for got in run_both_modes(engine, batch, params, rooted=True):
        references = check(got, substitution, site, fx["patterns"], fx["weights"], fx["parent_ids"], effective,
                           params, references=references, branches=False)


@pytest.mark.parametrize("shape,substitution,site", [
    ("ladder", "HKY", "weibull+4"), ("ladder", "GTR", "weibull+4"), ("ladder", "HKY", "weibull+32"),
    ("ladder", "GTR", "weibull+32"), ("random", "GTR", "weibull+4"), ("random", "HKY", "weibull+32")])
def test_thousand_taxa_rescaled(shape, substitution, site):
    """Site likelihoods of 1000 taxa underflow fp64; the ladder's pre-order partials need the
    walk's 2^-384 boost, whose scale the Phi accumulation must undo."""
    taxa = 1000
    tips, weights = trees.random_alignment(taxa, 96, 11, gap_fraction=0.01)
    rng = np.random.default_rng(13)
    parent_ids = (trees.ladder_topology(taxa) if shape == "ladder" else trees.random_unrooted_topology(taxa, rng))[None]
    lengths = np.maximum(rng.exponential(0.1, size=(1, 2 * taxa - 2)), 1e-6)
    params = np.array([random_row(substitution, site, rng)])
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "none"), tips, weights)
    got = engine.gradients(sbn.TreeBatch(parent_ids, lengths), params, True)
    check(got, substitution, site, tips, weights, parent_ids, lengths, params, branches=False)


@pytest.mark.parametrize("site", ["weibull+4", "weibull+32"])
def test_ambiguous_tips(site):
    """5 % ambiguous characters: the AMBIG + SUBST instantiations, plain and rescaled."""
    masks, weights = synthetic(masks=True)
    rng = np.random.default_rng(31)
    parent_ids, lengths = trees.random_tree_batch(21, 2, seed=32)
    params = np.array([random_row("GTR", site, rng) for _ in range(2)])
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", site, "none"), masks, weights, tip_encoding="masks")
    references = None
    for got in run_both_modes(engine, sbn.TreeBatch(parent_ids, lengths), params):
        references = check(got, "GTR", site, masks, weights, parent_ids, lengths, params, masks=True,
                           references=references)


@pytest.mark.parametrize("substitution,site,freqs", [
    ("GTR", "gamma+8", None), ("HKY", "gamma+8", None),
    ("GTR", "weibull+4", EXTREME_FREQS), ("HKY", "constant", EXTREME_FREQS)],
    ids=["GTR-gamma+8", "HKY-gamma+8", "GTR-weibull+4-extreme_freqs", "HKY-constant-extreme_freqs"])
def test_long_branches(substitution, site, freqs):
    """Branches of 50, 200 and 1000 expected substitutions, Gamma shape 0.2 (a fast last
    category) or frequencies (0.94, 0.02, 0.02, 0.02) (a wide eigenvalue spread): (l_k - l_l) tau
    reaches far beyond 709, where e^x - 1 overflows.  Phi must stay finite and exact."""
    tips, weights = synthetic(patterns=200)
    rng = np.random.default_rng(41)
    parent_ids, lengths = trees.random_tree_batch(21, 2, seed=42)
    lengths[:, [0, 5, 30]] = [50.0, 200.0, 1000.0]
    params = np.array([random_row(substitution, site, rng, freqs=freqs) for _ in range(2)])
    if site.startswith("gamma"):
        params[:, -1] = 0.2
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "none"), tips, weights)
    references = None
    for got in run_both_modes(engine, sbn.TreeBatch(parent_ids, lengths), params):
        references = check(got, substitution, site, tips, weights, parent_ids, lengths, params, references=references)


def test_zero_and_tiny_branches():
    """Lengths 0 and 1e-12 (Phi's diagonal tau e^{l tau} -> 0, its off-diagonal ratio at
    x -> 0), and a bifurcating input, whose root slide gives the root's second child length
    0 (the reference prunes the unslid tree: the same likelihood by the pulley principle)."""
    tips, weights = synthetic(patterns=200)
    rng = np.random.default_rng(51)
    parent_ids, lengths = trees.random_tree_batch(21, 2, seed=52)
    lengths[:, [1, 4, 22]] = 0.0
    lengths[:, [2, 7, 25]] = 1e-12
    rooted_ids, rooted_lengths = trees.random_tree_batch(21, 2, seed=53, rooted=True)
    for substitution, site in (("GTR", "weibull+4"), ("HKY", "constant")):
        params = np.array([random_row(substitution, site, rng) for _ in range(2)])
        engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "none"), tips, weights)
        for ids, lens in ((parent_ids, lengths), (rooted_ids, rooted_lengths)):
            for got in run_both_modes(engine, sbn.TreeBatch(ids, lens), params):
                check(got, substitution, site, tips, weights, ids, lens, params)


@pytest.mark.parametrize("site", ["constant", "weibull+4"])
def test_hky_with_kappa_one_and_uniform_frequencies(site):
    """JC69 as an HKY: exactly repeated eigenvalues, every off-diagonal ratio at x = 0 or nearly."""
    tips, weights = synthetic(patterns=200)
    parent_ids, lengths = trees.random_tree_batch(21, 2, seed=61)
    params = np.array([[0.25, 0.25, 0.25, 0.25, 1.0] + ([0.8] if site != "constant" else [])] * 2)
    engine = sbn.Engine(sbn.PhyloModelSpecification("HKY", site, "none"), tips, weights)
    references = None
    for got in run_both_modes(engine, sbn.TreeBatch(parent_ids, lengths), params):
        references = check(got, "HKY", site, tips, weights, parent_ids, lengths, params, references=references)


def test_graph_replay_with_new_parameters_and_lengths():
    """Repeated calls on one topology set replay a CUDA graph; every call brings new model
    parameters and branch lengths, and every call's result is the reference's."""
    tips, weights = synthetic()
    parent_ids, lengths = trees.random_tree_batch(21, 3, seed=71)
    rng = np.random.default_rng(72)
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+4", "none"), tips, weights)
    for call in range(4):
        params = np.array([random_row("GTR", "weibull+4", rng) for _ in range(3)])
        scaled = lengths * rng.uniform(0.5, 1.5, lengths.shape)
        _, walks_before = engine.walk_timing()
        got = engine.gradients(sbn.TreeBatch(parent_ids, scaled), params, True)
        if call == 3:
            assert engine.walk_timing()[1] == walks_before  # a replay: the graph's walk launch is not timed
        check(got, "GTR", "weibull+4", tips, weights, parent_ids, scaled, params)


def test_staged_pattern_ranges_finished_on_the_host():
    """stage / run / fetch over three pattern ranges, the raw sums (among them the [T][20]
    substitution sums) added, and sbnb_finish_gradients_analytic on the host."""
    tips, weights = synthetic()
    patterns, world = tips.shape[1], 3
    parent_ids, lengths = trees.random_tree_batch(21, 3, seed=81)
    rng = np.random.default_rng(82)
    spec = sbn.PhyloModelSpecification("HKY", "gamma+3", "none")
    params = np.array([random_row("HKY", "gamma+3", rng) for _ in range(3)])
    engine = sbn.Engine(spec, tips, weights, 0)
    batch = sbn.TreeBatch(parent_ids, lengths)
    total = None
    for rank in range(world):
        engine.set_pattern_range(*sharding.pattern_range(rank, world, patterns))
        staged = engine.stage(batch, params, substitution_analytic=True)
        staged.run(_capi.MODE_BRANCH_GRADIENT, True)
        parts = list(staged.fetch(gradients=True)) + [staged.fetch_substitution_sums()]
        staged.close()
        total = parts if total is None else [t + p for t, p in zip(total, parts)]
    engine.set_pattern_range(0, patterns)
    got = sharding.finish_gradients_analytic(spec, 21, batch, False, params, *total, engine.category_count)
    check(got, "HKY", "gamma+3", tips, weights, parent_ids, lengths, params)


def test_pattern_sharded_device_group():
    """Two pattern shards whose sums are added by the library (a repeated ordinal where the
    machine has one GPU: the same code path, one device)."""
    tips, weights = synthetic()
    parent_ids, lengths = trees.random_tree_batch(21, 3, seed=91)
    rng = np.random.default_rng(92)
    params = np.array([random_row("GTR", "weibull+8", rng) for _ in range(3)])
    devices = [0, 1] if _capi.load().sbnb_device_count() > 1 else [0, 0]
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+8", "none"), tips, weights, devices=devices,
                        shard_axis="patterns")
    got = engine.gradients(sbn.TreeBatch(parent_ids, lengths), params, True)
    check(got, "GTR", "weibull+8", tips, weights, parent_ids, lengths, params)
