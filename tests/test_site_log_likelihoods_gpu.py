"""Site log-likelihoods ([tree][pattern]) of the fused tree walk and of the BEAGLE-compatible
library against the exact per-site reference of tests/site_reference.py.

Bar: |s - ref| <= 1e-10 max(|ref|, 1) per entry.  The weighted sum of a call's matrix is its
log-likelihood to 1e-12, and that log-likelihood is bitwise what sbnb_log_likelihoods_* return.

Cases: JC69 / GTR / HKY x constant, weibull+K, gamma+K for K in {2, 3, 4, 5, 8, 16, 20, 32} (every
padded lane count), rescaling off and on, state tips, mask tips with ambiguous characters and
masks without; +I at p in {0, 0.5, 0.95}; pattern counts 1, 31, 513, 1007 with a guard region
after the output; weight-0 and split patterns; a 1000-taxon ladder; rooted time trees with
strict and relaxed clocks; the staged path and its refusals; pattern ranges; CUDA-graph replay;
device groups on both axes; tree- and pattern-sharded engines over two ranks; the BEAGLE
library's beagleGetSiteLogLikelihoods against the reference and against the walk at full size.
"""
import ctypes
import os
import socket

import numpy as np
import pytest

import libsbn_b200 as sbn
from libsbn_b200 import _capi, sharding, trees
from libsbn_b200 import beagle as bg
import beagle_reference as br
import site_reference as sr
from test_beagle_reference_gpu import _Ladder

pytestmark = pytest.mark.gpu

TAXA, PATTERNS = 11, 67
SUBSTITUTIONS = ["JC69", "GTR", "HKY"]
SITES = ["constant"] + [f"{family}+{k}" for family in ("weibull", "gamma") for k in (2, 3, 4, 5, 8, 16, 20, 32)]
TIP_MODES = ["states", "ambiguous", "masks"]  # masks: mask encoding without ambiguity (the state walk)


def row(substitution, site, rng, clock=False):
    out = {"JC69": [], "GTR": list(rng.dirichlet(np.ones(6) * 2)) + list(rng.dirichlet(np.ones(4) * 4)),
           "HKY": list(rng.dirichlet(np.ones(4) * 4)) + [rng.uniform(0.5, 4.0)]}[substitution]
    if not site.startswith("constant"):
        out.append(rng.uniform(0.3, 2.0))
    if site.endswith("+I"):
        out.append(0.0)  # (set by the caller)
    if clock:
        out.append(0.0)  # (the clock rate rides in the tree batch)
    return out


def params_for(substitution, site, count, seed, p=None, clock=False):
    rng = np.random.default_rng(seed)
    params = np.array([row(substitution, site, rng, clock) for _ in range(count)])
    if p is not None:
        params[:, params.shape[1] - 1 - clock] = p
    return params


def alignment(mode, taxa, patterns, seed):
    """(tips, weights, masks) in one of TIP_MODES."""
    rng = np.random.default_rng(seed + 1000)
    if mode == "ambiguous":
        tips, _ = trees.random_masked_alignment(taxa, patterns, seed, ambiguous_fraction=0.1, gap_fraction=0.03)
    else:
        tips, _ = trees.random_alignment(taxa, patterns, seed, gap_fraction=0.03)
        if mode == "masks":
            tips = np.where(tips >= 4, 15, 1 << np.minimum(tips, 3)).astype(np.uint8)
    return tips, rng.integers(1, 4, size=patterns).astype(np.float64), mode != "states"


def engine_for(substitution, site, tips, masks, weights, clock="none", **args):
    return sbn.Engine(sbn.PhyloModelSpecification(substitution, site, clock), tips, weights,
                      tip_encoding="masks" if masks else "states", **args)


def assert_sites(got, want):
    assert got.shape == want.shape
    error = np.abs(got - want) / np.maximum(np.abs(want), 1.0)
    assert np.all(error <= 1e-10), f"max error {np.max(error):.3e} at {np.unravel_index(np.argmax(error), error.shape)}"


def assert_sums(logl, sites, weights):
    np.testing.assert_allclose(sites @ weights, logl, rtol=1e-12)


def evaluate(engine, batch, params, rescaling, weights, rooted=False):
    """One site call: its log-likelihoods are bitwise the plain call's, its sites sum to them."""
    logl, sites = engine.site_log_likelihoods(batch, params, rescaling, rooted)
    assert np.array_equal(logl, engine.log_likelihoods(batch, params, rescaling, rooted))
    if not rooted:
        assert_sums(logl, sites, weights)
    return logl, sites


CASES = [(s, site, TIP_MODES[(i + j) % 3]) for i, site in enumerate(SITES) for j, s in enumerate(SUBSTITUTIONS)]


@pytest.mark.parametrize("substitution,site,mode", CASES, ids=[f"{s}-{m}-{t}" for s, m, t in CASES])
def test_models_and_kernel_variants(substitution, site, mode):
    tips, weights, masks = alignment(mode, TAXA, PATTERNS, seed=len(site) + SITES.index(site))
    parent_ids, lengths = trees.random_tree_batch(TAXA, 2, seed=SITES.index(site))
    params = params_for(substitution, site, 2, seed=SUBSTITUTIONS.index(substitution))
    engine = engine_for(substitution, site, tips, masks, weights)
    want = sr.matrix(substitution, site, tips, parent_ids, lengths, params, masks)
    for rescaling in (False, True):
        _, sites = evaluate(engine, sbn.TreeBatch(parent_ids, lengths), params, rescaling, weights)
        assert_sites(sites, want)


INVARIANT = [(s, m, p, TIP_MODES[i % 3]) for i, (s, m) in enumerate([("JC69", "constant+I"), ("GTR", "weibull+4+I"),
                                                                       ("HKY", "gamma+20+I"), ("GTR", "gamma+2+I")])
             for p in (0.0, 0.5, 0.95)]


@pytest.mark.parametrize("substitution,site,p,mode", INVARIANT)
def test_invariable_sites(substitution, site, p, mode):
    tips, weights, masks = alignment(mode, TAXA, PATTERNS, seed=21)
    tips = tips.copy()
    tips[:, :20] = tips[0, :20]  # constant columns, so that I_k > 0
    parent_ids, lengths = trees.random_tree_batch(TAXA, 2, seed=22)
    params = params_for(substitution, site, 2, seed=23, p=p)
    engine = engine_for(substitution, site, tips, masks, weights)
    want = sr.matrix(substitution, site, tips, parent_ids, lengths, params, masks)
    for rescaling in (False, True):
        _, sites = evaluate(engine, sbn.TreeBatch(parent_ids, lengths), params, rescaling, weights)
        assert_sites(sites, want)


@pytest.mark.parametrize("site", ["constant", "gamma+4", "weibull+32", "gamma+8"])
@pytest.mark.parametrize("patterns", [1, 31, 513, 1007])
def test_pattern_counts_leave_the_guard_region_intact(site, patterns):
    tips, weights, _ = alignment("states", TAXA, patterns, seed=patterns)
    parent_ids, lengths = trees.random_tree_batch(TAXA, 3, seed=31)
    params = params_for("GTR", site, 3, seed=32)
    engine = engine_for("GTR", site, tips, False, weights)
    batch = sbn.TreeBatch(parent_ids, lengths)
    want = sr.matrix("GTR", site, tips, parent_ids, lengths, params)
    for rescaling in (0, 1):
        out = np.full(3 * patterns + 1024, np.nan)
        logl = np.empty(3)
        struct = batch.as_struct()
        _capi.check(_capi.load().sbnb_site_log_likelihoods_unrooted(
            engine._handle, ctypes.byref(struct), _capi.as_double_ptr(params), rescaling, _capi.as_double_ptr(logl),
            _capi.as_double_ptr(out)))
        assert np.all(np.isnan(out[3 * patterns:]))
        sites = out[:3 * patterns].reshape(3, patterns)
        assert_sites(sites, want)
        assert_sums(logl, sites, weights)
        # NULL log-likelihoods: the matrix alone
        again = np.empty((3, patterns))
        _capi.check(_capi.load().sbnb_site_log_likelihoods_unrooted(
            engine._handle, ctypes.byref(struct), _capi.as_double_ptr(params), rescaling, None,
            _capi.as_double_ptr(again)))
        assert np.array_equal(again, sites)


def test_weight_zero_and_split_patterns():
    """Weight-0 patterns get their values; a pattern split into two copies with split weights gets
    two equal values and leaves logL as it was."""
    tips, weights, _ = alignment("states", 17, 300, seed=41)
    weights[::7] = 0.0
    parent_ids, lengths = trees.random_tree_batch(17, 2, seed=42)
    params = params_for("HKY", "gamma+4", 2, seed=43)
    batch = sbn.TreeBatch(parent_ids, lengths)
    want = sr.matrix("HKY", "gamma+4", tips, parent_ids, lengths, params)
    engine = engine_for("HKY", "gamma+4", tips, False, weights)
    split = np.concatenate([tips, tips[:, :40]], axis=1)
    split_weights = np.concatenate([weights * 1.0, weights[:40] * 0.75])
    split_weights[:40] *= 0.25
    split_engine = engine_for("HKY", "gamma+4", split, False, split_weights)
    for rescaling in (False, True):
        logl, sites = evaluate(engine, batch, params, rescaling, weights)
        assert_sites(sites[:, ::7], want[:, ::7])
        assert_sites(sites, want)
        split_logl, split_sites = evaluate(split_engine, batch, params, rescaling, split_weights)
        np.testing.assert_allclose(split_logl, logl, rtol=1e-12)
        if rescaling:  # (a pattern's power-of-two exponents may be decided with its tile neighbours)
            np.testing.assert_allclose(split_sites[:, 300:], split_sites[:, :40], rtol=1e-14)
        else:
            assert np.array_equal(split_sites[:, 300:], split_sites[:, :40])


def test_thousand_taxon_ladder():
    """Rescaled: finite and on the reference.  Unrescaled: sites that underflow are -inf, as their
    terms in the sum are; the others are on the reference."""
    taxa, patterns = 1000, 40
    tips, weights, _ = alignment("states", taxa, patterns, seed=51)
    parent_ids = trees.ladder_topology(taxa)[None, :]
    lengths = np.full((1, parent_ids.shape[1] + 1), 0.15)
    params = params_for("GTR", "weibull+4", 1, seed=52)
    engine = engine_for("GTR", "weibull+4", tips, False, weights)
    want = sr.matrix("GTR", "weibull+4", tips, parent_ids, lengths, params)
    batch = sbn.TreeBatch(parent_ids, lengths)
    _, sites = evaluate(engine, batch, params, True, weights)
    assert np.all(np.isfinite(sites)) and np.all(want < -745.0)
    assert_sites(sites, want)
    logl, sites = engine.site_log_likelihoods(batch, params, False)
    assert logl[0] == -np.inf and np.any(sites == -np.inf)
    finite = np.isfinite(sites)
    assert_sites(sites[finite], want[finite])


@pytest.mark.parametrize("substitution,site,relaxed", [("GTR", "weibull+4", False), ("HKY", "gamma+4+I", True),
                                                       ("JC69", "weibull+20", True), ("GTR", "constant", False)])
def test_rooted_time_trees(substitution, site, relaxed):
    tips, weights, masks = alignment("ambiguous" if relaxed else "states", TAXA, 201, seed=61)
    batch = trees.random_time_trees(TAXA, 3, seed=62, relaxed=relaxed)
    params = params_for(substitution, site, 3, seed=63, p=0.3 if site.endswith("+I") else None, clock=True)
    engine = engine_for(substitution, site, tips, masks, weights, clock="strict")
    want = sr.time_tree_matrix(substitution, site, tips, batch, params, masks)
    tree_batch = sbn.TreeBatch(**batch)
    jacobian = sharding.finish_log_likelihoods_rooted(TAXA, tree_batch, np.zeros(3))
    assert np.all(jacobian != 0.0)
    for rescaling in (False, True):
        logl, sites = evaluate(engine, tree_batch, params, rescaling, weights, rooted=True)
        assert_sites(sites, want)
        np.testing.assert_allclose(sites @ weights, logl - jacobian, rtol=1e-12)


def staged_case(patterns=1301, seed=71):
    tips, weights, _ = alignment("states", TAXA, patterns, seed=seed)
    parent_ids, lengths = trees.random_tree_batch(TAXA, 4, seed=seed + 1)
    params = params_for("GTR", "gamma+4", 4, seed=seed + 2)
    return tips, weights, sbn.TreeBatch(parent_ids, lengths), params


def test_staged_fetch_and_refusals():
    tips, weights, batch, params = staged_case()
    engine = engine_for("GTR", "gamma+4", tips, False, weights)
    plain = engine.stage(batch, params)
    plain.run(_capi.MODE_LOG_LIKELIHOOD, True)
    with pytest.raises(_capi.SbnbError, match="not staged") as refused:
        plain.fetch_site_log_likelihoods()
    assert refused.value.code == -1
    plain.close()
    staged = engine.stage(batch, params, site_log_likelihoods=True)
    with pytest.raises(_capi.SbnbError, match="not been run") as refused:
        staged.fetch_site_log_likelihoods()
    assert refused.value.code == -1
    for rescaling in (False, True):
        staged.run(_capi.MODE_BRANCH_GRADIENT, rescaling)
        with pytest.raises(_capi.SbnbError, match="gradient run") as refused:
            staged.fetch_site_log_likelihoods()
        assert refused.value.code == -1
        staged.run(_capi.MODE_LOG_LIKELIHOOD, rescaling)
        sites = staged.fetch_site_log_likelihoods()
        logl = staged.fetch()
        one_call_logl, one_call = engine.site_log_likelihoods(batch, params, rescaling)
        assert np.array_equal(sites, one_call) and np.array_equal(logl, one_call_logl)
    staged.close()


@pytest.mark.parametrize("rescaling", [False, True])
def test_pattern_ranges_are_columns_of_the_full_matrix(rescaling):
    tips, weights, batch, params = staged_case(seed=81)
    engine = engine_for("GTR", "gamma+4", tips, False, weights)
    _, full = engine.site_log_likelihoods(batch, params, rescaling)
    for begin, end in [(0, 700), (700, 1301), (13, 14), (5, 1290)]:
        engine.set_pattern_range(begin, end)
        logl, sites = engine.site_log_likelihoods(batch, params, rescaling)
        staged = engine.stage(batch, params, site_log_likelihoods=True)
        staged.run(_capi.MODE_LOG_LIKELIHOOD, rescaling)
        staged_sites = staged.fetch_site_log_likelihoods()
        staged.close()
        assert sites.shape == (4, end - begin) and np.array_equal(staged_sites, sites)
        assert_sums(logl, sites, weights[begin:end])
        if rescaling:
            np.testing.assert_allclose(sites, full[:, begin:end], rtol=1e-14)
        else:
            assert np.array_equal(sites, full[:, begin:end])
    engine.set_pattern_range(0, engine.pattern_count)
    staged = engine.stage(batch, params, site_log_likelihoods=True)
    engine.set_pattern_range(0, 100)
    with pytest.raises(_capi.SbnbError, match="pattern range has changed"):
        staged.run(_capi.MODE_LOG_LIKELIHOOD, rescaling)
    staged.close()


def test_graph_replay():
    """The same topologies five times (the later calls replay a CUDA graph) with new lengths: every
    call is on the reference and bitwise equal to an eager staged run."""
    tips, weights, batch, params = staged_case(patterns=257, seed=91)
    engine = engine_for("GTR", "gamma+4", tips, False, weights)
    for call in range(5):
        scaled = sbn.TreeBatch(batch.parent_ids, batch.branch_lengths * (1.0 + 0.2 * call))
        logl, sites = engine.site_log_likelihoods(scaled, params, True)
        assert_sites(sites, sr.matrix("GTR", "gamma+4", tips, scaled.parent_ids, scaled.branch_lengths, params))
        assert_sums(logl, sites, weights)
        staged = engine.stage(scaled, params, site_log_likelihoods=True)
        staged.run(_capi.MODE_LOG_LIKELIHOOD, True)
        assert np.array_equal(staged.fetch_site_log_likelihoods(), sites)
        assert np.array_equal(staged.fetch(), logl)
        staged.close()
        # the plain log-likelihood call on the same topologies keeps its own graph
        assert np.array_equal(engine.log_likelihoods(scaled, params, True), logl)


@pytest.mark.parametrize("axis", ["trees", "patterns"])
@pytest.mark.parametrize("rooted", [False, True])
def test_device_groups(axis, rooted):
    tips, weights, batch, params = staged_case(patterns=1001, seed=101)
    clock = "none"
    if rooted:
        batch = sbn.TreeBatch(**trees.random_time_trees(TAXA, 5, seed=102))
        params = params_for("GTR", "gamma+4", 5, seed=103, clock=True)
        clock = "strict"
    single = engine_for("GTR", "gamma+4", tips, False, weights, clock=clock)
    group = engine_for("GTR", "gamma+4", tips, False, weights, clock=clock, devices=[0, 0], shard_axis=axis)
    for rescaling in (False, True):
        logl, sites = single.site_log_likelihoods(batch, params, rescaling, rooted)
        group_logl, group_sites = group.site_log_likelihoods(batch, params, rescaling, rooted)
        np.testing.assert_allclose(group_logl, logl, rtol=1e-12)
        assert np.array_equal(group_logl, group.log_likelihoods(batch, params, rescaling, rooted))
        if rescaling:
            np.testing.assert_allclose(group_sites, sites, rtol=1e-14)
        else:
            assert np.array_equal(group_sites, sites)


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_worker(rank, world, port, result_path):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        tips, weights, batch, params = staged_case(patterns=1001, seed=111)
        spec = sbn.PhyloModelSpecification("GTR", "gamma+4", "none")
        out = {}
        for name, cls in (("trees", sharding.TreeShardedEngine), ("patterns", sharding.PatternShardedEngine)):
            logl, sites = cls(spec, tips, weights, device=0).site_log_likelihoods(batch, params, rescaling=True)
            out[name + "_logl"], out[name + "_sites"] = logl, sites
        if rank == 0:
            np.savez(result_path, **out)
    finally:
        dist.destroy_process_group()


def test_sharded_engines_over_two_ranks(tmp_path):
    import torch.multiprocessing as mp
    result = str(tmp_path / "sharded.npz")
    mp.spawn(_sharded_worker, args=(2, free_port(), result), nprocs=2, join=True)
    tips, weights, batch, params = staged_case(patterns=1001, seed=111)
    logl, sites = engine_for("GTR", "gamma+4", tips, False, weights).site_log_likelihoods(batch, params, True)
    got = np.load(result)
    for name in ("trees", "patterns"):
        np.testing.assert_allclose(got[name + "_logl"], logl, rtol=1e-12)
        np.testing.assert_allclose(got[name + "_sites"], sites, rtol=1e-14)


# ---- the BEAGLE-compatible library ----------------------------------------------------------

@pytest.mark.parametrize("categories", [1, 3, 4, 20])
def test_beagle_library_against_the_reference(categories):
    """A 700-taxon ladder, rescaled: beagleGetSiteLogLikelihoods is the reference per pattern (scale
    factors included), sums to the root call's logL, and is an error before any root call."""
    case = br.random_case(700, 61, categories, 130 + categories, "libsbn")
    case["post"], case["pre"] = bg.random_tree_operations(700, _Ladder(), True)
    _, _, _, freqs, q = bg.gtr_eigensystem()
    library = br.open_library(None, case)
    try:
        out = np.empty(case["P"])
        assert library.lib.beagleGetSiteLogLikelihoods(library.handle, out.ctypes.data_as(
            ctypes.POINTER(ctypes.c_double))) != 0
        logl, _, _, _ = br.evaluate(library, case)
        sites = library.site_log_likelihoods()
    finally:
        library.close()
    want = sr.beagle_case(case, q, freqs)
    assert np.all(want < -745.0)  # (far below the fp64 range without the scale factors)
    assert_sites(sites[None, :], want[None, :])
    assert abs(sites @ case["weights"] - logl) <= 1e-12 * abs(logl)


@pytest.mark.parametrize("taxa,patterns", [(100, 100000), (1000, 20000)])
def test_beagle_library_and_the_walk_agree_at_full_size(taxa, patterns):
    categories, shape = 4, 0.5
    N = 2 * taxa - 1
    rng = np.random.default_rng(20261022)
    states, _ = trees.random_alignment(taxa, patterns, 77, gap_fraction=0.01)
    weights = rng.integers(1, 4, size=patterns).astype(np.float64)
    post, pre = bg.random_tree_operations(taxa, rng, True)
    parent_ids = np.full(N - 1, -1, dtype=np.int32)
    for op in post:
        parent_ids[op[3]] = parent_ids[op[5]] = op[0]
    lengths = np.maximum(rng.exponential(0.1, size=N), 1e-6)
    lengths[N - 1] = 0.0
    evec, ivec, evals, freqs, q = bg.gtr_eigensystem()
    quantiles = (2.0 * np.arange(categories) + 1.0) / (2.0 * categories)
    rates = (-np.log(1.0 - quantiles)) ** (1.0 / shape)
    rates /= rates.mean()
    library = bg.Beagle(None, taxa, patterns, categories, True)
    library.set_tips(states.astype(np.int32), weights, True)
    library.set_model(evec, ivec, evals, freqs, rates, np.full(categories, 1.0 / categories))
    logl, _, _, _ = library.log_likelihood_and_gradient(post, pre, lengths, q, rates, freqs, True, per_site=False)
    sites = library.site_log_likelihoods()
    library.close()
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+4", "none"), states, weights)
    params = np.array([[0.05, 0.1, 0.15, 0.20, 0.25, 0.25, 0.1, 0.2, 0.3, 0.4, shape]])
    walk_logl, walk_sites = engine.site_log_likelihoods(sbn.TreeBatch(parent_ids[None, :], lengths[None, :]), params,
                                                        True)
    assert abs(walk_logl[0] - logl) <= 1e-10 * abs(logl)
    np.testing.assert_allclose(walk_sites[0], sites, rtol=1e-10)
