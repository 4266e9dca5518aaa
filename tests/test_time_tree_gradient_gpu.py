"""The time-tree gradient of the engine (the walk's edge sums, RootedFinishKernel on the
device, csrc/rooted.cpp on the host) against the exact reference of
tests/time_tree_reference.py: F = logL + log det J of ratios, root height, clock rates, site
shape and substitution coordinates, differentiated by the complex step.

Bars (as in test_subst_gradient_gpu.py): logL to 1e-10 relative; each gradient block of each
tree max |a - ref| <= 1e-9 max |ref|.  The walk sums ~1e4 fp64 terms per entry and the
finishing is O(n) with no cancellation beyond the reference's own, so its error is ~1e-13.
The scalar blocks (a strict clock, the site shape) are sums over edges of terms of both
signs; they keep the same relative bar, which holds on every case here, so none of them
is small from cancellation.  The engine's rooted gradient returns logL without the Jacobian (as
FatBeagle::Gradient does); rooted log_likelihoods add it.

Cases: every walk variant on batches of three dated trees of different topologies and date
sets; 130 trees (three blocks of RootedFinishKernel, repeated topologies with new dates);
relaxed clocks; 1000 taxa rescaled (directional and selected coordinates); ambiguous tips;
near-degenerate dates; CUDA-graph replay with new heights, rates and parameters; staged
pattern ranges finished on the host; device groups on both axes.
"""
import numpy as np
import pytest

import libsbn_b200 as sbn
from libsbn_b200 import _capi, sharding, trees
import time_tree_reference as tt
from test_subst_gradient_gpu import random_row, synthetic

pytestmark = pytest.mark.gpu

LOGL_RTOL = 1e-10
RTOL = 1e-9
SITES = ["constant", "weibull+2", "gamma+3", "weibull+4", "weibull+8", "gamma+16", "weibull+20", "weibull+32"]
# every site model with two substitution models, all three in turn
VARIANTS = [(s, m) for i, m in enumerate(SITES) for s in (["JC69", "GTR", "HKY"] * 2)[i % 3:i % 3 + 2]]


def time_row(substitution, site, rng):
    if substitution == "JC69":
        return ([rng.uniform(0.3, 2.0)] if site != "constant" else []) + [0.0]
    return random_row(substitution, site, rng, clock=True)


def references(substitution, site, tips, weights, batch, params, masks=False):
    return [tt.TimeTree(substitution, site, tips, weights, batch, t, params[t], masks).gradient()
            for t in range(len(params))]


def check(got, refs):
    for t, (g, (logl, _, want)) in enumerate(zip(got, refs)):
        assert abs(g.log_likelihood - logl) <= LOGL_RTOL * abs(logl), f"tree {t}"
        for key in want:
            a = g.gradient[key]
            assert a.shape == want[key].shape, key
            error = np.max(np.abs(a - want[key])) / np.max(np.abs(want[key]))
            assert error <= RTOL, f"tree {t} {key}: relative error {error:.3e}\n{a}\n{want[key]}"


def check_log_likelihoods(engine, batch, params, refs, rescaling):
    got = engine.log_likelihoods(sbn.TreeBatch(**batch), params, rescaling, rooted=True)
    want = np.array([logl + jacobian for logl, jacobian, _ in refs])
    assert np.max(np.abs(got - want) / np.abs(want)) <= LOGL_RTOL


def run(substitution, site, tips, weights, batch, params, masks=False, both=True, **engine_args):
    engine = sbn.Engine(sbn.PhyloModelSpecification(substitution, site, "strict"), tips, weights,
                        tip_encoding="masks" if masks else "states", **engine_args)
    refs = references(substitution, site, tips, weights, batch, params, masks)
    for rescaling in ((False, True) if both else (True,)):
        check(engine.gradients(sbn.TreeBatch(**batch), params, rescaling, rooted=True), refs)
    check_log_likelihoods(engine, batch, params, refs, True)
    return refs


@pytest.mark.parametrize("substitution,site", VARIANTS, ids=[f"{s}-{m}" for s, m in VARIANTS])
def test_every_walk_variant(substitution, site):
    """21 taxa x 509 patterns (a ragged last tile), three dated trees of different topologies
    and date sets, each with its own parameter row; plain and rescaled."""
    tips, weights = synthetic()
    seed = SITES.index(site) * 3 + len(substitution)
    batch = trees.random_time_trees(21, 3, seed=seed)
    rng = np.random.default_rng(seed)
    params = np.array([time_row(substitution, site, rng) for _ in range(3)])
    run(substitution, site, tips, weights, batch, params)


def test_many_trees():
    """130 trees over 40 topologies, each tree with its own dates, ratios and clock: three
    blocks of RootedFinishKernel, and per-tree strides beyond the first tree."""
    tips, weights = synthetic(patterns=64)
    batch = trees.random_time_trees(21, 130, seed=101, topology_count=40)
    rng = np.random.default_rng(102)
    params = np.array([time_row("HKY", "weibull+4", rng) for _ in range(130)])
    run("HKY", "weibull+4", tips, weights, batch, params, both=False)


@pytest.mark.parametrize("substitution,site", [("GTR", "weibull+4"), ("HKY", "gamma+8")])
def test_relaxed_clock(substitution, site):
    """rate_count 2n - 2: one rate per edge and one clock derivative per edge."""
    tips, weights = synthetic()
    batch = trees.random_time_trees(21, 3, seed=111 + len(site), relaxed=True)
    rng = np.random.default_rng(112)
    params = np.array([time_row(substitution, site, rng) for _ in range(3)])
    run(substitution, site, tips, weights, batch, params)


@pytest.mark.parametrize("ladder", [True, False], ids=["ladder", "random"])
def test_thousand_taxa_rescaled(ladder):
    """1000 dated taxa (the ladder takes the walk's pre-order boost): three seeded directional
    derivatives against sum a_i v_i to 1e-9 of sum |a_i v_i|, and the root height, the deepest
    ratio and ratios at epoch boundaries (both sides of the bounds test) exactly."""
    taxa = 1000
    tips, weights = trees.random_alignment(taxa, 96, 11, gap_fraction=0.01)
    batch = trees.random_time_trees(taxa, 1, seed=121 + ladder, ladder=ladder)
    rng = np.random.default_rng(122)
    params = np.array([time_row("GTR", "weibull+4", rng)])
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+4", "strict"), tips, weights)
    got = engine.gradients(sbn.TreeBatch(**batch), params, True, rooted=True)[0]
    tree = tt.TimeTree("GTR", "weibull+4", tips, weights, batch, 0, params[0])
    a = np.concatenate([got.gradient[key] for key, _ in tree.blocks])
    n, N = taxa, 2 * taxa - 1
    parent, bounds = batch["parent_ids"][0], batch["node_bounds"][0]
    depth = np.zeros(N, dtype=int)
    for node in range(N - 2, n - 1, -1):
        depth[node] = depth[parent[node]] + 1
    inner = [node for node in range(n, N - 1) if any(c >= n for c in np.flatnonzero(parent == node))]
    same = [node for node in inner if any(bounds[c] == bounds[node] for c in np.flatnonzero(parent == node) if c >= n)]
    other = [node for node in inner if any(bounds[c] != bounds[node] for c in np.flatnonzero(parent == node) if c >= n)]
    assert same and other
    selected = sorted({n - 2, int(np.argmax(depth[n:N - 1])), same[0] - n, other[0] - n, other[-1] - n})
    directions = np.random.default_rng(123).standard_normal((3, tree.size))
    logl, _, derivative = tree.evaluate(np.concatenate([directions, np.eye(tree.size)[selected]]))
    assert abs(got.log_likelihood - logl) <= LOGL_RTOL * abs(logl)
    for v, want in zip(directions, derivative[:3]):
        assert abs(a @ v - want) <= RTOL * np.sum(np.abs(a * v))
    for i, want in zip(selected, derivative[3:]):
        assert abs(a[i] - want) <= RTOL * abs(want), f"coordinate {i}"


@pytest.mark.parametrize("site", ["weibull+4", "weibull+32"])
def test_ambiguous_tips(site):
    masks, weights = synthetic(masks=True)
    batch = trees.random_time_trees(21, 3, seed=131)
    rng = np.random.default_rng(132)
    params = np.array([time_row("GTR", site, rng) for _ in range(3)])
    run("GTR", site, masks, weights, batch, params, masks=True)


def redate(batch, rng, ratios=None, root_gap=None):
    """The same topologies and bounds with new ratios (or ratios(t)), root heights and rates;
    the heights and lengths by the generator's float64 expression."""
    out = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in batch.items()}
    T, N = out["parent_ids"].shape[0], out["parent_ids"].shape[1] + 1
    n = (N + 1) // 2
    for t in range(T):
        r = out["height_ratios"][t]
        r[:n - 2] = rng.uniform(1e-3, 0.999, size=n - 2) if ratios is None else ratios(t)
        r[n - 2] = out["node_bounds"][t, N - 1] + (rng.uniform(0.2, 0.6) if root_gap is None else root_gap)
        h = tt.heights(out["parent_ids"][t], out["node_bounds"][t], r[None, :n - 2], r[n - 2])[0]
        out["node_heights"][t] = h
        out["branch_lengths"][t, :N - 1] = h[out["parent_ids"][t]] - h[:N - 1]
        out["rates"][t] = out["rates"][t] * rng.uniform(0.7, 1.4)
    return out


def test_near_degenerate_dates():
    """Ratios of 1e-3 (every cherry: its node almost on its bound) and 0.999 (every other node:
    almost at its parent), a root 1e-3 above the largest bound, and tips dated at their
    parent's bound.  (Chains of tiny ratios, where the heights lose the ratios to rounding,
    are left out: there the float64 heights and ratios disagree, not the gradient.)"""
    tips, weights = synthetic(patterns=200)
    base = trees.random_time_trees(21, 3, seed=141)
    rng = np.random.default_rng(142)

    def ratios(t):
        parent = base["parent_ids"][t]
        cherry = [all(c < 21 for c in np.flatnonzero(parent == node)) for node in range(21, 40)]
        return np.where(cherry, 1e-3, 0.999)
    batch = redate(base, rng, ratios=ratios, root_gap=1e-3)
    for t in range(3):
        parent, bounds = batch["parent_ids"][t], batch["node_bounds"][t]
        assert any(bounds[c] == bounds[parent[c]] for c in range(21))  # a tip at its parent's bound
    params = np.array([time_row("GTR", "weibull+4", rng) for _ in range(3)])
    run("GTR", "weibull+4", tips, weights, batch, params)


def test_graph_replay_with_new_heights_rates_and_parameters():
    """Four calls on one topology set replay a CUDA graph (the children arrays are not
    restaged); every call brings new ratios, root heights, rates and parameters."""
    tips, weights = synthetic()
    batch = trees.random_time_trees(21, 3, seed=151)
    rng = np.random.default_rng(152)
    engine = sbn.Engine(sbn.PhyloModelSpecification("HKY", "gamma+3", "strict"), tips, weights)
    for call in range(4):
        batch = redate(batch, rng)
        params = np.array([time_row("HKY", "gamma+3", rng) for _ in range(3)])
        _, walks_before = engine.walk_timing()
        got = engine.gradients(sbn.TreeBatch(**batch), params, True, rooted=True)
        if call == 3:
            assert engine.walk_timing()[1] == walks_before  # a replay: the graph's walk launch is not timed
        check(got, references("HKY", "gamma+3", tips, weights, batch, params))


@pytest.mark.parametrize("substitution,site,relaxed", [("GTR", "weibull+4", True), ("JC69", "gamma+3", False)])
def test_staged_pattern_ranges_finished_on_the_host(substitution, site, relaxed):
    """stage / run / fetch over three pattern ranges, the raw sums added, and the rooted host
    finishing: sbnb_finish_gradients_analytic (GTR) or sbnb_finish_gradients (JC69), and
    sbnb_finish_log_likelihoods_rooted."""
    tips, weights = synthetic()
    patterns, world, n = tips.shape[1], 3, tips.shape[0]
    batch = trees.random_time_trees(21, 3, seed=161, relaxed=relaxed)
    tree_batch = sbn.TreeBatch(**batch)
    rng = np.random.default_rng(162)
    spec = sbn.PhyloModelSpecification(substitution, site, "strict")
    params = np.array([time_row(substitution, site, rng) for _ in range(3)])
    engine = sbn.Engine(spec, tips, weights, 0)
    analytic = substitution != "JC69"
    total = None
    for rank in range(world):
        engine.set_pattern_range(*sharding.pattern_range(rank, world, patterns))
        staged = engine.stage(tree_batch, params, rooted=True, substitution_analytic=analytic)
        staged.run(_capi.MODE_BRANCH_GRADIENT, True)
        parts = list(staged.fetch(gradients=True)) + ([staged.fetch_substitution_sums()] if analytic else [])
        staged.close()
        total = parts if total is None else [t + p for t, p in zip(total, parts)]
    engine.set_pattern_range(0, patterns)
    if analytic:
        got = sharding.finish_gradients_analytic(spec, n, tree_batch, True, params, *total, engine.category_count)
    else:
        got = sharding.finish_gradients(spec, n, tree_batch, True, False, *total, engine.category_count)
    refs = references(substitution, site, tips, weights, batch, params)
    check(got, refs)
    with_jacobian = sharding.finish_log_likelihoods_rooted(n, tree_batch, total[0][:3].copy())
    want = np.array([logl + jacobian for logl, jacobian, _ in refs])
    assert np.max(np.abs(with_jacobian - want) / np.abs(want)) <= LOGL_RTOL


@pytest.mark.parametrize("axis", ["trees", "patterns"])
def test_device_groups(axis):
    """Five relaxed-clock dated trees through a two-member group (a repeated ordinal where the
    machine has one GPU: the same code path): the tree axis slices the rooted fields and the
    [rate_count]-wide clock rows per member, the pattern axis finishes on the host."""
    tips, weights = synthetic()
    batch = trees.random_time_trees(21, 5, seed=171, relaxed=True)
    rng = np.random.default_rng(172)
    params = np.array([time_row("GTR", "weibull+8", rng) for _ in range(5)])
    devices = [0, 1] if _capi.load().sbnb_device_count() > 1 else [0, 0]
    run("GTR", "weibull+8", tips, weights, batch, params, both=False, devices=devices, shard_axis=axis)
