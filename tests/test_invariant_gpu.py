"""Invariable sites (+I) on the fused tree walk against the exact reference of
tests/invariant_reference.py (complex step in every input, p included).

Bars (the project's): logL to 1e-10 relative; each gradient block of each tree
max |a - ref| <= 1e-8 max |ref|.  The finite-difference substitution gradient carries its
own truncation and rounding (|logL| eps / delta) and is held to the reference accordingly.

Cases: JC69 / GTR / HKY x constant+I / weibull+4+I / gamma+4+I / weibull+20+I (32 lanes) x
p in {0, 0.05, 0.5, 0.95}, rescaling off and on, state and mask tips; rooted trees with strict
and relaxed clocks; p = 0 against the plain spec; alignments with no constant pattern and
mostly constant ones; 1000 taxa rescaled; CUDA-graph replay; device groups on both axes;
staged pattern ranges finished on the host; PatternShardedEngine over two ranks.
"""
import os
import socket

import numpy as np
import pytest

import libsbn_b200 as sbn
from libsbn_b200 import sharding, trees
import invariant_reference as inv
from test_invariant_cpu import invariant_alignment

pytestmark = pytest.mark.gpu

LOGL_RTOL = 1e-10
RTOL = 1e-8
FD_RTOL = 1e-5
PS = [0.0, 0.05, 0.5, 0.95]
MODELS = [("JC69", "constant+I"), ("GTR", "weibull+4+I"), ("HKY", "gamma+4+I"), ("GTR", "weibull+20+I"),
          ("JC69", "weibull+4+I"), ("HKY", "constant+I")]


def random_row(substitution, site, p, rng, clock=False):
    row = {"JC69": [], "GTR": list(rng.dirichlet(np.ones(6) * 2)) + list(rng.dirichlet(np.ones(4) * 4)),
           "HKY": list(rng.dirichlet(np.ones(4) * 4)) + [rng.uniform(0.5, 4.0)]}[substitution]
    if not site.startswith("constant"):
        row.append(rng.uniform(0.3, 2.0))
    row.append(p)
    if clock:
        row.append(0.0)  # (the clock rate rides in the tree batch)
    return row


def params_for(substitution, site, p, count, seed, clock=False):
    rng = np.random.default_rng(seed)
    return np.array([random_row(substitution, site, p, rng, clock) for _ in range(count)])


def block_error(a, want):
    scale = np.max(np.abs(want))
    return np.max(np.abs(a - want)) / scale if scale > 0 else np.max(np.abs(a))


def check(got, refs, fd=False):
    for t, (g, (logl, want)) in enumerate(zip(got, refs)):
        assert abs(g.log_likelihood - logl) <= LOGL_RTOL * abs(logl), f"tree {t}: {g.log_likelihood} vs {logl}"
        for key, value in want.items():
            a = g.gradient[key]
            assert a.shape == value.shape, (key, a.shape, value.shape)
            if fd and key == "substitution_model":
                # central differences (delta 1e-6) of log-likelihoods: truncation plus rounding of |logL| x eps / delta
                assert np.max(np.abs(a - value)) <= FD_RTOL * np.max(np.abs(value)) + abs(logl) * 1e-12 / 1e-6
                continue
            bar = RTOL
            if key == "branch_lengths":  # the fixed node's entry is zeroed (fat_beagle.cpp:498-500)
                value = value.copy()
                value[a == 0.0] = 0.0
            error = block_error(a, value)
            assert error <= bar, f"tree {t} {key}: relative error {error:.3e}\n{a}\n{value}"


def unrooted_references(substitution, site, tips, weights, parent_ids, lengths, params, masks):
    out = []
    for t in range(len(params)):
        logl, want = inv.unrooted_gradient(substitution, site, tips, weights, parent_ids[t], lengths[t], params[t],
                                           masks)
        want["branch_lengths"] = np.append(want["branch_lengths"], 0.0)  # (the root entry)
        out.append((logl, want))
    return out


def slid(lengths, parent_ids):
    """The root slide of the reference's unrooted gradient, so that every edge derivative is
    comparable: bifurcating trees whose root's second child already has length 0."""
    lengths = lengths.copy()
    for t in range(len(lengths)):
        root = len(parent_ids[t])
        children = sorted(np.flatnonzero(parent_ids[t] == root))
        lengths[t, children[0]] += lengths[t, children[1]]
        lengths[t, children[1]] = 0.0
    return lengths


def unrooted_case(taxa=21, patterns=509, trees_=2, seed=3, masks=False, constant_fraction=0.3):
    tips, weights = invariant_alignment(taxa, patterns, seed, constant_fraction, masks)
    parent_ids, lengths = trees.random_tree_batch(taxa, trees_, seed=seed + 1, rooted=True)
    return tips, weights, parent_ids, slid(lengths, parent_ids)


def engine_for(substitution, site, tips, weights, masks, clock="none", **args):
    return sbn.Engine(sbn.PhyloModelSpecification(substitution, site, clock), tips, weights,
                      tip_encoding="masks" if masks else "states", **args)


CASES = [(s, m, p) for (s, m) in MODELS[:4] for p in PS]


@pytest.mark.parametrize("substitution,site,p", CASES, ids=[f"{s}-{m}-{p}" for s, m, p in CASES])
def test_unrooted_against_the_reference(substitution, site, p):
    masks = CASES.index((substitution, site, p)) % 2 == 1
    tips, weights, parent_ids, lengths = unrooted_case(masks=masks, seed=3 + len(site))
    params = params_for(substitution, site, p, 2, seed=int(p * 100) + len(substitution))
    engine = engine_for(substitution, site, tips, weights, masks)
    assert engine.param_count == params.shape[1]
    blocks = engine.param_block_map(params)
    assert np.array_equal(blocks["proportion invariant"][:, 0], params[:, -1])
    refs = unrooted_references(substitution, site, tips, weights, parent_ids, lengths, params, masks)
    batch = sbn.TreeBatch(parent_ids, lengths)
    for rescaling in (False, True):
        check(engine.gradients(batch, params, rescaling), refs)
        logl = engine.log_likelihoods(batch, params, rescaling)
        np.testing.assert_allclose(logl, [r[0] for r in refs], rtol=LOGL_RTOL)
    if substitution != "JC69":
        engine.set_substitution_gradient("fd")
        check(engine.gradients(batch, params, True), refs, fd=True)


@pytest.mark.parametrize("substitution,site", MODELS[4:])
def test_more_models(substitution, site):
    tips, weights, parent_ids, lengths = unrooted_case(masks=True, seed=8)
    params = params_for(substitution, site, 0.3, 2, seed=9)
    engine = engine_for(substitution, site, tips, weights, True)
    refs = unrooted_references(substitution, site, tips, weights, parent_ids, lengths, params, True)
    check(engine.gradients(sbn.TreeBatch(parent_ids, lengths), params, True), refs)


def rooted_refs(substitution, site, tips, weights, batch, params, masks):
    out = []
    for t in range(len(params)):
        logl, jacobian, want = inv.InvariantTimeTree(substitution, site, tips, weights, batch, t, params[t],
                                                     masks).gradient()
        out.append((logl, want, jacobian))
    return out


ROOTED = [("GTR", "weibull+4+I", 0.3, False), ("HKY", "constant+I", 0.5, True), ("JC69", "weibull+20+I", 0.05, True),
          ("GTR", "gamma+4+I", 0.95, False), ("HKY", "weibull+4+I", 0.0, True)]


@pytest.mark.parametrize("substitution,site,p,relaxed", ROOTED)
def test_rooted_against_the_reference(substitution, site, p, relaxed):
    masks = relaxed
    tips, weights = invariant_alignment(21, 509, seed=5, masks=masks)
    batch = trees.random_time_trees(21, 3, seed=7, relaxed=relaxed)
    params = params_for(substitution, site, p, 3, seed=8, clock=True)
    engine = engine_for(substitution, site, tips, weights, masks, clock="strict")
    refs = rooted_refs(substitution, site, tips, weights, batch, params, masks)
    for rescaling in (False, True):
        check(engine.gradients(sbn.TreeBatch(**batch), params, rescaling, rooted=True),
              [(logl, want) for logl, want, _ in refs])
    got = engine.log_likelihoods(sbn.TreeBatch(**batch), params, True, rooted=True)
    np.testing.assert_allclose(got, [logl + jacobian for logl, _, jacobian in refs], rtol=LOGL_RTOL)


def compare_plain(a, b, report):
    bitwise = a.log_likelihood == b.log_likelihood
    assert abs(a.log_likelihood - b.log_likelihood) <= 1e-12 * abs(b.log_likelihood)
    for key, value in b.gradient.items():
        got = a.gradient[key][:len(value)] if key == "site_model" else a.gradient[key]
        bitwise = bitwise and np.array_equal(got, value)
        assert np.max(np.abs(got - value)) <= 1e-12 * max(np.max(np.abs(value)), 1e-300), key
    report.append(bitwise)


@pytest.mark.parametrize("substitution,site", [("GTR", "weibull+4"), ("HKY", "constant"), ("JC69", "weibull+20")])
def test_p_zero_matches_the_plain_spec(substitution, site, capsys):
    tips, weights, parent_ids, lengths = unrooted_case(seed=12)
    params = params_for(substitution, site + "+I", 0.0, 2, seed=13)
    engine = engine_for(substitution, site + "+I", tips, weights, False)
    plain = engine_for(substitution, site, tips, weights, False)
    batch = sbn.TreeBatch(parent_ids, lengths)
    report = []
    for rescaling in (False, True):
        for a, b in zip(engine.gradients(batch, params, rescaling), plain.gradients(batch, params[:, :-1], rescaling)):
            compare_plain(a, b, report)
        np.testing.assert_allclose(engine.log_likelihoods(batch, params, rescaling),
                                   plain.log_likelihoods(batch, params[:, :-1], rescaling), rtol=1e-12)
    time_batch = trees.random_time_trees(21, 2, seed=14)
    clock_params = np.hstack([params, np.zeros((2, 1))])
    rooted = engine_for(substitution, site + "+I", tips, weights, False, clock="strict")
    rooted_plain = engine_for(substitution, site, tips, weights, False, clock="strict")
    for a, b in zip(rooted.gradients(sbn.TreeBatch(**time_batch), clock_params, True, rooted=True),
                    rooted_plain.gradients(sbn.TreeBatch(**time_batch), np.delete(clock_params, -2, axis=1), True,
                                           rooted=True)):
        compare_plain(a, b, report)
    with capsys.disabled():
        print(f"\n{substitution} {site}+I at p = 0: bitwise equal to {site} in {sum(report)} of {len(report)} trees")


@pytest.mark.parametrize("constant_fraction", [0.0, 0.9])
def test_no_constant_pattern_and_mostly_constant(constant_fraction):
    rng = np.random.default_rng(2)
    tips, _ = trees.random_alignment(21, 509, seed=21, gap_fraction=0.0)
    tips = tips.copy()
    if constant_fraction == 0.0:
        tips[0] = (tips[1] + 1) % 4  # no column has one state in every tip
    else:
        constant = rng.random(509) < constant_fraction
        tips[:, constant] = rng.integers(0, 4, size=509)[constant]
    weights = rng.integers(1, 4, size=509).astype(np.float64)
    parent_ids, lengths = trees.random_tree_batch(21, 2, seed=22, rooted=True)
    lengths = slid(lengths, parent_ids)
    params = params_for("GTR", "weibull+4+I", 0.4, 2, seed=23)
    engine = engine_for("GTR", "weibull+4+I", tips, weights, False)
    refs = unrooted_references("GTR", "weibull+4+I", tips, weights, parent_ids, lengths, params, False)
    check(engine.gradients(sbn.TreeBatch(parent_ids, lengths), params, True), refs)


def test_thousand_taxa_rescaled():
    """1000 taxa, p = 0.3, rescaling: finite, and logL and directional derivatives (edges,
    shape, p, substitution coordinates at once) match the reference."""
    taxa, patterns = 1000, 64
    tips, weights = invariant_alignment(taxa, patterns, seed=31, constant_fraction=0.5)
    parent_ids, lengths = trees.random_tree_batch(taxa, 1, seed=32, rooted=True)
    lengths = slid(lengths, parent_ids)
    params = params_for("GTR", "weibull+4+I", 0.3, 1, seed=33)
    engine = engine_for("GTR", "weibull+4+I", tips, weights, False)
    got = engine.gradients(sbn.TreeBatch(parent_ids, lengths), params, True)[0]
    for value in [got.log_likelihood] + list(got.gradient.values()):
        assert np.all(np.isfinite(value))
    model = inv.Model("GTR", "weibull+4+I", params[0])
    edges = 2 * taxa - 2
    rng = np.random.default_rng(34)
    directions = rng.normal(size=(3, edges + 2 + 8))
    # (no direction along the fixed node's edge, whose entry the engine zeroes)
    fixed = np.flatnonzero(got.gradient["branch_lengths"] == 0.0)
    directions[:, fixed[fixed < edges]] = 0.0
    stepped = np.broadcast_to(lengths[0], (3, edges + 1)).astype(np.complex128)
    stepped[:, :edges] += 1j * inv.STEP * directions[:, :edges]
    total = model.evaluate(tips, weights, parent_ids[0], stepped, directions[:, edges:edges + 2],
                           directions[:, edges + 2:], False)
    assert abs(got.log_likelihood - total[0].real) <= LOGL_RTOL * abs(total[0].real)
    flat = np.concatenate([got.gradient["branch_lengths"][:edges], got.gradient["site_model"],
                           got.gradient["substitution_model"]])
    want = total.imag / inv.STEP
    np.testing.assert_allclose(directions @ flat, want, rtol=1e-8)


def test_graph_replay():
    """The same topologies four times (the fourth and later calls replay a CUDA graph) with new
    lengths and parameters each time."""
    tips, weights, parent_ids, lengths = unrooted_case(seed=41)
    engine = engine_for("HKY", "gamma+4+I", tips, weights, False)
    for call in range(5):
        params = params_for("HKY", "gamma+4+I", [0.1, 0.6, 0.0, 0.3, 0.9][call], 2, seed=42 + call)
        scaled = lengths * (1.0 + 0.1 * call)
        got = engine.gradients(sbn.TreeBatch(parent_ids, scaled), params, True)
        if call in (0, 4):
            check(got, unrooted_references("HKY", "gamma+4+I", tips, weights, parent_ids, scaled, params, False))


def stack(results, key):
    return np.array([g.gradient[key] for g in results])


def assert_same(got, want, rtol=1e-12):
    np.testing.assert_allclose([g.log_likelihood for g in got], [g.log_likelihood for g in want], rtol=rtol)
    for key in want[0].gradient:
        a, b = stack(got, key), stack(want, key)
        assert np.max(np.abs(a - b)) <= rtol * np.max(np.abs(b)), key


@pytest.mark.parametrize("axis", ["trees", "patterns"])
@pytest.mark.parametrize("rooted", [False, True])
def test_device_groups(axis, rooted):
    tips, weights, parent_ids, lengths = unrooted_case(trees_=5, seed=51)
    site, substitution = "weibull+4+I", "GTR"
    if rooted:
        batch = sbn.TreeBatch(**trees.random_time_trees(21, 5, seed=52))
        params = params_for(substitution, site, 0.25, 5, seed=53, clock=True)
        clock = "strict"
    else:
        batch = sbn.TreeBatch(parent_ids, lengths)
        params = params_for(substitution, site, 0.25, 5, seed=53)
        clock = "none"
    single = engine_for(substitution, site, tips, weights, False, clock=clock)
    group = engine_for(substitution, site, tips, weights, False, clock=clock, devices=[0, 0], shard_axis=axis)
    want = single.gradients(batch, params, True, rooted=rooted)
    assert_same(group.gradients(batch, params, True, rooted=rooted), want)
    np.testing.assert_allclose(group.log_likelihoods(batch, params, True, rooted=rooted),
                               single.log_likelihoods(batch, params, True, rooted=rooted), rtol=1e-12)


@pytest.mark.parametrize("rooted", [False, True])
def test_staged_pattern_ranges_finished_on_the_host(rooted):
    tips, weights, parent_ids, lengths = unrooted_case(trees_=3, patterns=3001, seed=61)
    substitution, site = "HKY", "weibull+4+I"
    if rooted:
        batch = sbn.TreeBatch(**trees.random_time_trees(21, 3, seed=62, relaxed=True))
        params = params_for(substitution, site, 0.2, 3, seed=63, clock=True)
    else:
        batch = sbn.TreeBatch(parent_ids, lengths)
        params = params_for(substitution, site, 0.2, 3, seed=63)
    engine = engine_for(substitution, site, tips, weights, False, clock="strict" if rooted else "none")
    want = engine.gradients(batch, params, True, rooted=rooted)
    total = None
    for begin, end in [(0, 1234), (1234, 3001)]:
        engine.set_pattern_range(begin, end)
        staged = engine.stage(batch, params, rooted=rooted, substitution_analytic=True)
        staged.run(sbn._capi.MODE_BRANCH_GRADIENT, True)
        parts = list(staged.fetch(gradients=True)) + [staged.fetch_substitution_sums(), staged.fetch_invariant_sums()]
        staged.close()
        total = parts if total is None else [a + b for a, b in zip(total, parts)]
    engine.set_pattern_range(0, engine.pattern_count)
    logl, grad, rgrad, subst, invs = total
    got = sharding.finish_gradients_invariant(engine.specification, 21, batch, rooted, params, logl, grad, rgrad, subst,
                                              invs, engine.category_count, engine.site_gradient_size)
    assert_same(got, want, 1e-11)


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _pattern_worker(rank, world, port, result_path):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        tips, weights, parent_ids, lengths = unrooted_case(trees_=3, seed=71)
        params = params_for("GTR", "gamma+4+I", 0.35, 3, seed=72)
        spec = sbn.PhyloModelSpecification("GTR", "gamma+4+I", "none")
        engine = sharding.PatternShardedEngine(spec, tips, weights, device=0)
        got = engine.gradients(sbn.TreeBatch(parent_ids, lengths), params, rescaling=True)
        if rank == 0:
            np.savez(result_path, logl=[g.log_likelihood for g in got],
                     **{k: stack(got, k) for k in got[0].gradient})
    finally:
        dist.destroy_process_group()


def test_pattern_sharded_engine_host_all_reduce(tmp_path):
    import torch.multiprocessing as mp
    result = str(tmp_path / "sharded.npz")
    mp.spawn(_pattern_worker, args=(2, free_port(), result), nprocs=2, join=True)
    tips, weights, parent_ids, lengths = unrooted_case(trees_=3, seed=71)
    params = params_for("GTR", "gamma+4+I", 0.35, 3, seed=72)
    want = engine_for("GTR", "gamma+4+I", tips, weights, False).gradients(sbn.TreeBatch(parent_ids, lengths), params,
                                                                          True)
    got = np.load(result)
    np.testing.assert_allclose(got["logl"], [g.log_likelihood for g in want], rtol=1e-12)
    for key in want[0].gradient:
        b = stack(want, key)
        assert np.max(np.abs(got[key] - b)) <= 1e-11 * np.max(np.abs(b)), key
