"""The BEAGLE-compatible device library (libsbn_b200/csrc/beagle_shim.cu) against the exact reference
of tests/beagle_reference.py, through FatBeagle's call sequence with rescaling on: logL to 1e-10,
sums to 1e-9 of the largest, per-site derivatives to 1e-9 of each edge's largest entry, squares to
1e-9.

UpdatePartials picks an UpdatePartialsPipelinedKernel<PRE, CT, K, PADDED> instantiation from the
category count (CT lanes per pattern, the next power of two up to 16; PADDED when C < CT) or the
generic kernel above 16 categories.  The cases reach every one of them:
  * categories 1-5, 7-9, 12, 15-17 and 33: every CT, padded and not, and the generic kernel on both
    sides of the 16 categories EdgeDerivativesKernel stages in shared memory;
  * 40 taxa (39 ops, a multiple of no CT > 1, more than one staged chunk of 32, 16 or 8 ops, so the
    last group of logarithms is partly filled) and 301 patterns (a ragged last warp group and CTA
    at every CT), in libsbn's order, in node-id order and reordered depth first;
  * two patterns per thread (SBNB_BEAGLE_PATTERNS_PER_THREAD=2) on an odd pattern count;
  * a zero-rate and a zero-weight category, tip partials, nucleotide masks, a 1e-12 and a
    20-substitution branch;
  * 1000-taxon random and ladder trees (they underflow without rescaling), 40 003 patterns (the root
    and edge-derivative grids stride), one instance evaluated three times, and an op that writes the
    cumulative scale buffer itself.
The reference is the expensive side; each is computed once per module.
"""
import numpy as np
import pytest

import beagle_reference as br
from libsbn_b200.beagle import LIB_PATH as SHIM, random_tree_operations

pytestmark = pytest.mark.gpu

CATEGORIES = [1, 2, 3, 4, 5, 7, 8, 9, 12, 15, 16, 17, 33]
TAXA, PATTERNS = 40, 301


@pytest.fixture(scope="module")
def reference():
    """The reference of a case, computed once per key."""
    cache = {}

    def get(key, case, edges=None):
        if key not in cache:
            cache[key] = br.reference(case, edges)
        return cache[key]
    return get


def lanes(categories):
    return 1 << (categories - 1).bit_length()


@pytest.mark.parametrize("order", ["libsbn", "node_id", "depth_first"])
@pytest.mark.parametrize("categories", CATEGORIES)
def test_every_kernel_instantiation(categories, order, reference):
    case = br.random_case(TAXA, PATTERNS, categories, 1000 + categories, order)
    ops = len(case["post"])
    if categories <= 16:
        ct = lanes(categories)
        chunk = 32 if ct <= 4 else 16 if ct == 8 else 8
        warp_group, cta = 32 // ct, 8 * 32 // ct
        assert ops > chunk and (ct == 1 or ops % ct) and PATTERNS % warp_group and PATTERNS % cta
        assert PATTERNS > cta
    # (depth-first order is node_id's tree, ops reordered: the same reference)
    want = reference((categories, "libsbn" if order == "libsbn" else "node_id"), case)
    br.assert_matches(br.run_library(SHIM, case), want)


@pytest.mark.parametrize("categories", [1, 2, 4, 8, 16])
def test_two_patterns_per_thread(categories, monkeypatch):
    """K = 2 against the reference, and against K = 1 on the same instance: every pattern sees the
    same operations in the same order, so the bits are the same."""
    case = br.random_case(TAXA, 517, categories, 1100 + categories, "depth_first")
    beagle = br.open_library(SHIM, case)
    try:
        monkeypatch.setenv("SBNB_BEAGLE_PATTERNS_PER_THREAD", "2")
        two = br.evaluate(beagle, case)
        monkeypatch.delenv("SBNB_BEAGLE_PATTERNS_PER_THREAD")
        one = br.evaluate(beagle, case)
    finally:
        beagle.close()
    br.assert_matches(two, br.reference(case))
    assert two[0] == one[0]
    for a, b in zip(two[1:], one[1:]):
        np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("variant,categories", [("zero_rate_and_weight", 5), ("zero_rate_and_weight", 16),
                                                ("tip_partials", 5), ("tip_partials", 16), ("masks", 9),
                                                ("extreme_branches", 4), ("extreme_branches", 16)])
def test_model_and_input_edges(variant, categories):
    case = br.random_case(TAXA, PATTERNS, categories, 1200 + categories, "libsbn",
                          use_tip_states=variant != "tip_partials", masks=variant == "masks")
    saturated = None
    if variant == "zero_rate_and_weight":
        case = br.zero_rate_and_zero_weight(case)
    if variant == "extreme_branches":
        case, saturated = br.extreme_branches(case)
    br.assert_matches(br.run_library(SHIM, case), br.reference(case), saturated=saturated)


class _Ladder:
    """Stands in for the generator of random_tree_operations: always joins the last two roots, the
    newest subtree with the next taxon (a caterpillar, n - 1 ops deep)."""

    def integers(self, count):
        return count - 1


def sampled_edges(case, count, seed):
    """`count` edges, always both root children, the rest drawn."""
    root_children = [int(case["post"][-1][3]), int(case["post"][-1][5])]
    others = np.setdiff1d(np.arange(2 * case["n"] - 2), root_children)
    drawn = np.random.default_rng(seed).choice(others, count - 2, replace=False)
    return np.array(root_children + sorted(int(e) for e in drawn))


@pytest.mark.parametrize("categories", [4, 16])
@pytest.mark.parametrize("shape", ["random", "ladder"])
def test_deep_trees_rescaled(shape, categories):
    """1000 taxa, 501 patterns: the site likelihoods underflow fp64 many times over, so logL rests on
    the cumulative scale sums matching the reference's per-node log scale."""
    case = br.random_case(1000, 501, categories, 1300 + categories, "libsbn")
    if shape == "ladder":
        case["post"], case["pre"] = random_tree_operations(1000, _Ladder(), True)
    edges = sampled_edges(case, 8, categories)
    want = br.reference(case, edges)
    assert want[0] < -745.0 * np.sum(case["weights"])  # (each site likelihood below fp64's smallest)
    br.assert_matches(br.run_library(SHIM, case), want, edges)


@pytest.mark.parametrize("categories", [5, 16])
def test_wide_pattern_counts(categories):
    """40 003 patterns: more than the root kernel's 256 x 128 and the edge-derivative kernel's
    64 x 128 threads, so both go round their grid-stride loops."""
    case = br.random_case(30, 40003, categories, 1400 + categories, "libsbn")
    edges = sampled_edges(case, 4, categories)
    br.assert_matches(br.run_library(SHIM, case), br.reference(case, edges), edges)


@pytest.mark.parametrize("categories", [5, 17])
def test_instance_reuse(categories):
    """One instance, three evaluations (lengths, then category rates and weights change): each
    matches the reference of its own parameters."""
    case = br.random_case(TAXA, PATTERNS, categories, 1500 + categories, "node_id")
    beagle = br.open_library(SHIM, case)
    try:
        for step in br.reuse_sequence(beagle, case):
            br.assert_matches(br.evaluate(beagle, step), br.reference(step))
    finally:
        beagle.close()


@pytest.mark.parametrize("categories", [8, 16])
def test_op_that_writes_the_cumulative_buffer(categories):
    """The cumulative sums go through memory instead of registers (the first op's scale buffer is the
    cumulative buffer)."""
    case = br.random_case(TAXA, PATTERNS, categories, 1600 + categories, "depth_first")
    got = br.root_log_likelihood_first_op_writes_cumulative(SHIM, case)
    want = br.expected_first_op_writes_cumulative(case)
    assert abs(got - want) <= 1e-10 * abs(want)
