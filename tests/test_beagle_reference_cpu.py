"""The exact reference of tests/beagle_reference.py pinned on the CPU: against a 50-digit pruning
differentiated by central differences (mpmath), and the CPU restatement of the BEAGLE-compatible
library (oracle/beagle_cpu.cpp) against the reference at every category count the device library
has a kernel variant for, with unequal category weights, a zero-rate and a zero-weight category,
tip partials, nucleotide masks, extreme branches, instance reuse and an op that writes the
cumulative scale buffer.
"""
import os

import mpmath
import numpy as np
import pytest

from conftest import ROOT
import beagle_reference as br
from libsbn_b200.beagle import gtr_eigensystem

ORACLE = os.path.join(ROOT, "oracle", "_build", "libbeagle_oracle.so")
CATEGORIES = [1, 2, 3, 4, 5, 7, 8, 9, 12, 15, 16, 17, 33]
DIGITS = 50
DIFFERENCE_STEP = mpmath.mpf("1e-20")


def mp_site_log_likelihoods(q, freqs, rates, category_weights, tips, parents, lengths, masks):
    """[P] per-pattern log likelihoods, every step at DIGITS digits (lengths may be mpf)."""
    n = len(tips)
    node_count = len(parents) + 1
    children = [[] for _ in range(node_count)]
    for child, parent in enumerate(parents):
        children[parent].append(child)
    q = mpmath.matrix([[mpmath.mpf(float(x)) for x in row] for row in q])
    matrices = [[mpmath.expm(q * (mpmath.mpf(lengths[e]) * mpmath.mpf(float(r)))) for r in rates]
                for e in range(node_count - 1)]
    out = []
    for p in range(len(tips[0])):
        site = mpmath.mpf(0)
        for c in range(len(rates)):
            partial = {}
            for leaf in range(n):
                s = int(tips[leaf][p])
                partial[leaf] = ([mpmath.mpf((s >> i) & 1) for i in range(4)] if masks else
                                 [mpmath.mpf(1) if s >= 4 or s == i else mpmath.mpf(0) for i in range(4)])
            for node in range(n, node_count):
                vector = [mpmath.mpf(1)] * 4
                for child in children[node]:
                    m = matrices[child][c]
                    vector = [vector[i] * sum(m[i, s] * partial[child][s] for s in range(4)) for i in range(4)]
                partial[node] = vector
            site += mpmath.mpf(float(category_weights[c])) * sum(
                mpmath.mpf(float(freqs[i])) * partial[node_count - 1][i] for i in range(4))
        out.append(mpmath.log(site))
    return out


@pytest.mark.parametrize("categories,masks", [(1, False), (5, True), (16, False)])
def test_reference_against_50_digit_central_differences(categories, masks):
    """6 taxa, Dirichlet category weights, category 0 at rate 0 (more than one category), a 1e-12
    branch: logL, sums, squares and per-site derivatives to 1e-12."""
    case = br.random_case(6, 5, categories, 60 + categories, "libsbn", masks=masks)
    if categories > 1:
        case["rates"][0] = 0.0
    case["lengths"][1] = 1e-12
    logl, sums, squares, per_site = br.reference(case)
    _, _, _, freqs, q = gtr_eigensystem()
    parents = br.parent_ids(case["post"], case["n"])
    weights = [mpmath.mpf(float(w)) for w in case["weights"]]
    with mpmath.workdps(DIGITS):
        def sites(lengths):
            return mp_site_log_likelihoods(q, freqs, case["rates"], case["category_weights"], case["states"],
                                           parents, lengths, masks)
        base = [mpmath.mpf(float(t)) for t in case["lengths"]]
        want_logl = float(sum(w * s for w, s in zip(weights, sites(base))))
        want = []
        for e in range(len(parents)):
            up, down = list(base), list(base)
            up[e] += DIFFERENCE_STEP
            down[e] -= DIFFERENCE_STEP
            want.append([float((a - b) / (2 * DIFFERENCE_STEP)) for a, b in zip(sites(up), sites(down))])
    want = np.array(want)
    assert abs(logl - want_logl) <= 1e-12 * abs(want_logl)
    assert np.max(np.abs(per_site - want)) <= 1e-12 * np.max(np.abs(want))
    np.testing.assert_allclose(sums, want @ case["weights"], rtol=0, atol=1e-12 * np.max(np.abs(want @ case["weights"])))
    np.testing.assert_allclose(squares, (want * want) @ case["weights"], rtol=1e-12)


@pytest.mark.parametrize("categories", CATEGORIES)
def test_cpu_restatement_against_the_reference(categories):
    """Every category count of the device library's kernel table, the three op orders in turn, tip
    states, Dirichlet category weights, every edge."""
    order = ("libsbn", "node_id", "depth_first")[CATEGORIES.index(categories) % 3]
    case = br.random_case(14, 37, categories, 70 + categories, order)
    br.assert_matches(br.run_library(ORACLE, case), br.reference(case))


@pytest.mark.parametrize("variant,categories", [("zero_rate_and_weight", 5), ("zero_rate_and_weight", 16),
                                                ("tip_partials", 5), ("tip_partials", 16), ("masks", 9),
                                                ("extreme_branches", 4), ("extreme_branches", 16)])
def test_cpu_restatement_model_and_input_edges(variant, categories):
    case = br.random_case(14, 37, categories, 80 + categories, "libsbn", use_tip_states=variant != "tip_partials",
                          masks=variant == "masks")
    saturated = None
    if variant == "zero_rate_and_weight":
        case = br.zero_rate_and_zero_weight(case)
    if variant == "extreme_branches":
        case, saturated = br.extreme_branches(case)
    br.assert_matches(br.run_library(ORACLE, case), br.reference(case), saturated=saturated)


@pytest.mark.parametrize("categories", [5, 17])
def test_cpu_restatement_instance_reuse(categories):
    case = br.random_case(14, 37, categories, 90 + categories, "node_id")
    beagle = br.open_library(ORACLE, case)
    try:
        for case in br.reuse_sequence(beagle, case):
            br.assert_matches(br.evaluate(beagle, case), br.reference(case))
    finally:
        beagle.close()


@pytest.mark.parametrize("categories", [8, 16])
def test_cpu_restatement_first_op_writes_the_cumulative_buffer(categories):
    case = br.random_case(14, 37, categories, 100 + categories, "depth_first")
    assert br.root_log_likelihood_first_op_writes_cumulative(ORACLE, case) == pytest.approx(
        br.expected_first_op_writes_cumulative(case), rel=1e-10, abs=0)
