"""TEST INFRASTRUCTURE: an exact reference for the BEAGLE call sequence of libsbn_b200/beagle.py
(FatBeagle's log likelihood and branch gradient, fat_beagle.cpp:119-175).

The pruning is subst_reference.prune: complex128, every transition matrix scipy.linalg.expm(Q r_c t),
a real per-node rescaling.  It shares no formula with a BEAGLE implementation: no eigensystem, no
pre-order partials, no pre^T dQ post.  The derivative of the log likelihood of pattern k along edge e
is the complex step Im logL_k(t + i h e_e) / h (h = 1e-30) -- exact to fp64 rounding, nothing is
subtracted.  The edges are batched on prune's leading axis, and prune's pattern weights are the
identity so that it returns every pattern's log likelihood; BEAGLE's sums and sums of squares are
then g @ w and g^2 @ w.

The tree is the one the op lists describe, rooted where they root it: the library reports each root
child's edge on its own, so there is no root slide to repeat.  Q, the frequencies, the category
rates and the category weights are taken as the test hands them to the library.
"""
import ctypes

import numpy as np
import scipy.linalg

import subst_reference
from libsbn_b200.beagle import Beagle, depth_first_operations, gtr_eigensystem, random_tree_operations

STEP = subst_reference.STEP
# complex entries of one batched partial (J x C x patterns x 4): bounds prune's memory
_ENTRIES = 1 << 22
_PATTERNS = 1024  # patterns per prune call (the identity weights are patterns^2)


def parent_ids(post, n):
    """Parent of every node but the root, from a post-order op list (children below parents)."""
    parents = np.full(2 * n - 2, -1, dtype=np.int64)
    for op in post:
        parents[op[3]] = parents[op[5]] = op[0]
    assert np.all(parents >= 0)
    return parents


def log_likelihood_and_gradient(q, freqs, rates, category_weights, tips, weights, post, lengths, edges=None,
                                masks=False):
    """(logL, sums [E], squares [E], per-site derivatives [E][P]) over the edges `edges` (node ids;
    default: every edge), in that order.

    tips: [taxon][pattern] states (>= 4 missing) or, with masks, nucleotide masks; lengths: [nodes]
    indexed by node id (the library's matrix index)."""
    n, P = np.asarray(tips).shape
    parents = parent_ids(post, n)
    edges = np.arange(2 * n - 2) if edges is None else np.asarray(edges)
    lengths = np.asarray(lengths, dtype=np.float64)[:2 * n - 1]
    C = len(rates)
    weights = np.asarray(weights, dtype=np.float64)
    rows = [-1] + [int(e) for e in edges]  # -1: the unstepped evaluation
    per_row = max(1, _ENTRIES // (C * 4 * min(P, _PATTERNS)))
    site = np.zeros((len(rows), P), dtype=np.complex128)
    for r0 in range(0, len(rows), per_row):
        group = rows[r0:r0 + per_row]
        stepped = np.tile(lengths.astype(np.complex128), (len(group), 1))
        for j, e in enumerate(group):
            if e >= 0:
                stepped[j, e] += 1j * STEP
        qs = np.broadcast_to(np.asarray(q, dtype=np.complex128), (len(group), 4, 4))
        pis = np.broadcast_to(np.asarray(freqs, dtype=np.complex128), (len(group), 4))
        for p0 in range(0, P, _PATTERNS):
            p1 = min(P, p0 + _PATTERNS)
            site[r0:r0 + len(group), p0:p1] = subst_reference.prune(
                qs, pis, np.asarray(rates, dtype=np.float64), np.asarray(category_weights, dtype=np.float64),
                np.asarray(tips)[:, p0:p1], np.eye(p1 - p0), parents, stepped, masks)
    logl = float(site[0].real @ weights)
    g = site[1:].imag / STEP
    return logl, g @ weights, (g * g) @ weights, g


def first_op_scale(q, rates, tips, post, lengths):
    """[P] the largest entry, over categories and states, of the first op's product (P1 L1) o (P2 L2):
    what a rescaled first op stores in its scale buffer.  The first op of a post-order list has two
    tips below it (compact states, >= 4 missing)."""
    op = post[0]
    product = 1.0
    for child in (op[3], op[5]):
        states = np.asarray(tips[child]).astype(np.int64)
        columns = []
        for r in rates:
            m = scipy.linalg.expm(np.asarray(q) * (lengths[child] * r))
            columns.append(np.where(states[:, None] >= 4, 1.0, m[:, np.minimum(states, 3)].T))
        product = product * np.array(columns)  # [C][P][4]
    return product.max(axis=(0, 2))


def random_case(n, P, C, seed, order="libsbn", use_tip_states=True, masks=False, rescaling=True):
    """A seeded BEAGLE call sequence: a random rooted tree as op lists in `order` ("libsbn", "node_id",
    or "depth_first": node_id's post-order list reordered depth first), tips with 5 % missing states
    (or nucleotide masks, a fifth of them ambiguous), Dirichlet category weights and sorted Gamma
    category rates."""
    rng = np.random.default_rng(seed)
    if masks:
        states = (1 << rng.integers(0, 4, size=(n, P))).astype(np.int32)
        ambiguous = rng.random(states.shape) < 0.2
        states[ambiguous] = rng.integers(1, 16, size=int(ambiguous.sum()))
    else:
        states = rng.integers(0, 4, size=(n, P)).astype(np.int32)
        states[rng.random(states.shape) < 0.05] = 4
    post, pre = random_tree_operations(n, rng, rescaling, "node_id" if order == "depth_first" else order)
    if order == "depth_first":
        post = depth_first_operations(post, n)
    rates = np.sort(rng.gamma(2.0, 0.5, size=C))
    return dict(n=n, P=P, C=C, states=states, weights=rng.integers(1, 6, size=P).astype(np.float64),
                post=post, pre=pre, lengths=rng.exponential(0.1, size=2 * n - 1), rates=rates / rates.mean(),
                category_weights=rng.dirichlet(np.ones(C)), use_tip_states=use_tip_states and not masks,
                masks=masks, rescaling=rescaling)


def open_library(path, case):
    """A Beagle instance over the library at `path` (None: the device library) with the case's tips
    and model."""
    evec, ivec, evals, freqs, _ = gtr_eigensystem()
    beagle = Beagle(path, case["n"], case["P"], case["C"], case["use_tip_states"])
    beagle.set_tips(case["states"], case["weights"], case["use_tip_states"], case["masks"])
    beagle.set_model(evec, ivec, evals, freqs, case["rates"], case["category_weights"])
    return beagle


def evaluate(beagle, case):
    """The library's (logL, sums, squares, per-site derivatives) of the case."""
    _, _, _, freqs, q = gtr_eigensystem()
    return beagle.log_likelihood_and_gradient(case["post"], case["pre"], case["lengths"], q, case["rates"], freqs,
                                              case["rescaling"])


def run_library(path, case):
    beagle = open_library(path, case)
    try:
        return evaluate(beagle, case)
    finally:
        beagle.close()


def reuse_sequence(beagle, case):
    """Three evaluations on one instance, yielding each one's case once the instance is set for it:
    the case itself, new branch lengths, then new category rates and weights through
    beagleSetCategoryRates / beagleSetCategoryWeights (the evaluation's beagleUpdateTransitionMatrices
    recomputes the matrices from them)."""
    yield case
    rng = np.random.default_rng(case["C"])
    case = dict(case, lengths=rng.exponential(0.1, size=len(case["lengths"])))
    yield case
    rates = np.sort(rng.gamma(2.0, 0.5, size=case["C"]))
    case = dict(case, rates=rates / rates.mean(), category_weights=rng.dirichlet(np.ones(case["C"])))
    keep_r, rates_ptr = beagle._d(case["rates"])
    keep_w, weights_ptr = beagle._d(case["category_weights"])
    beagle.ok(beagle.lib.beagleSetCategoryRates(beagle.handle, rates_ptr))
    beagle.ok(beagle.lib.beagleSetCategoryWeights(beagle.handle, 0, weights_ptr))
    yield case


def root_log_likelihood_first_op_writes_cumulative(path, case):
    """The root logL of the case's post-order list after its first op is made to write its scale
    factors into the cumulative buffer (0) itself, so that the library cannot keep the cumulative sums
    of the call in registers and adds them up in memory, op by op."""
    n, N = case["n"], 2 * case["n"] - 1
    post = case["post"].copy()
    post[0][1] = 0
    beagle = open_library(path, case)
    try:
        keep_i, idx = beagle._i(np.arange(N - 1))
        keep_l, lens = beagle._d(case["lengths"][:N - 1])
        beagle.ok(beagle.lib.beagleUpdateTransitionMatrices(beagle.handle, 0, idx, None, None, lens, N - 1))
        beagle.ok(beagle.lib.beagleResetScaleFactors(beagle.handle, 0))
        keep_a, ops = beagle._i(post)
        beagle.ok(beagle.lib.beagleUpdatePartials(beagle.handle, ops, len(post), 0))
        keep_r, root = beagle._i([N - 1])
        keep_z, zero = beagle._i([0])
        logl = ctypes.c_double()
        beagle.ok(beagle.lib.beagleCalculateRootLogLikelihoods(beagle.handle, root, zero, zero, zero, 1,
                                                               ctypes.byref(logl)))
        return logl.value
    finally:
        beagle.close()


def expected_first_op_writes_cumulative(case):
    """What root_log_likelihood_first_op_writes_cumulative returns in BEAGLE's semantics: the first op
    stores its raw maxima m_k in the cumulative buffer and then, like every rescaled op, adds log m_k,
    so the buffer ends at m_k + sum_o log m_o,k and the root logL is the reference's + sum_k w_k m_k."""
    _, _, _, freqs, q = gtr_eigensystem()
    logl = log_likelihood_and_gradient(q, freqs, case["rates"], case["category_weights"], case["states"],
                                       case["weights"], case["post"], case["lengths"], [], case["masks"])[0]
    return logl + first_op_scale(q, case["rates"], case["states"], case["post"], case["lengths"]) @ case["weights"]


def reference(case, edges=None):
    """The reference's (logL, sums, squares, per-site derivatives) of the case over `edges`."""
    _, _, _, freqs, q = gtr_eigensystem()
    return log_likelihood_and_gradient(q, freqs, case["rates"], case["category_weights"], case["states"],
                                       case["weights"], case["post"], case["lengths"], edges, case["masks"])


def assert_matches(got, want, edges=None, logl_only=False, saturated=None):
    """A library's result against the reference's over `edges` (default: every edge): logL to 1e-10
    relative, sums to 1e-9 of the largest, per-site derivatives to 1e-9 of each edge's largest entry,
    squares to 1e-9 relative.  The per-site derivatives of the edge `saturated` (extreme_branches'
    long branch) are held to 1e-12 absolute instead, and its squares are not compared."""
    logl, sums, squares, per_site = got
    assert abs(logl - want[0]) <= 1e-10 * abs(want[0]), (logl, want[0])
    if logl_only:
        return
    edges = np.arange(len(sums)) if edges is None else np.asarray(edges)
    ref_sums, ref_squares, ref_per_site = want[1:]
    error = np.abs(sums[edges] - ref_sums)
    assert np.max(error) <= 1e-9 * np.max(np.abs(ref_sums)), (edges[np.argmax(error)], np.max(error))
    if saturated is not None:
        at = int(np.flatnonzero(edges == saturated)[0])
        assert np.max(np.abs(per_site[saturated] - ref_per_site[at])) <= 1e-12
        keep = edges != saturated
        edges, ref_squares, ref_per_site = edges[keep], ref_squares[keep], ref_per_site[keep]
    error = np.max(np.abs(per_site[edges] - ref_per_site), axis=1) / np.max(np.abs(ref_per_site), axis=1)
    assert np.max(error) <= 1e-9, (edges[np.argmax(error)], np.max(error))
    error = np.abs(squares[edges] - ref_squares) / np.abs(ref_squares)
    assert np.max(error) <= 1e-9, (edges[np.argmax(error)], np.max(error))


def zero_rate_and_zero_weight(case):
    """Category 0 at rate 0 (identity transition matrices) keeping its weight, the last category at
    weight 0."""
    case = dict(case, rates=case["rates"].copy(), category_weights=case["category_weights"].copy())
    case["rates"][0] = 0.0
    case["category_weights"][-1] = 0.0
    case["category_weights"] /= case["category_weights"].sum()
    return case


def extreme_branches(case):
    """A 1e-12 branch above a tip and a branch of 20 expected substitutions above an internal node,
    neither a child of the root; returns (case, the long branch's node id).

    Along the long branch a pattern's derivative is ~1e-11 and BEAGLE's pre^T dQ post / pre^T post
    reaches it by cancelling terms of order one: fp64 leaves ~1e-15 of it (2e-15 measured in the
    CPU restatement), so that edge is held to an absolute bar.  (On a root child the same holds for
    both root children: the two act as one edge.)"""
    n = case["n"]
    parents = parent_ids(case["post"], n)
    root = 2 * n - 2
    tip = next(v for v in range(n) if parents[v] != root)
    node = next(v for v in range(n, root) if parents[v] != root)
    case = dict(case, lengths=case["lengths"].copy())
    case["lengths"][tip] = 1e-12
    case["lengths"][node] = 20.0
    return case, node
