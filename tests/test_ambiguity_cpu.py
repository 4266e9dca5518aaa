"""Ambiguous nucleotides as partial tip states, on the host: the IUPAC mask table, the
masked-alignment generator, and the linearity the engine's ambiguous tips rest on, checked
on the CPU oracle (tests/ambiguity_oracle.py) against an independent NumPy pruning."""
import numpy as np
import pytest
from scipy.linalg import expm

import ambiguity_oracle
from libsbn_b200 import alignment, trees

IUPAC = {"A": "A", "C": "C", "G": "G", "T": "T", "U": "T", "R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT",
         "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT", "X": "ACGT", "?": "ACGT",
         "-": "ACGT"}


def test_iupac_mask_table():
    table = alignment.iupac_mask_table()
    for symbol, states in IUPAC.items():
        want = sum(1 << "ACGT".index(s) for s in states)
        assert table[symbol] == want, symbol
        assert table[symbol.lower()] == want, symbol
    assert len(table) == len(IUPAC) + sum(c.isalpha() for c in IUPAC)
    # the reference's table is unchanged: every degenerate code is the gap state
    states = alignment.symbol_table()
    assert all(states[c] == 4 for c in "RYSWKMBDHVNXU?-")


def test_iupac_encoding_and_its_error():
    sequences = {"a": "ACGTRYN-", "b": "acgtuk?x"}
    masks = alignment.encode(sequences, ["a", "b"], ambiguity=True)
    assert masks.tolist() == [[1, 2, 4, 8, 5, 10, 15, 15], [1, 2, 4, 8, 8, 12, 15, 15]]
    assert alignment.encode(sequences, ["a"]).tolist() == [[0, 1, 2, 3, 4, 4, 4, 4]]  # (the reference's table)
    with pytest.raises(RuntimeError, match=r"^Symbol 'J' not known\.$"):
        alignment.encode({"a": "ACJT"}, ["a"], ambiguity=True)


def test_masked_alignment_generator():
    masks, weights = trees.random_masked_alignment(40, 5000, seed=3, ambiguous_fraction=0.1, gap_fraction=0.02)
    again, _ = trees.random_masked_alignment(40, 5000, seed=3, ambiguous_fraction=0.1, gap_fraction=0.02)
    assert np.array_equal(masks, again) and weights.shape == (5000,)
    assert masks.min() >= 1 and masks.max() <= 15
    ambiguous = ~np.isin(masks, [1, 2, 4, 8, 15])
    assert abs(ambiguous.mean() - 0.1) < 0.01 and abs((masks == 15).mean() - 0.02) < 0.005
    assert set(np.unique(masks[ambiguous])) == {3, 5, 6, 7, 9, 10, 11, 12, 13, 14}
    states = trees.masks_to_states(masks)
    assert np.array_equal(trees.states_to_masks(states)[~ambiguous], masks[~ambiguous])
    assert (states[ambiguous] == 4).all()


@pytest.mark.parametrize("rooted", [False, True], ids=["unrooted", "rooted"])
def test_mask_oracle_without_ambiguity_is_the_state_oracle(oracle, rooted):
    """Masks that are single states or 15, every pattern through the per-pattern path of the
    mask oracle (which strips the rooted Jacobian from every call), against one state call."""
    from conftest import load_fixture
    if rooted:
        fx = load_fixture("flua_jc69_strict")
        states, weights = fx["patterns"][:, :40], fx["weights"][:40]
        args = (fx["parent_ids"], fx["branch_lengths"], np.array([[0.8, 0.0]]))
        kwargs = dict(rooted=True, rates=fx["rates"], node_heights=fx["node_heights"], node_bounds=fx["node_bounds"],
                      height_ratios=fx["height_ratios"])
        substitution = "JC69"
    else:
        states, weights = trees.random_alignment(9, 60, seed=2, gap_fraction=0.1)
        parent_ids, lengths = trees.random_tree_batch(9, 2, seed=3)
        row = [0.1, 0.2, 0.3, 0.1, 0.2, 0.1, 0.3, 0.2, 0.25, 0.25, 0.6]
        args, kwargs, substitution = (parent_ids, lengths, np.tile(row, (2, 1))), {}, "GTR"
    want = oracle.gradients(substitution, "weibull+4", states, weights, *args, rescaling=True, **kwargs)
    got = ambiguity_oracle.gradients(oracle, substitution, "weibull+4", trees.states_to_masks(states), weights, *args,
                                     rescaling=True, batch_unambiguous=False, **kwargs)
    for key in ambiguity_oracle.KEYS:
        scale = max(np.max(np.abs(want[key])), 1e-300)
        # (the oracle's substitution gradient is central differences at delta 1e-6, whose
        #  rounding differs between one call and a sum of per-pattern calls)
        tol = 1e-6 if key == "substitution_model" else 1e-9
        assert np.max(np.abs(got[key] - want[key])) <= tol * scale, key


def pruning_log_likelihood(parent_ids, lengths, tip_partials, q, freqs):
    """log L of one site by Felsenstein pruning on the tree as given (a trifurcating root is
    fine): NumPy and scipy only, nothing shared with the oracle."""
    n = tip_partials.shape[0]
    node_count = lengths.shape[0]
    partial = {i: tip_partials[i] for i in range(n)}
    for node in range(n, node_count):
        value = np.ones(4)
        for child in np.flatnonzero(parent_ids == node):
            value = value * (expm(q * lengths[child]) @ partial[child])
        partial[node] = value
    return float(np.log(freqs @ partial[node_count - 1]))


def test_linearity_on_the_oracle(oracle):
    """One pattern with R (A or G) at tip 0: L_R = L_A + L_G, and for every leaf edge
    grad log L_R = (L_A grad log L_A + L_G grad log L_G) / (L_A + L_G), with L_R and its
    derivatives from an independent pruning (central differences for the gradient)."""
    taxa = 7
    parent_ids, lengths = trees.random_tree_batch(taxa, 1, seed=8)
    column = np.array([5, 2, 8, 1, 4, 15, 10], dtype=np.uint8)  # R at tip 0, Y at tip 6
    weights = np.ones(1)
    combinations = ambiguity_oracle.expand(column)  # [4][taxa]: A or G at tip 0, C or T at tip 6
    by_state = {state: [oracle.gradients("JC69", "constant", c[:, None], weights, parent_ids, lengths)
                        for c in combinations[combinations[:, 0] == state]] for state in (0, 2)}
    l = {s: sum(np.exp(g["log_likelihood"][0]) for g in by_state[s]) for s in by_state}
    masked = ambiguity_oracle.gradients(oracle, "JC69", "constant", column[:, None], weights, parent_ids, lengths,
                                        None)
    assert abs(np.exp(masked["log_likelihood"][0]) - (l[0] + l[2])) <= 1e-13 * (l[0] + l[2])
    grad = {s: sum(np.exp(g["log_likelihood"][0]) * g["branch"][0] for g in by_state[s]) / l[s] for s in by_state}
    identity = (l[0] * grad[0] + l[2] * grad[2]) / (l[0] + l[2])
    assert np.allclose(masked["branch"][0], identity, rtol=1e-12, atol=0)

    q = (np.ones((4, 4)) - 4 * np.eye(4)) / 3
    freqs = np.full(4, 0.25)
    tips = ((column[:, None] >> np.arange(4)) & 1).astype(np.float64)
    tree, t = parent_ids[0], lengths[0]
    log_l = pruning_log_likelihood(tree, t, tips, q, freqs)
    assert abs(log_l - masked["log_likelihood"][0]) <= 1e-12 * abs(log_l)
    for edge in range(taxa):  # leaf ids and their edges are the same before and after detrifurcation
        if masked["branch"][0][edge] == 0.0:  # the fixed node of an unrooted tree
            continue
        h = 1e-5
        up, down = t.copy(), t.copy()
        up[edge] += h
        down[edge] -= h
        fd = (pruning_log_likelihood(tree, up, tips, q, freqs) - pruning_log_likelihood(tree, down, tips, q, freqs))
        assert abs(fd / (2 * h) - identity[edge]) <= 1e-7 * max(1.0, abs(identity[edge])), edge
