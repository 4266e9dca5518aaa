"""Small invocations of the pipelined partial-update kernels of the BEAGLE-compatible device library
(op lists over two staged chunks, depth-first order = register forwarding, 1 / 2 / 3 / 4 / 8 categories)
and of site-pattern compression (alignments over several 64-taxon chunks of the tile kernels, with and
without repeats; 65 taxa x 129 sites; a retry under seed 1 after a key collision under seed 0; more than
1024 scan blocks), for compute-sanitizer:

  compute-sanitizer --tool memcheck  python tools/sanitizer_cases_shim_patterns.py
  compute-sanitizer --tool racecheck python tools/sanitizer_cases_shim_patterns.py

Results are compared with the CPU restatements (site patterns: tests/site_pattern_reference.py)
inside the sanitized run.
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from libsbn_b200 import beagle  # noqa: E402
from libsbn_b200.site_pattern import SitePattern  # noqa: E402
from oracle import site_pattern as restatement  # noqa: E402
import site_pattern_reference as reference  # noqa: E402
from test_beagle_shim import _depth_first  # noqa: E402

ORACLE = os.path.join(ROOT, "oracle", "_build", "libbeagle_oracle.so")


def beagle_case(categories, depth_first):
    rng = np.random.default_rng(categories + 10 * depth_first)
    n, P = 41, 515
    states = rng.integers(0, 4, size=(n, P)).astype(np.int32)
    states[rng.random(states.shape) < 0.05] = 4
    weights = rng.integers(1, 6, size=P).astype(np.float64)
    post, pre = beagle.random_tree_operations(n, rng, True)
    if depth_first:
        post = _depth_first(post, n)
    lengths = rng.exponential(0.1, size=2 * n - 1)
    evec, ivec, evals, freqs, q = beagle.gtr_eigensystem()
    rates = np.sort(rng.gamma(2.0, 0.5, size=categories))
    rates /= rates.mean()
    results = []
    for path in (None, ORACLE):
        instance = beagle.Beagle(path, n, P, categories, True)
        instance.set_tips(states, weights, True)
        instance.set_model(evec, ivec, evals, freqs, rates, np.full(categories, 1.0 / categories))
        results.append(instance.log_likelihood_and_gradient(post, pre, lengths, q, rates, freqs, True))
        instance.close()
    e_logl = abs(results[0][0] - results[1][0]) / abs(results[1][0])
    e_grad = np.max(np.abs(results[0][1] - results[1][1])) / np.max(np.abs(results[1][1]))
    print(f"BEAGLE library C={categories} depth_first={int(depth_first)} (40 + 80 ops): logL rel.err {e_logl:.1e} "
          f"derivative rel.err {e_grad:.1e}", flush=True)
    assert e_logl < 1e-12 and e_grad < 1e-10


def pattern_case(taxa, sites, distinct):
    rng = np.random.default_rng(taxa + sites)
    alphabet = np.frombuffer(b"ACGTacgt-N?RYKM", dtype=np.uint8)
    pool = alphabet[rng.integers(0, alphabet.size, size=(taxa, distinct))]
    sequences = [bytes(row) for row in pool[:, rng.integers(0, distinct, size=sites)]]
    got = SitePattern(sequences)
    want_patterns, want_weights = restatement.compress(sequences)
    assert np.array_equal(got.patterns, want_patterns) and np.array_equal(got.weights, want_weights)
    print(f"site patterns {taxa} taxa x {sites} sites: {got.pattern_count} patterns, equal to the restatement", flush=True)


def pattern_reference_case(what, pool, picks, key_bits=None):
    if key_bits is not None:
        os.environ["SBNB_DEBUG_PATTERN_KEY_BITS"] = str(key_bits)
    try:
        got = SitePattern(reference.alignment(pool, picks))
    finally:
        os.environ.pop("SBNB_DEBUG_PATTERN_KEY_BITS", None)
    want_patterns, want_weights = reference.by_construction(pool, picks)
    assert np.array_equal(got.patterns, want_patterns) and np.array_equal(got.weights, want_weights)
    print(f"site patterns, {what}: {got.pattern_count} patterns, equal to the reference", flush=True)


if __name__ == "__main__":
    for categories, depth_first in ((4, True), (4, False), (8, True), (2, True), (1, True), (3, True)):
        beagle_case(categories, depth_first)
    pattern_case(130, 5000, 300)    # three 64-taxon chunks, every pattern repeats
    pattern_case(69, 987, 987)      # hardly any repeats
    pattern_case(20, 3001, 40)      # ragged last tile
    rng = np.random.default_rng(65)
    pattern_reference_case("65 taxa x 129 sites", reference.pool_columns(65, 129, rng),
                           reference.site_picks("prefix1", 129, 129, rng))
    index, bits = reference.find_rehash_case((True, False, None, None), "states")
    pattern_reference_case(f"seed 0 collides at {bits}-bit keys, seed 1 is clean",
                           *reference.rehash_alignment(index, "states"), key_bits=bits)
    sites = 1_048_577
    pattern_reference_case("12 taxa x 1048577 sites (1025 scan blocks)",
                           reference.pool_columns(12, sites, rng, digit_rows=12),
                           reference.site_picks("prefix1", sites, sites, rng))
