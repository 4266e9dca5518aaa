"""Cost of the site log-likelihood matrix (profiles/r05_site_log_likelihoods_bench.json).

On 100 taxa x 100k patterns, GTR + Gamma 4 and GTR + Gamma 32, rescaling on, `--trees` random trees:
- the logL-only walk, ms per tree from the engine's own CUDA events around each walk launch, of a
  batch staged without and with the site matrix (arms alternated, each `--repeats` times, so that
  the spread between repeats is visible next to the difference);
- the one-call sbnb_site_log_likelihoods_unrooted end to end (the [T][P] matrix copied to the host)
  next to sbnb_log_likelihoods_unrooted, host clock around calls that end in a synchronise;
- the BEAGLE-compatible library's RootLogLikelihoodKernel device time (torch.profiler), with the
  per-pattern store (this tree's libhmsbeagle_b200.so) and, given `--beagle-before` (a build of the
  library without it), before it, arms alternated.
The card's name, power limit and maximum SM clock are read in the same run.

    python tools/site_log_likelihoods_bench.py [--beagle-before PATH] > profiles/r05_site_log_likelihoods_bench.json
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from categories_bench import GTR_ROW, card  # noqa: E402

SHAPE = 0.5


def walk_ms(engine, staged, tree_count, steps, warmup):
    from libsbn_b200 import _capi
    for _ in range(warmup):
        staged.run(_capi.MODE_LOG_LIKELIHOOD, True)
    engine.walk_timing(reset=True)
    for _ in range(steps):
        staged.run(_capi.MODE_LOG_LIKELIHOOD, True)
    total, launches = engine.walk_timing(reset=True)
    return total / max(launches, 1) / tree_count


def fused_walk(categories, taxa, patterns, tree_count, steps, warmup, repeats):
    import libsbn_b200 as sbn
    from libsbn_b200 import trees
    states, weights = trees.random_alignment(taxa, patterns, seed=3, gap_fraction=0.01)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=4)
    params = np.tile(np.array(GTR_ROW[:10] + [SHAPE]), (tree_count, 1))
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", f"gamma+{categories}", "none"), states, weights)
    batch = sbn.TreeBatch(parent_ids, lengths)
    arms = {"plain": engine.stage(batch, params), "with_sites": engine.stage(batch, params, site_log_likelihoods=True)}
    runs = {name: [] for name in arms}
    for _ in range(repeats):
        for name, staged in arms.items():
            runs[name].append(walk_ms(engine, staged, tree_count, steps, warmup))
    for staged in arms.values():
        staged.close()
    # one-call entry points, end to end (the first calls run eagerly, later ones replay a CUDA graph)
    calls = {"log_likelihoods_ms": [], "site_log_likelihoods_ms": []}
    for _ in range(repeats):
        for key, call in (("log_likelihoods_ms", lambda: engine.log_likelihoods(batch, params, True)),
                          ("site_log_likelihoods_ms", lambda: engine.site_log_likelihoods(batch, params, True))):
            for _ in range(warmup + 2):
                call()
            start = time.perf_counter()
            for _ in range(steps):
                call()
            calls[key].append((time.perf_counter() - start) * 1e3 / steps)
    engine.close()
    plain, sites = np.mean(runs["plain"]), np.mean(runs["with_sites"])
    row = {"categories": categories, "walk_ms_per_tree": runs, "with_sites_over_plain": float(sites / plain),
           "one_call": calls, "matrix_bytes": tree_count * patterns * 8}
    print(json.dumps({"categories": categories, "with_sites_over_plain": row["with_sites_over_plain"]}),
          file=sys.stderr)
    return row


def beagle_root(paths, taxa, patterns, categories, calls, repeats):
    """RootLogLikelihoodKernel device time (us per call) of each library, arms alternated."""
    import torch
    from libsbn_b200 import beagle, trees
    rng = np.random.default_rng(7)
    states, _ = trees.random_alignment(taxa, patterns, seed=8, gap_fraction=0.01)
    weights = np.ones(patterns)
    post, pre = beagle.random_tree_operations(taxa, rng, True)
    lengths = np.maximum(rng.exponential(0.1, size=2 * taxa - 1), 1e-6)
    evec, ivec, evals, freqs, q = beagle.gtr_eigensystem()
    rates = np.ones(categories) if categories == 1 else np.sort(rng.gamma(2.0, 0.5, size=categories))
    rates /= rates.mean()
    libraries = {}
    for name, path in paths.items():
        library = beagle.Beagle(path, taxa, patterns, categories, True)
        library.set_tips(states.astype(np.int32), weights, True)
        library.set_model(evec, ivec, evals, freqs, rates, np.full(categories, 1.0 / categories))
        library.log_likelihood_and_gradient(post, pre, lengths, q, rates, freqs, True, per_site=False)
        libraries[name] = library
    N = 2 * taxa - 1
    root, zero, cum = (np.array([v], dtype=np.int32) for v in (N - 1, 0, 0))
    pointer = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int))

    def root_calls(library):
        out = ctypes.c_double()
        for _ in range(calls):
            library.ok(library.lib.beagleCalculateRootLogLikelihoods(library.handle, pointer(root), pointer(zero),
                                                                     pointer(zero), pointer(cum), 1,
                                                                     ctypes.byref(out)))
        return out.value

    results = {name: [] for name in libraries}
    values = {}
    for _ in range(repeats):
        for name, library in libraries.items():
            root_calls(library)  # warm-up
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as profile:
                values[name] = root_calls(library)
            for event in profile.key_averages():
                if "RootLogLikelihoodKernel" in event.key:
                    total = getattr(event, "device_time_total", None) or getattr(event, "cuda_time_total")
                    results[name].append(total / event.count)
    for library in libraries.values():
        library.close()
    return {"workload": f"{taxa} taxa x {patterns} patterns x {categories} categories, one root call per step, "
                        f"{calls} calls per profile", "us_per_call": results, "log_likelihoods": values}


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--categories", default="4,32")
    parser.add_argument("--taxa", type=int, default=100)
    parser.add_argument("--patterns", type=int, default=100000)
    parser.add_argument("--trees", type=int, default=64)
    parser.add_argument("--steps", type=int, default=5)
    parser.add_argument("--warmup", type=int, default=2)
    parser.add_argument("--repeats", type=int, default=3)
    parser.add_argument("--beagle-before", default=None,
                        help="a libhmsbeagle_b200.so built without the per-pattern store, for the before arm")
    args = parser.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("site_log_likelihoods_bench.py measures on a CUDA device; none is available")
    rows = [fused_walk(int(c), args.taxa, args.patterns, args.trees, args.steps, args.warmup, args.repeats)
            for c in args.categories.split(",")]
    from libsbn_b200 import beagle
    paths = {"after": beagle.LIB_PATH}
    if args.beagle_before:
        paths = {"before": os.path.abspath(args.beagle_before), "after": beagle.LIB_PATH}
    library = beagle_root(paths, args.taxa, args.patterns, 4, 50, args.repeats)
    print(json.dumps({
        "workload": f"{args.taxa} taxa x {args.patterns} patterns, GTR + Gamma (shape {SHAPE}), rescaling on, "
                    f"{args.trees} random trees per batch, {args.steps} timed steps after {args.warmup} warm-up; "
                    f"arms alternated, {args.repeats} repeats each",
        "card": card(), "walk": rows, "beagle_root_log_likelihoods": library}))


if __name__ == "__main__":
    main()
