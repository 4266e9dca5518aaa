"""Cost of ambiguous tips on the fused tree walk, and of masked site-pattern compression
(profiles/r04_ambiguity_bench.json).

For 4 and 32 rate categories, on 100 taxa x 100k patterns, GTR + Weibull, rescaling on, and
alignments with 0 %, 1e-4 %, 1 % and 10 % ambiguous tip characters (trees.random_masked_alignment;
1e-4 % is ~10 characters of 10M: the ambiguous walk's fixed cost, with next to no divergence):
  * the walk over the masks (the ambiguous variant whenever some tip is ambiguous);
  * the state walk on the same alignment with its ambiguous characters turned into gaps;
each as logL+gradient, logL-only and logL+gradient with the analytic substitution gradient
evals/s from CUDA events around `--steps` runs of `--trees` trees, and walk ms per tree from
the engine's own events around each walk launch.  The two arms run alternately, each arm
twice, so that the spread between repeats is visible next to the difference.
Then site-pattern compression of 1000 taxa x 1M sites (IUPAC characters, 1 % degenerate) in
state mode and masked mode: device ms from the library's own events.

    python tools/ambiguity_bench.py [--categories 4,32 --fractions 0,0.000001,0.01,0.1 --trees 64 --steps 3]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from categories_bench import GTR_ROW, card  # noqa: E402


def walk(engine, tree_count, parent_ids, lengths, steps, warmup):
    import torch
    import libsbn_b200 as sbn
    from libsbn_b200 import _capi
    stream = torch.cuda.ExternalStream(engine.stream)
    batch = sbn.TreeBatch(parent_ids, lengths)
    params = np.tile(np.array(GTR_ROW), (tree_count, 1))

    def measure(staged, mode):
        for _ in range(warmup):
            staged.run(mode, True)
        engine.walk_timing(reset=True)
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            start.record()
            for _ in range(steps):
                staged.run(mode, True)
            stop.record()
        stop.synchronize()
        walk_ms, walks = engine.walk_timing(reset=True)
        ms = start.elapsed_time(stop)
        return {"evals_per_s": tree_count * steps / (ms * 1e-3),
                "walk_ms_per_tree": walk_ms / max(walks, 1) / tree_count}

    staged = engine.stage(batch, params)
    out = {"logl_plus_gradient": measure(staged, _capi.MODE_BRANCH_GRADIENT),
           "logl_only": measure(staged, _capi.MODE_LOG_LIKELIHOOD)}
    staged.close()
    staged = engine.stage(batch, params, substitution_analytic=True)
    out["logl_plus_gradient_with_substitution"] = measure(staged, _capi.MODE_BRANCH_GRADIENT)
    staged.close()
    return out


def walk_rows(categories, fractions, taxa, patterns, tree_count, steps, warmup):
    import libsbn_b200 as sbn
    from libsbn_b200 import trees
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=4)
    spec = sbn.PhyloModelSpecification("GTR", f"weibull+{categories}", "none")
    rows = []
    for fraction in fractions:
        masks, weights = trees.random_masked_alignment(taxa, patterns, seed=3, ambiguous_fraction=fraction,
                                                       gap_fraction=0.01)
        engines = {"masks": sbn.Engine(spec, masks, weights, tip_encoding="masks"),
                   "states_ambiguous_as_gaps": sbn.Engine(spec, trees.masks_to_states(masks), weights)}
        runs = {name: [] for name in engines}
        for _ in range(2):
            for name, engine in engines.items():
                runs[name].append(walk(engine, tree_count, parent_ids, lengths, steps, warmup))
        for engine in engines.values():
            engine.close()
        ambiguous = float(np.mean(~np.isin(masks, [1, 2, 4, 8, 15])))
        row = {"categories": categories, "ambiguous_fraction": ambiguous, "runs": runs}
        row["masks_over_states_walk_ms"] = {
            mode: float(np.mean([r[mode]["walk_ms_per_tree"] for r in runs["masks"]]) /
                        np.mean([r[mode]["walk_ms_per_tree"] for r in runs["states_ambiguous_as_gaps"]]))
            for mode in runs["masks"][0]}
        rows.append(row)
        print(json.dumps(row), file=sys.stderr)
    return rows


def compression(taxa, sites, repeats):
    import libsbn_b200 as sbn
    rng = np.random.default_rng(7)
    characters = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=(taxa, sites))]
    degenerate = rng.random((taxa, sites)) < 0.01
    characters[degenerate] = np.frombuffer(b"RYSWKMBDHVN-", dtype=np.uint8)[rng.integers(0, 12, int(degenerate.sum()))]
    characters = np.ascontiguousarray(characters)
    out = {}
    for name, ambiguity in (("states", False), ("masks", True)):
        times = []
        for _ in range(repeats + 1):
            pattern = sbn.SitePattern(characters, ambiguity=ambiguity)
            times.append(pattern.device_ms)
        out[name] = {"device_ms_median": float(np.median(times[1:])), "device_ms": times[1:],
                     "pattern_count": int(pattern.pattern_count)}
    return out


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--categories", default="4,32")
    parser.add_argument("--fractions", default="0,0.000001,0.01,0.1")
    parser.add_argument("--taxa", type=int, default=100)
    parser.add_argument("--patterns", type=int, default=100000)
    parser.add_argument("--trees", type=int, default=64)
    parser.add_argument("--steps", type=int, default=3)
    parser.add_argument("--warmup", type=int, default=1)
    parser.add_argument("--compression-taxa", type=int, default=1000)
    parser.add_argument("--compression-sites", type=int, default=1000000)
    parser.add_argument("--compression-repeats", type=int, default=3)
    args = parser.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("ambiguity_bench.py measures on a CUDA device; none is available")
    fractions = [float(f) for f in args.fractions.split(",")]
    rows = []
    for categories in (int(c) for c in args.categories.split(",")):
        rows += walk_rows(categories, fractions, args.taxa, args.patterns, args.trees, args.steps, args.warmup)
    print(json.dumps({
        "workload": f"{args.taxa} taxa x {args.patterns} patterns, GTR + Weibull, rescaling on, "
                    f"{args.trees} random trees per staged batch, {args.steps} timed steps after {args.warmup} "
                    "warm-up; each arm run twice, alternating",
        "card": card(), "walk": rows,
        "compression": {"workload": f"{args.compression_taxa} taxa x {args.compression_sites} sites, 1 % degenerate",
                        **compression(args.compression_taxa, args.compression_sites, args.compression_repeats)}}))


if __name__ == "__main__":
    main()
