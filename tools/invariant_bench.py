"""Cost of invariable sites (+I) on the fused tree walk (profiles/r05_invariant_bench.json).

For 4 and 32 rate categories, on 100 taxa x 100k patterns (20 % of the columns constant),
GTR + Gamma against GTR + Gamma + I (p = 0.2), rescaling on, `--trees` random trees per staged
batch: logL-only, logL+gradient, and logL+gradient with the analytic substitution gradient,
evals/s from CUDA events around `--steps` runs, and walk ms per tree from the engine's own
events around each walk launch.  The two arms run alternately, each twice, so that the
spread between repeats is visible next to the difference.  The card's name and power limit
are read in the same run.

    python tools/invariant_bench.py [--categories 4,32 --trees 64 --steps 3] > profiles/r05_invariant_bench.json
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

PINV = 0.2
SHAPE = 0.5


def walk(engine, row, tree_count, parent_ids, lengths, steps, warmup):
    import torch
    import libsbn_b200 as sbn
    from libsbn_b200 import _capi
    stream = torch.cuda.ExternalStream(engine.stream)
    batch = sbn.TreeBatch(parent_ids, lengths)
    params = np.tile(np.array(row), (tree_count, 1))

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
    out = {"logl_only": measure(staged, _capi.MODE_LOG_LIKELIHOOD),
           "logl_plus_gradient": measure(staged, _capi.MODE_BRANCH_GRADIENT)}
    staged.close()
    staged = engine.stage(batch, params, substitution_analytic=True)
    out["logl_plus_gradient_with_substitution"] = measure(staged, _capi.MODE_BRANCH_GRADIENT)
    staged.close()
    return out


def rows_for(categories, taxa, patterns, tree_count, steps, warmup):
    import libsbn_b200 as sbn
    from libsbn_b200 import trees
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=4)
    states, weights = trees.random_alignment(taxa, patterns, seed=3, gap_fraction=0.01)
    rng = np.random.default_rng(5)
    states = states.copy()
    constant = rng.random(patterns) < 0.2
    states[:, constant] = rng.integers(0, 4, size=patterns)[constant]
    site = f"gamma+{categories}"
    arms = {site: (sbn.Engine(sbn.PhyloModelSpecification("GTR", site, "none"), states, weights),
                   GTR_ROW[:10] + [SHAPE]),
            site + "+I": (sbn.Engine(sbn.PhyloModelSpecification("GTR", site + "+I", "none"), states, weights),
                          GTR_ROW[:10] + [SHAPE, PINV])}
    runs = {name: [] for name in arms}
    for _ in range(2):
        for name, (engine, row) in arms.items():
            runs[name].append(walk(engine, row, tree_count, parent_ids, lengths, steps, warmup))
    for engine, _ in arms.values():
        engine.close()
    row = {"categories": categories, "runs": runs}
    row["invariant_over_plain_walk_ms"] = {
        mode: float(np.mean([r[mode]["walk_ms_per_tree"] for r in runs[site + "+I"]]) /
                    np.mean([r[mode]["walk_ms_per_tree"] for r in runs[site]]))
        for mode in runs[site][0]}
    print(json.dumps(row["invariant_over_plain_walk_ms"]), file=sys.stderr)
    return row


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--categories", default="4,32")
    parser.add_argument("--taxa", type=int, default=100)
    parser.add_argument("--patterns", type=int, default=100000)
    parser.add_argument("--trees", type=int, default=64)
    parser.add_argument("--steps", type=int, default=3)
    parser.add_argument("--warmup", type=int, default=1)
    args = parser.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("invariant_bench.py measures on a CUDA device; none is available")
    rows = [rows_for(int(c), args.taxa, args.patterns, args.trees, args.steps, args.warmup)
            for c in args.categories.split(",")]
    print(json.dumps({
        "workload": f"{args.taxa} taxa x {args.patterns} patterns (20 % constant columns), GTR + Gamma "
                    f"(shape {SHAPE}) against GTR + Gamma + I (p = {PINV}), rescaling on, {args.trees} random trees "
                    f"per staged batch, {args.steps} timed steps after {args.warmup} warm-up; each arm run twice, "
                    "alternating",
        "card": card(), "walk": rows}))


if __name__ == "__main__":
    main()
