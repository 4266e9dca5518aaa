"""Throughput of the fused tree walk across rate-category counts, next to the BEAGLE-compatible
device library at the same counts (profiles/r03_categories_bench.json).

For every count, on 100 taxa x 100k patterns, GTR + Weibull:
  * the fused walk behind the C ABI (staged batch, inputs resident on the device): logL+gradient
    (branch lengths and site model; and with the analytic substitution gradient as well) and
    logL-only evals/s from CUDA events around `--steps` runs of `--trees` trees, and walk kernel
    ms per tree from the engine's own events around each walk launch;
  * libhmsbeagle_b200.so driven by FatBeagle's call sequence (tools/beagle_shim_bench.py): device
    ms of beagleUpdatePartials + beagleUpdatePrePartials + beagleCalculateEdgeDerivatives for one
    tree, i.e. one logL + gradient evaluation.
Counts that are not powers of two run padded (17-31 on 32 lanes), so 20 costs what 32 costs.

    python tools/categories_bench.py [--categories 4,16,20,32 --trees 64 --steps 3 --warmup 1 --no-beagle]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

GTR_ROW = [0.05, 0.1, 0.15, 0.20, 0.25, 0.25, 0.1, 0.2, 0.3, 0.4, 0.5]


def card():
    """Name, power limit and maximum SM clock of GPU 0, read in the same run as the numbers."""
    query = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = (cell.strip() for cell in line.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.SubprocessError, ValueError):
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "not read", "max_sm_clock": "not read"}


def fused_walk(categories, taxa, patterns, tree_count, steps, warmup):
    import torch
    import libsbn_b200 as sbn
    from libsbn_b200 import _capi, trees
    states, weights = trees.random_alignment(taxa, patterns, seed=3)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=4)
    params = np.tile(np.array(GTR_ROW), (tree_count, 1))
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", f"weibull+{categories}", "none"), states, weights)
    stream = torch.cuda.ExternalStream(engine.stream)
    batch = sbn.TreeBatch(parent_ids, lengths)

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
        return {"evals_per_s": tree_count * steps / (ms * 1e-3), "ms_per_step": ms / steps,
                "walk_ms_per_tree": walk_ms / max(walks, 1) / tree_count}

    staged = engine.stage(batch, params)
    out = {"logl_plus_gradient": measure(staged, _capi.MODE_BRANCH_GRADIENT),
           "logl_only": measure(staged, _capi.MODE_LOG_LIKELIHOOD)}
    staged.close()
    # what Engine.gradients runs for GTR: the branch-length sweep also accumulates the sums of the
    # exact substitution-parameter gradient
    staged = engine.stage(batch, params, substitution_analytic=True)
    out["logl_plus_gradient_with_substitution"] = measure(staged, _capi.MODE_BRANCH_GRADIENT)
    staged.close()
    engine.close()
    return out


def beagle_library(categories, taxa, patterns, repeats):
    import beagle_shim_bench
    got = beagle_shim_bench._measure(taxa, patterns, categories, repeats, "libsbn", probe=False)
    return {key: got[key]["ms"] for key in ("update_partials", "update_pre_partials", "edge_derivatives")} | {
        "device_ms_per_logl_plus_gradient": got["device_ms_per_logl_plus_gradient"],
        "call_sequence_ms": got["branch_gradient_call_sequence_ms"]}


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--categories", default="4,16,20,32")
    parser.add_argument("--taxa", type=int, default=100)
    parser.add_argument("--patterns", type=int, default=100000)
    parser.add_argument("--trees", type=int, default=64)
    parser.add_argument("--steps", type=int, default=3)
    parser.add_argument("--warmup", type=int, default=1)
    parser.add_argument("--repeats", type=int, default=3, help="BEAGLE call sequences per count (median)")
    parser.add_argument("--no-beagle", action="store_true")
    args = parser.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("categories_bench.py measures on a CUDA device; none is available")
    rows = []
    for categories in (int(c) for c in args.categories.split(",")):
        row = {"categories": categories,
               "fused_walk": fused_walk(categories, args.taxa, args.patterns, args.trees, args.steps, args.warmup)}
        if not args.no_beagle:
            row["beagle_library"] = beagle_library(categories, args.taxa, args.patterns, args.repeats)
            row["fused_walk_speedup_in_device_time"] = (row["beagle_library"]["device_ms_per_logl_plus_gradient"] /
                                                         row["fused_walk"]["logl_plus_gradient"]["walk_ms_per_tree"])
        rows.append(row)
    print(json.dumps({
        "workload": f"{args.taxa} taxa x {args.patterns} patterns, GTR + Weibull, rescaling on; fused walk: "
                    f"{args.trees} random trees per staged batch, {args.steps} timed steps after {args.warmup} warm-up",
        "card": card(), "library": os.environ.get("SBNB_LIBRARY", "libsbn_b200/lib/libsbn_b200.so"),
        "rows": rows}))


if __name__ == "__main__":
    main()
