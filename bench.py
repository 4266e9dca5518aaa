"""bench.py -- BASELINE.json's headline metric on BASELINE.json's configs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[3]): synthetic 100 taxa x 100,000 site
patterns, GTR + 4 rate categories (the reference's "weibull+4"), a batch of 1024
random unrooted topologies, rescaling on, SHARDED BY TREE across the ranks -- strong
scaling: 1024 trees in total, rank r evaluates trees [r, r+1) x 1024 / N; trees are
independent, so there is no data-path collective.

A "step" is one pass of the hot path over the batch: per tree, the log-likelihood and
all 2n-2 branch-length derivatives, i.e. one BranchGradientInternals-equivalent
(reference src/fat_beagle.cpp:119-175).  --dump-outputs DIR writes what the last timed
step computed, as sbnb_batch_fetch returns it: log_likelihoods [T], raw branch_gradients
and rate_gradients [T][2n-1] (fp64 .npy files; the inputs are seeded, so two builds can
be compared output for output).

  value    : batch staged in HBM, only the kernels in the timed region (CUDA events on
             the engine's stream, barrier + synchronize on both sides, max over ranks).
  e2e      : the public call -- host arrays in, PhyloGradient arrays out -- per step:
             host-side schedule generation, H2D from page-locked staging, kernels, D2H,
             host finishing.  `e2e_full_phylo_gradients` is the same through the
             reference's full GTR phylo_gradients semantics (+ 16 finite-difference
             log-likelihood sweeps per tree, fat_beagle.cpp:400-465).
  roofline : the tree-walk kernel against the bound that binds it.  The fused walk keeps
             O(log n) partials on chip, so its DRAM traffic (measured in this run with
             ncu's dram__bytes_{read,write}.sum on a 148-tree probe launch) is a
             fraction of the reference schedule's ALGORITHMIC bytes (SURVEY.md 8d:
             (10n-14) x 32 C P per tree): achieved = measured bytes / CUDA-event kernel
             time against the measured HBM copy bandwidth, frac <= 1; the
             algorithmic-bytes equivalent is reported beside it (it exceeds the HBM peak).
  config5  : BASELINE.json configs[4] -- 1000 taxa x 1M site patterns, HKY + 4
             categories, 8 trees, SITE PATTERNS sharded across the ranks with one NCCL
             sum-all-reduce of the per-tree log-likelihoods and gradient sums.
  small_problem : BASELINE.json configs[0..1] -- DS1 (27 taxa x 934 patterns) x 100
             topologies: call latency of JC69 log_likelihoods and of the full GTR+weibull4
             phylo_gradients at 10 and 100 trees, beside the CPU oracle port on all cores.
  partial_update : BASELINE.json's second metric -- partial-update HBM GB/s against the measured
             peak -- on the op-at-a-time schedule where it is directly meaningful: the
             BEAGLE-compatible device library (libhmsbeagle_b200.so, the inner boundary) running
             FatBeagle's call sequence for one tree at the headline size, bytes by SURVEY.md 8d.
  gp       : BASELINE.json configs[2] -- generalized pruning on the DS1 subsplit DAG: device time
             of each op program of the reference's schedule, and the unmodified python
             `gp_instance` over this library beside the reference's own Eigen code on the host.
  cpu_baseline / --impl reference: the UNMODIFIED reference host code (oracle/_ref, its
             own python module, thread pool = host cores) over the BEAGLE-equivalent CPU
             kernels of oracle/beagle_cpu.cpp, at the FULL pattern count on one tree per
             core.  The reference exposes BranchGradientInternals only inside
             phylo_gradients(); with JC69 + weibull+4 that call is exactly 2 of them per
             tree and nothing else (fat_beagle.cpp:467-503; the 4x4 kernels do not
             depend on the substitution model), so evals/s = 2 x trees / time.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tree logL+branch-gradient evals/sec"
UNIT = "evals/s"
GTR_ROW = [0.05, 0.1, 0.15, 0.20, 0.25, 0.25, 0.1, 0.2, 0.3, 0.4, 0.5]  # rates, freqs, Weibull shape
WALK_KERNEL = "TreeWalkOeKernel<C=4,K=4,GRAD,RESCALE>"
WALK_KERNEL_REGEX = r"regex:TreeWalkOeKernel<\(int\)4, \(int\)4, \(bool\)1"
FP64_PEAK = 148 * 64 * 2 * 1.965e9  # non-tensor fp64: 64 DFMA / clk / SM x 148 SMs x 1.965 GHz
FLOPS_PER_PATTERN_CATEGORY = 26.1e3  # logL + gradient at 100 taxa (SURVEY.md 8d)


def workload(args, seed=4):
    from libsbn_b200 import trees
    states, weights = trees.random_alignment(args.taxa, args.patterns, seed=20261017, gap_fraction=0.01)
    parent_ids, lengths = trees.random_tree_batch(args.taxa, args.trees, seed=seed, mean_branch_length=0.1)
    params = np.tile(np.array(GTR_ROW), (args.trees, 1))
    return states, weights, parent_ids, lengths, params


def config_of(args, world=1):
    return {
        "workload": f"synthetic {args.taxa} taxa x {args.patterns} site patterns, GTR+weibull4 (4 rate "
                    f"categories), {args.trees} random unrooted topologies in total, logL + branch gradients, "
                    "rescaling on (BASELINE.json configs[3])",
        "taxa": args.taxa, "patterns": args.patterns, "categories": 4, "trees": args.trees,
        "trees_per_gpu": args.trees // max(world, 1),
        "sharding": "trees across ranks (rank r evaluates a contiguous slice of the batch), no data-path "
                    "collective",
        "l2": "no flush needed: each step streams the post-order arena and per-tree operand blocks "
              "(> 1 GB) through a 126 MB L2",
    }


# --------------------------------------------------------------------------- clocks

class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, sm_max, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            try:
                sm.append(float(row[1])), sm_max.append(float(row[2])), power.append(float(row[3]))
            except (ValueError, IndexError):
                continue
            for name, value in zip(names, row[5:9]):
                if value.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        busy = [c for c, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": max(sm_max), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


# --------------------------------------------------------------------------- reference arm

def reference_worker(args):
    """Child process: times the reference python module found in args.module_dir (or the
    oracle port when there is none) and prints one JSON object.  Isolated in a process
    of its own because the reference prints per-thread banners on stdout and because two
    builds of the module (same name) cannot live in one interpreter."""
    from libsbn_b200 import trees
    states, weights, parent_ids, lengths, _ = workload(args)
    cores, steps = args.cores, args.steps
    out = {"cores": cores, "trees": int(args.trees), "patterns": int(args.patterns)}
    libsbn = None
    if args.module_dir and os.path.isdir(args.module_dir):
        sys.path.insert(0, args.module_dir)
        try:
            import libsbn  # the reference's own python module
        except ImportError:
            libsbn = None
    saved = os.dup(1)
    os.dup2(2, 1)  # everything the libraries print goes to stderr
    try:
        if libsbn is not None:
            with tempfile.TemporaryDirectory() as tmp:
                names = [f"t{i}" for i in range(args.taxa)]
                with open(os.path.join(tmp, "a.fasta"), "w") as f:
                    for name, row in zip(names, states):
                        f.write(f">{name}\n{''.join('ACGT-'[s] for s in row)}\n")
                with open(os.path.join(tmp, "t.nwk"), "w") as f:
                    for ids, bl in zip(parent_ids, lengths):
                        f.write(trees.newick(ids, bl, names) + "\n")
                inst = libsbn.unrooted_instance("bench")
                inst.read_newick_file(os.path.join(tmp, "t.nwk"))
                inst.read_fasta_file(os.path.join(tmp, "a.fasta"))
                inst.prepare_for_phylo_likelihood(libsbn.PhyloModelSpecification("JC69", "weibull+4", "none"),
                                                  cores, [], True)
                inst.get_phylo_model_param_block_map()["Weibull shape"][:] = GTR_ROW[10]
                inst.set_rescaling(True)
                times = []
                for _ in range(args.warmup + steps):
                    t0 = time.perf_counter()
                    inst.phylo_gradients()
                    times.append(time.perf_counter() - t0)
            out.update(kind="reference", times=times[args.warmup:],
                       how="unmodified reference python module (oracle/_ref) over BEAGLE-equivalent CPU kernels; "
                           "JC69+weibull4 phylo_gradients() = exactly 2 BranchGradientInternals per tree on the "
                           "same trees and alignment (the 4x4 kernels do not depend on the substitution model)")
        else:
            from oracle import phylo
            shape = np.full((args.trees, 1), GTR_ROW[10])
            times = []
            for _ in range(args.warmup + steps):
                t0 = time.perf_counter()
                phylo.gradients("JC69", "weibull+4", states, weights, parent_ids, lengths, shape, rescaling=True,
                                threads=cores)
                times.append(time.perf_counter() - t0)
            out.update(kind="port", times=times[args.warmup:],
                       how="oracle port (oracle/phylo_oracle.cpp), JC69+weibull4: 2 BranchGradientInternals per "
                           "tree, same 4x4 kernels as GTR")
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    print(json.dumps(out))


def time_reference(args, module_dir, trees, steps, warmup):
    """Runs reference_worker in a subprocess; returns (evals/s, detail dict)."""
    cores = os.cpu_count() or 1
    command = [sys.executable, os.path.abspath(__file__), "--_reference-worker", "--module-dir", module_dir or "",
               "--cores", str(cores), "--taxa", str(args.taxa), "--patterns", str(args.patterns),
               "--trees", str(trees), "--steps", str(steps), "--warmup", str(warmup)]
    done = subprocess.run(command, capture_output=True, text=True, timeout=3000, cwd=ROOT)
    if done.returncode != 0:
        raise RuntimeError(f"reference worker failed: {done.stderr[-2000:]}")
    result = json.loads(done.stdout.strip().splitlines()[-1])
    rates = [2.0 * trees / t for t in result["times"]]
    detail = {"kind": result["kind"], "cores": cores, "how": result["how"],
              "sample": f"{trees} trees (one per core) x all {args.patterns} patterns, {len(rates)} timed "
                        f"phylo_gradients() calls of 2 BranchGradientInternals per tree",
              "evals_per_s_per_call": rates,
              "spread": (max(rates) - min(rates)) / float(np.mean(rates)) if rates else None}
    return float(2.0 * trees * len(result["times"]) / sum(result["times"])), detail


def reference_trees(args):
    return int(min(args.trees, max(os.cpu_count() or 1, 1)))


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    trees = reference_trees(args)
    t0 = time.perf_counter()
    value, detail = time_reference(args, os.path.join(ROOT, "oracle", "_ref"), trees, max(args.steps, 1),
                                   max(args.warmup, 1 if args.patterns >= 50000 else 0))
    elapsed = time.perf_counter() - t0
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / max(args.steps, 1),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_of(args),
        "cpu_baseline": dict(detail, value=value, unit=UNIT),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- legs of our arm

def measure_traffic(args):
    """DRAM bytes of ONE gradient-walk launch on a 148-tree batch of the same workload,
    measured in this run by ncu (two metrics, one pass set; the number printed by the
    probe process itself is discarded).  Returns (bytes per tree, source) or (None, why)."""
    probe_trees = 148
    with tempfile.TemporaryDirectory() as tmp:
        log = os.path.join(tmp, "traffic.csv")
        command = ["ncu", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none",
                   "--print-units", "base",
                   "--kernel-name-base", "demangled", "-k", WALK_KERNEL_REGEX, "-c", "1", "--csv",
                   "--log-file", log, sys.executable, os.path.abspath(__file__), "--_traffic-probe",
                   "--taxa", str(args.taxa), "--patterns", str(args.patterns), "--trees", str(probe_trees)]
        try:
            subprocess.run(command, capture_output=True, text=True, timeout=600, cwd=ROOT)
            total = 0.0
            found = 0
            for row in open(log):
                cells = [c.strip('"') for c in row.strip().split('","')]
                if len(cells) > 3 and cells[-3].startswith("dram__bytes_"):
                    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}[cells[-2]]
                    total += float(cells[-1].replace(",", "")) * scale
                    found += 1
            if found == 2 and total > 0:
                return total / probe_trees, (f"ncu dram__bytes_read.sum + dram__bytes_write.sum of one "
                                             f"{WALK_KERNEL} launch on {probe_trees} trees, measured in this run")
        except (OSError, subprocess.SubprocessError, ValueError, KeyError):
            pass
    return committed_traffic(args)


def committed_traffic(args):
    """DRAM bytes per tree of the committed ncu capture of the same kernel and workload."""
    name = "r02_treewalk_v6_ncu_summary.json"
    profile = os.path.join(ROOT, "profiles", name)
    if os.path.exists(profile) and (args.taxa, args.patterns) == (100, 100000):
        summary = json.load(open(profile))
        return summary.get("dram_bytes_per_tree"), (f"profiles/{name} (ncu --set full on 148 trees of this "
                                                    f"workload, kernel source {summary.get('git_sha', '?')}; "
                                                    "not measured in this run)")
    return None, "not measured"


def traffic_probe(args):
    """The process measure_traffic() profiles: one gradient launch, nothing else."""
    import libsbn_b200 as sbn
    from libsbn_b200 import _capi
    states, weights, parent_ids, lengths, params = workload(args)
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+4", "none"), states, weights, 0)
    staged = engine.stage(sbn.TreeBatch(parent_ids, lengths), params)
    staged.run(_capi.MODE_BRANCH_GRADIENT, True)
    staged.fetch()


def config5_alignment(taxa, begin, end, block=125000):
    """Columns [begin, end) of the configs[4] alignment: iid uniform {A,C,G,T} with 1 % gap
    states, generated in byte arithmetic block by block (seed (5, block index)), so every
    rank builds exactly its own range of the same alignment."""
    parts = []
    for b in range(begin // block, (end + block - 1) // block):
        rng = np.random.default_rng([5, b])
        states = rng.integers(0, 4, size=(taxa, block), dtype=np.uint8)
        states[rng.integers(0, 100, size=(taxa, block), dtype=np.uint8) == 0] = 4
        lo, hi = max(begin, b * block), min(end, (b + 1) * block)
        parts.append(states[:, lo - b * block:hi - b * block])
    return np.ascontiguousarray(np.concatenate(parts, axis=1))


def config5_leg(args, world, rank, local_rank, timed, dist):
    """BASELINE.json configs[4], site patterns sharded across the ranks."""
    import torch
    import libsbn_b200 as sbn
    from libsbn_b200 import sharding, trees
    taxa, patterns, tree_count = args.config5_taxa, args.config5_patterns, args.config5_trees
    begin, end = sharding.pattern_range(rank, world, patterns)
    local_states = config5_alignment(taxa, begin, end)
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=5)
    # row layout (blocks sorted by name, as the reference does): 4 frequencies, kappa; Weibull shape
    params = np.tile(np.array([0.1, 0.2, 0.3, 0.4, 2.0, 0.5]), (tree_count, 1))
    spec = sbn.PhyloModelSpecification("HKY", "weibull+4", "none")
    # every rank's engine holds only its own columns; the reduction is the sharded engine's
    engine = sharding.PatternShardedEngine(spec, local_states, np.ones(end - begin), local_rank, presharded=True)
    batch = sbn.TreeBatch(parent_ids, lengths)
    step = lambda: engine.gradients(batch, params, rescaling=True, substitution_gradient=False)
    result = step()
    engine.engine.walk_timing(reset=True)
    steps = max(1, min(args.steps, 3))
    ms = timed(step, steps)
    walk_ms, walk_samples = engine.engine.walk_timing(reset=True)
    kernel_ms = walk_ms / max(walk_samples, 1)
    result = step()
    logl = np.array([g.log_likelihood for g in result])
    leg = {
        "workload": f"synthetic {taxa} taxa x {patterns} site patterns, HKY+weibull4, {tree_count} trees, logL + "
                    "branch gradients, rescaling on (BASELINE.json configs[4])",
        "sharding": f"site patterns across {world} rank(s), {end - begin} per GPU; one NCCL sum-all-reduce of "
                    f"[{tree_count}] logL + [{tree_count} x {2 * taxa - 1}] x 2 gradient sums per call"
                    if world > 1 else "one GPU holds all site patterns (no collective)",
        "value": tree_count * steps / (ms * 1e-3), "unit": UNIT, "ms_per_call": ms / steps,
        "timing": "CUDA events on the engine's stream around the public call (staging + walk + all-reduce + "
                  "host finishing), max over ranks",
        "kernel_ms_this_rank": kernel_ms,
        "algorithmic_GBps_all_gpus": (10 * taxa - 14) * 32 * 4 * patterns * tree_count / (ms / steps * 1e-3) / 1e9,
        "mean_log_likelihood": float(np.mean(logl)),
    }
    if world > 1:
        mine = torch.tensor(logl, device="cuda", dtype=torch.float64)
        others = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(others, mine)
        leg["ranks_agree_bitwise"] = bool(all(torch.equal(o, mine) for o in others))
    if rank == 0:
        # oracle check of this run's inputs: tree 0 over a pattern range inside rank 0's shard
        from oracle import phylo
        lo, hi = 1000, 1300
        sub = sbn.Engine(spec, local_states[:, lo:hi], np.ones(hi - lo), local_rank)
        got = sub.gradients(sbn.TreeBatch(parent_ids[:1], lengths[:1]), params[:1], rescaling=True,
                            substitution_gradient=False)[0]
        raw = np.array([1, 2, 1, 1, 2, 1.0])
        want = phylo.gradients("GTR", "weibull+4", local_states[:, lo:hi], np.ones(hi - lo), parent_ids[:1],
                               lengths[:1], np.array([list(raw / raw.sum()) + [0.1, 0.2, 0.3, 0.4, 0.5]]),
                               rescaling=True)
        leg["oracle_check"] = {
            "what": f"tree 0 over patterns [{lo}, {hi}) of this run's alignment against the CPU oracle",
            "logl_rel_err": float(abs(got.log_likelihood - want["log_likelihood"][0]) / abs(want["log_likelihood"][0])),
            "gradient_rel_err": float(np.max(np.abs(got.gradient["branch_lengths"] - want["branch"][0])) /
                                      np.max(np.abs(want["branch"][0])))}
        assert leg["oracle_check"]["logl_rel_err"] < 1e-10 and leg["oracle_check"]["gradient_rel_err"] < 1e-8
    return leg


def small_problem_leg(local_rank):
    """DS1 x 100 topologies from the committed reference fixtures: call latency through
    the C ABI with host buffers, beside the CPU oracle port on all host cores."""
    import libsbn_b200 as sbn
    from oracle import phylo
    golden = os.path.join(ROOT, "tests", "golden")
    cores = os.cpu_count() or 1
    out = {"what": "DS1 (27 taxa x 934 site patterns), wall time of one public call with host buffers (median of "
                   "20 after 3 warm-up calls; the trees of a call are unchanged between calls, the branch lengths "
                   "are not)", "cpu": f"oracle port (oracle/phylo_oracle.cpp) on {cores} threads, median of 5",
           "cases": []}
    cases = [("JC69 log_likelihoods (configs[0])", "ds1_100_topologies_jc69", False),
             ("GTR+weibull4 phylo_gradients: logL + branch + site-model + substitution-model gradients (configs[1])",
              "ds1_100_topologies_gtr_weibull4", True)]
    for label, name, gradient in cases:
        with np.load(os.path.join(golden, name + ".npz"), allow_pickle=False) as data:
            fx = {k: (data[k].item() if data[k].ndim == 0 else data[k]) for k in data.files}
        spec = sbn.PhyloModelSpecification(fx["substitution"], fx["site"], fx["clock"])
        engine = sbn.Engine(spec, fx["patterns"], fx["weights"], local_rank)
        rng = np.random.default_rng(0)
        for tree_count in (10, 100):
            ids, params = fx["parent_ids"][:tree_count], fx["params"][:tree_count]
            base = fx["branch_lengths"][:tree_count]

            def call(lengths):
                batch = sbn.TreeBatch(ids, lengths)
                return engine.gradients(batch, params, True) if gradient else \
                    engine.log_likelihoods(batch, params, False)

            def cpu(lengths):
                if gradient:
                    return phylo.gradients(fx["substitution"], fx["site"], fx["patterns"], fx["weights"], ids,
                                           lengths, params, rescaling=True, threads=cores)
                return phylo.log_likelihoods(fx["substitution"], fx["site"], fx["patterns"], fx["weights"], ids,
                                             lengths, params, rescaling=False, threads=cores)

            def median_seconds(f, repeats, warmup):
                samples = []
                for i in range(warmup + repeats):
                    lengths = base * (1.0 + 0.01 * rng.random(base.shape))  # new lengths, same topologies
                    lengths[:, -1] = base[:, -1]
                    t0 = time.perf_counter()
                    f(lengths)
                    samples.append(time.perf_counter() - t0)
                return float(np.median(samples[warmup:]))

            gpu_s, cpu_s = median_seconds(call, 20, 3), median_seconds(cpu, 5, 1)
            out["cases"].append({"case": label, "trees": tree_count, "gpu_us_per_call": gpu_s * 1e6,
                                 "gpu_trees_per_s": tree_count / gpu_s, "cpu_us_per_call": cpu_s * 1e6,
                                 "cpu_trees_per_s": tree_count / cpu_s, "speedup": cpu_s / gpu_s})
    return out


def partial_update_leg(local_rank):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import beagle_shim_bench
    return beagle_shim_bench.measure(device=local_rank)


def gp_leg(local_rank):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gp_bench
    import gp_kernel_time
    out = {"device_ms_per_program": gp_kernel_time.measure(device=local_rank)}
    try:
        out["python_gp_instance"] = gp_bench.measure(repeats=5, iterations=5)
    except (OSError, RuntimeError, subprocess.SubprocessError, ValueError) as error:  # (artefacts not built)
        out["python_gp_instance"] = {"unavailable": str(error)[:200]}
    return out


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(directory, **per_tree):
    """Writes each per-tree array (first axis = trees) as directory/<name>.npy in fp64, so
    that two builds run with the same arguments -- hence the same seeded inputs -- can be
    compared output for output.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of
    the trees is written, and tree_index.npy says which."""
    trees = len(next(iter(per_tree.values())))
    row_bytes = sum(8 * np.asarray(a)[0].size for a in per_tree.values())
    keep = np.arange(trees)
    if trees * row_bytes > DUMP_LIMIT_BYTES:
        sample = (DUMP_LIMIT_BYTES - 4096) // (row_bytes + 8)  # (4096: room for the .npy headers)
        keep = np.sort(np.random.default_rng(0).choice(trees, sample, replace=False))
        per_tree = dict(per_tree, tree_index=keep)
    os.makedirs(directory, exist_ok=True)
    for name, array in per_tree.items():
        array = np.asarray(array) if name == "tree_index" else np.asarray(array)[keep]
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(array, dtype=np.float64))


# --------------------------------------------------------------------------- our arm

def run_ours(args):
    import torch
    import torch.distributed as dist
    import libsbn_b200 as sbn
    from libsbn_b200 import _capi, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    # stdout carries exactly one JSON line.  Libraries write to file descriptor 1 behind
    # Python's back (NCCL prints its version banner there in this image), so for the
    # duration of the run descriptor 1 points at stderr and the line goes to the saved one.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    states, weights, parent_ids, lengths, params = workload(args)
    begin, end = sharding.shard_range(rank, world, args.trees)
    shard = sbn.TreeBatch(parent_ids[begin:end], lengths[begin:end])
    shard_params = params[begin:end]
    engine = sbn.Engine(sbn.PhyloModelSpecification("GTR", "weibull+4", "none"), states, weights, local_rank)
    stream = torch.cuda.ExternalStream(engine.stream, device=local_rank)

    def timed(body, steps):
        """CUDA events on the engine's stream around `steps` calls of body(); max over ranks."""
        barrier()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            start.record()
            for _ in range(steps):
                body()
            stop.record()
        stop.synchronize()
        barrier()
        timed.local_ms = start.elapsed_time(stop)
        return max_over_ranks(timed.local_ms)

    # ---- value: inputs resident in HBM, kernels only ---------------------------------
    staged = engine.stage(shard, shard_params)
    run = lambda: staged.run(_capi.MODE_BRANCH_GRADIENT, True)
    for _ in range(args.warmup):
        run()
    engine.walk_timing(reset=True)
    launches_before = engine.launch_count
    with ClockSampler(local_rank) as clocks:
        ms = timed(run, args.steps)
    ms_local = timed.local_ms
    launches = engine.launch_count - launches_before
    walk_ms, walk_samples = engine.walk_timing(reset=True)
    value = args.trees * args.steps / (ms * 1e-3)
    logl_check, branch_gradients, rate_gradients = staged.fetch(gradients=True)
    local_trees = end - begin
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, log_likelihoods=logl_check[:local_trees],
                     branch_gradients=branch_gradients, rate_gradients=rate_gradients)

    # ---- roofline of the dominant kernel (gradient tree walk), this rank's launch -----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_source = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_source = 6650.0, "fallback (B200_PROFILING.md)"
    kernel_ms = walk_ms / max(walk_samples, 1)
    algorithmic_bytes = staged.algorithmic_bytes(_capi.MODE_BRANCH_GRADIENT)
    if world == 1 and not args.no_traffic_probe:
        traffic_per_tree, traffic_source = measure_traffic(args)
    else:
        # (ncu profiles one process on one GPU: multi-rank runs quote the committed capture)
        traffic_per_tree, traffic_source = committed_traffic(args)
    flops = FLOPS_PER_PATTERN_CATEGORY * (args.taxa / 100.0) * args.patterns * 4 * local_trees
    fp64_floor_ms = flops / FP64_PEAK * 1e3
    roofline = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_source,
                "kernel": WALK_KERNEL, "kernel_ms": kernel_ms,
                "kernel_share_of_step": walk_ms / (ms_local if world > 1 else ms),
                "traffic_source": traffic_source,
                "algorithmic_bytes_per_launch": algorithmic_bytes,
                "algorithmic_equiv_GBps": algorithmic_bytes / (kernel_ms * 1e-3) / 1e9,
                "algorithmic_equiv_frac": algorithmic_bytes / (kernel_ms * 1e-3) / 1e9 / peak,
                "fp64": {"flops_per_launch": flops, "peak_TFLOPs": FP64_PEAK / 1e12, "floor_ms": fp64_floor_ms,
                         "frac": fp64_floor_ms / kernel_ms},
                "note": "the fused walk keeps O(log n) partials on chip: its DRAM traffic (`traffic`, measured) is "
                        "a fraction of the ALGORITHMIC bytes of the reference's op-at-a-time schedule "
                        "((10n-14) x 32 C P per tree, every partial through HBM).  achieved = measured traffic / "
                        "kernel time and frac = achieved / peak are the kernel's real HBM utilisation = its "
                        "fraction of the bound that binds it (the HBM floor is above the fp64 floor); "
                        "algorithmic_equiv_* restate the speed in the reference schedule's bytes (> peak: not "
                        "an HBM measurement)"}
    if traffic_per_tree:
        traffic = traffic_per_tree * local_trees
        roofline.update(traffic=traffic, achieved=traffic / (kernel_ms * 1e-3) / 1e9,
                        frac=traffic / (kernel_ms * 1e-3) / 1e9 / peak,
                        hbm_floor_ms=traffic / (peak * 1e9) * 1e3)
    else:
        roofline.update(traffic=None, achieved=roofline["algorithmic_equiv_GBps"],
                        frac=roofline["algorithmic_equiv_frac"])

    # ---- the same batch, log-likelihood only (post-order sweep + root reduction) -----
    run_logl = lambda: staged.run(_capi.MODE_LOG_LIKELIHOOD, True)
    for _ in range(2):
        run_logl()
    engine.walk_timing(reset=True)
    logl_ms = timed(run_logl, args.steps)
    logl_walk_ms, logl_samples = engine.walk_timing(reset=True)
    logl_bytes = staged.algorithmic_bytes(_capi.MODE_LOG_LIKELIHOOD)
    logl_kernel_ms = logl_walk_ms / max(logl_samples, 1)
    logl_flops = 60.0 * (args.taxa - 1) * args.patterns * 4 * local_trees
    logl_only = {"value": args.trees * args.steps / (logl_ms * 1e-3), "unit": "logL evals/s",
                 "ms_per_step": logl_ms / args.steps,
                 "algorithmic_equiv_GBps": logl_bytes / (logl_kernel_ms * 1e-3) / 1e9,
                 "fp64_frac": logl_flops / FP64_PEAK * 1e3 / logl_kernel_ms,
                 "note": "no partial leaves the chip: bound by fp64 issue, not by HBM"}
    assert np.allclose(staged.fetch()[:local_trees], logl_check[:local_trees], rtol=1e-12)
    staged.close()

    # ---- e2e: the public call with host buffers ----------------------------------------
    call = lambda: engine.gradients(shard, shard_params, rescaling=True, substitution_gradient=False)
    for _ in range(min(args.warmup, 2)):
        results = call()
    h2d_before, d2h_before = engine.transfer_bytes
    e2e_steps = max(1, min(args.steps, 5))
    e2e_ms = timed(call, e2e_steps)
    h2d_after, d2h_after = engine.transfer_bytes
    e2e_value = args.trees * e2e_steps / (e2e_ms * 1e-3)
    assert np.allclose([g.log_likelihood for g in results], logl_check[:len(results)], rtol=1e-12)
    e2e = {"value": e2e_value, "unit": UNIT, "steps": e2e_steps,
           "h2d_bytes_per_step": int(max_over_ranks((h2d_after - h2d_before) / e2e_steps) * world),
           "d2h_bytes_per_step": int(max_over_ranks((d2h_after - d2h_before) / e2e_steps) * world)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(args, world), "clocks": clocks.summary(), "e2e": e2e,
        "gpu_launches": int(launches) * world, "roofline": roofline, "log_likelihood_only": logl_only,
        "mean_log_likelihood": float(np.mean(logl_check[:local_trees])),
    }

    if not args.quick:
        # ---- the reference's full GTR phylo_gradients through the public call ------------
        full = lambda: engine.gradients(shard, shard_params, rescaling=True, substitution_gradient=True)
        line["e2e_full_phylo_gradients"] = {
            "unit": "trees/s",
            "what": "logL + branch + site-model + substitution-model gradients through the public call; the "
                    "substitution block either exactly, inside the gradient sweep (analytic: W = sum of w/lik "
                    "(V^T T)(V^-1 L)^T o Phi over edges, categories and patterns, contracted with V^-1 dQ/dtheta V "
                    "on the host), or by the reference's 16 central-difference log-likelihood sweeps per tree "
                    "(finite_differences; fat_beagle.cpp:400-465)"}
        for mode, key in (("analytic", "analytic"), ("fd", "finite_differences")):
            engine.set_substitution_gradient(mode)
            full()
            full_steps = max(1, min(args.steps, 2))
            full_ms = timed(full, full_steps)
            line["e2e_full_phylo_gradients"][key] = {
                "value": args.trees * full_steps / (full_ms * 1e-3),
                "ms_per_tree_per_gpu": full_ms / full_steps / max(local_trees, 1)}
        engine.set_substitution_gradient("analytic")
        line["e2e_full_phylo_gradients"]["value"] = line["e2e_full_phylo_gradients"]["analytic"]["value"]

        # ---- weak scaling beside the strong headline (N > 1) ---------------------------
        if world > 1:
            _, _, ids_w, lengths_w, params_w = workload(args, seed=4 + rank)
            staged_w = engine.stage(sbn.TreeBatch(ids_w, lengths_w), params_w)
            run_w = lambda: staged_w.run(_capi.MODE_BRANCH_GRADIENT, True)
            run_w()
            weak_steps = max(1, min(args.steps, 3))
            weak_ms = timed(run_w, weak_steps)
            staged_w.close()
            line["weak_scaling"] = {"value": args.trees * world * weak_steps / (weak_ms * 1e-3), "unit": UNIT,
                                    "trees_per_gpu": args.trees,
                                    "what": f"{args.trees} trees on EVERY rank (rank r's batch drawn with seed 4 + r)"}

        # ---- BASELINE configs[4]: site patterns sharded, NCCL all-reduce ---------------
        line["config5"] = config5_leg(args, world, rank, local_rank, timed, dist)

        # ---- BASELINE configs[0..1]: the small-problem regime (one GPU) ----------------
        if world == 1:
            line["small_problem"] = small_problem_leg(local_rank)
            # ---- BASELINE's second metric on the materialised (BEAGLE-compatible) schedule,
            #      and configs[2]: generalized pruning on the DS1 DAG ----------------------
            line["partial_update"] = partial_update_leg(local_rank)
            line["gp"] = gp_leg(local_rank)

    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        sample_trees = reference_trees(args)
        cpu_value, detail = time_reference(args, os.path.join(ROOT, "oracle", "_ref"), sample_trees, 3, 1)
        line["cpu_baseline"] = dict(detail, value=cpu_value, unit=UNIT)
        v3_dir = os.path.join(ROOT, "oracle", "_ref", "v3")
        if os.path.isdir(v3_dir):
            try:
                v3_value, v3_detail = time_reference(args, v3_dir, sample_trees, 2, 1)
                line["cpu_baseline"]["x86_64_v3_build"] = {
                    "value": v3_value, "unit": UNIT, "spread": v3_detail["spread"],
                    "what": "the same measurement with the BEAGLE-equivalent kernels compiled -march=x86-64-v3 "
                            "(AVX2 + FMA, auto-vectorised) instead of the SSE2-class default"}
            except (RuntimeError, subprocess.SubprocessError, ValueError):
                pass
    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=5)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--impl", default="ours", choices=["ours", "reference"])
    parser.add_argument("--taxa", type=int, default=100)
    parser.add_argument("--patterns", type=int, default=100000)
    parser.add_argument("--trees", type=int, default=1024)
    parser.add_argument("--config5-taxa", type=int, default=1000)
    parser.add_argument("--config5-patterns", type=int, default=1000000)
    parser.add_argument("--config5-trees", type=int, default=8)
    parser.add_argument("--no-cpu-baseline", action="store_true")
    parser.add_argument("--no-traffic-probe", action="store_true")
    parser.add_argument("--quick", action="store_true",
                        help="headline, logL-only and e2e legs only (development A/B runs)")
    parser.add_argument("--dump-outputs", metavar="DIR", default=None,
                        help="write the log-likelihoods and gradients of the last timed step as DIR/<name>.npy")
    # internal modes (child processes of this script)
    parser.add_argument("--_reference-worker", dest="reference_worker", action="store_true", help=argparse.SUPPRESS)
    parser.add_argument("--_traffic-probe", dest="traffic_probe", action="store_true", help=argparse.SUPPRESS)
    parser.add_argument("--module-dir", default="", help=argparse.SUPPRESS)
    parser.add_argument("--cores", type=int, default=1, help=argparse.SUPPRESS)
    args = parser.parse_args()
    if args.steps < 1:
        parser.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        parser.error("--dump-outputs needs --impl ours in a single process")
    args.warmup = max(args.warmup, 0)
    if args.reference_worker:
        reference_worker(args)
    elif args.traffic_probe:
        traffic_probe(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
