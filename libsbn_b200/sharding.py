"""Multi-GPU sharding of the likelihood path: one process per GPU, the two
natural axes of SURVEY.md 8(e) / BASELINE.json's north star.

* Tree axis (`TreeShardedEngine`): the trees of a collection are independent
  (the reference already fans them over a thread pool, fat_beagle.hpp:119-149),
  so rank r evaluates a contiguous slice and the per-tree results are
  all-gathered.  No data-path collective.
* Site-pattern axis (`PatternShardedEngine`): every rank holds a contiguous
  range of site patterns and walks ALL trees over it; the per-pattern ratios of
  the edge derivatives are formed before the reduction, so the only exchange is
  one sum-all-reduce of [T] log-likelihoods and [T x (2n-1)] gradient sums
  (fp64), after which every rank runs the O(n) host finishing
  (sbnb_finish_gradients).  With the nccl backend the all-reduce runs in place on
  the engine's device result arrays, ordered on the engine's stream; with gloo
  (CPU tests) it runs on host copies.

`torch.distributed` is plumbing here: process group, NCCL over NVLink, gloo on CPU.
"""
import ctypes

import numpy as np

from . import _capi
from .engine import Engine, PhyloGradient, TreeBatch


def shard_range(rank, world, count):
    """Contiguous, balanced [begin, end) of `count` units for `rank` of `world`."""
    if not (0 <= rank < world):
        raise RuntimeError(f"rank {rank} out of range for world size {world}.")
    return rank * count // world, (rank + 1) * count // world


def pattern_range(rank, world, pattern_count):
    """Pattern shard of a rank; every rank must own at least one pattern
    (sbnb_engine_set_pattern_range rejects an empty range)."""
    if pattern_count < world:
        raise RuntimeError(f"Cannot shard {pattern_count} site patterns over {world} ranks.")
    return shard_range(rank, world, pattern_count)


def _dist():
    import torch.distributed as dist
    return dist


def _world():
    dist = _dist()
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size(), dist.get_backend()
    return 0, 1, None


def all_reduce_sum_host(*arrays):
    """Sum-all-reduce of host fp64 arrays (in place) over the default process
    group: one flat buffer, one collective.  gloo reduces on the host; with nccl
    the buffer takes a round trip through the current CUDA device."""
    rank, world, backend = _world()
    if world == 1:
        return
    import torch
    flat = np.concatenate([a.ravel() for a in arrays])
    tensor = torch.from_numpy(flat)
    if backend == "nccl":
        tensor = tensor.cuda()
    _dist().all_reduce(tensor, op=_dist().ReduceOp.SUM)
    flat = tensor.cpu().numpy()
    offset = 0
    for a in arrays:
        a[...] = flat[offset:offset + a.size].reshape(a.shape)
        offset += a.size


def all_gather_rows(local, total_rows):
    """local: this rank's [shard_range rows, width] fp64 slab -> [total_rows, width] on every rank."""
    rank, world, backend = _world()
    if world == 1:
        return local
    import torch
    width = local.shape[1]
    counts = [shard_range(r, world, total_rows)[1] - shard_range(r, world, total_rows)[0] for r in range(world)]
    if local.shape[0] != counts[rank]:
        raise RuntimeError(f"rank {rank} holds {local.shape[0]} rows, expected {counts[rank]}.")
    padded = np.zeros((max(counts), width))
    padded[:local.shape[0]] = local
    tensor = torch.from_numpy(padded)
    if backend == "nccl":
        tensor = tensor.cuda()
    gathered = [torch.empty_like(tensor) for _ in range(world)]
    _dist().all_gather(gathered, tensor)
    return np.concatenate([g.cpu().numpy()[:c] for g, c in zip(gathered, counts)], axis=0)


class _DeviceArrayView:
    """A device fp64 array owned by libsbn_b200.so, exposed to torch through
    __cuda_array_interface__ so that NCCL can reduce it in place."""

    def __init__(self, pointer, count):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (pointer, False),
                                         "version": 2, "strides": None}


class TreeShardedEngine:
    """Engine whose batch calls evaluate this rank's slice of the trees and
    all-gather the per-tree results, so every rank returns the whole batch."""

    def __init__(self, specification, patterns, weights, device=0, tip_encoding="states"):
        self.rank, self.world, self.backend = _world()
        self.engine = Engine(specification, patterns, weights, device, tip_encoding=tip_encoding)

    def local_slice(self, trees, params):
        begin, end = shard_range(self.rank, self.world, trees.tree_count)
        return begin, end, trees.slice(begin, end), (None if params is None else params[begin:end])

    def log_likelihoods(self, trees, params=None, rescaling=False, rooted=False):
        _, _, local_trees, local_params = self.local_slice(trees, params)
        local = self.engine.log_likelihoods(local_trees, local_params, rescaling, rooted)
        return all_gather_rows(local[:, None], trees.tree_count)[:, 0]

    def site_log_likelihoods(self, trees, params=None, rescaling=False, rooted=False):
        """(logL [T], site log-likelihoods [T][P]) on every rank: the local rows, all-gathered."""
        _, _, local_trees, local_params = self.local_slice(trees, params)
        logl, sites = self.engine.site_log_likelihoods(local_trees, local_params, rescaling, rooted)
        rows = all_gather_rows(np.concatenate([logl[:, None], sites], axis=1), trees.tree_count)
        return rows[:, 0].copy(), np.ascontiguousarray(rows[:, 1:])

    def gradients(self, trees, params=None, rescaling=False, rooted=False, substitution_gradient=True):
        _, _, local_trees, local_params = self.local_slice(trees, params)
        local = self.engine.gradients(local_trees, local_params, rescaling, rooted, substitution_gradient)
        return gather_gradients(local, trees.tree_count, self._keys(rooted, substitution_gradient, trees))

    def _keys(self, rooted, substitution_gradient, trees):
        """(key, width) of every gradient block, known without looking at local
        results (a rank may own zero trees)."""
        n = self.engine.taxon_count
        spec = self.engine.specification
        keys = [("ratios_root_height", n - 1), ("clock_model", trees.rate_count)] if rooted \
            else [("branch_lengths", 2 * n - 1)]
        fd = {"GTR": 8, "HKY": 4}.get(spec.substitution, 0) if substitution_gradient else 0
        if fd:
            keys.append(("substitution_model", fd))
        if self.engine.category_count > 1 or self.engine.invariant:
            keys.append(("site_model", self.engine.site_gradient_size))
        return keys


def gather_gradients(local, tree_count, keys):
    """Packs PhyloGradients into rows, all-gathers, unpacks."""
    width = 1 + sum(w for _, w in keys)
    rows = np.zeros((len(local), width))
    for i, g in enumerate(local):
        rows[i, 0] = g.log_likelihood
        offset = 1
        for key, w in keys:
            rows[i, offset:offset + w] = g.gradient[key]
            offset += w
    rows = all_gather_rows(rows, tree_count)
    out = []
    for row in rows:
        gradient, offset = {}, 1
        for key, w in keys:
            gradient[key] = row[offset:offset + w].copy()
            offset += w
        out.append(PhyloGradient(float(row[0]), gradient))
    return out


def finish_gradients(specification, taxon_count, trees, rooted, with_substitution_fd, log_likelihoods,
                     branch_gradients, rate_gradients, category_count):
    """sbnb_finish_gradients: raw (already reduced) sums -> PhyloGradients.  Host only."""
    lib = _capi.load()
    T, n = trees.tree_count, taxon_count
    fd_size = {"GTR": 8, "HKY": 4}.get(specification.substitution, 0) if with_substitution_fd else 0
    buffers = {"log_likelihood": np.zeros(T)}
    if rooted:
        buffers["ratios_root_height"] = np.zeros((T, n - 1))
        buffers["clock_model"] = np.zeros((T, trees.rate_count))
    else:
        buffers["branch_lengths"] = np.zeros((T, 2 * n - 1))
    if fd_size:
        buffers["substitution_model"] = np.zeros((T, fd_size))
    if category_count > 1:
        buffers["site_model"] = np.zeros((T, 1))
    out = _capi.GradientOutStruct()
    for key, value in buffers.items():
        setattr(out, key, _capi.as_double_ptr(value))
    struct = trees.as_struct()
    log_likelihoods = np.ascontiguousarray(log_likelihoods, dtype=np.float64)
    branch_gradients = np.ascontiguousarray(branch_gradients, dtype=np.float64)
    rate_gradients = None if rate_gradients is None else np.ascontiguousarray(rate_gradients, dtype=np.float64)
    _capi.check(lib.sbnb_finish_gradients(
        specification.substitution.encode(), specification.site.encode(), specification.clock.encode(), n,
        ctypes.byref(struct), int(rooted), int(bool(fd_size)), _capi.as_double_ptr(log_likelihoods),
        _capi.as_double_ptr(branch_gradients), _capi.as_double_ptr(rate_gradients), ctypes.byref(out)))
    return [PhyloGradient(float(buffers["log_likelihood"][t]),
                          {k: v[t].copy() for k, v in buffers.items() if k != "log_likelihood"}) for t in range(T)]


def finish_gradients_analytic(specification, taxon_count, trees, rooted, params, log_likelihoods,
                              branch_gradients, rate_gradients, substitution_sums, category_count):
    """sbnb_finish_gradients_analytic: raw (already reduced) sums, among them the [T][20]
    substitution sums -> PhyloGradients with an exact "substitution_model" block.  Host only."""
    lib = _capi.load()
    T, n = trees.tree_count, taxon_count
    size = {"GTR": 8, "HKY": 4}.get(specification.substitution, 0)
    buffers = {"log_likelihood": np.zeros(T)}
    if rooted:
        buffers["ratios_root_height"] = np.zeros((T, n - 1))
        buffers["clock_model"] = np.zeros((T, trees.rate_count))
    else:
        buffers["branch_lengths"] = np.zeros((T, 2 * n - 1))
    if size:
        buffers["substitution_model"] = np.zeros((T, size))
    if category_count > 1:
        buffers["site_model"] = np.zeros((T, 1))
    out = _capi.GradientOutStruct()
    for key, value in buffers.items():
        setattr(out, key, _capi.as_double_ptr(value))
    struct = trees.as_struct()
    as_array = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    params, log_likelihoods, branch_gradients = as_array(params), as_array(log_likelihoods), as_array(branch_gradients)
    rate_gradients, substitution_sums = as_array(rate_gradients), as_array(substitution_sums)
    _capi.check(lib.sbnb_finish_gradients_analytic(
        specification.substitution.encode(), specification.site.encode(), specification.clock.encode(), n,
        ctypes.byref(struct), int(rooted), _capi.as_double_ptr(params), _capi.as_double_ptr(log_likelihoods),
        _capi.as_double_ptr(branch_gradients), _capi.as_double_ptr(rate_gradients),
        _capi.as_double_ptr(substitution_sums), ctypes.byref(out)))
    return [PhyloGradient(float(buffers["log_likelihood"][t]),
                          {k: v[t].copy() for k, v in buffers.items() if k != "log_likelihood"}) for t in range(T)]


def finish_gradients_invariant(specification, taxon_count, trees, rooted, params, log_likelihoods,
                               branch_gradients, rate_gradients, substitution_sums, invariant_sums, category_count,
                               site_gradient_size):
    """sbnb_finish_gradients_invariant: raw (already reduced) sums of a +I model, among them the
    [T][5] invariant sums (and, if not None, the [T][20] substitution sums) -> PhyloGradients whose
    "site_model" row ends with d logL / d proportion invariant.  Host only."""
    lib = _capi.load()
    T, n = trees.tree_count, taxon_count
    size = {"GTR": 8, "HKY": 4}.get(specification.substitution, 0) if substitution_sums is not None else 0
    buffers = {"log_likelihood": np.zeros(T)}
    if rooted:
        buffers["ratios_root_height"] = np.zeros((T, n - 1))
        buffers["clock_model"] = np.zeros((T, trees.rate_count))
    else:
        buffers["branch_lengths"] = np.zeros((T, 2 * n - 1))
    if size:
        buffers["substitution_model"] = np.zeros((T, size))
    buffers["site_model"] = np.zeros((T, site_gradient_size))
    out = _capi.GradientOutStruct()
    for key, value in buffers.items():
        setattr(out, key, _capi.as_double_ptr(value))
    struct = trees.as_struct()
    as_array = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    params, log_likelihoods, branch_gradients = as_array(params), as_array(log_likelihoods), as_array(branch_gradients)
    rate_gradients = as_array(rate_gradients) if category_count > 1 else None
    substitution_sums, invariant_sums = as_array(substitution_sums), as_array(invariant_sums)
    _capi.check(lib.sbnb_finish_gradients_invariant(
        specification.substitution.encode(), specification.site.encode(), specification.clock.encode(), n,
        ctypes.byref(struct), int(rooted), _capi.as_double_ptr(params), _capi.as_double_ptr(log_likelihoods),
        _capi.as_double_ptr(branch_gradients), _capi.as_double_ptr(rate_gradients),
        _capi.as_double_ptr(substitution_sums), _capi.as_double_ptr(invariant_sums), ctypes.byref(out)))
    return [PhyloGradient(float(buffers["log_likelihood"][t]),
                          {k: v[t].copy() for k, v in buffers.items() if k != "log_likelihood"}) for t in range(T)]


def finish_log_likelihoods_rooted(taxon_count, trees, log_likelihoods):
    """sbnb_finish_log_likelihoods_rooted: + log-det Jacobian (fat_beagle.cpp:82-94), in place."""
    struct = trees.as_struct()
    _capi.check(_capi.load().sbnb_finish_log_likelihoods_rooted(taxon_count, ctypes.byref(struct),
                                                                 _capi.as_double_ptr(log_likelihoods)))
    return log_likelihoods


class PatternShardedEngine:
    """Engine restricted to this rank's range of site patterns; batch calls walk
    ALL trees over the local patterns and sum-all-reduce the raw results."""

    def __init__(self, specification, patterns, weights, device=0, presharded=False, tip_encoding="states"):
        """presharded: `patterns` / `weights` are already this rank's columns only (an
        alignment too large to build on every rank); otherwise every rank passes the
        whole alignment and keeps its range of it.  tip_encoding as for Engine."""
        self.rank, self.world, self.backend = _world()
        self.specification = specification
        self.engine = Engine(specification, patterns, weights, device, tip_encoding=tip_encoding)
        self.presharded = presharded
        if presharded:
            self.begin, self.end = 0, self.engine.pattern_count
        else:
            self.begin, self.end = pattern_range(self.rank, self.world, self.engine.pattern_count)
            if self.world > 1:
                self.engine.set_pattern_range(self.begin, self.end)

    def _reduce(self, staged, arrays_wanted, substitution_sums=False, invariant_sums=False):
        """All-reduce of the raw result arrays of a finished run, then fetch
        (arrays_wanted: 1 = log-likelihoods, 3 = + edge and rate derivatives;
        substitution_sums: + the [T][20] sums of the analytic substitution gradient;
        invariant_sums: + the [T][5] sums of a +I model, which follow them on the device)."""
        lib = _capi.load()
        if self.world > 1 and self.backend == "nccl":
            import torch
            pointers = [ctypes.c_void_p() for _ in range(3)]
            _capi.check(lib.sbnb_batch_device_results(staged._handle, *[ctypes.byref(p) for p in pointers]))
            # The three result arrays are one contiguous fp64 array on the device:
            # [evaluations] log-likelihoods, [T x (2n-1)] edge derivatives and, with more than
            # one rate category, [T x (2n-1)] rate derivatives -- one collective.
            T, N = staged.tree_count, staged.node_count
            if invariant_sums:
                count = lib.sbnb_batch_evaluation_count(staged._handle) + 2 * T * N + \
                    (_capi.SUBSTITUTION_SUMS + _capi.INVARIANT_SUMS) * T
            elif substitution_sums:
                count = lib.sbnb_batch_evaluation_count(staged._handle) + 2 * T * N + _capi.SUBSTITUTION_SUMS * T
            elif arrays_wanted > 1:
                count = lib.sbnb_batch_evaluation_count(staged._handle) + (2 if pointers[2].value else 1) * T * N
            else:
                count = T
            stream = torch.cuda.ExternalStream(self.engine.stream, device=self.engine.device)
            with torch.cuda.stream(stream):  # NCCL is ordered after the walk kernels on the engine's stream
                view = torch.as_tensor(_DeviceArrayView(pointers[0].value, count), device=f"cuda:{self.engine.device}")
                _dist().all_reduce(view, op=_dist().ReduceOp.SUM)
            stream.synchronize()
            result = staged.fetch(gradients=arrays_wanted > 1)
            if substitution_sums:
                result = (*result, staged.fetch_substitution_sums())
            return (*result, staged.fetch_invariant_sums()) if invariant_sums else result
        result = staged.fetch(gradients=arrays_wanted > 1)
        arrays = list(result) if arrays_wanted > 1 else [result]
        if substitution_sums:
            arrays.append(staged.fetch_substitution_sums())
        if invariant_sums:
            arrays.append(staged.fetch_invariant_sums())
        all_reduce_sum_host(*arrays)
        return tuple(arrays) if arrays_wanted > 1 else arrays[0]

    def log_likelihoods(self, trees, params=None, rescaling=False, rooted=False):
        staged = self.engine.stage(trees, params, rooted=rooted)
        staged.run(_capi.MODE_LOG_LIKELIHOOD, rescaling)
        logl = self._reduce(staged, 1)
        staged.close()
        if rooted:
            finish_log_likelihoods_rooted(self.engine.taxon_count, trees, logl)
        return logl

    def site_log_likelihoods(self, trees, params=None, rescaling=False, rooted=False):
        """(logL [T], site log-likelihoods [T][pattern_count]) on every rank: the log-likelihoods
        sum-all-reduced, this rank's [T][P_r] columns all-gathered (transposed: the ranks' rows are
        their pattern ranges, which follow shard_range)."""
        if self.presharded:
            raise RuntimeError("site_log_likelihoods needs the whole alignment on every rank (presharded=False).")
        staged = self.engine.stage(trees, params, rooted=rooted, site_log_likelihoods=True)
        staged.run(_capi.MODE_LOG_LIKELIHOOD, rescaling)
        logl = self._reduce(staged, 1)
        local = staged.fetch_site_log_likelihoods()
        staged.close()
        if rooted:
            finish_log_likelihoods_rooted(self.engine.taxon_count, trees, logl)
        return logl, np.ascontiguousarray(all_gather_rows(np.ascontiguousarray(local.T), self.engine.pattern_count).T)

    def gradients(self, trees, params=None, rescaling=False, rooted=False, substitution_gradient=True):
        wanted = substitution_gradient and self.specification.substitution in ("GTR", "HKY")
        analytic = wanted and self.engine.substitution_gradient_mode == "analytic"
        fd = wanted and not analytic
        staged = self.engine.stage(trees, params, rooted=rooted, substitution_fd=fd, substitution_analytic=analytic)
        staged.run(_capi.MODE_BRANCH_GRADIENT, rescaling)
        if self.engine.invariant:
            if fd:
                staged.close()
                raise RuntimeError("A +I site model takes the analytic substitution gradient across pattern shards.")
            arrays = self._reduce(staged, 3, substitution_sums=analytic, invariant_sums=True)
            staged.close()
            logl, grad, rgrad = arrays[:3]
            return finish_gradients_invariant(self.specification, self.engine.taxon_count, trees, rooted,
                                              self.engine._params(params, trees.tree_count), logl, grad, rgrad,
                                              arrays[3] if analytic else None, arrays[-1], self.engine.category_count,
                                              self.engine.site_gradient_size)
        if analytic:
            logl, grad, rgrad, sums = self._reduce(staged, 3, substitution_sums=True)
            staged.close()
            return finish_gradients_analytic(self.specification, self.engine.taxon_count, trees, rooted,
                                             self.engine._params(params, trees.tree_count), logl, grad, rgrad, sums,
                                             self.engine.category_count)
        logl, grad, rgrad = self._reduce(staged, 3)
        staged.close()
        return finish_gradients(self.specification, self.engine.taxon_count, trees, rooted, fd, logl, grad, rgrad,
                                self.engine.category_count)


__all__ = ["TreeShardedEngine", "PatternShardedEngine", "shard_range", "pattern_range", "all_reduce_sum_host",
           "all_gather_rows", "finish_gradients", "finish_gradients_analytic", "finish_gradients_invariant",
           "finish_log_likelihoods_rooted", "gather_gradients", "TreeBatch"]
