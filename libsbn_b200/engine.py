"""Host-side mirror of the reference's likelihood `Engine` (src/engine.hpp:26-53)
over the C ABI of libsbn_b200.so.

Method names, argument meaning and error behaviour follow the reference:
`log_likelihoods`, `unrooted_log_likelihoods`, `gradients` take a tree
collection, a trees x params row-major parameter matrix and a `rescaling` flag
and return one value / one PhyloGradient per tree; failures raise RuntimeError
(the reference's Failwith).  Trees are passed in flat form (`TreeBatch`).
"""
import ctypes
import os
from dataclasses import dataclass, field
from typing import Dict, Optional

import numpy as np

from . import _capi


@dataclass
class PhyloModelSpecification:
    """src/phylo_model.hpp:13-17."""
    substitution: str = "JC69"
    site: str = "constant"
    clock: str = "none"


@dataclass
class PhyloGradient:
    """src/tree_gradient.hpp:10-19."""
    log_likelihood: float
    gradient: Dict[str, np.ndarray] = field(default_factory=dict)


@dataclass
class TreeBatch:
    """A tree collection in flat form (see include/sbn_b200.h, sbnb_tree_batch).

    parent_ids[t] is Node::ParentIdVector of tree t, branch_lengths[t] is indexed
    by node id.  The rooted fields mirror RootedTree's members.
    """
    parent_ids: np.ndarray
    branch_lengths: np.ndarray
    rates: Optional[np.ndarray] = None
    node_heights: Optional[np.ndarray] = None
    node_bounds: Optional[np.ndarray] = None
    height_ratios: Optional[np.ndarray] = None
    rate_count: int = 1

    def __post_init__(self):
        self.parent_ids = np.ascontiguousarray(self.parent_ids, dtype=np.int32)
        self.branch_lengths = np.ascontiguousarray(self.branch_lengths, dtype=np.float64)
        if self.parent_ids.ndim != 2 or self.branch_lengths.ndim != 2:
            raise RuntimeError("parent_ids and branch_lengths must be 2-D (trees x nodes).")
        if self.parent_ids.shape[0] != self.branch_lengths.shape[0] or \
                self.parent_ids.shape[1] + 1 != self.branch_lengths.shape[1]:
            raise RuntimeError("parent_ids must be [T][nodes-1] and branch_lengths [T][nodes].")
        for name in ("rates", "node_heights", "node_bounds", "height_ratios"):
            value = getattr(self, name)
            if value is not None:
                setattr(self, name, np.ascontiguousarray(value, dtype=np.float64))

    @property
    def tree_count(self):
        return self.parent_ids.shape[0]

    @property
    def node_count(self):
        return self.branch_lengths.shape[1]

    def slice(self, begin, end):
        """Trees [begin, end) -- the tree-sharding axis."""
        pick = lambda a: None if a is None else a[begin:end]
        return TreeBatch(self.parent_ids[begin:end], self.branch_lengths[begin:end], pick(self.rates),
                         pick(self.node_heights), pick(self.node_bounds), pick(self.height_ratios),
                         self.rate_count)

    def as_struct(self):
        s = _capi.TreeBatchStruct()
        s.tree_count = self.tree_count
        s.node_count = self.node_count
        s.parent_ids = _capi.as_int32_ptr(self.parent_ids)
        s.branch_lengths = _capi.as_double_ptr(self.branch_lengths)
        s.rates = _capi.as_double_ptr(self.rates)
        s.node_heights = _capi.as_double_ptr(self.node_heights)
        s.node_bounds = _capi.as_double_ptr(self.node_bounds)
        s.height_ratios = _capi.as_double_ptr(self.height_ratios)
        s.rate_count = self.rate_count
        return s


class StagedBatch:
    """A tree collection staged in device memory (sbnb_batch)."""

    def __init__(self, engine, handle, tree_count, node_count):
        self._engine = engine
        self._handle = handle
        self.tree_count = tree_count
        self.node_count = node_count  # 2n-1

    def run(self, mode=_capi.MODE_LOG_LIKELIHOOD, rescaling=False):
        """Enqueue one pass on the engine's stream (no copies, no sync)."""
        _capi.check(_capi.load().sbnb_batch_run(self._engine._handle, self._handle, mode, int(rescaling)))

    def fetch(self, gradients=False):
        lib = _capi.load()
        count = lib.sbnb_batch_evaluation_count(self._handle)
        logl = np.empty(count, dtype=np.float64)
        grad = np.empty((self.tree_count, self.node_count)) if gradients else None
        rgrad = np.empty((self.tree_count, self.node_count)) if gradients else None
        _capi.check(lib.sbnb_batch_fetch(self._engine._handle, self._handle, _capi.as_double_ptr(logl),
                                         _capi.as_double_ptr(grad), _capi.as_double_ptr(rgrad)))
        return (logl, grad, rgrad) if gradients else logl

    def fetch_substitution_sums(self):
        """[T][20] sums of the analytic substitution gradient (batch staged for them)."""
        sums = np.empty((self.tree_count, _capi.SUBSTITUTION_SUMS))
        _capi.check(_capi.load().sbnb_batch_fetch_substitution_sums(self._engine._handle, self._handle,
                                                                    _capi.as_double_ptr(sums)))
        return sums

    def fetch_invariant_sums(self):
        """[T][5] sums of the invariant class (D, E_A..E_T) of the last gradient run of a +I model."""
        sums = np.empty((self.tree_count, _capi.INVARIANT_SUMS))
        _capi.check(_capi.load().sbnb_batch_fetch_invariant_sums(self._engine._handle, self._handle,
                                                                 _capi.as_double_ptr(sums)))
        return sums

    def algorithmic_bytes(self, mode):
        return _capi.load().sbnb_batch_algorithmic_bytes(self._handle, mode)

    def close(self):
        if self._handle:
            _capi.load().sbnb_batch_destroy(self._engine._handle, self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    """B200 likelihood engine for one alignment and one phylo-model specification."""

    def __init__(self, specification, patterns, weights, device=0, devices=None, shard_axis="trees",
                 tip_encoding="states"):
        """device: one CUDA ordinal; or devices=[...]: a device group inside the library
        (sbnb_engine_create_multi: one host thread + stream per GPU), sharded by
        "trees" or by "patterns" (SURVEY.md 8e).  tip_encoding: "states" (0..3 = ACGT,
        anything >= 4 a gap) or "masks" (nucleotide masks, bit 0 = A .. bit 3 = T: an
        ambiguous character such as R = 5 enters as the partial vector of its states)."""
        lib = _capi.load()
        encoding = _capi.tip_encoding(tip_encoding)
        patterns = np.ascontiguousarray(patterns, dtype=np.uint8)
        weights = np.ascontiguousarray(weights, dtype=np.float64)
        if patterns.ndim != 2 or weights.shape != (patterns.shape[1],):
            raise RuntimeError("patterns must be [taxon][pattern] and weights [pattern].")
        self.specification = specification
        self.tip_encoding = tip_encoding
        self.taxon_count, self.pattern_count = patterns.shape
        handle = ctypes.c_void_p()
        common = (specification.substitution.encode(), specification.site.encode(),
                  specification.clock.encode(), self.taxon_count, self.pattern_count,
                  patterns.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), _capi.as_double_ptr(weights))
        common = common[:6] + (encoding,) + common[6:]
        if devices is None:
            _capi.check(lib.sbnb_engine_create_encoded(*common, device, ctypes.byref(handle)))
        else:
            if shard_axis not in ("trees", "patterns"):
                raise RuntimeError("shard_axis must be 'trees' or 'patterns'.")
            ordinals = np.ascontiguousarray(devices, dtype=np.int32)
            axis = _capi.SHARD_TREES if shard_axis == "trees" else _capi.SHARD_PATTERNS
            _capi.check(lib.sbnb_engine_create_multi_encoded(*common, _capi.as_int32_ptr(ordinals), len(ordinals),
                                                             axis, ctypes.byref(handle)))
            device = int(ordinals[0])
        self._handle = handle
        self.device = device
        self.device_count = lib.sbnb_engine_device_count(handle)
        self.substitution_gradient_mode = "fd" if os.environ.get("SBNB_SUBSTITUTION_GRADIENT") == "fd" else "analytic"
        self.param_count = lib.sbnb_engine_param_count(handle)
        self.category_count = lib.sbnb_engine_category_count(handle)
        self.invariant = specification.site.endswith("+I")
        # entries of a tree's "site_model" gradient: [shape | proportion invariant]
        self.site_gradient_size = max(1, self.param_block("entire site")[1])

    def set_substitution_gradient(self, mode):
        """'analytic' (default): exact d logL / d (substitution parameters) inside the
        gradient sweep; 'fd': the reference's 16 central-difference log-likelihood
        sweeps (fat_beagle.cpp:400-465)."""
        modes = {"analytic": _capi.SUBSTITUTION_ANALYTIC, "fd": _capi.SUBSTITUTION_FINITE_DIFFERENCES}
        if mode not in modes:
            raise RuntimeError("substitution gradient mode must be 'analytic' or 'fd'.")
        _capi.check(_capi.load().sbnb_engine_set_substitution_gradient(self._handle, modes[mode]))
        self.substitution_gradient_mode = mode

    def close(self):
        if getattr(self, "_handle", None):
            _capi.load().sbnb_engine_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- Engine::GetPhyloModelBlockSpecification --------------------------------
    def param_block(self, key):
        start, length = ctypes.c_int32(), ctypes.c_int32()
        _capi.check(_capi.load().sbnb_engine_param_block(self._handle, key.encode(), ctypes.byref(start),
                                                         ctypes.byref(length)))
        return start.value, length.value

    def param_block_map(self, params):
        """Views into a trees x params matrix by block name (get_phylo_model_param_block_map)."""
        out = {}
        for key in ("GTR rates", "frequencies", "kappa", "Weibull shape", "Gamma shape", "proportion invariant",
                    "clock rate", "entire substitution", "entire site", "entire clock", "entire"):
            try:
                start, length = self.param_block(key)
            except _capi.SbnbError:
                continue
            out[key] = params[:, start:start + length]
        return out

    def _params(self, params, tree_count):
        if params is None:
            params = np.zeros((tree_count, self.param_count))
        params = np.ascontiguousarray(params, dtype=np.float64)
        if params.shape != (tree_count, self.param_count):
            raise RuntimeError(
                f"phylo_model_params must be {tree_count} x {self.param_count}, got {params.shape}.")
        return params

    # -- the five Engine methods (engine.hpp:33-47) -----------------------------
    def log_likelihoods(self, trees, params=None, rescaling=False, rooted=False):
        """Engine::LogLikelihoods for an unrooted (default) or rooted collection."""
        lib = _capi.load()
        params = self._params(params, trees.tree_count)
        out = np.empty(trees.tree_count, dtype=np.float64)
        fn = lib.sbnb_log_likelihoods_rooted if rooted else lib.sbnb_log_likelihoods_unrooted
        struct = trees.as_struct()
        _capi.check(fn(self._handle, ctypes.byref(struct), _capi.as_double_ptr(params), int(rescaling),
                       _capi.as_double_ptr(out)))
        return out

    def unrooted_log_likelihoods(self, trees, params=None, rescaling=False):
        """Engine::UnrootedLogLikelihoods(RootedTreeCollection)."""
        params = self._params(params, trees.tree_count)
        out = np.empty(trees.tree_count, dtype=np.float64)
        struct = trees.as_struct()
        _capi.check(_capi.load().sbnb_unrooted_log_likelihoods_of_rooted(
            self._handle, ctypes.byref(struct), _capi.as_double_ptr(params), int(rescaling),
            _capi.as_double_ptr(out)))
        return out

    def gradients(self, trees, params=None, rescaling=False, rooted=False, substitution_gradient=True):
        """Engine::Gradients: one PhyloGradient per tree.  substitution_gradient=False
        skips the 16 finite-difference log-likelihood sweeps of a GTR model."""
        lib = _capi.load()
        T, n = trees.tree_count, self.taxon_count
        params = self._params(params, T)
        spec = self.specification
        fd_size = {"GTR": 8, "HKY": 4}.get(spec.substitution, 0) if substitution_gradient else 0
        buffers = {"log_likelihood": np.zeros(T)}
        if rooted:
            buffers["ratios_root_height"] = np.zeros((T, n - 1))
            buffers["clock_model"] = np.zeros((T, trees.rate_count))
        else:
            buffers["branch_lengths"] = np.zeros((T, 2 * n - 1))
        if fd_size:
            buffers["substitution_model"] = np.zeros((T, fd_size))
        if self.category_count > 1 or self.invariant:
            buffers["site_model"] = np.zeros((T, self.site_gradient_size))
        out = _capi.GradientOutStruct()
        for key, value in buffers.items():
            setattr(out, key, _capi.as_double_ptr(value))
        fn = lib.sbnb_gradients_rooted if rooted else lib.sbnb_gradients_unrooted
        struct = trees.as_struct()
        _capi.check(fn(self._handle, ctypes.byref(struct), _capi.as_double_ptr(params), int(rescaling),
                       ctypes.byref(out)))
        results = []
        for t in range(T):
            gradient = {k: v[t].copy() for k, v in buffers.items() if k != "log_likelihood"}
            results.append(PhyloGradient(float(buffers["log_likelihood"][t]), gradient))
        return results

    # -- staged form -------------------------------------------------------------
    def stage(self, trees, params=None, rooted=False, substitution_fd=False, substitution_analytic=False):
        params = self._params(params, trees.tree_count)
        flags = (_capi.STAGE_ROOTED if rooted else 0) | (_capi.STAGE_SUBSTITUTION_FD if substitution_fd else 0) | \
            (_capi.STAGE_SUBSTITUTION_ANALYTIC if substitution_analytic else 0)
        handle = ctypes.c_void_p()
        struct = trees.as_struct()
        _capi.check(_capi.load().sbnb_batch_stage(self._handle, ctypes.byref(struct),
                                                  _capi.as_double_ptr(params), flags, ctypes.byref(handle)))
        return StagedBatch(self, handle, trees.tree_count, 2 * self.taxon_count - 1)

    def set_pattern_range(self, begin, end):
        _capi.check(_capi.load().sbnb_engine_set_pattern_range(self._handle, begin, end))

    @property
    def stream(self):
        return _capi.load().sbnb_engine_stream(self._handle)

    @property
    def transfer_bytes(self):
        """(host->device, device->host) bytes copied so far."""
        h2d, d2h = ctypes.c_int64(), ctypes.c_int64()
        _capi.check(_capi.load().sbnb_engine_transfer_bytes(self._handle, ctypes.byref(h2d), ctypes.byref(d2h)))
        return h2d.value, d2h.value

    def walk_timing(self, reset=False):
        """(total ms, launches) of the tree-walk kernel since the last reset,
        from CUDA events around each launch; waits for outstanding launches."""
        total, samples = ctypes.c_double(), ctypes.c_int64()
        _capi.check(_capi.load().sbnb_engine_walk_timing(self._handle, ctypes.byref(total),
                                                         ctypes.byref(samples), int(reset)))
        return total.value, samples.value

    @property
    def launch_count(self):
        return _capi.load().sbnb_engine_launch_count(self._handle)
