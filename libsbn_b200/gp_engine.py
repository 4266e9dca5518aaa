"""Host-side mirror of the reference's GPEngine (src/gp_engine.hpp:20-207) over
the C ABI of include/sbn_b200_gp.h.

Same method names and argument meaning as the reference (snake_case of
ProcessOperations, SetBranchLengths, GetPerGPCSPLogLikelihoods, ...); a failed
Assert inside an operation surfaces as RuntimeError like the reference's
Failwith (sugar.hpp:67-78).  The op program is the flat int32 encoding of
GPOperationVector (gp_operation.hpp:25-171) described in the header; `GPOperations`
below builds it with the reference's op names.  There is no CPU fallback: every
call runs on the device or raises.
"""
import ctypes

import numpy as np

from . import _capi


class GPOperations:
    """Encoders, one per reference GPOperation struct (gp_operation.hpp:25-171)."""

    @staticmethod
    def ZeroPLV(dest):
        return [0, dest]

    @staticmethod
    def SetToStationaryDistribution(dest, root_gpcsp_idx):
        return [1, dest, root_gpcsp_idx]

    @staticmethod
    def IncrementWithWeightedEvolvedPLV(dest, gpcsp, src):
        return [2, dest, gpcsp, src]

    @staticmethod
    def Multiply(dest, src1, src2):
        return [3, dest, src1, src2]

    @staticmethod
    def Likelihood(dest, child, parent):
        return [4, dest, child, parent]

    @staticmethod
    def OptimizeBranchLength(leafward, rootward, gpcsp):
        return [5, leafward, rootward, gpcsp]

    @staticmethod
    def UpdateSBNProbabilities(start, stop):
        return [6, start, stop]

    @staticmethod
    def ResetMarginalLikelihood():
        return [7]

    @staticmethod
    def IncrementMarginalLikelihood(stationary_times_prior, rootsplit, p):
        return [8, stationary_times_prior, rootsplit, p]

    @staticmethod
    def PrepForMarginalization(dest, src_vector):
        return [9, dest, len(src_vector), *src_vector]

    @staticmethod
    def program(operations):
        """Concatenates encoded operations into one int32 program."""
        words = [w for op in operations for w in op]
        return np.array(words, dtype=np.int32)


def schedule_program(plv_count, gpcsp_count, program):
    """The schedule the device runs for `program` (sbnb_gp_schedule_program; host only): runs of
    increments into one PLV fused (internal kind 10; bit 30 of word 0 = "fresh" / count-only ZeroPLV), the
    records re-ordered by dependency level, the first record of a batch tagged with its length in bits 8..15."""
    import ctypes
    program = np.ascontiguousarray(program, dtype=np.int32)
    out = np.empty_like(program)
    count = ctypes.c_int64(0)
    _capi.check(_capi.load().sbnb_gp_schedule_program(int(plv_count), int(gpcsp_count), _capi.as_int32_ptr(program),
                                                      program.size, _capi.as_int32_ptr(out), ctypes.byref(count)))
    return out[:count.value].copy()


def _tips(tips):
    """QuartetTipVector (quartet_hybrid_request.hpp): records (tip_node_id, plv_idx, gpcsp_idx)."""
    array = np.ascontiguousarray(np.array(tips, dtype=np.int32).reshape(-1, 3))
    return array, _capi.as_int32_ptr(array), array.shape[0]


class GPEngine:
    """GPEngine::GPEngine (gp_engine.cpp:9-46) with PLVs resident in HBM instead of an mmapped file."""

    default_rescaling_threshold = 1e-40  # gp_engine.hpp:86
    default_branch_length = 0.1  # gp_engine.hpp:87

    def __init__(self, tip_states, pattern_weights, site_count, plv_count, gpcsp_count,
                 rescaling_threshold=default_rescaling_threshold, sbn_prior=None,
                 unconditional_node_probabilities=None, inverted_sbn_prior=None, device=0, tip_encoding="states"):
        """tip_encoding: "states" (0..3 = ACGT, 4 = gap) or "masks" (nucleotide masks 1..15:
        leaf PLV entry s = bit s of the tip's mask)."""
        self._lib = _capi.load()
        encoding = _capi.tip_encoding(tip_encoding)
        tip_states = np.ascontiguousarray(tip_states, dtype=np.uint8)
        if tip_states.ndim != 2:
            raise ValueError("tip_states must be [taxon][pattern]")
        weights = np.ascontiguousarray(pattern_weights, dtype=np.float64)
        if weights.shape != (tip_states.shape[1],):
            raise ValueError("pattern_weights must have one entry per site pattern")

        def optional(vector, length, name):
            if vector is None or len(vector) == 0:
                return None
            vector = np.ascontiguousarray(vector, dtype=np.float64)
            if vector.shape != (length,):
                raise ValueError(f"{name} must have length {length}")
            return vector

        self.taxon_count, self.pattern_count = tip_states.shape
        self.plv_count, self.gpcsp_count = int(plv_count), int(gpcsp_count)
        nodes = None if unconditional_node_probabilities is None else np.ascontiguousarray(
            unconditional_node_probabilities, dtype=np.float64)
        self.node_count = 0 if nodes is None else nodes.shape[0]
        prior = optional(sbn_prior, self.gpcsp_count, "sbn_prior")
        inverted = optional(inverted_sbn_prior, self.gpcsp_count, "inverted_sbn_prior")
        handle = ctypes.c_void_p()
        _capi.check(self._lib.sbnb_gp_create_encoded(
            self.taxon_count, self.pattern_count, tip_states.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
            encoding, _capi.as_double_ptr(weights), int(site_count), self.plv_count, self.gpcsp_count,
            float(rescaling_threshold), _capi.as_double_ptr(prior), _capi.as_double_ptr(nodes), self.node_count,
            _capi.as_double_ptr(inverted), int(device), ctypes.byref(handle)))
        self._handle = handle

    def close(self):
        if getattr(self, "_handle", None):
            self._lib.sbnb_gp_destroy(self._handle)
            self._handle = None

    def __del__(self):
        self.close()

    def set_substitution_model(self, substitution, params=()):
        """"JC69" (the reference's only GP model, gp_engine.hpp:143-154), "GTR" (6 rates + 4 frequencies) or
        "HKY" (4 frequencies + kappa): an addition to the reference's interface."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        _capi.check(self._lib.sbnb_gp_set_substitution_model(self._handle, substitution.encode(),
                                                             _capi.as_double_ptr(params), params.size))

    def set_site_model(self, site, params=()):
        """"constant", "weibull+K" or "gamma+K" (K = 1, 2, 4, 8) rate categories: an addition to the
        reference's interface.  Resets the PLVs; get_plv then returns [pattern][K * 4]."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        _capi.check(self._lib.sbnb_gp_set_site_model(self._handle, site.encode(), _capi.as_double_ptr(params),
                                                     params.size))

    @property
    def category_count(self):
        return int(self._lib.sbnb_gp_category_count(self._handle))

    # ---- ProcessOperations (gp_engine.cpp:167-171)
    def process_operations(self, program):
        program = np.ascontiguousarray(program, dtype=np.int32)
        _capi.check(self._lib.sbnb_gp_process_operations(self._handle, _capi.as_int32_ptr(program), program.size))

    # ---- setters / getters (gp_engine.cpp:193-235)
    def _get(self, function, count):
        out = np.empty(count, dtype=np.float64)
        _capi.check(function(self._handle, _capi.as_double_ptr(out)))
        return out

    def _set(self, function, values, count, what):
        values = np.ascontiguousarray(values, dtype=np.float64)
        if values.shape != (count,):
            raise RuntimeError(f"Size mismatch in GPEngine::{what}.")
        _capi.check(function(self._handle, _capi.as_double_ptr(values)))

    def set_branch_lengths(self, branch_lengths):
        self._set(self._lib.sbnb_gp_set_branch_lengths, branch_lengths, self.gpcsp_count, "SetBranchLengths")

    def set_branch_lengths_to_constant(self, branch_length):
        _capi.check(self._lib.sbnb_gp_set_branch_lengths_to_constant(self._handle, float(branch_length)))

    def get_branch_lengths(self):
        return self._get(self._lib.sbnb_gp_get_branch_lengths, self.gpcsp_count)

    def reset_log_marginal_likelihood(self):
        _capi.check(self._lib.sbnb_gp_reset_log_marginal_likelihood(self._handle))

    def get_log_marginal_likelihood(self):
        return float(self._get(self._lib.sbnb_gp_get_log_marginal_likelihood, 1)[0])

    def get_per_gpcsp_log_likelihoods(self, start=0, length=None):
        length = self.gpcsp_count - start if length is None else length
        out = np.empty(length, dtype=np.float64)
        _capi.check(self._lib.sbnb_gp_get_per_gpcsp_log_likelihoods(self._handle, int(start), int(length),
                                                                    _capi.as_double_ptr(out)))
        return out

    def get_per_gpcsp_components_of_full_log_marginal(self):
        return self._get(self._lib.sbnb_gp_get_per_gpcsp_components_of_full_log_marginal, self.gpcsp_count)

    def get_log_likelihood_matrix(self):
        return self._get(self._lib.sbnb_gp_get_log_likelihood_matrix,
                         self.gpcsp_count * self.pattern_count).reshape(self.gpcsp_count, self.pattern_count)

    def get_sbn_parameters(self):
        return self._get(self._lib.sbnb_gp_get_sbn_parameters, self.gpcsp_count)

    def set_sbn_parameters(self, q):
        self._set(self._lib.sbnb_gp_set_sbn_parameters, q, self.gpcsp_count, "SetSBNParameters")

    def get_hybrid_marginals(self):
        return self._get(self._lib.sbnb_gp_get_hybrid_marginals, self.gpcsp_count)

    def set_hybrid_marginals(self, values):
        self._set(self._lib.sbnb_gp_set_hybrid_marginals, values, self.gpcsp_count, "SetHybridMarginals")

    # ---- LogLikelihoodAndDerivative (gp_engine.cpp:244-266); op = OptimizeBranchLength fields
    def log_likelihood_and_derivative(self, leafward, rootward, gpcsp):
        out = np.empty(2, dtype=np.float64)
        _capi.check(self._lib.sbnb_gp_log_likelihood_and_derivative(self._handle, int(leafward), int(rootward),
                                                                    int(gpcsp), _capi.as_double_ptr(out)))
        return float(out[0]), float(out[1])

    # ---- SetTransitionMatrixToHaveBranchLength + GetTransitionMatrix (gp_engine.cpp:173-176)
    def transition_matrix(self, branch_length):
        out = np.empty(16, dtype=np.float64)
        _capi.check(self._lib.sbnb_gp_transition_matrix(self._handle, float(branch_length), _capi.as_double_ptr(out)))
        return out.reshape(4, 4)

    # ---- quartet hybrid marginals (gp_engine.cpp:396-460)
    def calculate_quartet_hybrid_likelihoods(self, central_gpcsp, rootward_tips, sister_tips, rotated_tips,
                                             sorted_tips):
        lists = [_tips(t) for t in (rootward_tips, sister_tips, rotated_tips, sorted_tips)]
        count = 1
        for _, _, n in lists:
            count *= n
        out = np.empty(count, dtype=np.float64)
        args = [x for _, pointer, n in lists for x in (pointer, n)]
        _capi.check(self._lib.sbnb_gp_quartet_hybrid_likelihoods(self._handle, int(central_gpcsp), *args,
                                                                 _capi.as_double_ptr(out)))
        return out

    def process_quartet_hybrid_request(self, central_gpcsp, rootward_tips, sister_tips, rotated_tips, sorted_tips):
        lists = [_tips(t) for t in (rootward_tips, sister_tips, rotated_tips, sorted_tips)]
        args = [x for _, pointer, n in lists for x in (pointer, n)]
        _capi.check(self._lib.sbnb_gp_process_quartet_hybrid_request(self._handle, int(central_gpcsp), *args))

    # ---- diagnostics
    def get_plv(self, plv_idx):
        width = 4 * self.category_count
        out = np.empty(self.pattern_count * width, dtype=np.float64)
        _capi.check(self._lib.sbnb_gp_get_plv(self._handle, int(plv_idx), _capi.as_double_ptr(out)))
        return out.reshape(self.pattern_count, width)

    def get_rescaling_counts(self):
        out = np.empty(self.plv_count, dtype=np.int32)
        _capi.check(self._lib.sbnb_gp_get_rescaling_counts(self._handle, _capi.as_int32_ptr(out)))
        return out

    @property
    def launch_plan(self):
        """The interpreter's launch plan (sbnb_gp_debug_launch_plan): threads per CTA, CTAs, whether the
        grid is one cluster, and whether matrices / rescaling counts sit in shared memory."""
        out = np.zeros(6, dtype=np.int32)
        _capi.check(self._lib.sbnb_gp_debug_launch_plan(self._handle, _capi.as_int32_ptr(out)))
        return {"threads": int(out[0]), "blocks": int(out[1]), "cluster": bool(out[2]),
                "shared_matrices": bool(out[3]), "shared_counts": bool(out[4]), "scratch": int(out[5])}

    @property
    def launch_count(self):
        return int(self._lib.sbnb_gp_launch_count(self._handle))

    @property
    def last_kernel_ms(self):
        return float(self._lib.sbnb_gp_last_kernel_ms(self._handle))


def estimate_branch_lengths(engine, branch_length_optimization, populate_plvs, marginal_likelihood, tol, max_iter):
    """GPInstance::EstimateBranchLengths (gp_instance.cpp:129-175) over already
    scheduled programs.  Returns the marginal log likelihood after each pass."""
    engine.process_operations(populate_plvs)
    engine.process_operations(marginal_likelihood)
    current = engine.get_log_marginal_likelihood()
    trace = [current]
    per_iteration = np.concatenate([np.asarray(branch_length_optimization, dtype=np.int32),
                                    np.asarray(populate_plvs, dtype=np.int32),
                                    np.asarray(marginal_likelihood, dtype=np.int32)])
    for _ in range(max_iter):
        engine.process_operations(per_iteration)  # the three programs of one iteration in one launch
        updated = engine.get_log_marginal_likelihood()
        trace.append(updated)
        if abs(current - updated) < tol:
            break
        current = updated
    return trace
