"""Host mirror of the reference's SitePattern (src/site_pattern.hpp): an alignment
compressed into unique site patterns and their multiplicities, computed on the
device through sbnb_compress_site_patterns (include/sbn_b200_patterns.h).

    pattern = SitePattern(sequences)          # list of equal-length strings, leaf-id order,
                                              # or a C-contiguous uint8 array [taxon][site] of characters
    engine = Engine(spec, pattern.patterns, pattern.weights)

    pattern = SitePattern(sequences, ambiguity=True)   # IUPAC nucleotide masks
    engine = Engine(spec, pattern.patterns, pattern.weights, tip_encoding="masks")
"""
import ctypes

import numpy as np

from . import _capi


class SitePattern:
    """patterns: uint8 [taxon][pattern] (0..3 = ACGT, 4 = gap; with ambiguity=True the
    IUPAC nucleotide masks 1..15), weights: float64 [pattern]; patterns are in order of
    first appearance in the alignment."""

    def __init__(self, sequences, device=0, ambiguity=False):
        if isinstance(sequences, np.ndarray) and sequences.ndim == 2 and sequences.dtype == np.uint8:
            # the characters as they lie in memory: no host copy
            keep = np.ascontiguousarray(sequences)
            rows, length = range(keep.shape[0]), keep.shape[1]
            flat = keep.ctypes.data_as(ctypes.c_char_p)
        else:
            rows = [s.encode() if isinstance(s, str) else (s if isinstance(s, bytes) else bytes(s)) for s in sequences]
            if rows:
                length = len(rows[0])
                if any(len(r) != length for r in rows):
                    # Alignment::Length (alignment.hpp) asserts this in the reference
                    raise RuntimeError("Sequences of the alignment are not all of the same length.")
                flat = b"".join(rows)
        if not len(rows):
            raise RuntimeError("Site pattern compression needs at least one sequence.")
        self.sequence_count, self.site_count = len(rows), length
        patterns = np.empty(max(len(rows) * length, 1), dtype=np.uint8)
        weights = np.empty(max(length, 1), dtype=np.float64)
        count, device_ms = ctypes.c_int64(), ctypes.c_double()
        encoding = _capi.TIPS_NUCLEOTIDE_MASKS if ambiguity else _capi.TIPS_STATES
        _capi.check(_capi.load().sbnb_compress_site_patterns_encoded(
            len(rows), length, flat, encoding, device, patterns.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
            _capi.as_double_ptr(weights), ctypes.byref(count), ctypes.byref(device_ms)))
        self.ambiguity = ambiguity
        self.pattern_count = count.value
        # (no second copy of an alignment that did not shrink)
        self.patterns = patterns[:len(rows) * count.value].reshape(len(rows), count.value)
        self.weights = weights[:count.value]
        if count.value < length:
            self.patterns, self.weights = self.patterns.copy(), self.weights.copy()
        self.device_ms = device_ms.value
