"""The inner drop-in boundary (SURVEY.md 8b): libsbn_b200/lib/libhmsbeagle_b200.so, the 17
BEAGLE entry points of include/libhmsbeagle/beagle.h on the device
(libsbn_b200/csrc/beagle_shim.cu).

  * CPU: the library exports every function the header declares and fails loudly without a device;
  * GPU: the same call sequence -- the one fat_beagle.cpp makes for a log likelihood and a branch
    gradient (fat_beagle.cpp:50-70, 119-175) -- through the device library and through the CPU
    restatement (oracle/beagle_cpu.cpp, the test oracle pinned to the reference's goldens):
    compact tips and tip partials, gaps, 1 / 3 / 4 rate categories, rescaling on and off, a
    ragged pattern count;
  * GPU: the reference's own doctest suite, EVERY reference source unmodified (fat_beagle.cpp
    and engine.cpp included), linked against the device library (integration/Makefile).
"""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT
import test_integration_gpu as integration

from libsbn_b200.beagle import (Beagle, LIB_PATH as SHIM, depth_first_operations, gtr_eigensystem,
                                random_tree_operations)

ORACLE = os.path.join(ROOT, "oracle", "_build", "libbeagle_oracle.so")


def _declared():
    header = open(os.path.join(ROOT, "include", "libhmsbeagle", "beagle.h")).read()
    return sorted(set(re.findall(r"^int (beagle[A-Za-z]+)\(", header, flags=re.M)))


def test_library_exports_every_declared_symbol():
    declared = _declared()
    assert len(declared) == 17
    lib = ctypes.CDLL(SHIM)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in beagle.h but not exported"


def test_no_device_means_no_resource_not_a_cpu_fallback():
    import libsbn_b200._capi as capi
    if capi.load().sbnb_device_count() > 0:
        pytest.skip("a CUDA device is present")
    lib = ctypes.CDLL(SHIM)
    handle = lib.beagleCreateInstance(3, 7, 3, 4, 10, 1, 10, 1, 8, None, 0, 0, 0, None)
    assert handle == -6  # BEAGLE_ERROR_NO_RESOURCE


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["libsbn", "node_id"])
@pytest.mark.parametrize("categories,use_tip_states,rescaling", [(1, True, False), (4, True, True), (4, False, False),
                                                                 (3, True, True), (4, True, False), (20, True, True)])
def test_device_library_against_the_cpu_restatement(categories, use_tip_states, rescaling, order):
    rng = np.random.default_rng(categories * 10 + use_tip_states * 2 + rescaling)
    n, P = 13, 1003
    states = rng.integers(0, 4, size=(n, P)).astype(np.int32)
    states[rng.random(states.shape) < 0.05] = 4
    weights = rng.integers(1, 6, size=P).astype(np.float64)
    post, pre = random_tree_operations(n, rng, rescaling, order)
    lengths = rng.exponential(0.1, size=2 * n - 1)
    evec, ivec, evals, freqs, q = gtr_eigensystem()
    rates = np.sort(rng.gamma(2.0, 0.5, size=categories))
    rates /= rates.mean()
    proportions = np.full(categories, 1.0 / categories)
    results = []
    for path in (SHIM, ORACLE):
        beagle = Beagle(path, n, P, categories, use_tip_states)
        beagle.set_tips(states, weights, use_tip_states)
        beagle.set_model(evec, ivec, evals, freqs, rates, proportions)
        results.append(beagle.log_likelihood_and_gradient(post, pre, lengths, q, rates, freqs, rescaling))
        # a second evaluation on the same instance with other lengths (buffers are reused)
        results.append(beagle.log_likelihood_and_gradient(post, pre, lengths * 1.7, q, rates, freqs, rescaling))
        beagle.close()
    for ours, want in ((results[0], results[2]), (results[1], results[3])):
        assert abs(ours[0] - want[0]) <= 1e-12 * abs(want[0])
        np.testing.assert_allclose(ours[1], want[1], rtol=1e-10, atol=1e-9)
        np.testing.assert_allclose(ours[2], want[2], rtol=1e-10, atol=1e-9)
        np.testing.assert_allclose(ours[3], want[3], rtol=1e-10, atol=1e-11)


@pytest.mark.gpu
def test_reference_doctest_suite_passes_over_the_device_beagle_library():
    """reference src/doctest.cpp with EVERY reference source unmodified -- fat_beagle.cpp, engine.cpp,
    site_pattern.cpp, ... -- and libhmsbeagle replaced by libhmsbeagle_b200.so at link time."""
    integration._compare_with_reference_build("doctest_beagle", ("likelihood", "gradients", "time trees"), 42,
                                              reference_name="doctest")
    with open(integration._artefact("doctest_beagle"), "rb") as handle:
        binary = handle.read()
    assert b"beagleUpdatePrePartials" in binary  # the reference's FatBeagle is what runs


@pytest.mark.gpu
@pytest.mark.parametrize("categories,variant", [(4, "depth_first"), (4, "cumulative_is_written"), (2, "depth_first"),
                                                (8, "depth_first"), (1, "both_children_forwarded")])
def test_partial_update_op_lists_the_pipelined_kernel_special_cases(categories, variant):
    """Op lists longer than one staged chunk, in depth-first order (register forwarding at nearly every
    op), with an op whose scale buffer IS the cumulative buffer (the sums then go through memory), and
    with an op whose two children are both the previous destination: root log likelihoods through the
    device library and the CPU restatement."""
    rng = np.random.default_rng(categories * 7 + len(variant))
    n, P = 41, 515
    states = rng.integers(0, 4, size=(n, P)).astype(np.int32)
    states[rng.random(states.shape) < 0.05] = 4
    weights = rng.integers(1, 4, size=P).astype(np.float64)
    post, _ = random_tree_operations(n, rng, True, "node_id")
    post = depth_first_operations(post, n)
    assert len(post) == n - 1 > 32
    if variant == "cumulative_is_written":
        post[5][1] = 0
    if variant == "both_children_forwarded":
        post[7][3] = post[7][5] = post[6][0]
        post[7][4] = post[7][6] = post[6][0]
    lengths = rng.exponential(0.1, size=2 * n - 1)
    evec, ivec, evals, freqs, q = gtr_eigensystem()
    rates = np.sort(rng.gamma(2.0, 0.5, size=categories))
    rates /= rates.mean()
    values = []
    for path in (SHIM, ORACLE):
        beagle = Beagle(path, n, P, categories, True)
        beagle.set_tips(states, weights, True)
        beagle.set_model(evec, ivec, evals, freqs, rates, np.full(categories, 1.0 / categories))
        keep_i, idx = beagle._i(np.arange(2 * n - 2))
        keep_l, lens = beagle._d(lengths[:2 * n - 2])
        beagle.ok(beagle.lib.beagleUpdateTransitionMatrices(beagle.handle, 0, idx, None, None, lens, 2 * n - 2))
        for repeat in range(2):  # (the second call adds onto the cumulative buffer the first one left)
            if repeat == 0:
                beagle.ok(beagle.lib.beagleResetScaleFactors(beagle.handle, 0))
            keep_a, ops = beagle._i(post)
            beagle.ok(beagle.lib.beagleUpdatePartials(beagle.handle, ops, len(post), 0))
            keep_r, root = beagle._i([2 * n - 2])
            keep_z, zero = beagle._i([0])
            logl = ctypes.c_double()
            beagle.ok(beagle.lib.beagleCalculateRootLogLikelihoods(beagle.handle, root, zero, zero, zero, 1,
                                                                   ctypes.byref(logl)))
            values.append(logl.value)
        beagle.close()
    assert np.all(np.isfinite(values))
    np.testing.assert_allclose(values[:2], values[2:], rtol=1e-13)
