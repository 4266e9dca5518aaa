"""Host side of 17 to 32 rate categories (no device needed): the discretised Weibull and
Gamma tables the fused walk reads, the host finishing of raw sums, and the refusal of counts
the walk cannot hold (one category per lane of a 32-lane warp)."""
import ctypes

import numpy as np
import pytest

import libsbn_b200 as sbn
from libsbn_b200 import _capi


def site_tables(site, shape):
    """Category rates, weights and d rate / d shape of a JC69 + `site` model."""
    lib = _capi.load()
    count = int(site.split("+")[1])
    out = {k: np.zeros(count) for k in ("rates", "weights", "drates")}
    row = np.array([shape])
    _capi.check(lib.sbnb_debug_model_tables(b"JC69", site.encode(), b"none", _capi.as_double_ptr(row),
                                            None, None, None, None, None,
                                            *[_capi.as_double_ptr(out[k]) for k in ("rates", "weights", "drates")]))
    return out


@pytest.mark.parametrize("count", [17, 20, 32])
@pytest.mark.parametrize("shape", [0.1, 0.5, 1.3, 7.0])
def test_weibull_tables(count, shape):
    """site_model.cpp:37-62: median discretisation, rates normalised to mean 1."""
    t = site_tables(f"weibull+{count}", shape)
    quantiles = (2.0 * np.arange(count) + 1.0) / (2.0 * count)
    rates = (-np.log(1.0 - quantiles)) ** (1.0 / shape)
    np.testing.assert_allclose(t["rates"], rates / rates.mean(), rtol=1e-12, atol=1e-300)
    assert np.array_equal(t["weights"], np.full(count, 1.0 / count))
    assert abs(t["rates"].mean() - 1) < 1e-14
    h = 1e-6 * shape
    numeric = (site_tables(f"weibull+{count}", shape + h)["rates"] -
               site_tables(f"weibull+{count}", shape - h)["rates"]) / (2 * h)
    np.testing.assert_allclose(t["drates"], numeric, rtol=1e-6, atol=1e-9 * np.abs(numeric).max())


@pytest.mark.parametrize("count", [17, 20, 32])
@pytest.mark.parametrize("shape", [0.1, 0.5, 1.3, 7.0])
def test_gamma_tables(count, shape):
    """Discrete Gamma against scipy.stats.gamma.ppf (oracle/phylo.py), which shares no code
    with the library's incomplete-gamma inverse."""
    from oracle import phylo
    t = site_tables(f"gamma+{count}", shape)
    rates, derivative = phylo.gamma_rates(shape, count)
    np.testing.assert_allclose(t["rates"], rates, rtol=1e-11, atol=1e-300)
    assert np.array_equal(t["weights"], np.full(count, 1.0 / count))
    assert abs(t["rates"].mean() - 1) < 1e-14
    assert np.abs(t["drates"] - derivative).max() <= 1e-6 * np.abs(derivative).max()
    h = 1e-6 * shape
    numeric = (site_tables(f"gamma+{count}", shape + h)["rates"] -
               site_tables(f"gamma+{count}", shape - h)["rates"]) / (2 * h)
    np.testing.assert_allclose(t["drates"], numeric, rtol=1e-5, atol=1e-8 * np.abs(numeric).max())


def test_host_finishing_takes_32_categories():
    """sbnb_finish_gradients (what ranks run after all-reducing raw sums) parses the model
    and finishes the site-model gradient the same way at 32 categories as at 4."""
    from libsbn_b200 import sharding, trees
    taxa, tree_count = 9, 3
    parent_ids, lengths = trees.random_tree_batch(taxa, tree_count, seed=1)
    batch = sbn.TreeBatch(parent_ids, lengths)
    rng = np.random.default_rng(2)
    N = 2 * taxa - 1
    logl, grad, rgrad = rng.normal(size=tree_count), rng.normal(size=(tree_count, N)), rng.normal(size=(tree_count, N))
    finished = [sharding.finish_gradients(sbn.PhyloModelSpecification("GTR", site, "none"), taxa, batch, False, False,
                                          logl, grad, rgrad, count)
                for site, count in (("weibull+4", 4), ("weibull+32", 32), ("gamma+32", 32))]
    for other in finished[1:]:
        for a, b in zip(other, finished[0]):
            assert a.log_likelihood == b.log_likelihood and set(a.gradient) == {"branch_lengths", "site_model"}
            assert all(np.array_equal(a.gradient[k], b.gradient[k]) for k in b.gradient)


@pytest.mark.parametrize("site", ["weibull+33", "gamma+33", "weibull+0", "gamma+100"])
def test_counts_outside_1_to_32_are_rejected_on_the_host(site):
    lib = _capi.load()
    out = (ctypes.c_double * 16)()
    code = lib.sbnb_debug_model_tables(b"JC69", site.encode(), b"none", (ctypes.c_double * 1)(0.5), out,
                                       None, None, None, None, None, None, None)
    message = lib.sbnb_last_error().decode()
    assert code == -1 and "out of range [1,32]" in message and site in message
    assert "libhmsbeagle_b200.so" in message
