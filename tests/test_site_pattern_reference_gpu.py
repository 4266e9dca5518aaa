"""Site-pattern compression on the device (libsbn_b200/csrc/site_pattern.cu) against the exact
reference (tests/site_pattern_reference.py) at the edges of its kernels.  Every result must be
the reference's exactly: the patterns byte for byte and in order, the weights bit for bit.

- taxon counts around the groups of 8 / 16 taxa of HashKernel and the 64-row chunks of
  TileKernel, times site counts around the groups of 4 sites, the 128-site tiles and the
  1024-site scan blocks, with first appearances that do and do not take EmitKernel's
  32-bit store;
- more than 1024 scan blocks (the carry of ScanSumsKernel);
- 65,536 sites and patterns, where the copies switch from one 2-D copy to row-by-row copies;
- key collisions (SBNB_DEBUG_PATTERN_KEY_BITS) predicted by the key mirror: a seed that
  collides must be retried without leaving stale state behind, a pair of columns that differ
  in one taxon must never be merged, and four colliding seeds must be refused;
- every byte value in both encodings, and which of several unknown characters is reported;
- every input form, and the refusals of the C ABI.
"""
import ctypes

import numpy as np
import pytest

import site_pattern_reference as ref
from libsbn_b200 import _capi
from libsbn_b200.site_pattern import SitePattern
from oracle import site_pattern as restatement

pytestmark = pytest.mark.gpu

TAXA = [1, 7, 8, 9, 15, 16, 17, 63, 64, 65, 128, 129]
SITES = [1, 3, 4, 5, 127, 128, 129, 1023, 1024, 1025]


def device(sequences, encoding):
    got = SitePattern(sequences, ambiguity=encoding == "masks")
    return got.patterns, got.weights


def assert_exact(got, want):
    patterns, weights = got
    assert patterns.dtype == np.uint8 and weights.dtype == np.float64
    assert patterns.shape == want[0].shape, (patterns.shape, want[0].shape)
    assert np.array_equal(patterns, want[0]), "patterns differ"
    assert np.array_equal(weights, want[1]), "weights differ"


def grid_case(taxa, sites, regime, encoding):
    rng = np.random.default_rng([taxa, sites, ref.REGIMES.index(regime), ref.ENCODINGS.index(encoding)])
    size = ref.pool_size(regime, sites)
    pool = ref.pool_columns(taxa, size, rng, encoding)
    return ref.alignment(pool, ref.site_picks(regime, sites, size, rng))


@pytest.mark.parametrize("sites", SITES)
@pytest.mark.parametrize("taxa", TAXA)
def test_boundary_grid(taxa, sites):
    for e, encoding in enumerate(ref.ENCODINGS):
        regime = ref.REGIMES[(TAXA.index(taxa) + SITES.index(sites) + 3 * e) % len(ref.REGIMES)]
        rows = grid_case(taxa, sites, regime, encoding)
        assert_exact(device(rows, encoding), ref.compress(rows, encoding))


@pytest.mark.parametrize("regime", ref.REGIMES)
def test_every_regime_on_a_subset_of_the_grid(regime):
    for taxa in (8, 64, 129):
        for sites in (5, 129, 1025):
            for encoding in ref.ENCODINGS:
                rows = grid_case(taxa, sites, regime, encoding)
                assert_exact(device(rows, encoding), ref.compress(rows, encoding))


@pytest.mark.parametrize("sites,regime", [(1_048_576, "distinct"), (1_048_577, "prefix1"), (3_200_003, "random")])
def test_scan_carry(sites, regime):
    """Exactly 1024 scan blocks of 1024 sites, then more: first appearances in blocks >= 1024 get
    the carry of ScanSumsKernel's second pass."""
    for encoding in ref.ENCODINGS:
        rng = np.random.default_rng([sites, ref.ENCODINGS.index(encoding)])
        pool = ref.pool_columns(12, sites, rng, encoding, digit_rows=12)
        picks = ref.site_picks(regime, sites, sites, rng)
        _, first = ref.first_uses(picks, sites)
        assert (first[-1] >= 1024 * 1024) == (sites > 1024 * 1024)
        assert_exact(device(ref.alignment(pool, picks), encoding), ref.by_construction(pool, picks, encoding))


@pytest.mark.parametrize("patterns", [65_535, 65_536, 65_537])
def test_pattern_counts_around_the_row_by_row_copy(patterns):
    for encoding in ref.ENCODINGS:
        rng = np.random.default_rng([patterns, ref.ENCODINGS.index(encoding)])
        pool = ref.pool_columns(8, patterns, rng, encoding)
        picks = ref.site_picks("cover", patterns + 12_345, patterns, rng)
        want = ref.by_construction(pool, picks, encoding)
        assert want[0].shape[1] == patterns
        assert_exact(device(ref.alignment(pool, picks), encoding), want)


@pytest.mark.parametrize("sites", [65_535, 65_536])
@pytest.mark.parametrize("regime", ["distinct", "prefix2", "random"])
def test_site_counts_around_the_row_by_row_copy(sites, regime):
    for encoding in ref.ENCODINGS:
        rng = np.random.default_rng([sites, ref.REGIMES.index(regime), ref.ENCODINGS.index(encoding)])
        size = ref.pool_size(regime, sites)
        pool = ref.pool_columns(17, size, rng, encoding)
        picks = ref.site_picks(regime, sites, size, rng)
        assert_exact(device(ref.alignment(pool, picks), encoding), ref.by_construction(pool, picks, encoding))


def test_the_bench_shape():
    """1000 taxa x 1M sites with 50k patterns, as bench.py compresses them."""
    rng = np.random.default_rng(20261022)
    pool = ref.pool_columns(1000, 50_000, rng, "states")
    picks = ref.site_picks("cover", 1_000_000, 50_000, rng)
    assert_exact(device(ref.alignment(pool, picks), "states"), ref.by_construction(pool, picks, "states"))


# ---- key collisions, as the mirror predicts them ---------------------------------------------

def with_key_bits(monkeypatch, bits, sequences, encoding):
    monkeypatch.setenv("SBNB_DEBUG_PATTERN_KEY_BITS", str(bits))
    try:
        return device(sequences, encoding)
    finally:
        monkeypatch.delenv("SBNB_DEBUG_PATTERN_KEY_BITS")


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
@pytest.mark.parametrize("target,seed", [((True, False, None, None), 1), ((True, True, True, False), 3)])
def test_a_later_seed_gives_the_exact_result(monkeypatch, encoding, target, seed):
    index, bits = ref.find_rehash_case(target, encoding)
    pool, picks = ref.rehash_alignment(index, encoding)
    want = ref.by_construction(pool, picks, encoding)
    assert ref.expected_outcome(want[0], encoding, bits) == seed
    assert_exact(with_key_bits(monkeypatch, bits, ref.alignment(pool, picks), encoding), want)


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
def test_four_colliding_seeds_are_refused(monkeypatch, encoding):
    # the widest keys at which every seed collides in this family
    index, bits = ref.find_rehash_case((True, True, True, True), encoding, bit_range=range(26, 13, -1))
    pool, picks = ref.rehash_alignment(index, encoding)
    assert ref.expected_outcome(ref.by_construction(pool, picks, encoding)[0], encoding, bits) is None
    assert ref.expected_outcome(ref.by_construction(pool, picks, encoding)[0], encoding, bits + 1) is not None
    with pytest.raises(_capi.SbnbError, match=r"^Site pattern hashing collided under four seeds\.$") as info:
        with_key_bits(monkeypatch, bits, ref.alignment(pool, picks), encoding)
    assert info.value.code == -3


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
@pytest.mark.parametrize("family", ["12 taxa", "129 taxa"])
def test_key_width_sweep_matches_the_mirror(monkeypatch, encoding, family):
    """At every width from 8 to 24 bits the device succeeds exactly when the mirror finds a clean seed.
    Each family member is the first whose sweep includes a width where seed 0 collides and a later one is clean."""
    shape = {} if family == "12 taxa" else dict(taxa=129, sites=3000, distinct=600)
    index, _ = ref.find_rehash_case((True, False, None, None), encoding, range(8, 25), **shape)
    pool, picks = ref.rehash_alignment(index, encoding, **shape)
    rows = ref.alignment(pool, picks)
    want = ref.by_construction(pool, picks, encoding)
    outcomes = {}
    for bits in range(8, 25):
        outcomes[bits] = ref.expected_outcome(want[0], encoding, bits)
        if outcomes[bits] is None:
            with pytest.raises(_capi.SbnbError, match="collided under four seeds"):
                with_key_bits(monkeypatch, bits, rows, encoding)
        else:
            assert_exact(with_key_bits(monkeypatch, bits, rows, encoding), want)
    # the sweep crosses from refusals to rehashes
    assert outcomes[8] is None and any(o not in (None, 0) for o in outcomes.values())


def pair_alignment(a, b, sites=37):
    picks = np.random.default_rng(sites).integers(0, 2, size=sites)
    picks[:2] = [1, 0]
    return ref.alignment(np.stack([a, b], axis=1), picks), picks


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
@pytest.mark.parametrize("taxon", [0, 63, 64, 128])
def test_columns_differing_in_one_taxon_are_never_merged(monkeypatch, encoding, taxon):
    """Two columns of 129 taxa that differ only at `taxon` share a 5-bit key under seeds 0-2:
    the verification must see the difference in whichever 64-row chunk it lies."""
    a, b = ref.find_colliding_pair(129, taxon, encoding, 5, (True, True, True, False))
    rows, picks = pair_alignment(a, b)
    want = ref.by_construction(np.stack([a, b], axis=1), picks, encoding)
    assert want[0].shape[1] == 2 and ref.expected_outcome(want[0], encoding, 5) == 3
    assert_exact(with_key_bits(monkeypatch, 5, rows, encoding), want)


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
def test_a_pair_colliding_under_every_seed_is_refused(monkeypatch, encoding):
    """The mirror predicts a 4-bit collision under all four seeds for this one pair (a chance of
    2^-16 if its keys were not the device's): the device must refuse it."""
    a, b = ref.find_colliding_pair(129, 64, encoding, 4, (True, True, True, True))
    rows, _ = pair_alignment(a, b)
    with pytest.raises(_capi.SbnbError, match="collided under four seeds"):
        with_key_bits(monkeypatch, 4, rows, encoding)
    assert_exact(device(rows, encoding), ref.compress(rows, encoding))


# ---- characters --------------------------------------------------------------------------------

@pytest.mark.parametrize("encoding", ref.ENCODINGS)
def test_every_byte_value(encoding):
    """Each byte alone at the last site (135 sites: a partial group of 4) of the last taxon
    (13 taxa: a partial group of 8) of an otherwise valid alignment."""
    rng = np.random.default_rng(ref.ENCODINGS.index(encoding))
    base = ref.pool_columns(13, 135, rng, encoding)
    wrong = []
    for byte in range(256):
        rows = base.copy()
        rows[12, 134] = byte
        sequences = [bytes(r) for r in rows]
        if ref.TABLES[encoding][byte] != ref.UNKNOWN:
            got, want = device(sequences, encoding), ref.compress(rows, encoding)
            if not (np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])):
                wrong.append((byte, "result"))
            continue
        try:
            device(sequences, encoding)
            wrong.append((byte, "accepted"))
        except _capi.SbnbError as error:
            if error.code != -1 or str(error) != ref.unknown_message(byte):
                wrong.append((byte, error.code, str(error)))
        if encoding == "states":
            with pytest.raises(RuntimeError) as info:
                restatement.compress(sequences)
            assert str(info.value) == ref.unknown_message(byte)
    assert not wrong


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
def test_the_first_of_several_unknown_characters_is_named(encoding):
    rng = np.random.default_rng(40 + ref.ENCODINGS.index(encoding))
    unknown = np.flatnonzero(ref.TABLES[encoding] == ref.UNKNOWN)
    base = ref.pool_columns(40, 5000, rng, encoding)
    cases = []
    for _ in range(12):  # scattered over threads and blocks
        rows = base.copy()
        count = rng.integers(2, 30)
        rows[rng.integers(0, 40, size=count), rng.integers(0, 5000, size=count)] = rng.choice(unknown, size=count)
        cases.append(rows)
    rows = base.copy()  # a later taxon at an earlier site, and two in one thread's group of 4 sites
    rows[[30, 7, 7], [2, 4093, 4094]] = [ord("!"), ord("#"), 0xff]
    cases.append(rows)
    for rows in cases:
        t, s = ref.first_unknown(rows, encoding)
        with pytest.raises(_capi.SbnbError) as info:
            device(rows, encoding)
        assert info.value.code == -1 and str(info.value) == ref.unknown_message(rows[t, s])
        if encoding == "states":
            with pytest.raises(RuntimeError) as oracle_info:
                restatement.compress([bytes(r) for r in rows])
            assert str(oracle_info.value) == str(info.value)
    assert str(info.value) == "Symbol '#' not known."


# ---- inputs and refusals -------------------------------------------------------------------------

@pytest.mark.parametrize("encoding", ref.ENCODINGS)
def test_every_input_form_gives_the_same_result(encoding):
    rng = np.random.default_rng(11)
    wide = ref.pool_columns(21, 2 * 300 + 7, rng, encoding)
    rows = np.ascontiguousarray(wide[3:, 5:5 + 2 * 300:2])
    want = ref.compress(rows, encoding)
    tall = np.concatenate([wide[:3, :300], rows])
    forms = {
        "str": [bytes(r).decode("ascii") for r in rows],
        "bytes": [bytes(r) for r in rows],
        "bytearray": [bytearray(r) for r in rows],
        "C array": rows,
        "Fortran array": np.asfortranarray(rows),
        "strided slice": wide[3:, 5:5 + 2 * 300:2],
        "offset view": tall[3:],  # C-contiguous, starting 900 bytes into its buffer
    }
    assert not forms["strided slice"].flags["C_CONTIGUOUS"] and not forms["Fortran array"].flags["C_CONTIGUOUS"]
    assert forms["offset view"].flags["C_CONTIGUOUS"] and forms["offset view"].base is tall
    for name, sequences in forms.items():
        got = device(sequences, encoding)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), name


def test_a_device_index_out_of_range_is_refused():
    lib = _capi.load()
    devices = lib.sbnb_device_count()
    patterns, weights, count = np.empty(8, np.uint8), np.empty(4), ctypes.c_int64(-7)
    for device_index in (devices, devices + 5, -1):
        code = lib.sbnb_compress_site_patterns(2, 4, b"ACGTACGT", device_index,
                                               patterns.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
                                               _capi.as_double_ptr(weights), ctypes.byref(count), None)
        assert code == -1 and lib.sbnb_last_error() == b"CUDA device index out of range." and count.value == -7
