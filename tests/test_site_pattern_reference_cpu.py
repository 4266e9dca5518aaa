"""The exact site-pattern reference (tests/site_pattern_reference.py) checked without a device:
its tables against the library's Python tables, its compression against a column-by-column
dictionary and the NumPy restatement, the construction generators against its compression,
the key mirror's invariants and the determinism of its case searches.  Also the C-ABI
refusals that come before any device is touched, and the decoding of error messages."""
import ctypes
import types

import numpy as np
import pytest

import site_pattern_reference as ref
from libsbn_b200 import _capi, alignment
from oracle import site_pattern as restatement


def dictionary_compress(rows, encoding):
    """Column by column through a dict, the way SitePattern::Compress does, in first-appearance order."""
    table = ref.TABLES[encoding]
    index, patterns, weights = {}, [], []
    for column in np.asarray(rows).T:
        key = bytes(table[column])
        if key not in index:
            index[key] = len(patterns)
            patterns.append(table[column])
            weights.append(0.0)
        weights[index[key]] += 1.0
    return np.array(patterns, np.uint8).T.reshape(rows.shape[0], -1), np.array(weights)


def test_state_table_is_the_library_s_and_the_restatement_s():
    assert np.array_equal(ref.STATE_TABLE, restatement.symbol_table())
    table = np.full(256, ref.UNKNOWN, np.uint8)
    for c, v in alignment.symbol_table().items():
        table[ord(c)] = v
    assert np.array_equal(ref.STATE_TABLE, table)
    # only a c g t are known in lower case; U is a gap
    assert list(ref.STATE_TABLE[np.frombuffer(b"acgtU-?", np.uint8)]) == [0, 1, 2, 3, 4, 4, 4]
    assert (ref.STATE_TABLE[np.frombuffer(b"nrxyu", np.uint8)] == ref.UNKNOWN).all()
    assert np.count_nonzero(ref.STATE_TABLE != ref.UNKNOWN) == 23


def test_mask_table_is_the_iupac_table():
    table = np.full(256, ref.UNKNOWN, np.uint8)
    for c, v in alignment.iupac_mask_table().items():
        table[ord(c)] = v
    assert np.array_equal(ref.MASK_TABLE, table)
    # U = T and lower-case IUPAC codes are known; no byte maps to 0
    assert list(ref.MASK_TABLE[np.frombuffer(b"UurnXx?-", np.uint8)]) == [8, 8, 5, 15, 15, 15, 15, 15]
    assert np.count_nonzero(ref.MASK_TABLE != ref.UNKNOWN) == 36 and 0 not in ref.MASK_TABLE
    assert (ref.MASK_TABLE[128:] == ref.UNKNOWN).all() and (ref.STATE_TABLE[128:] == ref.UNKNOWN).all()


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
@pytest.mark.parametrize("taxa", [1, 7, 16, 17, 65])
def test_compression_equals_a_column_dictionary(encoding, taxa):
    rng = np.random.default_rng(taxa)
    pool = ref.pool_columns(taxa, 40, rng, encoding, digit_rows=2)  # 25 distinct digit columns at most
    rows = ref.alignment(pool, rng.integers(0, 40, size=300))
    patterns, weights = ref.compress(rows, encoding)
    want_patterns, want_weights = dictionary_compress(rows, encoding)
    assert np.array_equal(patterns, want_patterns) and np.array_equal(weights, want_weights)
    if encoding == "states":
        oracle_patterns, oracle_weights = restatement.compress([bytes(r) for r in rows])
        assert np.array_equal(patterns, oracle_patterns) and np.array_equal(weights, oracle_weights)


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
@pytest.mark.parametrize("regime", ref.REGIMES + ("cover",))
@pytest.mark.parametrize("taxa,sites", [(1, 3), (8, 129), (9, 1025), (64, 128), (129, 517)])
def test_construction_equals_compression(encoding, regime, taxa, sites):
    rng = np.random.default_rng([taxa, sites, ref.REGIMES.index(regime) if regime in ref.REGIMES else 9])
    size = ref.pool_size(regime, sites) if regime != "cover" else max(1, sites // 4)
    size = min(size, 5 ** min(taxa, 8))  # distinct pool columns only
    if regime in ("distinct",) or regime.startswith("prefix"):
        sites = min(sites, size)
    pool = ref.pool_columns(taxa, size, rng, encoding)
    picks = ref.site_picks(regime, sites, size, rng)
    rows = ref.alignment(pool, picks)
    assert np.array_equal(rows, pool[:, picks])
    want = ref.compress(rows, encoding)
    got = ref.by_construction(pool, picks, encoding)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    if regime == "cover":
        assert got[0].shape[1] == size


def test_construction_equals_compression_at_a_million_sites():
    rng = np.random.default_rng(7)
    pool = ref.pool_columns(12, 900_000, rng, "masks", digit_rows=12)
    picks = ref.site_picks("random", 1_100_000, 900_000, rng)
    rows = ref.alignment(pool, picks)
    got, want = ref.by_construction(pool, picks, "masks"), ref.compress(rows, "masks")
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_the_regimes_control_the_store_path():
    """'distinct' writes every group of four with one word per taxon; 'prefixK' never does."""
    for sites in (4, 5, 127, 128, 129, 1023, 1024, 1025):
        used, first = ref.first_uses(ref.site_picks("distinct", sites, sites, None), sites)
        assert ref.word_store_groups(first, sites) == sites // 4
        for k in (1, 2, 3):
            picks = ref.site_picks(f"prefix{k}", sites, sites, None)
            used, first = ref.first_uses(picks, sites)
            assert used.size == sites - k and ref.word_store_groups(first, sites) == 0


@pytest.mark.parametrize("patterns", [65_535, 65_536, 65_537])
def test_the_pattern_count_is_exact(patterns):
    rng = np.random.default_rng(patterns)
    pool = ref.pool_columns(8, patterns, rng)
    picks = ref.site_picks("cover", patterns + 12_345, patterns, rng)
    got, weights = ref.by_construction(pool, picks)
    assert got.shape == (8, patterns) and weights.sum() == picks.size
    assert np.unique(ref._column_ids(got)).size == patterns


def test_unknown_characters_are_reported_first_in_taxon_site_order():
    rows = ref.as_rows([b"ACGTACGT", b"ACGZACGT", b"AJGTACGT"])
    assert ref.first_unknown(rows, "states") == (1, 3)
    with pytest.raises(RuntimeError, match=r"^Symbol 'Z' not known\.$"):
        ref.compress(rows, "masks")
    with pytest.raises(RuntimeError, match=r"^Symbol 'Z' not known\.$"):
        restatement.compress([bytes(r) for r in rows])
    assert ref.unknown_message(0xe9) == "Symbol '\\xe9' not known."
    assert ref.unknown_message(0) == "Symbol '\\x00' not known."
    assert ref.unknown_message(ord(" ")) == "Symbol ' ' not known."
    assert ref.unknown_message(0x7f) == "Symbol '\\x7f' not known."
    for byte in range(256):
        if ref.STATE_TABLE[byte] == ref.UNKNOWN:
            with pytest.raises(RuntimeError) as info:
                restatement.compress([b"ACGT", b"AC" + bytes([byte]) + b"T"])
            assert str(info.value) == ref.unknown_message(byte)


def test_key_mirror_padding_and_width():
    """Taxa missing from the last group of 8 hash as 'A' (field 0 for states, 1 for masks), so a
    column keeps its key when rows of 'A' are appended up to the group's end -- but not beyond."""
    rng = np.random.default_rng(3)
    for encoding in ref.ENCODINGS:
        rows = ref.pool_columns(5, 200, rng, encoding, digit_rows=3)
        padded = np.concatenate([rows, np.full((3, 200), ord("A"), np.uint8)])
        longer = np.concatenate([padded, np.full((1, 200), ord("A"), np.uint8)])
        table = ref.TABLES[encoding]
        for seed in range(4):
            keys = ref.column_keys(table[rows], encoding, seed)
            assert np.array_equal(keys, ref.column_keys(table[padded], encoding, seed))
            assert not np.array_equal(keys, ref.column_keys(table[longer], encoding, seed))
            assert np.array_equal(ref.column_keys(table[rows], encoding, seed, 13), keys & np.uint64(0x1fff))
            # (widths clamp to 1..63, as the device's hook does)
            assert np.array_equal(ref.column_keys(table[rows], encoding, seed, 99), keys & np.uint64(2 ** 63 - 1))
            assert np.array_equal(ref.column_keys(table[rows], encoding, seed, 0), keys & np.uint64(1))
        # the seeds give different keys
        assert len({ref.column_keys(table[rows], encoding, seed)[0] for seed in range(4)}) == 4


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
def test_rehash_case_search_is_deterministic(encoding):
    for target, outcome in (((True, False, None, None), 1), ((True, True, True, False), 3),
                            ((True, True, True, True), None)):
        index, bits = ref.find_rehash_case(target, encoding)
        assert (index, bits) == ref.find_rehash_case(target, encoding)
        pool, picks = ref.rehash_alignment(index, encoding)
        patterns, _ = ref.by_construction(pool, picks, encoding)
        got = ref.colliding_seeds(patterns, encoding, bits)
        assert all(t is None or t == g for t, g in zip(target, got))
        assert ref.expected_outcome(patterns, encoding, bits) == outcome
        assert ref.expected_outcome(patterns, encoding, None) == 0  # the whole key: no collision


@pytest.mark.parametrize("encoding", ref.ENCODINGS)
def test_colliding_pair_search(encoding):
    target = (True, True, True, False)
    a, b = ref.find_colliding_pair(129, 64, encoding, 5, target)
    again = ref.find_colliding_pair(129, 64, encoding, 5, target)
    assert np.array_equal(a, again[0]) and np.array_equal(b, again[1])
    table = ref.TABLES[encoding]
    assert list(np.flatnonzero(table[a] != table[b])) == [64]
    pair = table[np.stack([a, b], axis=1)]
    assert ref.colliding_seeds(pair, encoding, 5) == target
    assert ref.expected_outcome(pair, encoding, 5) == 3


# ---- the C ABI refuses before touching a buffer or a device -------------------------------------

def _call(taxa, sites, encoding=None):
    lib = _capi.load()
    count = ctypes.c_int64(-7)
    if encoding is None:
        code = lib.sbnb_compress_site_patterns(taxa, sites, None, 0, None, None, ctypes.byref(count), None)
    else:
        code = lib.sbnb_compress_site_patterns_encoded(taxa, sites, None, encoding, 0, None, None,
                                                       ctypes.byref(count), None)
    return code, lib.sbnb_last_error().decode(), count.value


@pytest.mark.parametrize("encoding", [None, _capi.TIPS_STATES, _capi.TIPS_NUCLEOTIDE_MASKS])
def test_sizes_are_refused_before_any_buffer_is_read(encoding):
    """NULL buffers: a refusal that came any later would name them (or fault)."""
    for taxa in (0, -1, -2 ** 31):
        assert _call(taxa, 10, encoding) == (-1, "Site pattern compression needs at least one sequence.", -7)
    for sites in (2 ** 30, 2 ** 40, -1):
        assert _call(3, sites, encoding) == (-1, "Site count out of range [0, 2^30).", -7)


def test_an_unknown_tip_encoding_is_refused():
    for encoding in (-1, 2):
        assert _call(3, 10, encoding) == (-1, "Unknown tip encoding.", -7)


def test_error_messages_are_decoded_without_failing(monkeypatch):
    """A message that is not UTF-8 still raises the SbnbError, with the odd byte escaped."""
    monkeypatch.setattr(_capi, "load", lambda: types.SimpleNamespace(sbnb_last_error=lambda: b"Symbol '\xe9' not known."))
    with pytest.raises(_capi.SbnbError) as info:
        _capi.check(-1)
    assert info.value.code == -1 and str(info.value) == "Symbol '\\xe9' not known."
