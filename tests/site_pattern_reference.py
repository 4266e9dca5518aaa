"""Exact site-pattern compression for the tests of include/sbn_b200_patterns.h.

Written independently of the library (libsbn_b200/csrc/site_pattern.cu) and of the
restatement (oracle/site_pattern.py):
- `STATE_TABLE` / `MASK_TABLE`: the two symbol tables, all 256 byte values;
- `compress`: patterns in order of first appearance and their weights through `np.unique`
  over columns (a column packed into one integer when it fits, so that multi-million-site
  alignments stay cheap);
- `pool_columns` / `site_picks` / `by_construction`: an alignment built as `pool[:, picks]`
  from distinct pool columns, whose answer is known without looking at its columns: the
  pool columns in order of first use, weighted by `bincount(picks)`;
- `column_keys`: a NumPy mirror of the device's 64-bit column key (HashKernel + Mix + the
  SBNB_DEBUG_PATTERN_KEY_BITS mask), so that a test knows in advance under which of the
  four seeds two different columns share a key and the device must rehash;
- deterministic searches for alignments and column pairs with a chosen collision pattern.
"""
import numpy as np

UNKNOWN = 255
ENCODINGS = ("states", "masks")


def _table(entries):
    table = np.full(256, UNKNOWN, np.uint8)
    for characters, value in entries:
        for c in characters:
            table[ord(c)] = value
    return table


# GetSymbolTable (site_pattern.cpp:15-45): A C G T in either case; the gap and the degenerate
# codes in upper case only, all as state 4 (U too); everything else unknown.
STATE_TABLE = _table([("Aa", 0), ("Cc", 1), ("Gg", 2), ("Tt", 3), ("-NX?BDHKMRSUVWY", 4)])
# IUPAC nucleotide masks (bit 0 = A, 1 = C, 2 = G, 3 = T) in either case; U = T; N X ? - = 15.
MASK_TABLE = _table([("Aa", 1), ("Cc", 2), ("Gg", 4), ("Tt", 8), ("Uu", 8), ("Rr", 5), ("Yy", 10), ("Ss", 6),
                     ("Ww", 9), ("Kk", 12), ("Mm", 3), ("Bb", 14), ("Dd", 13), ("Hh", 11), ("Vv", 7),
                     ("NnXx?-", 15)])
TABLES = {"states": STATE_TABLE, "masks": MASK_TABLE}
# characters known in each encoding
ALPHABETS = {name: np.flatnonzero(table != UNKNOWN).astype(np.uint8) for name, table in TABLES.items()}
# base-5 digit -> characters that stand for it; the five sets are distinct symbols in both encodings
DIGIT_CHARACTERS = [b"Aa", b"Cc", b"Gg", b"Tt", b"-NX?"]


def as_rows(sequences):
    """Equal-length str / bytes rows or a uint8 [taxon][site] array -> uint8 [taxon][site]."""
    if isinstance(sequences, np.ndarray):
        return np.asarray(sequences, np.uint8)
    rows = [np.frombuffer(s.encode() if isinstance(s, str) else bytes(s), np.uint8) for s in sequences]
    return np.array(rows, np.uint8).reshape(len(rows), -1)


def unknown_message(byte):
    """The message of an unknown character: printable ASCII verbatim, any other byte as \\xHH."""
    text = chr(byte) if 0x20 <= byte <= 0x7e else f"\\x{int(byte):02x}"
    return f"Symbol '{text}' not known."


def first_unknown(rows, encoding):
    """(taxon, site) of the first unknown character in (taxon, site) order, or None."""
    where = np.flatnonzero(TABLES[encoding][rows] == UNKNOWN)
    return None if where.size == 0 else divmod(int(where[0]), rows.shape[1])


def _column_ids(symbols):
    """One comparable value per column: packed 4-bit fields when they fit 64 bits, else raw bytes."""
    n = symbols.shape[0]
    if n <= 16:
        ids = np.zeros(symbols.shape[1], np.uint64)
        for t in range(n):
            ids |= symbols[t].astype(np.uint64) << np.uint64(4 * t)
        return ids
    return np.ascontiguousarray(symbols.T).view(np.dtype((np.void, n)))[:, 0]


def compress(sequences, encoding="states"):
    """-> (patterns uint8 [taxon][pattern], weights float64), patterns in order of first appearance.
    An unknown character raises RuntimeError with the message of the first one in (taxon, site) order."""
    rows = as_rows(sequences)
    where = first_unknown(rows, encoding)
    if where is not None:
        raise RuntimeError(unknown_message(rows[where]))
    symbols = TABLES[encoding][rows]
    if rows.shape[1] == 0:
        return np.zeros((rows.shape[0], 0), np.uint8), np.zeros(0)
    _, first, counts = np.unique(_column_ids(symbols), return_index=True, return_counts=True)
    order = np.argsort(first)
    return np.ascontiguousarray(symbols[:, first[order]]), counts[order].astype(np.float64)


# ---- alignments by construction --------------------------------------------------------------

def pool_columns(taxa, count, rng, encoding="states", digit_rows=8):
    """uint8 [taxa][count] characters.  `digit_rows` randomly placed taxa (all of them if fewer)
    hold the base-5 digits of distinct integers, so the columns are distinct symbol columns in
    both encodings while count <= 5 ** digit_rows; beyond that they repeat.  The other taxa
    hold random known characters of the encoding (which may stand for the same symbol)."""
    d = min(taxa, digit_rows)
    capacity = 5 ** d
    if count <= capacity:
        values = rng.choice(capacity, size=count, replace=False)
    else:
        values = rng.integers(0, capacity, size=count)
    pool = ALPHABETS[encoding][rng.integers(0, ALPHABETS[encoding].size, size=(taxa, count))]
    spelled = np.array([[c[v % len(c)] for v in range(4)] for c in DIGIT_CHARACTERS], np.uint8)  # [digit][variant]
    for i, t in enumerate(rng.permutation(taxa)[:d]):
        pool[t] = spelled[(values // 5 ** i) % 5, rng.integers(0, 4, size=count)]
    return pool


def site_picks(regime, sites, pool_size, rng):
    """int64 [sites] pool indices.  Regimes (first appearances relative to the device's groups of 4):
    'distinct'  every site a new column (needs pool_size >= sites);
    'prefixK'   (K = 1..3) column 0 K + 1 times, then new columns: the first index of every later
                group of four first appearances is K short of a multiple of 4;
    'runs'      each column repeated 1..5 times in a row;
    'random'    uniform draws from the pool;
    'cover'     uniform draws in which every pool column appears (needs pool_size <= sites)."""
    if regime == "distinct":
        return np.arange(sites)
    if regime.startswith("prefix"):
        k = int(regime[len("prefix"):])
        return np.concatenate([np.zeros(min(k + 1, sites), np.int64), np.arange(1, max(sites - k, 1))])[:sites]
    if regime == "runs":
        runs = np.repeat(np.arange(sites), rng.integers(1, 6, size=sites))[:sites]
        return runs % pool_size
    if regime == "random":
        return rng.integers(0, pool_size, size=sites)
    if regime == "cover":
        picks = rng.integers(0, pool_size, size=sites)
        picks[rng.choice(sites, size=pool_size, replace=False)] = rng.permutation(pool_size)
        return picks
    raise ValueError(regime)


REGIMES = ("distinct", "prefix1", "prefix2", "prefix3", "runs", "random")


def pool_size(regime, sites):
    return max(1, sites // 3) if regime == "random" else sites


def alignment(pool, picks):
    """pool[:, picks], gathered row by row (several times faster than one 2-D gather at 1000 x 1M)."""
    out = np.empty((pool.shape[0], picks.size), np.uint8)
    for t in range(pool.shape[0]):
        out[t] = pool[t][picks]
    return out


def first_uses(picks, pool_size):
    """The pool indices in order of first use, and the site of each first use."""
    first = np.full(pool_size, picks.size, np.int64)
    np.minimum.at(first, picks, np.arange(picks.size))
    used = np.flatnonzero(first < picks.size)
    used = used[np.argsort(first[used])]
    return used, first[used]


def by_construction(pool, picks, encoding="states"):
    """The exact answer for the alignment pool[:, picks] when the pool columns are distinct symbol columns."""
    used, _ = first_uses(picks, pool.shape[1])
    weights = np.bincount(picks, minlength=pool.shape[1])[used].astype(np.float64)
    return np.ascontiguousarray(TABLES[encoding][pool[:, used]]), weights


def word_store_groups(first_sites, sites):
    """How many groups of 4 sites EmitKernel writes with one 32-bit store per taxon: all four are
    first appearances of consecutive patterns, the first of them a multiple of 4."""
    flags = np.zeros((sites + 3) // 4 * 4, bool)
    flags[first_sites] = True
    index = np.cumsum(flags) - 1  # the pattern index of a first appearance
    group_flags = flags.reshape(-1, 4)
    group_index = index.reshape(-1, 4)
    return int(np.sum(group_flags.all(axis=1) & (group_index[:, 0] % 4 == 0)))


# ---- mirror of the device column key ---------------------------------------------------------

_M32 = np.uint64(0xffffffff)
_GOLDEN = 0x9e3779b97f4a7c15


def _rotl32(x, r):
    return ((x << np.uint64(r)) | (x >> np.uint64(32 - r))) & _M32


def _hash_step(h, word, c1, c2, r1, r2, m, add):
    k = (word * np.uint64(c1)) & _M32
    k = (_rotl32(k, r1) * np.uint64(c2)) & _M32
    h = h ^ k
    return (_rotl32(h, r2) * np.uint64(m) + np.uint64(add)) & _M32


def _mix(x):  # splitmix64 finaliser, wrapping uint64
    x = x ^ (x >> np.uint64(30))
    x = x * np.uint64(0xbf58476d1ce4e5b9)
    x = x ^ (x >> np.uint64(27))
    x = x * np.uint64(0x94d049bb133111eb)
    return x ^ (x >> np.uint64(31))


def fields(symbols, encoding):
    """The 4-bit field the device hashes per symbol: states symbol & 0xf (unknown 0xf), masks the mask (unknown 0)."""
    symbols = np.asarray(symbols, np.uint8)
    if encoding == "masks":
        return np.where(symbols == UNKNOWN, 0, symbols).astype(np.uint8)
    return symbols & np.uint8(0xf)


def column_keys(symbols, encoding, seed, bits=None):
    """uint64 [columns]: the device's key of each symbol column [taxon][column] under seed 0..3,
    cut to the low `bits` bits as SBNB_DEBUG_PATTERN_KEY_BITS=bits does (None: the whole key)."""
    f = fields(symbols, encoding)
    n, count = f.shape
    pad = np.uint64(1 if encoding == "masks" else 0)  # taxa missing from the last group of 8 read as 'A'
    s = (seed * _GOLDEN) % 2 ** 64
    ha = np.full(count, (0x811c9dc5 ^ (s & 0xffffffff)), np.uint64)
    hb = np.full(count, (0x9e3779b9 + (s >> 32)) & 0xffffffff, np.uint64)
    for g in range(0, n, 8):
        packed = np.zeros(count, np.uint64)
        for i in range(8):
            field = f[g + i].astype(np.uint64) if g + i < n else pad
            packed |= field << np.uint64(4 * i)
        ha = _hash_step(ha, packed, 0xcc9e2d51, 0x1b873593, 15, 13, 5, 0xe6546b64)
        hb = _hash_step(hb, packed, 0x85ebca6b, 0xc2b2ae35, 16, 11, 9, 0x7f4a7c15)
    key = _mix(((ha << np.uint64(32)) | hb) + np.uint64(_GOLDEN))
    if bits is not None:
        key &= np.uint64((1 << max(1, min(63, bits))) - 1)
    key[key == np.uint64(2 ** 64 - 1)] = 0
    return key


def colliding_seeds(patterns, encoding, bits):
    """For distinct symbol columns `patterns` [taxon][pattern]: per seed 0..3, whether two of them share a key."""
    return tuple(bool(np.unique(column_keys(patterns, encoding, seed, bits)).size < patterns.shape[1])
                 for seed in range(4))


def expected_outcome(patterns, encoding, bits):
    """The first seed under which no two patterns share a key (the device succeeds there), or None (it refuses)."""
    clean = [not c for c in colliding_seeds(patterns, encoding, bits)]
    return clean.index(True) if any(clean) else None


# ---- deterministic case searches -------------------------------------------------------------

def rehash_alignment(index, encoding, taxa=12, sites=4000, distinct=1500):
    """Alignment `index` of a family for the rehash tests: `distinct` pool columns drawn over `sites`."""
    rng = np.random.default_rng([20261022, index, ENCODINGS.index(encoding)])
    pool = pool_columns(taxa, distinct, rng, encoding)
    picks = site_picks("cover", sites, distinct, rng)
    return pool, picks


def find_rehash_case(target, encoding, bit_range=range(14, 27), tries=40, **family):
    """-> (index, bits) of the first rehash_alignment(index, encoding, **family) and key width whose
    per-seed collision pattern matches `target` (a 4-tuple of True / False / None = either)."""
    for index in range(tries):
        pool, picks = rehash_alignment(index, encoding, **family)
        patterns = TABLES[encoding][pool]
        for bits in bit_range:
            got = colliding_seeds(patterns, encoding, bits)
            if all(t is None or t == g for t, g in zip(target, got)):
                return index, bits
    raise LookupError(f"no rehash case with collisions {target}")


def find_colliding_pair(taxa, taxon, encoding, bits, target, batch=1 << 15, batches=64):
    """Two character columns [taxa] that differ only at `taxon` and share a `bits`-bit key under
    exactly the seeds marked True in `target` (4 booleans).  Deterministic."""
    rng = np.random.default_rng([taxa, taxon, bits, ENCODINGS.index(encoding)] + [int(t) for t in target])
    alphabet = ALPHABETS[encoding]
    table = TABLES[encoding]
    for _ in range(batches):
        a = alphabet[rng.integers(0, alphabet.size, size=(taxa, batch))]
        b = a.copy()
        replacement = alphabet[rng.integers(0, alphabet.size, size=batch)]
        b[taxon] = replacement
        ok = table[replacement] != table[a[taxon]]
        match = ok.copy()
        for seed in range(4):
            same = column_keys(table[a], encoding, seed, bits) == column_keys(table[b], encoding, seed, bits)
            match &= same == bool(target[seed])
        hit = np.flatnonzero(match)
        if hit.size:
            return a[:, hit[0]].copy(), b[:, hit[0]].copy()
    raise LookupError(f"no pair at taxon {taxon} with collisions {target}")
