"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): NumPy restatement of the
reference's SitePattern::Compress (src/site_pattern.cpp:77-115) and symbol table
(site_pattern.cpp:15-45).  Only tests/ and bench code may import it.

The reference emits patterns in the iteration order of a libstdc++ unordered_map;
that order is an accident of the hash, so this restatement (like the CUDA path)
emits them in order of first appearance, and the tests pin the SET of (pattern,
weight) pairs against the reference's own output (tests/golden)."""
import numpy as np

SYMBOLS = {c: i for i, c in enumerate("ACGT")}
SYMBOLS.update({c.lower(): i for i, c in enumerate("ACGT")})
SYMBOLS.update({c: 4 for c in "-NX?BDHKMRSUVWY"})


def symbol_table():
    table = np.full(256, 255, dtype=np.uint8)
    for c, v in SYMBOLS.items():
        table[ord(c)] = v
    return table


def symbol_text(byte):
    """A character as the error message writes it: printable ASCII verbatim, other bytes as \\xHH."""
    return chr(byte) if 0x20 <= byte <= 0x7e else f"\\x{int(byte):02x}"


def compress(sequences):
    """sequences: equal-length strings in leaf-id order -> (patterns uint8 [taxon][pattern], weights)."""
    rows = np.array([np.frombuffer(s.encode() if isinstance(s, str) else s, dtype=np.uint8) for s in sequences])
    symbols = symbol_table()[rows]
    if (symbols == 255).any():
        t, k = np.argwhere(symbols == 255)[np.lexsort(np.argwhere(symbols == 255).T[::-1])][0]
        raise RuntimeError(f"Symbol '{symbol_text(rows[t, k])}' not known.")
    if rows.shape[1] == 0:
        return np.zeros((rows.shape[0], 0), np.uint8), np.zeros(0)
    _, first, counts = np.unique(symbols, axis=1, return_index=True, return_counts=True)
    order = np.argsort(first)
    return np.ascontiguousarray(symbols[:, first[order]]), counts[order].astype(np.float64)
