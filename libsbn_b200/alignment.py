"""Host-side alignment handling: FASTA parsing and the DNA symbol table.

Mirrors the reference's Alignment::ReadFasta (src/alignment.cpp:41-73) and
SitePattern::GetSymbolTable (src/site_pattern.cpp:16-46): every non-ACGT symbol is a
gap (state 4).  The IUPAC table keeps what a degenerate nucleotide says instead: the
set of states it allows, as a mask (bit 0 = A, 1 = C, 2 = G, 3 = T).  Compressing identical columns into weighted site patterns
(SitePattern::Compress) is done on the device: libsbn_b200.site_pattern.SitePattern.
"""
import numpy as np

_SYMBOLS = {c: i for i, c in enumerate("ACGT")}
_SYMBOLS.update({c.lower(): i for c, i in list(_SYMBOLS.items())})
_GAPS = "-NX?BDHKMRSUVWY"


# IUPAC nucleotide codes -> masks of the states they allow; U = T; N X ? - = 15 (missing)
_IUPAC = {"A": 1, "C": 2, "G": 4, "T": 8, "U": 8, "R": 5, "Y": 10, "S": 6, "W": 9, "K": 12, "M": 3,
          "B": 14, "D": 13, "H": 11, "V": 7, "N": 15, "X": 15}
_IUPAC.update({c.lower(): m for c, m in list(_IUPAC.items())})
_IUPAC.update({"?": 15, "-": 15})


def iupac_mask_table():
    """{character: nucleotide mask} of the IUPAC codes, upper and lower case."""
    return dict(_IUPAC)


def symbol_table():
    """SitePattern::GetSymbolTable (site_pattern.cpp:16-46)."""
    table = dict(_SYMBOLS)
    table.update({c: 4 for c in _GAPS})
    return table


def read_fasta(path):
    """Alignment::ReadFasta: {taxon name: sequence}; all sequences same length."""
    data, taxon, chunks = {}, None, []
    with open(path) as handle:
        for line in handle:
            line = line.rstrip("\n").rstrip("\r")
            if not line:
                continue
            if line[0] == ">":
                if taxon:
                    data[taxon] = "".join(chunks)
                taxon, chunks = line[1:], []
            else:
                chunks.append(line)
    if taxon:
        data[taxon] = "".join(chunks)
    if len({len(s) for s in data.values()}) > 1:
        raise RuntimeError("Sequences of the alignment are not all the same length.")
    return data


def encode(sequences, taxon_names, ambiguity=False):
    """Sequences (dict name -> str) in leaf-id order -> uint8 [taxon][site]: states
    (the reference's table), or with ambiguity=True nucleotide masks (the IUPAC table)."""
    table = iupac_mask_table() if ambiguity else symbol_table()
    lut = np.full(256, 255, dtype=np.uint8)
    for symbol, state in table.items():
        lut[ord(symbol)] = state
    rows = []
    for name in taxon_names:
        if name not in sequences:
            raise RuntimeError(f"Taxon {name} not found in alignment.")
        row = lut[np.frombuffer(sequences[name].encode("ascii"), dtype=np.uint8)]
        if (row == 255).any():
            bad = sequences[name][int(np.argmax(row == 255))]
            raise RuntimeError(f"Symbol '{bad}' not known.")
        rows.append(row)
    return np.stack(rows)


def sequences_in_leaf_order(sequences, taxon_names):
    """Sequences (dict name -> str) as a list in leaf-id order."""
    for name in taxon_names:
        if name not in sequences:
            raise RuntimeError(f"Taxon {name} not found in alignment.")
    return [sequences[name] for name in taxon_names]


def site_patterns_of_fasta(path, taxon_names, device=0, ambiguity=False):
    """FASTA -> (patterns [taxon][P], weights [P]); the compression runs on the
    device (SitePattern::Compress, include/sbn_b200_patterns.h).  ambiguity=True gives
    nucleotide masks (Engine(..., tip_encoding="masks"))."""
    from .site_pattern import SitePattern
    pattern = SitePattern(sequences_in_leaf_order(read_fasta(path), taxon_names), device, ambiguity)
    return pattern.patterns, pattern.weights
