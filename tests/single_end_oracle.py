"""Single-end demux (FRENDER_SINGLE_END=1) in the CPU oracle's terms: route_pairs (F:774-810) over one file, the key
taken from each record's own header.  Test infrastructure, kept beside the tests so that oracle/ keeps restating the
reference alone."""
import gzip

import frender_oracle as O


def route_single(lines, table, roles):
    """Route 4-line records of one file by the demux key of their own header.  Returns {sink name: R1 bytes}; a
    trailing partial record is padded with "" (F:719-723), an unknown key is SystemExit (F:807-810)."""
    text = list(lines)              # every record is its own mate: the key of route_pairs' R2 header is its own
    return {name: r1 for name, (r1, _) in O.route_pairs(text, text, table, roles).items()}


def demux_file_single(path, table, roles):
    """route_single over one fastq.gz file opened in text mode (F:776)."""
    with gzip.open(path, "rt") as handle:
        return route_single(handle, table, roles)
