"""Demux with index reads (FRENDER_INDEX_READS=1) in the CPU oracle's terms: route_pairs (F:774-810) with the zip()
of the 4-line groupers (F:719-723, F:777) taken over N files instead of two.  Test infrastructure, kept beside the
tests so that oracle/ keeps restating the reference alone."""
import frender_oracle as O


def groups(lines):
    """The reference's 4-line grouper (F:719-723): a trailing partial record is padded with ""."""
    block = []
    for line in lines:
        block.append(line)
        if len(block) == 4:
            yield block
            block = []
    if block:
        yield block + [""] * (4 - len(block))


def route_mates(mates, key_mate, table, roles):
    """Route the 4-line records of N files together: record i of every file goes to the sink of the demux key of
    record i of file `key_mate` (R2 in a paired run, R1 in a single-end one).  The loop ends with the shortest file.
    Returns {sink name: (bytes of file 0, bytes of file 1, ...)}; an unknown key is SystemExit (F:807-810)."""
    sinks = {name: [[] for _ in mates] for name in roles.values() if name}
    have_samples = any(not r.startswith("#") for r in roles)
    for recs in zip(*(groups(lines) for lines in mates)):
        key = O.demux_key(recs[key_mate][0])
        if key not in table:
            raise SystemExit(f"Couldn't find barcode {key} in supplied frender result file!")
        kind, sid = table[key]
        if kind == "demuxable" and have_samples:
            name = roles[sid]
        elif kind == "index_hop" and roles["#hop"]:
            name = roles["#hop"]
        elif kind == "ambiguous" and roles["#amb"]:
            name = roles["#amb"]
        elif kind == "undetermined" and roles["#und"]:
            name = roles["#und"]
        else:
            raise SystemExit("Unrecognized read type found in supplied frender result file!")
        for out, rec in zip(sinks[name], recs):
            out.extend(rec)
    return {n: tuple("".join(part).encode() for part in parts) for n, parts in sinks.items()}
