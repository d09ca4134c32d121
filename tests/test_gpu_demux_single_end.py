"""Single-end demux (frb_route_set_mates(ctx, 1), FRENDER_SINGLE_END=1): the one-mate stream against the oracle's
route_single, its output formats, the API rules of the setting, and frender demux on R1 files alone against the
reference's golden R1 sinks and against paired runs."""
import ctypes
import gzip
import hashlib
import os
import random
import zlib
from argparse import Namespace

import numpy as np
import pytest

import single_end_oracle as SE
from frender_b200 import bgzf

pytestmark = pytest.mark.gpu

KINDS = ["demuxable", "index_hop", "ambiguous", "undetermined"]


def make_single(rng, n, n_keys=40, half=8):
    """n single-end records keyed by index pairs of half+half symbols, and a results table over the keys."""
    bases = "ACGTN"
    keys = ["".join(rng.choice(bases) for _ in range(half)) + "+" + "".join(rng.choice(bases) for _ in range(half))
            for _ in range(n_keys)]
    recs = []
    for i in range(n):
        k, ln = rng.choice(keys), rng.randint(1, 300)
        recs.append(f"@M0:{i}:FC:1:{rng.randint(1, 99999)}:{rng.randint(1, 99999)} 1:N:0:{k}\n{'A' * ln}\n+\n"
                    f"{'F' * ln}\n")
    table = {k: (KINDS[j % 4], f"S{j % 7}" if j % 4 == 0 else "") for j, k in enumerate(keys)}
    return "".join(recs), table


def load(ctx, table, roles):
    """The results table on the device; returns the sink names in sink-id order."""
    from frender_b200.engine import pack_keys, pack_keys2
    names = sorted({n for n in roles.values() if n})
    sid = {n: i for i, n in enumerate(names)}
    role_of = {"index_hop": "#hop", "ambiguous": "#amb", "undetermined": "#und"}
    keys = list(table)
    routes = np.array([sid[roles[table[k][1]] if table[k][0] == "demuxable" else roles[role_of[table[k][0]]]]
                       for k in keys], np.uint32)
    if ctx.wide:
        lo, hi = pack_keys2(keys)
        ctx.route_load(lo, routes, len(names), keys_hi=hi)
    else:
        ctx.route_load(pack_keys(keys), routes, len(names))
    return names


def stream_single(ctx, text, table, roles, cut, mode="plain"):
    """Push `text` in pieces of cut() bytes through a single-end stream, two chunks in flight.  Returns the cells of
    every popped chunk ([R1 bytes per sink]) and the records routed."""
    names = load(ctx, table, roles)
    ctx.route_gzip(mode != "plain", bgzf=mode == "bgzf")
    ctx.route_mates(1)
    ctx.route_reset()
    data = text.encode()
    chunks, pos, queued, total = [], 0, 0, 0

    def take():
        nonlocal total
        o1, o2, off1, off2, n, _, c2 = ctx.route_pop()
        assert len(o2) == 0 and not off2.any() and c2 == 0
        total += n
        chunks.append([o1[off1[i]:off1[i + 1]].tobytes() for i in range(len(names))])

    try:
        while True:
            piece = data[pos:pos + cut()]
            pos += len(piece)
            final = 1 if pos >= len(data) else 0
            ctx.route_push(piece, None, final)
            queued += 1
            if queued == 2:
                take()
                queued -= 1
            if final:
                break
        while queued:
            take()
            queued -= 1
    finally:
        ctx.route_reset()                               # after an error, the chunk still in flight is dropped
        ctx.route_gzip(False)
        ctx.route_mates(2)
    return names, chunks, total


def joined(names, chunks):
    return {n: b"".join(c[i] for c in chunks) for i, n in enumerate(names)}


@pytest.fixture(scope="module")
def ctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=16)
    yield c
    c.close()


@pytest.fixture(scope="module")
def wctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=16, wide=True)
    yield c
    c.close()


CASES = ["random_cuts", "tiny_cuts", "one_mb", "no_final_newline", "partial_tail", "shorter_than_a_record", "empty"]


@pytest.mark.parametrize("width", ["narrow", "wide"])
@pytest.mark.parametrize("case", CASES)
def test_single_end_stream_matches_the_oracle(ctx, wctx, case, width):
    import frender_oracle as O
    rng = random.Random(sum(case.encode()) + (7 if width == "wide" else 0))
    c = wctx if width == "wide" else ctx
    text, table = make_single(rng, 6000 if case != "one_mb" else 20000, half=12 if width == "wide" else 8)
    if case == "no_final_newline":
        text = text[:-1]
    elif case == "partial_tail":
        text = text[:-rng.randint(5, 40)]
    elif case == "shorter_than_a_record":
        text = text[:text.index("\n", text.index("\n") + 1) + 3]    # header, sequence, 2 bytes of the '+' line
    elif case == "empty":
        text = ""
    roles = O.sink_names(table)
    want = SE.route_single(text.splitlines(keepends=True), table, roles)
    cut = {"tiny_cuts": lambda: rng.randint(1, 3000), "one_mb": lambda: 1 << 20}.get(
        case, lambda: rng.randint(50_000, 500_000))
    names, chunks, total = stream_single(c, text, table, roles, cut)
    got = joined(names, chunks)
    assert total == sum(v.count(b"\n@M0:") + (1 if v.startswith(b"@M0:") else 0) for v in want.values())
    for name in names:
        assert got[name] == want.get(name, b""), f"{case}/{width}: sink {name}"


def test_single_end_header_cut_inside_the_key(ctx):
    """A small text cut in two at many places around its middle, headers and keys included: a record cut anywhere
    is routed from the carried bytes."""
    import frender_oracle as O
    rng = random.Random(3)
    text, table = make_single(rng, 40)
    roles = O.sink_names(table)
    want = SE.route_single(text.splitlines(keepends=True), table, roles)
    for at in range(len(text) // 2 - 60, len(text) // 2 + 60, 7):
        cuts = iter([at, len(text)])
        names, chunks, _ = stream_single(ctx, text, table, roles, lambda: next(cuts))
        got = joined(names, chunks)
        assert all(got[n] == want.get(n, b"") for n in names), at


def test_single_end_unknown_key_has_the_references_message(ctx):
    import frender_oracle as O
    from frender_b200 import _lib
    from frender_b200.engine import FrbError
    rng = random.Random(5)
    text, table = make_single(rng, 500)
    roles = O.sink_names(table)
    lost = text.splitlines()[4 * 321].rsplit(":", 1)[1]
    del table[lost]
    with pytest.raises(FrbError) as err:
        stream_single(ctx, text, table, roles, lambda: 1 << 20)
    assert err.value.code == _lib.ERR_KEY_NOT_FOUND
    assert err.value.message == f"Couldn't find barcode {lost} in supplied frender result file!"
    ctx.route_reset()


def test_single_end_record_longer_than_the_chunk(ctx):
    import frender_oracle as O
    from frender_b200 import _lib
    from frender_b200.engine import FrbError
    rng = random.Random(9)
    text, table = make_single(rng, 100)
    key = next(iter(table))
    text += f"@long 1:N:0:{key}\n{'A' * (3 << 20)}\n+\n{'F' * (3 << 20)}\n"
    roles = O.sink_names(table)
    with pytest.raises(FrbError) as err:
        stream_single(ctx, text, table, roles, lambda: 1 << 20)
    assert err.value.code == _lib.ERR_ARG
    ctx.route_reset()


# ---- formats ---------------------------------------------------------------------------------------------------------
def whole_blocks(cell):
    """The bytes of a run of whole BGZF blocks (no EOF block), each block checked against its ISIZE."""
    out = []
    for pos, bsize, isize in bgzf.iter_blocks(cell):
        assert isize > 0
        data = zlib.decompress(bytes(cell[pos:pos + bsize + 1]), 31)
        assert len(data) == isize
        out.append(data)
    return b"".join(out)


@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_single_end_formats_agree(ctx, wctx, width):
    import frender_oracle as O
    c = wctx if width == "wide" else ctx
    text, table = make_single(random.Random(21), 30000, half=12 if width == "wide" else 8)
    roles = O.sink_names(table)
    runs = {}
    for mode in ("plain", "gzip", "bgzf"):
        rng = random.Random(4)                          # the same pushes in every format (none larger than the
        runs[mode] = stream_single(c, text, table, roles, lambda: rng.randint(100_000, 1 << 20), mode)  # 1 MB buffers)
    names, plain, total = runs["plain"]
    assert total == 30000
    for mode, unpack in (("gzip", lambda b: zlib.decompress(b, 31)), ("bgzf", whole_blocks)):
        _, cells, n = runs[mode]
        assert n == total and len(cells) == len(plain)
        for chunk_p, chunk_z in zip(plain, cells):
            for p, z in zip(chunk_p, chunk_z):
                assert (unpack(z) if z else b"") == p, mode
    want = SE.route_single(text.splitlines(keepends=True), table, roles)
    assert joined(names, plain) == {n: want.get(n, b"") for n in names}


# ---- API rules -------------------------------------------------------------------------------------------------------
def test_set_mates_rules(ctx):
    import frender_oracle as O
    from frender_b200 import _lib
    from frender_b200._lib import lib
    from frender_b200.engine import FrbError
    rng = random.Random(13)
    text, table = make_single(rng, 2000)
    roles = O.sink_names(table)
    load(ctx, table, roles)
    for bad in (0, 3):
        assert lib.frb_route_set_mates(ctx._h, bad) == _lib.ERR_ARG
    ctx.route_mates(1)
    ctx.route_reset()
    with pytest.raises(FrbError) as err:              # R2 in a single-end stream
        ctx.route_push(text.encode(), b"@x\n", 1)
    assert err.value.code == _lib.ERR_ARG
    # no switch while a chunk is in flight
    ctx.route_push(text.encode(), None, 1)
    assert lib.frb_route_set_mates(ctx._h, 2) == _lib.ERR_STATE
    assert ctx.route_pop()[4] == 2000
    ctx.route_reset()                                   # the setting survives a reset
    ctx.route_push(text.encode(), None, 1)
    assert ctx.route_pop()[4] == 2000
    ctx.route_mates(2)
    ctx.route_reset()


def test_route_pair_and_paired_streams_after_single_end(ctx):
    """frb_route_pair routes pairs while the stream is single-end (and keeps the setting); a paired stream after
    switching back gives the cells of a fresh context."""
    import frender_oracle as O
    from frender_b200.engine import Context
    from test_gpu_route import make_pair, stream
    rng = random.Random(17)
    t1, t2, table = make_pair(rng, 3000, crop_tail=5)
    roles = O.sink_names(table)
    want = O.route_pairs(t1.splitlines(keepends=True), t2.splitlines(keepends=True), table, roles)
    names = load(ctx, table, roles)
    ctx.route_mates(1)
    o1, o2, off1, off2, pairs, used1, used2 = ctx.route_pair(t1.encode(), t2.encode(), 3)
    assert pairs == 3000 and used1 == len(t1) and used2 == len(t2)
    for i, n in enumerate(names):
        assert (bytes(o1[off1[i]:off1[i + 1]]), bytes(o2[off2[i]:off2[i + 1]])) == want[n]
    ctx.route_reset()                                   # the setting is kept: R1 alone is accepted
    ctx.route_push(t1.encode(), None, 1)
    assert ctx.route_pop()[4] == 3000
    # still single-end: R1 alone routes by its own headers (R1 and R2 carry the same keys here)
    single = SE.route_single(t1.splitlines(keepends=True), table, roles)
    got_names, chunks, _ = stream_single(ctx, t1, table, roles, lambda: 1 << 20)
    assert joined(got_names, chunks) == {n: single.get(n, b"") for n in got_names}
    # back to pairs: the same cells as a fresh context
    cuts = lambda r: (lambda: r.randint(100_000, 300_000))  # noqa: E731
    got, total = stream(ctx, t1, t2, table, roles, cuts(random.Random(1)), cuts(random.Random(2)))
    fresh = Context(0, table_log2=16)
    try:
        ref, ref_total = stream(fresh, t1, t2, table, roles, cuts(random.Random(1)), cuts(random.Random(2)))
    finally:
        fresh.close()
    assert got == ref and total == ref_total == 3000


# ---- frender demux ---------------------------------------------------------------------------------------------------
def run_demux(res, out, files, flags=None):
    from frender_b200.cli import frender_demux
    flags = flags or {}
    frender_demux(Namespace(r=str(res), d=str(out), o=flags.get("o"), no_index_hop=flags.get("i", False),
                            no_ambiguous=flags.get("a", False), no_undeter=False, no_samples=False,
                            files=[str(f) for f in files]))


def decompressed(out):
    return {n: gzip.open(out / n, "rb").read() for n in sorted(os.listdir(out))}


@pytest.mark.parametrize("device", ["1", "0"])
@pytest.mark.parametrize("level", ["6", "gpu", "bgzf"])
@pytest.mark.parametrize("name", ["c1", "c1_ia", "c4"])
def test_cli_single_end_golden(golden, tmp_path, monkeypatch, name, level, device):
    from conftest import unb64
    from frender_b200 import synth
    case = golden["demux"][name]
    scan = golden["scan"][case["scan_case"]]
    spec = synth.make_spec(scan["config"], n_samples=scan["n_samples"])
    r1 = tmp_path / "Undetermined_S0_L001_R1_001.fastq.gz"
    r1.write_bytes(gzip.compress(synth.generate_big(spec, 0, case["reads"], 1), 1))
    (tmp_path / "results.csv").write_bytes(unb64(case["results_csv"]))
    monkeypatch.setenv("FRENDER_SINGLE_END", "1")
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", level)
    monkeypatch.setenv("FRB_GZ_DEVICE", device)
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "1")
    run_demux(tmp_path / "results.csv", tmp_path / "out", [tmp_path], case["flags"])
    want = {f: v for f, v in case["sinks"].items() if f.endswith("_R1.fq.gz")}
    got = decompressed(tmp_path / "out")
    assert sorted(got) == sorted(want)                  # no R2 file
    for fname, w in want.items():
        assert len(got[fname]) == w["bytes"], fname
        assert hashlib.sha256(got[fname]).hexdigest() == w["sha256"], fname
    if level == "bgzf":
        for fname in got:
            blob = (tmp_path / "out" / fname).read_bytes()
            assert blob.endswith(bgzf.EOF_BLOCK)
            list(bgzf.iter_blocks(blob))


@pytest.fixture(scope="module")
def c4_lane(tmp_path_factory):
    from frender_b200 import synth
    from test_gpu_demux_gz import gz, scan_results
    d = tmp_path_factory.mktemp("c4se")
    spec = synth.make_spec("C4")
    r1, r2 = d / "L_S0_L001_R1_001.fastq.gz", d / "L_S0_L001_R2_001.fastq.gz"
    r1.write_bytes(gz(synth.generate_big(spec, 0, 200_000, 1), 6))
    r2.write_bytes(gz(synth.generate_big(spec, 0, 200_000, 2), 6))
    return d, scan_results(d, r1, spec), r1, r2


@pytest.mark.parametrize("level", ["6", "bgzf"])
def test_cli_single_end_equals_paired_r1(c4_lane, tmp_path, monkeypatch, level):
    _, res, r1, r2 = c4_lane
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", level)
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "1")
    monkeypatch.delenv("FRENDER_SINGLE_END", raising=False)
    run_demux(res, tmp_path / "paired", [r1, r2])
    monkeypatch.setenv("FRENDER_SINGLE_END", "1")
    run_demux(res, tmp_path / "single", [r1])
    paired, single = decompressed(tmp_path / "paired"), decompressed(tmp_path / "single")
    assert sorted(single) == sorted(n for n in paired if n.endswith("_R1.fq.gz"))
    assert sum(len(v) for v in single.values()) > 10 << 20
    for name in single:
        assert single[name] == paired[name], name


def test_cli_single_end_two_gpus(golden, tmp_path, monkeypatch):
    """FRENDER_GPUS=2 with three R1 files: every sink decompresses to what the one-GPU run writes."""
    from conftest import unb64
    from frender_b200 import synth
    from frender_b200._lib import lib
    from frender_b200.cli import main
    n = ctypes.c_int()
    lib.frb_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs")
    case = golden["demux"]["c1"]
    scan = golden["scan"][case["scan_case"]]
    spec = synth.make_spec(scan["config"], n_samples=scan["n_samples"])
    files = []
    for lane, (g0, g1) in enumerate([(0, 1200), (1200, 2100), (2100, 3000)], start=1):
        p = tmp_path / f"Undetermined_S0_L00{lane}_R1_001.fastq.gz"
        p.write_bytes(gzip.compress(synth.generate_big(spec, g0, g1, 1), 1))
        files.append(str(p))
    (tmp_path / "results.csv").write_bytes(unb64(case["results_csv"]))
    monkeypatch.setenv("FRENDER_SINGLE_END", "1")
    main(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "one")] + files)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    main(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "two")] + files)
    one, two = decompressed(tmp_path / "one"), decompressed(tmp_path / "two")
    assert sorted(one) == sorted(f for f in case["sinks"] if f.endswith("_R1.fq.gz"))
    assert one == two
