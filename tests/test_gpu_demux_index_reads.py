"""Demux with index reads (frb_route_set_mates2, FRENDER_INDEX_READS=1): the C-ABI rules of the N-mate stream, the
stream against the N-mate oracle through host bytes, device spans and host zlib, the sink limit of a 4-mate stream,
four span readers at once, and frender demux in every output format, with wide keys, single-end and on two GPUs."""
import ctypes
import gzip
import os
import random
import zlib
from argparse import Namespace

import numpy as np
import pytest

import frender_oracle as O
import index_reads_oracle as IR
from frender_b200 import bgzf

pytestmark = pytest.mark.gpu

KINDS = ["demuxable", "index_hop", "ambiguous", "undetermined"]


def make_lane(rng, n, n_keys=40, half=8):
    """R1, R2, I1, I2 texts of n records keyed by index pairs of half+half symbols (the index reads carry the two
    halves as their sequence), and a results table over the keys."""
    bases = "ACGTN"
    keys = ["".join(rng.choice(bases) for _ in range(half)) + "+" + "".join(rng.choice(bases) for _ in range(half))
            for _ in range(n_keys)]
    texts = [[], [], [], []]
    for i in range(n):
        k = rng.choice(keys)
        a, b = k.split("+")
        l1, l2 = rng.randint(1, 300), rng.randint(1, 300)
        name = f"@M0:{i}:FC:1:{rng.randint(1, 99999)}:{rng.randint(1, 99999)}"
        texts[0].append(f"{name} 1:N:0:{k}\n{'A' * l1}\n+\n{'F' * l1}\n")
        texts[1].append(f"{name} 2:N:0:{k}\n{'C' * l2}\n+\n{'#' * l2}\n")
        texts[2].append(f"{name} 1:N:0:{k}\n{a}\n+\n{'F' * len(a)}\n")
        texts[3].append(f"{name} 2:N:0:{k}\n{b}\n+\n{':' * len(b)}\n")
    table = {k: (KINDS[j % 4], f"S{j % 7}" if j % 4 == 0 else "") for j, k in enumerate(keys)}
    return ["".join(t) for t in texts], table


def load(ctx, table, roles):
    from test_gpu_demux_single_end import load as load_table
    return load_table(ctx, table, roles)


def lines(text):
    return text.splitlines(keepends=True)


def reads_of(texts, single):
    """(the texts in mate order, the key mate) of a lane: R1, R2, I1, I2, or R1, I1, I2 when single-end."""
    return ([texts[0]] + texts[2:], 0) if single else (texts, 1)


def stream_mates(ctx, readers, table, roles, key_mate, window=1 << 20, mode="plain"):
    """Push the mates' readers (read(n) -> bytes or GzSpan, .eof) through a stream of len(readers) mates, two chunks
    in flight, every mate reading `window` - what it has not had routed yet (the chunk in flight included).  Returns
    {sink: tuple of the mates' bytes} and the records routed."""
    names = load(ctx, table, roles)
    M = len(readers)
    ctx.route_gzip(mode != "plain", bgzf=mode == "bgzf")
    ctx.route_mates(M, key_mate)
    ctx.route_reset(window)
    out = {n: [bytearray() for _ in range(M)] for n in names}
    unpack = {"plain": bytes, "gzip": lambda b: zlib.decompress(b, 31),
              "bgzf": lambda b: b"".join(zlib.decompress(bytes(b[p:p + s + 1]), 31) for p, s, _ in bgzf.iter_blocks(b))}
    total, flags, sizes, carry = 0, [], [], [0] * M

    def take():
        nonlocal total, carry
        outs, offs, n, carry = ctx.route_popv()
        total += n
        for i, name in enumerate(names):
            for m in range(M):
                cell = outs[m][offs[m][i]:offs[m][i + 1]]
                out[name][m].extend(unpack[mode](cell.tobytes()) if len(cell) else b"")

    try:
        while True:
            ahead = [sum(s[m] for s in sizes) for m in range(M)]
            got = [r.read(max(window - c - a, 1)) if not r.eof else b"" for r, c, a in zip(readers, carry, ahead)]
            flags.append(sum(1 << m for m, r in enumerate(readers) if r.eof))
            sizes.append([len(g) for g in got])
            ctx.route_pushv(got, flags[-1])
            if len(flags) == 2:
                take()
                was = flags.pop(0)
                sizes.pop(0)
                if any(was >> m & 1 and carry[m] == 0 for m in range(M)):
                    break
            if all(r.eof for r in readers):
                break
        while flags:
            take()
            flags.pop(0)
    finally:
        ctx.route_reset()
        ctx.route_gzip(False)
        ctx.route_mates(2)
    return {n: tuple(bytes(b) for b in v) for n, v in out.items()}, total


class Cuts:
    """A text read in pieces of random size (at most what is asked for)."""

    def __init__(self, text, rng):
        self.data, self.pos, self.rng, self.eof = text.encode(), 0, rng, False

    def read(self, n):
        piece = self.data[self.pos:self.pos + self.rng.randint(1, n)]
        self.pos += len(piece)
        self.eof = self.pos >= len(self.data)
        return piece


@pytest.fixture(scope="module")
def ctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=16)
    yield c
    c.close()


# ---- C-ABI -------------------------------------------------------------------------------------------------------
def test_set_mates2_rules(ctx):
    from frender_b200 import _lib
    from frender_b200._lib import lib
    from frender_b200.engine import FrbError
    texts, table = make_lane(random.Random(1), 500)
    roles = O.sink_names(table)
    load(ctx, table, roles)
    for mates, key in ((0, 0), (5, 1), (3, -1), (3, 3), (1, 1)):
        assert lib.frb_route_set_mates2(ctx._h, mates, key) == _lib.ERR_ARG, (mates, key)
    assert lib.frb_route_set_mates(ctx._h, 3) == _lib.ERR_ARG
    ctx.route_mates(4, 1)
    ctx.route_reset()
    # a 4-mate stream takes the vector calls only
    with pytest.raises(FrbError) as err:
        ctx.route_push(texts[0].encode(), texts[1].encode(), 3)
    assert err.value.code == _lib.ERR_STATE
    ctx.route_pushv([t.encode() for t in texts], 15)
    assert lib.frb_route_set_mates2(ctx._h, 2, 1) == _lib.ERR_STATE        # a chunk in flight
    with pytest.raises(FrbError) as err:
        ctx.route_pop()
    assert err.value.code == _lib.ERR_STATE
    outs, offs, n, carry = ctx.route_popv()
    assert n == 500 and carry == [0, 0, 0, 0]
    want = IR.route_mates([lines(t) for t in texts], 1, table, roles)
    names = sorted({v for v in roles.values() if v})
    for i, name in enumerate(names):
        assert tuple(outs[m][offs[m][i]:offs[m][i + 1]].tobytes() for m in range(4)) == want.get(name, (b"",) * 4)
    ctx.route_mates(2)
    ctx.route_reset()


@pytest.mark.parametrize("mates", [1, 2])
def test_pushv_popv_equal_push_pop_on_golden_c1(ctx, golden, mates):
    from conftest import unb64
    from frender_b200 import synth
    case = golden["demux"]["c1"]
    scan = golden["scan"][case["scan_case"]]
    spec = synth.make_spec(scan["config"], n_samples=scan["n_samples"])
    r1, r2 = synth.generate_big(spec, 0, case["reads"], 1), synth.generate_big(spec, 0, case["reads"], 2)
    import tempfile
    with tempfile.NamedTemporaryFile("wb", suffix=".csv", delete=False) as fh:
        fh.write(unb64(case["results_csv"]))
    table = O.parse_results_file(fh.name)
    os.unlink(fh.name)
    roles = O.sink_names(table)
    names = load(ctx, table, roles)
    runs = []
    for vector in (False, True):
        ctx.route_mates(mates)
        ctx.route_reset(1 << 20)
        cells = []
        for k in range(0, max(len(r1), len(r2)), 300_000):
            a, b = r1[k:k + 300_000], r2[k:k + 300_000]
            final = (1 if k + 300_000 >= len(r1) else 0) | (2 if k + 300_000 >= len(r2) else 0)
            if vector:
                ctx.route_pushv([a, b][:mates], final)
                outs, offs, n, carry = ctx.route_popv()
            else:
                ctx.route_push(a, b if mates == 2 else None, final)
                o1, o2, off1, off2, n, c1, c2 = ctx.route_pop()
                outs, offs, carry = [o1, o2][:mates], [off1, off2][:mates], [c1, c2][:mates]
            cells.append((n, list(carry), [[o[f[i]:f[i + 1]].tobytes() for i in range(len(names))]
                                          for o, f in zip(outs, offs)]))
        runs.append(cells)
    ctx.route_mates(2)
    ctx.route_reset()
    assert runs[0] == runs[1]
    assert sum(c[0] for c in runs[0]) == case["reads"]


def test_sink_limit_of_a_four_mate_stream(ctx):
    from frender_b200 import _lib
    from frender_b200._lib import lib
    from frender_b200.engine import FrbError, pack_keys
    texts, _ = make_lane(random.Random(2), 300)
    keys = sorted({ln.rsplit(":", 1)[1] for ln in texts[1].splitlines()[0::4]})
    limit = (227 << 10) // 16                                                # 14,528
    for n_sinks in (limit, limit + 1):
        ctx.route_mates(2)
        ids = np.full(len(keys), n_sinks - 1, np.uint32)                     # every record in the last sink
        ctx.route_load(pack_keys(keys), ids, n_sinks)
        if n_sinks > limit:
            assert lib.frb_route_set_mates2(ctx._h, 4, 1) == _lib.ERR_ARG
            assert lib.frb_route_set_mates2(ctx._h, 3, 1) == _lib.OK        # 3 mates take 16,384 sinks
            ctx.route_mates(2)
            continue
        ctx.route_mates(4, 1)
        ctx.route_reset()
        ctx.route_pushv([t.encode() for t in texts], 15)
        outs, offs, n, _ = ctx.route_popv()
        assert n == 300
        for m in range(4):
            assert offs[m][n_sinks - 1] == 0 and outs[m].tobytes() == texts[m].encode()
    # a table with too many sinks for a 4-mate stream is refused when it is loaded
    ctx.route_mates(2)
    ctx.route_load(pack_keys(keys), np.zeros(len(keys), np.uint32), limit)
    ctx.route_mates(4, 1)
    with pytest.raises(FrbError) as err:
        ctx.route_load(pack_keys(keys), np.zeros(len(keys), np.uint32), limit + 1)
    assert err.value.code == _lib.ERR_ARG
    ctx.route_mates(2)
    ctx.route_reset()


@pytest.mark.parametrize("mode", ["plain", "gzip", "bgzf"])
def test_route_pair_then_a_four_mate_stream(mode):
    """frb_route_pair builds a fresh context's stream for a plain pair (two mates, no gzip buffers); the 4-mate
    stream pushed after it gets the buffers of its index-read mates and of its format before its first chunk, and
    routes as the oracle does, for one chunk and for a whole stream after it."""
    from frender_b200.engine import Context
    rng = random.Random(61)
    texts, table = make_lane(rng, 3000)
    roles = O.sink_names(table)
    unpack = {"plain": bytes, "gzip": lambda b: zlib.decompress(b, 31),
              "bgzf": lambda b: b"".join(zlib.decompress(bytes(b[p:p + s + 1]), 31) for p, s, _ in bgzf.iter_blocks(b))}
    c = Context(0, table_log2=16)
    try:
        names = load(c, table, roles)
        c.route_gzip(mode != "plain", bgzf=mode == "bgzf")
        c.route_mates(4, 1)
        o1, o2, off1, off2, pairs, used1, used2 = c.route_pair(texts[0].encode(), texts[1].encode(), 3)
        pair = O.route_pairs(lines(texts[0]), lines(texts[1]), table, roles)
        assert pairs == 3000 and used1 == len(texts[0]) and used2 == len(texts[1])
        for i, n in enumerate(names):
            assert (bytes(o1[off1[i]:off1[i + 1]]), bytes(o2[off2[i]:off2[i + 1]])) == pair.get(n, (b"", b""))
        want = IR.route_mates([lines(t) for t in texts], 1, table, roles)
        c.route_reset(1 << 20)
        c.route_pushv([t.encode() for t in texts], 15)
        outs, offs, n, carry = c.route_popv()
        assert n == 3000 and carry == [0, 0, 0, 0]
        for i, name in enumerate(names):
            cells = [outs[m][offs[m][i]:offs[m][i + 1]].tobytes() for m in range(4)]
            assert tuple(unpack[mode](x) if x else b"" for x in cells) == want.get(name, (b"",) * 4), name
        got, total = stream_mates(c, [Cuts(t, rng) for t in texts], table, roles, 1, mode=mode)
        assert total == 3000 and got == {k: want.get(k, (b"",) * 4) for k in got}
    finally:
        c.close()


# ---- the stream against the oracle ---------------------------------------------------------------------------------
CASES = ["equal", "index_shorter", "partial_tails", "crlf"]


def lane_files(tmp_path, texts, crlf=False):
    paths = []
    for read, t in zip(("R1", "R2", "I1", "I2"), texts):
        p = tmp_path / f"L_S1_L001_{read}_001.fastq.gz"
        data = t.replace("\n", "\r\n") if crlf and read == "I1" else t
        p.write_bytes(gzip.compress(data.encode(), 6))
        paths.append(p)
    return paths


@pytest.mark.parametrize("single", [False, True])
@pytest.mark.parametrize("inflate", ["device", "zlib"])
@pytest.mark.parametrize("case", CASES)
def test_stream_matches_the_oracle(ctx, tmp_path, case, inflate, single):
    from frender_b200.cli import DeviceTextChunks, TextChunks
    rng = random.Random(sum(case.encode()) + 3 * single)
    texts, table = make_lane(rng, 12000)
    if case == "index_shorter":
        texts[2] = texts[2][:texts[2].index("@M0:7000:") + 11]             # a partial record, then the file ends
    elif case == "partial_tails":
        texts = [t[:-rng.randint(2, 9)] for t in texts]
    roles = O.sink_names(table)
    paths = lane_files(tmp_path, texts, crlf=case == "crlf")
    mates, key = reads_of(paths, single)
    with_text = [gzip.open(p, "rt").read() for p in mates]                  # text mode (F:776)
    want = IR.route_mates([lines(t) for t in with_text], key, table, roles)
    readers = [DeviceTextChunks(ctx, m, p) if inflate == "device" else TextChunks(p) for m, p in enumerate(mates)]
    wrapped = [RandomSizes(r, rng) for r in readers]
    try:
        got, total = stream_mates(ctx, wrapped, table, roles, key)
    finally:
        for r in readers:
            if isinstance(r, DeviceTextChunks):
                r.close()
    names = sorted(got)
    assert total == (7001 if case == "index_shorter" else 12000)
    for name in names:
        assert got[name] == want.get(name, (b"",) * len(mates)), f"{case}: sink {name}"


class RandomSizes:
    """A reader asked for random amounts up to what the stream wants."""

    def __init__(self, reader, rng):
        self.r, self.rng = reader, rng

    @property
    def eof(self):
        return self.r.eof

    def read(self, n):
        return self.r.read(self.rng.randint(max(1, n // 8), n))


@pytest.mark.parametrize("mode", ["gzip", "bgzf"])
def test_stream_formats_match_the_oracle(ctx, mode):
    rng = random.Random(31)
    texts, table = make_lane(rng, 20000)
    roles = O.sink_names(table)
    want = IR.route_mates([lines(t) for t in texts], 1, table, roles)
    got, total = stream_mates(ctx, [Cuts(t, rng) for t in texts], table, roles, 1, mode=mode)
    assert total == 20000
    assert got == {n: want.get(n, (b"",) * 4) for n in got}


def test_four_span_readers_at_once(ctx, tmp_path):
    from frender_b200 import synth
    spec = synth.make_spec("C4")
    texts = [synth.generate_big(spec, 0, 60_000, 1), synth.generate_big(spec, 0, 60_000, 2),
             synth.generate_big(spec, 0, 60_000, 1, index_read=1), synth.generate_big(spec, 0, 60_000, 1, index_read=2)]
    paths = []
    for k, t in enumerate(texts):
        p = tmp_path / f"m{k}.fastq.gz"
        p.write_bytes(gzip.compress(t, 6))
        paths.append(p)
        ctx.gz_open(k, p)
    got = [bytearray() for _ in texts]
    try:
        done = [False] * 4
        while not all(done):
            for k in range(4):
                if not done[k]:
                    span = ctx.gz_read(k, 1 << 20, copy=True)
                    assert not span.declined
                    got[k].extend(span.data[:span.size])
                    done[k] = span.size == 0 or span.eof
    finally:
        for k in range(4):
            ctx.gz_close(k)
    for k, t in enumerate(texts):
        assert bytes(got[k]) == zlib.decompress(paths[k].read_bytes(), 31), k


# ---- frender demux -------------------------------------------------------------------------------------------------
def run_demux(res, out, files):
    from frender_b200.cli import frender_demux
    frender_demux(Namespace(r=str(res), d=str(out), o=None, no_index_hop=False, no_ambiguous=False, no_undeter=False,
                            no_samples=False, files=[str(f) for f in files]))


def results_csv(path, table):
    with open(path, "w") as fh:
        fh.write("idx1,idx2,reads,matched_idx1,matched_idx2,read_type,sample_name\n")
        for k, (kind, sid) in table.items():
            a, b = k.split("+")
            fh.write(f"{a},{b},1,{a},{b},{kind},{sid}\n")
    return path


def decompressed(out):
    return {n: gzip.open(out / n, "rb").read() for n in sorted(os.listdir(out))}


def expected_files(texts, table, single):
    roles = O.sink_names(table)
    mates, key = reads_of(texts, single)
    reads = (["R1"] if single else ["R1", "R2"]) + ["I1", "I2"]
    want = IR.route_mates([lines(t) for t in mates], key, table, roles)
    names = {v for v in roles.values() if v}
    return {f"{n}_frender-demux_{r}.fq.gz": want.get(n, (b"",) * len(reads))[m]
            for n in names for m, r in enumerate(reads)}


@pytest.mark.parametrize("level", ["6", "gpu", "bgzf"])
def test_cli_every_format(tmp_path, monkeypatch, level):
    texts, table = make_lane(random.Random(41), 30000)
    d = tmp_path / "in"
    d.mkdir()
    lane_files(d, texts)
    res = results_csv(tmp_path / "results.csv", table)
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", level)
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "1")
    monkeypatch.delenv("FRENDER_INDEX_READS", raising=False)
    run_demux(res, tmp_path / "plain", [d / "L_S1_L001_R1_001.fastq.gz", d / "L_S1_L001_R2_001.fastq.gz"])
    monkeypatch.setenv("FRENDER_INDEX_READS", "1")
    run_demux(res, tmp_path / "out", [d])
    got = decompressed(tmp_path / "out")
    assert got == expected_files(texts, table, False)
    # the R1 / R2 sinks are the files of the run without index reads, byte for byte
    plain = sorted(os.listdir(tmp_path / "plain"))
    assert plain == sorted(n for n in got if n.endswith(("_R1.fq.gz", "_R2.fq.gz")))
    for name in plain:
        assert (tmp_path / "out" / name).read_bytes() == (tmp_path / "plain" / name).read_bytes(), name
    if level == "bgzf":
        for name in got:
            blob = (tmp_path / "out" / name).read_bytes()
            assert blob.endswith(bgzf.EOF_BLOCK)
            assert sum(isize for _, _, isize in bgzf.iter_blocks(blob)) == len(got[name])


def test_cli_wide_lane(tmp_path, monkeypatch):
    texts, table = make_lane(random.Random(43), 8000, half=12)
    d = tmp_path / "in"
    d.mkdir()
    lane_files(d, texts)
    res = results_csv(tmp_path / "results.csv", table)
    monkeypatch.setenv("FRENDER_INDEX_READS", "1")
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "1")
    run_demux(res, tmp_path / "out", [d])
    assert decompressed(tmp_path / "out") == expected_files(texts, table, False)


@pytest.mark.parametrize("inflate", ["1", "0"])
def test_cli_single_end_with_index_reads(tmp_path, monkeypatch, inflate):
    texts, table = make_lane(random.Random(47), 20000)
    d = tmp_path / "in"
    d.mkdir()
    paths = lane_files(d, texts)
    os.unlink(paths[1])                                                     # no R2
    res = results_csv(tmp_path / "results.csv", table)
    monkeypatch.setenv("FRENDER_INDEX_READS", "1")
    monkeypatch.setenv("FRENDER_SINGLE_END", "1")
    monkeypatch.setenv("FRB_GZ_DEVICE", inflate)
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "1")
    run_demux(res, tmp_path / "out", [d])
    assert decompressed(tmp_path / "out") == expected_files(texts, table, True)


def test_cli_two_gpus(tmp_path, monkeypatch):
    """FRENDER_GPUS=2 with three lanes: every sink of every read decompresses to what the one-GPU run writes."""
    from frender_b200._lib import lib
    from frender_b200.cli import main
    n = ctypes.c_int()
    lib.frb_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs")
    rng = random.Random(53)
    d = tmp_path / "in"
    d.mkdir()
    tables = {}
    for lane in range(1, 4):
        texts, table = make_lane(rng, 3000, n_keys=20)
        tables.update(table)
        for read, t in zip(("R1", "R2", "I1", "I2"), texts):
            (d / f"L_S1_L00{lane}_{read}_001.fastq.gz").write_bytes(gzip.compress(t.encode(), 1))
    res = results_csv(tmp_path / "results.csv", tables)
    monkeypatch.setenv("FRENDER_INDEX_READS", "1")
    main(["demux", "-r", str(res), "-d", str(tmp_path / "one"), str(d)])
    monkeypatch.setenv("FRENDER_GPUS", "2")
    main(["demux", "-r", str(res), "-d", str(tmp_path / "two"), str(d)])
    one, two = decompressed(tmp_path / "one"), decompressed(tmp_path / "two")
    assert any(n.endswith("_I2.fq.gz") for n in one)
    assert one == two
