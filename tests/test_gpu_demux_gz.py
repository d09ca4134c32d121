"""Device inflate of the demux inputs: the span reader (frb_gz_open / frb_gz_read) returns exactly the text zlib
does, in spans of exactly the size asked for; it hands a file back to zlib behind the text it already returned; the
demux stream takes device spans; `frender demux` writes byte-identical sinks with FRB_GZ_DEVICE=1 and =0."""
import csv
import gzip
import hashlib
import os
import random
import re
import zlib
from argparse import Namespace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MIB = 1 << 20


@pytest.fixture(scope="module")
def ctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=16)
    yield c
    c.close()


def fastq(n_reads, seed=0, mate=1, config="C2"):
    from frender_b200 import synth
    return synth.generate_big(synth.make_spec(config, seed=1234 + seed), 0, n_reads, mate)


def gz(data, level=6):
    z = zlib.compressobj(level, zlib.DEFLATED, 31)
    return z.compress(data) + z.flush()


def read_spans(ctx, path, rng=None, size=None, may_decline=False):
    """All spans of the file (random sizes of 1 B .. 4 MiB, or `size`), fetched to the host: (text, spans, sizes);
    None when the device path declined the file (only where may_decline)."""
    ctx.gz_open(0, path)
    try:
        spans, sizes = [], []
        while True:
            want = size or rng.choice([1, 2, 17, 4095, 65536, 999_999, 4 * MIB, rng.randint(1, 4 * MIB)])
            s = ctx.gz_read(0, want, copy=True)
            if s.declined and may_decline:
                assert s.delivered == sum(x.size for x in spans)
                return None
            assert not s.declined, path
            spans.append(s)
            sizes.append(want)
            if s.eof or s.size == 0:
                break
        after = ctx.gz_read(0, 1000, copy=True)
        assert after.size == 0 and not after.declined
        return b"".join(s.data for s in spans), spans, sizes
    finally:
        ctx.gz_close(0)


def check_exact(spans, sizes, text):
    """Every span but the last has the size asked for; eof is set on the last one only; delivered counts them."""
    assert all(s.size == w for s, w in zip(spans[:-1], sizes[:-1]))
    assert [s.eof for s in spans].count(True) == 1 and spans[-1].eof
    assert spans[-1].delivered == len(text)


def bgzf(data, block=65280):
    return b"".join(gz(data[i:i + block], 6) for i in range(0, len(data), block)) or gz(b"")


def files_for_reader():
    big = fastq(60_000)                                    # ~ 20 MB of text
    return {
        "level1": (gz(big, 1), None),
        "level6": (gz(big, 6), None),
        "level9": (gz(big[:6 * MIB], 9), None),
        "multi_member": (b"".join(gz(big[i:i + 3 * MIB], 1 + i % 9) for i in range(0, len(big), 3 * MIB)), None),
        "bgzf_like": (bgzf(big[:8 * MIB]), None),
        "stored": (gz(big[:3 * MIB], 0), None),
        "empty": (gz(b""), None),
        "tiny": (gz(b"@r 1:N:0:A+C\nA\n+\nF\n"), None),
        "pieces_1MiB": (gz(big, 1), "1"),                 # > 3 MiB compressed: several pieces
        "one_and_a_bit_pieces": (gz(big[:5 * MIB + 123_457], 1), "1"),   # between 1 and 1.5 pieces
    }


@pytest.fixture(scope="module")
def reader_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("reader")
    out = {}
    for name, (blob, piece) in files_for_reader().items():
        p = d / f"{name}.fastq.gz"
        p.write_bytes(blob)
        out[name] = (str(p), piece)
    return out


@pytest.mark.parametrize("name", ["level1", "level6", "level9", "multi_member", "bgzf_like", "stored", "empty", "tiny",
                                  "pieces_1MiB", "one_and_a_bit_pieces"])
def test_reader_equals_zlib(ctx, reader_files, name, monkeypatch):
    path, piece = reader_files[name]
    if piece:
        monkeypatch.setenv("FRB_GZ_PIECE_MB", piece)
    want = gzip.decompress(open(path, "rb").read())
    if name == "one_and_a_bit_pieces":
        assert MIB < os.path.getsize(path) < 1.5 * MIB
    if name == "pieces_1MiB":
        assert os.path.getsize(path) > 3 * MIB
    rng = random.Random(sum(name.encode()))
    got = read_spans(ctx, path, rng, may_decline=name in ("empty", "stored"))   # as frb_gz_inflate may
    if got is None:
        return
    text, spans, sizes = got
    assert text == want
    check_exact(spans, sizes, want)


# ---- hand-back -------------------------------------------------------------------------------------------------------
def test_cr_in_a_late_piece_is_handed_back(ctx, tmp_path, monkeypatch):
    from frender_b200.cli import DeviceTextChunks, TextChunks
    monkeypatch.setenv("FRB_GZ_PIECE_MB", "1")
    text = fastq(60_000)
    at = len(text) - 2 * MIB
    at = text.index(b"\n", at)
    text = text[:at] + b"\r\n" + text[at + 1:]
    path = tmp_path / "cr.fastq.gz"
    path.write_bytes(gz(text, 1))
    ctx.gz_open(0, path)
    got, declined = [], None
    while True:
        s = ctx.gz_read(0, 1_000_000, copy=True)
        if s.declined:
            declined = s
            break
        assert s.size == 1_000_000
        got.append(s.data)
    ctx.gz_close(0)
    assert got and declined.delivered == sum(map(len, got)) and declined.delivered < at
    assert b"".join(got) == text[:declined.delivered]
    # the CLI's reader: device spans, then zlib in text mode behind them -- the bytes TextChunks alone gives
    dev = DeviceTextChunks(ctx, 1, path)
    host = TextChunks(path)
    cuts = [700_000, 1, 3 * MIB, 65_536]
    parts, want, k = [], [], 0
    while not (dev.eof and host.eof):
        n = cuts[k % len(cuts)]
        k += 1
        a, b = dev.read(n), host.read(n)
        parts.append(_span_bytes(ctx, a) if hasattr(a, "ptr") else a)   # a device span, or zlib's bytes
        want.append(b)
        assert dev.eof == host.eof
    dev.close()
    assert not dev.on_device
    assert parts == want
    assert b"".join(parts) == text.replace(b"\r\n", b"\n")


def _span_bytes(ctx, span):
    """A device span's bytes, read back through the driver API."""
    import ctypes
    from frender_b200._lib import lib
    out = np.empty(max(span.size, 1), np.uint8)
    if span.size:
        assert lib.frb_d2h(ctx._h, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(span.ptr), span.size) == 0
    return out[:span.size].tobytes()


@pytest.mark.parametrize("blob", [b"", b"hello", b"\x1f\x8b\x08" + b"\0" * 10, b"not a gzip file at all, longer"])
def test_not_gzip_or_tiny_is_declined_at_once(ctx, tmp_path, blob):
    path = tmp_path / "x.gz"
    path.write_bytes(blob)
    ctx.gz_open(0, path)
    s = ctx.gz_read(0, 4096)
    ctx.gz_close(0)
    assert s.declined and s.delivered == 0 and s.size == 0


def test_missing_file_is_declined(ctx, tmp_path):
    ctx.gz_open(1, tmp_path / "nope.gz")
    s = ctx.gz_read(1, 10)
    ctx.gz_close(1)
    assert s.declined and s.delivered == 0


def test_staging_overflow_in_a_late_piece(ctx, tmp_path, monkeypatch, capfd):
    monkeypatch.setenv("FRB_GZ_PIECE_MB", "1")
    monkeypatch.setenv("FRB_GZ_EXPAND", "2")
    monkeypatch.setenv("FRB_GZ_VERBOSE", "1")
    head = fastq(30_000)
    runs = b"".join(f"@run:{i} 1:N:0:ACGT+TTGA\n{'A' * 3000}\n+\n{'F' * 3000}\n".encode() for i in range(3000))
    text = head + runs + fastq(5000, seed=1)
    path = tmp_path / "runs.fastq.gz"
    path.write_bytes(gz(text, 6))
    got, spans, sizes = read_spans(ctx, str(path), random.Random(5))
    assert got == text
    check_exact(spans, sizes, text)
    err = capfd.readouterr().err
    assert re.search(r"gz: piece [1-9]\d* chunk \d+ of \d+: status", err), "no staging overflow in a late piece"


# ---- span lifetime through the demux stream --------------------------------------------------------------------------
def device_stream(ctx, p1, p2, table, roles, cut, pieces_between=True):
    """The demux stream fed with device spans of both mates (several read and pushed before a pop)."""
    from frender_b200.engine import pack_keys
    names = sorted({n for n in roles.values() if n})
    sid = {n: i for i, n in enumerate(names)}
    role_of = {"index_hop": "#hop", "ambiguous": "#amb", "undetermined": "#und"}
    keys = list(table)
    routes = np.array([sid[roles[table[k][1]] if table[k][0] == "demuxable" else roles[role_of[table[k][0]]]]
                       for k in keys], np.uint32)
    ctx.route_load(pack_keys(keys), routes, len(names))
    ctx.route_reset(cut)
    out = {n: (bytearray(), bytearray()) for n in names}
    ctx.gz_open(0, p1)
    ctx.gz_open(1, p2)
    queued, eof = 0, [False, False]

    def take():
        o1, o2, off1, off2 = ctx.route_pop()[:4]
        for n, i in sid.items():
            out[n][0].extend(o1[off1[i]:off1[i + 1]].tobytes())
            out[n][1].extend(o2[off2[i]:off2[i + 1]].tobytes())

    while not all(eof):
        spans = []
        for m in (0, 1):
            s = ctx.gz_read(m, cut)
            assert not s.declined
            eof[m] = eof[m] or s.eof or s.size == 0
            spans.append(s)
        ctx.route_push(spans[0], spans[1], (1 if eof[0] else 0) | (2 if eof[1] else 0))
        queued += 1
        if queued == 2:
            take()
            queued -= 1
    while queued:
        take()
        queued -= 1
    ctx.gz_close(0)
    ctx.gz_close(1)
    return {n: (bytes(a), bytes(b)) for n, (a, b) in out.items()}


@pytest.mark.parametrize("cut", [300_000, 16 * MIB])
def test_device_spans_through_the_stream_vs_oracle(ctx, tmp_path, monkeypatch, cut):
    """Pieces of 1 MiB: small cuts read many spans of one piece, large ones span several pieces; two chunks are in
    flight while the readers inflate further, so text buffers are reused under queued copies."""
    import frender_oracle as O
    from test_gpu_route import make_pair
    monkeypatch.setenv("FRB_GZ_PIECE_MB", "1")
    rng = random.Random(cut)
    t1, t2, table = make_pair(rng, 120_000, r2_records=110_000, crop_tail=5)
    p1, p2 = tmp_path / "a_R1.fastq.gz", tmp_path / "a_R2.fastq.gz"
    p1.write_bytes(gz(t1.encode(), 6))
    p2.write_bytes(gz(t2.encode(), 6))
    assert os.path.getsize(p1) > 2 * MIB
    roles = O.sink_names(table)
    want = O.route_pairs(t1.splitlines(keepends=True), t2.splitlines(keepends=True), table, roles)
    got = device_stream(ctx, p1, p2, table, roles, cut)
    for name, (w1, w2) in want.items():
        assert got[name][0] == w1, f"R1 of sink {name}"
        assert got[name][1] == w2, f"R2 of sink {name}"


def test_route_push_mixed_device_and_host_mates_vs_oracle(ctx, tmp_path):
    """R1 from device spans, R2 as host bytes, in the same stream."""
    import frender_oracle as O
    from frender_b200.engine import pack_keys
    from test_gpu_route import make_pair
    rng = random.Random(11)
    t1, t2, table = make_pair(rng, 8000, crop_tail=3)
    p1 = tmp_path / "m_R1.fastq.gz"
    p1.write_bytes(gz(t1.encode(), 1))
    roles = O.sink_names(table)
    want = O.route_pairs(t1.splitlines(keepends=True), t2.splitlines(keepends=True), table, roles)
    names = sorted({n for n in roles.values() if n})
    sid = {n: i for i, n in enumerate(names)}
    role_of = {"index_hop": "#hop", "ambiguous": "#amb", "undetermined": "#und"}
    routes = np.array([sid[roles[table[k][1]] if table[k][0] == "demuxable" else roles[role_of[table[k][0]]]]
                       for k in table], np.uint32)
    ctx.route_load(pack_keys(list(table)), routes, len(names))
    ctx.route_reset(1 * MIB)
    ctx.gz_open(0, p1)
    b2 = t2.encode()
    out = {n: (bytearray(), bytearray()) for n in names}
    p2, queued, e1 = 0, 0, False

    def take():
        o1, o2, off1, off2 = ctx.route_pop()[:4]
        for n, i in sid.items():
            out[n][0].extend(o1[off1[i]:off1[i + 1]].tobytes())
            out[n][1].extend(o2[off2[i]:off2[i + 1]].tobytes())

    while True:
        s = ctx.gz_read(0, rng.randint(1, 200_000))
        e1 = e1 or s.eof
        d2 = b2[p2:p2 + rng.randint(1, 200_000)]
        p2 += len(d2)
        final = (1 if e1 else 0) | (2 if p2 >= len(b2) else 0)
        ctx.route_push(s, d2, final)
        queued += 1
        if queued == 2:
            take()
            queued -= 1
        if final == 3:
            break
    while queued:
        take()
        queued -= 1
    ctx.gz_close(0)
    for name, (w1, w2) in want.items():
        assert bytes(out[name][0]) == w1 and bytes(out[name][1]) == w2, name


# ---- frender demux: FRB_GZ_DEVICE=1 against =0 -----------------------------------------------------------------------
def beside(tmp_path, r1):
    """R1 next to a damaged or altered R2 in tmp_path (demux pairs the mates of one directory)."""
    link = tmp_path / r1.name
    os.symlink(r1, link)
    return link


def run_demux(res, out, files):
    from frender_b200.cli import frender_demux
    frender_demux(Namespace(r=str(res), d=str(out), o=None, no_index_hop=False, no_ambiguous=False, no_undeter=False,
                            no_samples=False, files=[str(f) for f in files]))


def sink_bytes(out):
    return {n: (out / n).read_bytes() for n in sorted(os.listdir(out))}


def scan_results(d, r1, spec, wide=False):
    """frender scan of R1, written as the results CSV demux reads."""
    from frender_b200.cli import frender_scan
    (d / "SampleSheet.csv").write_text(spec.sheet_csv())
    old = os.getcwd()
    os.chdir(d)
    try:
        frender_scan(Namespace(n=1, rc=True, c=1, s=None, o="res", p=None, b="SampleSheet.csv", files=[str(r1)]))
    finally:
        os.chdir(old)
    src = next(f for f in os.listdir(d) if f.startswith("frender-scan-results_"))
    rows = list(csv.reader(open(d / src, newline="")))
    order = [rows[0].index(c) for c in ("idx1", "idx2", "reads", "matched_idx1", "matched_idx2", "read_type",
                                        "sample_name", "demux_ok")]
    with open(d / "results.csv", "w", newline="") as fh:
        csv.writer(fh).writerows([[r[i] for i in order] for r in rows])
    return d / "results.csv"


@pytest.fixture(scope="module")
def c4_lane(tmp_path_factory):
    from frender_b200 import synth
    d = tmp_path_factory.mktemp("c4")
    spec = synth.make_spec("C4")
    t1, t2 = synth.generate_big(spec, 0, 200_000, 1), synth.generate_big(spec, 0, 200_000, 2)
    r1, r2 = d / "L_S0_L001_R1_001.fastq.gz", d / "L_S0_L001_R2_001.fastq.gz"
    r1.write_bytes(gz(t1, 6))
    r2.write_bytes(gz(t2, 6))
    res = scan_results(d, r1, spec)
    return d, res, r1, r2, t1, t2


@pytest.fixture
def count_reads(monkeypatch):
    """gz_read calls that returned device text."""
    from frender_b200.engine import Context
    real = Context.gz_read
    n = {"device": 0}

    def counted(self, *a, **k):
        s = real(self, *a, **k)
        if not s.declined and s.size:
            n["device"] += 1
        return s
    monkeypatch.setattr(Context, "gz_read", counted)
    return n


def both_ways(tmp_path, monkeypatch, res, files, count):
    outs = {}
    for dev in ("0", "1"):
        monkeypatch.setenv("FRB_GZ_DEVICE", dev)
        before = count["device"]
        out = tmp_path / f"out{dev}"
        run_demux(res, out, files)
        outs[dev] = sink_bytes(out)
        if dev == "0":
            assert count["device"] == before
    return outs


@pytest.mark.parametrize("level", ["6", "gpu"])
@pytest.mark.parametrize("chunk_mb", ["0", "64"])
def test_cli_device_inflate_byte_identical(c4_lane, tmp_path, monkeypatch, count_reads, level, chunk_mb):
    d, res, r1, r2, _, _ = c4_lane
    monkeypatch.setenv("FRB_GZ_PIECE_MB", "1")
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", level)
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", chunk_mb)               # 0: MIN_CHUNK
    outs = both_ways(tmp_path, monkeypatch, res, [r1, r2], count_reads)
    assert outs["0"] == outs["1"] and len(outs["1"]) > 4
    assert count_reads["device"] >= 2 * (2 if chunk_mb == "64" else 20)


def test_cli_device_inflate_short_r2(c4_lane, tmp_path, monkeypatch, count_reads):
    d, res, r1, _, _, t2 = c4_lane
    cut = t2.index(b"\n@", len(t2) * 2 // 3) + 1
    short = tmp_path / "L_S0_L001_R2_001.fastq.gz"
    short.write_bytes(gz(t2[:cut], 1))
    monkeypatch.setenv("FRB_GZ_PIECE_MB", "1")
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "0")
    outs = both_ways(tmp_path, monkeypatch, res, [beside(tmp_path, r1), short], count_reads)
    assert outs["0"] == outs["1"] and count_reads["device"] > 0


def test_cli_one_mate_handed_back_mid_file(c4_lane, tmp_path, monkeypatch, count_reads):
    """CRLF in the second half of R2 only: R2 goes to zlib part way, R1 stays on the device."""
    import frender_b200.cli as cli
    d, res, r1, _, _, t2 = c4_lane
    half = len(t2) // 2
    crlf = tmp_path / "L_S0_L001_R2_001.fastq.gz"
    crlf.write_bytes(gz(t2[:half] + t2[half:].replace(b"\n", b"\r\n"), 6))
    monkeypatch.setenv("FRB_GZ_PIECE_MB", "1")
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "0")
    handed = []
    real = cli.DeviceTextChunks.read

    def watch(self, size):
        was = self.on_device
        out = real(self, size)
        if was and not self.on_device:
            handed.append((self.slot, self.host is not None))
        return out
    monkeypatch.setattr(cli.DeviceTextChunks, "read", watch)
    outs = both_ways(tmp_path, monkeypatch, res, [beside(tmp_path, r1), crlf], count_reads)
    assert outs["0"] == outs["1"]
    assert handed == [(1, True)]
    assert count_reads["device"] > 50


def test_cli_device_inflate_wide_pair(tmp_path, monkeypatch, count_reads):
    from frender_b200.synth import generate_big
    from test_gpu_wide import spec_12x12
    spec = spec_12x12()
    r1, r2 = tmp_path / "W_S0_L001_R1_001.fastq.gz", tmp_path / "W_S0_L001_R2_001.fastq.gz"
    r1.write_bytes(gz(generate_big(spec, 0, 30_000, 1), 1))
    r2.write_bytes(gz(generate_big(spec, 0, 30_000, 2), 1))
    res = scan_results(tmp_path, r1, spec)
    assert any(len(row[0]) + len(row[1]) > 21 for row in csv.reader(open(res)))
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "0")
    outs = both_ways(tmp_path, monkeypatch, res, [r1, r2], count_reads)
    assert outs["0"] == outs["1"] and count_reads["device"] > 0


def test_cli_device_inflate_golden_c4(golden, tmp_path, monkeypatch, count_reads):
    from conftest import unb64
    from frender_b200 import synth
    case = golden["demux"]["c4"]
    scan = golden["scan"][case["scan_case"]]
    spec = synth.make_spec(scan["config"], n_samples=scan["n_samples"])
    p1 = tmp_path / "Undetermined_S0_L001_R1_001.fastq.gz"
    p2 = tmp_path / "Undetermined_S0_L001_R2_001.fastq.gz"
    p1.write_bytes(gzip.compress(synth.generate_big(spec, 0, case["reads"], 1), 1))
    p2.write_bytes(gzip.compress(synth.generate_big(spec, 0, case["reads"], 2), 1))
    (tmp_path / "results.csv").write_bytes(unb64(case["results_csv"]))
    monkeypatch.setenv("FRB_GZ_DEVICE", "1")
    run_demux(tmp_path / "results.csv", tmp_path / "out", [p1, p2])
    assert count_reads["device"] > 0
    assert sorted(os.listdir(tmp_path / "out")) == sorted(case["sinks"])
    for fname, want in case["sinks"].items():
        raw = gzip.open(tmp_path / "out" / fname, "rb").read()
        assert len(raw) == want["bytes"], fname
        assert hashlib.sha256(raw).hexdigest() == want["sha256"], fname


@pytest.mark.parametrize("damage", ["truncated", "crc_flipped"])
def test_cli_damaged_mate_same_error(c4_lane, tmp_path, monkeypatch, damage):
    d, res, r1, r2, _, _ = c4_lane
    blob = bytearray(r2.read_bytes())
    if damage == "truncated":
        blob = blob[:len(blob) * 3 // 4]
    else:
        blob[-8] ^= 0x5A
    bad = tmp_path / "L_S0_L001_R2_001.fastq.gz"
    bad.write_bytes(bytes(blob))
    r1 = beside(tmp_path, r1)
    monkeypatch.setenv("FRB_GZ_PIECE_MB", "1")
    monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "0")
    errors = {}
    for dev in ("0", "1"):
        monkeypatch.setenv("FRB_GZ_DEVICE", dev)
        with pytest.raises(Exception) as exc:
            run_demux(res, tmp_path / f"out{dev}", [r1, bad])
        errors[dev] = (type(exc.value), str(exc.value))
    assert errors["0"] == errors["1"], errors
