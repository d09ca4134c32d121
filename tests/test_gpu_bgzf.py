"""BGZF written on the device: frb_gz_deflate_bgzf gives complete BGZF files whose blocks inflate one by one, the
demux stream in BGZF format returns runs of whole blocks that decompress to plain mode's cells, `frender demux` with
FRENDER_GZIP_LEVEL=bgzf writes BGZF sinks with the reference's bytes, and the device inflate reads BGZF back."""
import ctypes
import gzip
import hashlib
import os
import random
import zlib

import numpy as np
import pytest

from frender_b200 import bgzf

pytestmark = pytest.mark.gpu

KIB, MIB = 1024, 1 << 20
BLOCK = 49152


@pytest.fixture(scope="module")
def ctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=16)
    yield c
    c.close()


def fastq(n_bytes, binned):
    from frender_b200 import synth
    spec = synth.make_spec("C2")
    data = synth.generate_big(spec, 0, n_bytes // 300 + 1)[:n_bytes]
    return synth.binned_qualities(data, 7) if binned else data


def text_like(n, seed):
    rng = random.Random(seed)
    words = [bytes(rng.choice(b"ACGTNacgtn:+@ \n") for _ in range(rng.randint(1, 12))) for _ in range(300)]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words)
    return bytes(out[:n])


def check_blocks(buf, want, eof=True):
    """buf is whole BGZF blocks (and the EOF block at the end when eof) holding `want`: every block within the size
    limits, its deflate data inflating on its own to bytes that match its CRC-32 and ISIZE.  Returns the block
    count (EOF block excluded)."""
    blocks = list(bgzf.iter_blocks(buf))
    if eof:
        assert buf[-28:] == bgzf.EOF_BLOCK and blocks[-1] == (len(buf) - 28, 27, 0)
        blocks = blocks[:-1]
    pos, got = 0, []
    for off, bsize, isize in blocks:
        assert off == pos and bsize + 1 <= 65536
        assert 0 < isize <= BLOCK
        blk = bytes(buf[off:off + bsize + 1])
        d = zlib.decompressobj(-15)
        raw = d.decompress(blk[18:-8]) + d.flush()
        assert d.eof and not d.unused_data
        crc, n = np.frombuffer(blk[-8:], "<u4")
        assert len(raw) == isize == n and zlib.crc32(raw) == crc
        got.append(raw)
        pos = off + bsize + 1
    assert pos == len(buf) - (28 if eof else 0)
    # every block but the cell's last is full: blocks are cut every 49,152 input bytes
    assert all(len(r) == BLOCK for r in got[:-1])
    assert b"".join(got) == want
    return len(blocks)


CASES = {
    "1": lambda: b"A",
    "16383": lambda: text_like(16383, 1),
    "16384": lambda: text_like(16384, 2),
    "16385": lambda: text_like(16385, 3),
    "49151": lambda: text_like(49151, 4),
    "49152": lambda: text_like(49152, 5),
    "49153": lambda: text_like(49153, 6),
    "3x49152+7": lambda: text_like(3 * 49152 + 7, 7),
    "random1MiB": lambda: np.random.default_rng(1).integers(0, 256, 1 << 20, np.uint8).tobytes(),
    "run1M": lambda: b"\x00" * (1 << 20),
    "fastq8MB_allF": lambda: fastq(8 << 20, False),
    "fastq8MB_binned": lambda: fastq(8 << 20, True),
}


@pytest.mark.parametrize("name", list(CASES))
def test_gz_deflate_bgzf_round_trips(ctx, name):
    from frender_b200._lib import lib
    data = CASES[name]()
    z = ctx.gz_deflate(data, bgzf=True)
    assert len(z) <= lib.frb_gz_deflate_bgzf_bound(len(data))
    assert gzip.decompress(z) == data
    assert check_blocks(z, data) == -(-len(data) // BLOCK)


def test_gz_deflate_bgzf_of_nothing_is_the_eof_block(ctx):
    from frender_b200._lib import lib
    assert ctx.gz_deflate(b"", bgzf=True) == bgzf.EOF_BLOCK
    assert lib.frb_gz_deflate_bgzf_bound(0) == 28


def test_gz_deflate_bgzf_refuses_a_small_buffer(ctx):
    from frender_b200 import _lib
    data = np.frombuffer(b"x" * 1000, np.uint8)
    out = np.empty(_lib.lib.frb_gz_deflate_bgzf_bound(1000) - 1, np.uint8)
    n = ctypes.c_uint64()
    rc = _lib.lib.frb_gz_deflate_bgzf(ctx._h, data.ctypes.data, 1000, out.ctypes.data, out.size, ctypes.byref(n))
    assert rc == _lib.ERR_ARG


def test_gz_deflate_bgzf_is_deterministic_and_compresses(ctx):
    data = fastq(8 << 20, True)
    a, b = ctx.gz_deflate(data, bgzf=True), ctx.gz_deflate(data, bgzf=True)
    assert a == b
    assert len(data) / len(a) > 2.4, len(data) / len(a)
    # the gzip member of the same bytes is not changed by the BGZF layout living next to it
    assert zlib.decompress(ctx.gz_deflate(data), 31) == data


# ---- the demux stream in BGZF format -------------------------------------------------------------------------------
def chunk_cells(ctx, t1, t2, table, roles, cuts, mode, pack):
    """Push the texts in the given (cut1, cut2) pieces, two chunks in flight, in mode "plain", "gzip" or "bgzf";
    returns one list of cells per popped chunk: [(R1 bytes, R2 bytes) per sink]."""
    names = sorted({n for n in roles.values() if n})
    sid = {n: i for i, n in enumerate(names)}
    role_of = {"index_hop": "#hop", "ambiguous": "#amb", "undetermined": "#und"}
    keys = list(table)
    routes = np.array([sid[roles[table[k][1]] if table[k][0] == "demuxable" else roles[role_of[table[k][0]]]]
                       for k in keys], np.uint32)
    lo, hi = pack(keys)
    ctx.route_load(lo, routes, len(names), keys_hi=hi)
    ctx.route_gzip(mode != "plain", bgzf=mode == "bgzf")
    ctx.route_reset()
    b1, b2 = t1.encode(), t2.encode()
    chunks, p1, p2, queued = [], 0, 0, 0

    def take():
        o1, o2, off1, off2 = ctx.route_pop()[:4]
        chunks.append([(o1[off1[i]:off1[i + 1]].tobytes(), o2[off2[i]:off2[i + 1]].tobytes()) for i in range(len(names))])

    for n1, n2 in cuts:
        d1, d2 = b1[p1:p1 + n1], b2[p2:p2 + n2]
        p1, p2 = p1 + len(d1), p2 + len(d2)
        final = (1 if p1 >= len(b1) else 0) | (2 if p2 >= len(b2) else 0)
        ctx.route_push(d1, d2, final)
        queued += 1
        if queued == 2:
            take()
            queued -= 1
        if final == 3:
            break
    while queued:
        take()
        queued -= 1
    ctx.route_gzip(False)
    return chunks


def assert_blocks_match(plain, packed):
    assert len(plain) == len(packed)
    for chunk_p, chunk_z in zip(plain, packed):
        for (p1, p2), (z1, z2) in zip(chunk_p, chunk_z):
            for p, z in ((p1, z1), (p2, z2)):
                if not p:
                    assert z == b""
                else:
                    check_blocks(z, p, eof=False)


@pytest.mark.parametrize("case", ["even", "r2_short", "r1_short_partial", "tiny_cuts", "big_cells"])
def test_bgzf_stream_matches_plain_stream(ctx, case):
    import frender_oracle as O
    from frender_b200.engine import pack_keys
    from test_gpu_deflate import cut_list
    from test_gpu_route import make_pair
    rng = random.Random(sum(case.encode()) + 5)
    n = 6000
    if case == "r2_short":
        t1, t2, table = make_pair(rng, n, r2_records=n - 1500)
    elif case == "r1_short_partial":
        t2, t1, table = make_pair(rng, n, r2_records=n - 2500, crop_tail=7)
    else:
        t1, t2, table = make_pair(rng, 30_000 if case == "big_cells" else n)
    roles = O.sink_names(table)
    if case == "big_cells":   # a few chunks of MBs: cells of many blocks
        cuts = [(len(t1) // 3 + 11, len(t2) // 3 + 5)] * 4
    else:
        cuts = cut_list(rng, case == "tiny_cuts", len(t1), len(t2))
    pack = lambda keys: (pack_keys(keys), None)
    plain = chunk_cells(ctx, t1, t2, table, roles, cuts, "plain", pack=pack)
    packed = chunk_cells(ctx, t1, t2, table, roles, cuts, "bgzf", pack=pack)
    assert_blocks_match(plain, packed)
    assert any(z1 for chunk in packed for z1, _ in chunk)
    if case == "big_cells":
        assert max(len(list(bgzf.iter_blocks(z1))) for chunk in packed for z1, _ in chunk) > 3


def test_bgzf_stream_on_a_wide_context():
    import frender_oracle as O
    from frender_b200.engine import Context, pack_keys2
    from test_gpu_deflate import cut_list
    from test_gpu_wide import wide_pair
    rng = random.Random(78)
    t1, t2, table = wide_pair(rng, 5000, crop_tail=3)
    roles = O.sink_names(table)
    cuts = cut_list(rng, False, len(t1), len(t2))
    wctx = Context(0, table_log2=16, wide=True)
    try:
        plain = chunk_cells(wctx, t1, t2, table, roles, cuts, "plain", pack=pack_keys2)
        packed = chunk_cells(wctx, t1, t2, table, roles, cuts, "bgzf", pack=pack_keys2)
    finally:
        wctx.close()
    assert_blocks_match(plain, packed)


def test_bgzf_format_switch_only_between_chunks(ctx):
    """Refused while a chunk is in flight (either direction); kept by route_reset; route_pair stays plain; an
    unknown format is refused; gzip mode after BGZF gives members again."""
    import frender_oracle as O
    from frender_b200 import _lib
    from frender_b200.engine import FrbError, pack_keys
    from test_gpu_route import make_pair
    rng = random.Random(4)
    t1, t2, table = make_pair(rng, 400)
    roles = O.sink_names(table)
    pack = lambda k: (pack_keys(k), None)
    chunks = chunk_cells(ctx, t1, t2, table, roles, [(len(t1), len(t2))], "plain", pack=pack)
    ctx.route_gzip(True, bgzf=True)
    ctx.route_reset()
    ctx.route_push(t1.encode(), t2.encode(), 3)
    for on, as_bgzf in ((False, False), (True, False), (True, True)):
        with pytest.raises(FrbError) as err:
            ctx.route_gzip(on, bgzf=as_bgzf)
        assert err.value.code == _lib.ERR_STATE
    o1, o2, off1, off2 = ctx.route_pop()[:4]
    cells = [(o1[off1[i]:off1[i + 1]].tobytes(), o2[off2[i]:off2[i + 1]].tobytes()) for i in range(len(off1) - 1)]
    assert_blocks_match(chunks, [cells])
    o1, o2, off1, off2, pairs = ctx.route_pair(t1.encode(), t2.encode(), 3)[:5]
    assert pairs == 400 and [(o1[off1[i]:off1[i + 1]], o2[off2[i]:off2[i + 1]]) for i in range(len(off1) - 1)] == chunks[0]
    assert _lib.lib.frb_route_set_gz_format(ctx._h, 3) == _lib.ERR_ARG
    gz_chunks = chunk_cells(ctx, t1, t2, table, roles, [(len(t1), len(t2))], "gzip", pack=pack)
    for (p1, p2), (z1, z2) in zip(chunks[0], gz_chunks[0]):
        assert (zlib.decompress(z1, 31) if z1 else b"") == p1 and (zlib.decompress(z2, 31) if z2 else b"") == p2
    ctx.route_gzip(False)


# ---- frender demux with FRENDER_GZIP_LEVEL=bgzf --------------------------------------------------------------------
def run_cli(argv, cwd):
    from frender_b200.cli import main
    old = os.getcwd()
    os.chdir(cwd)
    try:
        main(argv)
    finally:
        os.chdir(old)


def assert_bgzf_file(raw):
    blocks = list(bgzf.iter_blocks(raw))
    assert raw.endswith(bgzf.EOF_BLOCK) and raw.count(bgzf.EOF_BLOCK) == 1
    assert all(isize for _, _, isize in blocks[:-1])
    return len(blocks) - 1


@pytest.mark.parametrize("chunk_mb", ["64", "0"])
def test_cli_demux_bgzf_golden_c4(golden, tmp_path, chunk_mb, monkeypatch):
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
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", "bgzf")
    if chunk_mb == "0":
        monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "0")
        import frender_b200.cli as cli
        monkeypatch.setattr(cli, "MIN_CHUNK", 50_000, raising=False)
    run_cli(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "out"), str(p1), str(p2)], tmp_path)
    assert sorted(os.listdir(tmp_path / "out")) == sorted(case["sinks"])
    most = 0
    for fname, want in case["sinks"].items():
        raw = (tmp_path / "out" / fname).read_bytes()
        text = gzip.decompress(raw)
        assert len(text) == want["bytes"], fname
        assert hashlib.sha256(text).hexdigest() == want["sha256"], fname
        n_blocks = assert_bgzf_file(raw)
        if not want["bytes"]:
            assert raw == bgzf.EOF_BLOCK
        most = max(most, n_blocks)
    assert most > 1


def test_cli_demux_bgzf_empty_sink(tmp_path, monkeypatch):
    """A sink that receives no record is exactly the 28-byte EOF block."""
    rows = ("idx1,idx2,reads,matched_idx1,matched_idx2,read_type,sample_name,demux_ok\r\n"
            "AAAA,CCCC,1,AAAA,CCCC,demuxable,S1,True\r\nGGGG,TTTT,1,GGGG,TTTT,demuxable,S2,True\r\n")
    (tmp_path / "r.csv").write_text(rows)
    rec = lambda k, n: f"@r:1 {n}:N:0:{k}\nACGT\n+\nFFFF\n".encode()
    (tmp_path / "x_R1_001.fastq.gz").write_bytes(gzip.compress(rec("AAAA+CCCC", 1) * 3))
    (tmp_path / "x_R2_001.fastq.gz").write_bytes(gzip.compress(rec("AAAA+CCCC", 2) * 3))
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", "bgzf")
    run_cli(["demux", "-r", str(tmp_path / "r.csv"), "-d", str(tmp_path / "o"),
             str(tmp_path / "x_R1_001.fastq.gz"), str(tmp_path / "x_R2_001.fastq.gz")], tmp_path)
    full = (tmp_path / "o" / "S1_frender-demux_R2.fq.gz").read_bytes()
    assert gzip.decompress(full) == rec("AAAA+CCCC", 2) * 3 and assert_bgzf_file(full) == 1
    assert (tmp_path / "o" / "S2_frender-demux_R1.fq.gz").read_bytes() == bgzf.EOF_BLOCK


def test_cli_demux_bgzf_pairs_on_two_gpus(golden, tmp_path, monkeypatch):
    """FRENDER_GPUS=2 with three lane pairs in bgzf mode: every sink is byte for byte the one-GPU run's file."""
    from conftest import unb64
    from frender_b200 import synth
    from frender_b200._lib import lib
    n = ctypes.c_int()
    lib.frb_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs")
    case = golden["demux"]["c1"]
    scan = golden["scan"][case["scan_case"]]
    spec = synth.make_spec(scan["config"], n_samples=scan["n_samples"])
    files = []
    for lane, (g0, g1) in enumerate([(0, 1200), (1200, 2100), (2100, 3000)], start=1):
        for mate in (1, 2):
            p = tmp_path / f"Undetermined_S0_L00{lane}_R{mate}_001.fastq.gz"
            p.write_bytes(gzip.compress(synth.generate_big(spec, g0, g1, mate), 1))
            files.append(str(p))
    (tmp_path / "results.csv").write_bytes(unb64(case["results_csv"]))
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", "bgzf")
    run_cli(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "one")] + files, tmp_path)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    run_cli(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "two")] + files, tmp_path)
    names = sorted(os.listdir(tmp_path / "one"))
    assert names == sorted(os.listdir(tmp_path / "two")) == sorted(case["sinks"])
    for name in names:
        one = (tmp_path / "one" / name).read_bytes()
        assert one == (tmp_path / "two" / name).read_bytes(), name
        assert_bgzf_file(one)


# ---- reading BGZF back on the device -------------------------------------------------------------------------------
def spans_of(ctx, path):
    """The whole text through the span reader (random span sizes); asserts it never declined."""
    rng = random.Random(5)
    ctx.gz_open(0, path)
    try:
        out = []
        while True:
            s = ctx.gz_read(0, rng.choice([17, 65536, 999_999, 4 * MIB]), copy=True)
            assert not s.declined, path
            out.append(s.data)
            if s.eof or s.size == 0:
                return b"".join(out)
    finally:
        ctx.gz_close(0)


def tally(ctx, path):
    ctx.reset()
    reads, _, raw = ctx.scan_gz(path, 0)
    return reads, raw, list(ctx.counter()["total"].items())


def test_device_inflate_reads_our_bgzf(ctx, tmp_path):
    from frender_b200 import synth
    text = synth.generate_big(synth.make_spec("C2", seed=1234), 0, 60_000, 1)   # ~ 20 MB
    assert len(text) > 15 * MIB
    z = ctx.gz_deflate(text, bgzf=True)
    check_blocks(z, text)
    (tmp_path / "bgzf").mkdir()
    (tmp_path / "zlib").mkdir()
    p_b = tmp_path / "bgzf" / "Undetermined_S0_L001_R1_001.fastq.gz"
    p_z = tmp_path / "zlib" / "Undetermined_S0_L001_R1_001.fastq.gz"
    p_b.write_bytes(z)
    p_z.write_bytes(gzip.compress(text, 6))
    assert spans_of(ctx, p_b) == text
    assert ctx.gz_inflate(p_b, len(text) + 1) == text            # None would mean the device path declined
    assert tally(ctx, p_b) == tally(ctx, p_z)


def test_golden_scan_case_as_bgzf_gives_the_same_tally(ctx, golden, golden_dir, tmp_path):
    from frender_b200.engine import tally_barcodes
    case = golden["scan"]["c2"]
    files = []
    for f in case["files"]:
        text = gzip.decompress(open(os.path.join(golden_dir, f"c2__{f}"), "rb").read())
        z = ctx.gz_deflate(text, bgzf=True)
        check_blocks(z, text)
        path = tmp_path / f"c2__{f}"
        path.write_bytes(z)
        assert ctx.gz_inflate(path, len(text) + 1) == text
        files.append(str(path))
    counter = tally_barcodes(1, files, case["sample"], ctx=ctx)
    counter = {k.split("__", 1)[-1]: v for k, v in counter.items()}
    assert {k: [list(x) for x in v.items()] for k, v in counter.items()} == case["tally"]
