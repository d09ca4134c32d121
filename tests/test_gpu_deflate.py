"""The device gzip writer: frb_gz_deflate round-trips through zlib (which checks CRC-32 and ISIZE), the demux stream
in gzip mode returns members that decompress to plain mode's cells, and `frender demux` with FRENDER_GZIP_LEVEL=gpu
writes sinks that decompress to the reference's bytes."""
import ctypes
import gzip
import hashlib
import os
import random
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KIB = 1024


@pytest.fixture(scope="module")
def ctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=16)
    yield c
    c.close()


def bound(n):
    from frender_b200._lib import lib
    return lib.frb_gz_deflate_bound(n)


def far_repeats(back):
    """Random bytes whose only repeat is a 64-byte block exactly `back` bytes behind its first copy."""
    rng = np.random.default_rng(back)
    block = rng.integers(0, 256, 64, np.uint8).tobytes()
    return block + rng.integers(0, 256, back - 64, np.uint8).tobytes() + block + rng.integers(0, 256, 999, np.uint8).tobytes()


def fastq(n_bytes, binned):
    from frender_b200 import synth
    spec = synth.make_spec("C2")
    data = synth.generate_big(spec, 0, n_bytes // 300 + 1)[:n_bytes]
    return synth.binned_qualities(data, 7) if binned else data


def text_like(n, seed):
    """Bytes with repeats at every distance class: words drawn from a small vocabulary."""
    rng = random.Random(seed)
    words = [bytes(rng.choice(b"ACGTNacgtn:+@ \n") for _ in range(rng.randint(1, 12))) for _ in range(300)]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words)
    return bytes(out[:n])


CASES = {
    "empty": lambda: b"",
    "1": lambda: b"A",
    "2": lambda: b"AC",
    "3": lambda: b"ACG",
    "run257": lambda: b"F" * 257,
    "run258": lambda: b"F" * 258,
    "run259": lambda: b"F" * 259,
    "run1M": lambda: b"\x00" * (1 << 20),
    "random1MiB": lambda: np.random.default_rng(1).integers(0, 256, 1 << 20, np.uint8).tobytes(),
    "all256": lambda: bytes(range(256)),
    "64K-1": lambda: text_like(64 * KIB - 1, 1),
    "64K": lambda: text_like(64 * KIB, 2),
    "64K+1": lambda: text_like(64 * KIB + 1, 3),
    "3x64K+17": lambda: text_like(3 * 64 * KIB + 17, 4),
    "back32768": lambda: far_repeats(32768),
    "back32769": lambda: far_repeats(32769),
    "fastq8MB_allF": lambda: fastq(8 << 20, False),
    "fastq8MB_binned": lambda: fastq(8 << 20, True),
}


@pytest.mark.parametrize("name", list(CASES))
def test_gz_deflate_round_trips(ctx, name):
    data = CASES[name]()
    z = ctx.gz_deflate(data)
    assert z[:10] == bytes.fromhex("1f8b0800000000000003")
    assert len(z) <= bound(len(data))
    assert zlib.decompress(z, 31) == data
    if not data:
        assert len(z) == 20


def test_gz_deflate_is_deterministic_and_compresses(ctx):
    data = fastq(8 << 20, True)
    a, b = ctx.gz_deflate(data), ctx.gz_deflate(data)
    assert a == b
    assert len(data) / len(a) >= 2.5, len(data) / len(a)


def test_gz_deflate_refuses_a_small_buffer(ctx):
    from frender_b200 import _lib
    data = np.frombuffer(b"x" * 1000, np.uint8)
    out = np.empty(bound(1000) - 1, np.uint8)
    n = ctypes.c_uint64()
    rc = _lib.lib.frb_gz_deflate(ctx._h, data.ctypes.data, 1000, out.ctypes.data, out.size, ctypes.byref(n))
    assert rc == _lib.ERR_ARG


# ---- the demux stream in gzip mode ---------------------------------------------------------------------------------
def chunk_cells(ctx, t1, t2, table, roles, cuts, gzip_mode, pack):
    """Push the texts in the given (cut1, cut2) pieces, two chunks in flight; returns one list of cells per popped
    chunk: [(R1 bytes, R2 bytes) per sink]."""
    names = sorted({n for n in roles.values() if n})
    sid = {n: i for i, n in enumerate(names)}
    role_of = {"index_hop": "#hop", "ambiguous": "#amb", "undetermined": "#und"}
    keys = list(table)
    routes = np.array([sid[roles[table[k][1]] if table[k][0] == "demuxable" else roles[role_of[table[k][0]]]]
                       for k in keys], np.uint32)
    lo, hi = pack(keys)
    ctx.route_load(lo, routes, len(names), keys_hi=hi)
    ctx.route_gzip(gzip_mode)
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


def cut_list(rng, tiny, n1, n2):
    lo1, hi1, lo2, hi2 = (1, 3000, 1, 3000) if tiny else (100_000, 400_000, 50_000, 500_000)
    cuts, a, b = [], 0, 0
    while a < n1 or b < n2:
        c = (rng.randint(lo1, hi1), rng.randint(lo2, hi2))
        cuts.append(c)
        a, b = a + c[0], b + c[1]
    return cuts


def assert_members_match(plain, packed):
    assert len(plain) == len(packed)
    for chunk_p, chunk_z in zip(plain, packed):
        for (p1, p2), (z1, z2) in zip(chunk_p, chunk_z):
            for p, z in ((p1, z1), (p2, z2)):
                if not p:
                    assert z == b""
                else:
                    assert zlib.decompress(z, 31) == p


@pytest.mark.parametrize("case", ["even", "r2_short", "r1_short_partial", "r2_partial_tail", "tiny_cuts"])
def test_gzip_stream_matches_plain_stream(ctx, case):
    """The cases of test_stream_matches_the_oracle: every popped member decompresses to the plain-mode cell."""
    import frender_oracle as O
    from frender_b200.engine import pack_keys
    from test_gpu_route import make_pair
    rng = random.Random(sum(case.encode()))
    n = 6000
    if case == "r2_short":
        t1, t2, table = make_pair(rng, n, r2_records=n - 1500)
    elif case == "r1_short_partial":
        t2, t1, table = make_pair(rng, n, r2_records=n - 2500, crop_tail=7)
    elif case == "r2_partial_tail":
        t1, t2, table = make_pair(rng, n, crop_tail=3)
    else:
        t1, t2, table = make_pair(rng, n)
    roles = O.sink_names(table)
    cuts = cut_list(rng, case == "tiny_cuts", len(t1), len(t2))
    pack = lambda keys: (pack_keys(keys), None)
    plain = chunk_cells(ctx, t1, t2, table, roles, cuts, False, pack=pack)
    packed = chunk_cells(ctx, t1, t2, table, roles, cuts, True, pack=pack)
    assert_members_match(plain, packed)
    assert any(z1 for chunk in packed for z1, _ in chunk)


def test_gzip_stream_on_a_wide_context():
    """12+12, 21+20, 10+10 and 42-symbol keys: the encoder runs behind the wide router unchanged."""
    import frender_oracle as O
    from frender_b200.engine import Context, pack_keys2
    from test_gpu_wide import wide_pair
    rng = random.Random(77)
    t1, t2, table = wide_pair(rng, 5000, crop_tail=3)
    roles = O.sink_names(table)
    cuts = cut_list(rng, False, len(t1), len(t2))
    wctx = Context(0, table_log2=16, wide=True)
    try:
        plain = chunk_cells(wctx, t1, t2, table, roles, cuts, False, pack=pack_keys2)
        packed = chunk_cells(wctx, t1, t2, table, roles, cuts, True, pack=pack_keys2)
    finally:
        wctx.close()
    assert_members_match(plain, packed)


def test_gzip_mode_switch_only_between_chunks(ctx):
    """Refused while a chunk is in flight; kept by route_reset; route_pair stays plain."""
    import frender_oracle as O
    from frender_b200 import _lib
    from frender_b200.engine import FrbError, pack_keys
    from test_gpu_route import make_pair
    rng = random.Random(3)
    t1, t2, table = make_pair(rng, 400)
    roles = O.sink_names(table)
    chunks = chunk_cells(ctx, t1, t2, table, roles, [(len(t1), len(t2))], False, pack=lambda k: (pack_keys(k), None))
    ctx.route_gzip(True)
    ctx.route_reset()
    ctx.route_push(t1.encode(), t2.encode(), 3)
    with pytest.raises(FrbError) as err:
        ctx.route_gzip(False)
    assert err.value.code == _lib.ERR_STATE
    o1, o2, off1, off2 = ctx.route_pop()[:4]
    cells = [(o1[off1[i]:off1[i + 1]].tobytes(), o2[off2[i]:off2[i + 1]].tobytes()) for i in range(len(off1) - 1)]
    assert_members_match(chunks, [cells])
    o1, o2, off1, off2, pairs = ctx.route_pair(t1.encode(), t2.encode(), 3)[:5]
    assert pairs == 400 and [(o1[off1[i]:off1[i + 1]], o2[off2[i]:off2[i + 1]]) for i in range(len(off1) - 1)] == chunks[0]
    ctx.route_gzip(False)


# ---- frender demux with FRENDER_GZIP_LEVEL=gpu ---------------------------------------------------------------------
def run_cli(argv, cwd):
    from frender_b200.cli import main
    old = os.getcwd()
    os.chdir(cwd)
    try:
        main(argv)
    finally:
        os.chdir(old)


@pytest.mark.parametrize("chunk_mb", ["64", "0"])
def test_cli_demux_gpu_gzip_golden_c4(golden, tmp_path, chunk_mb, monkeypatch):
    """The golden C4 case: same file names, every sink decompresses to the reference's bytes; with a tiny chunk the
    files hold many members."""
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
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", "gpu")
    if chunk_mb == "0":
        monkeypatch.setenv("FRENDER_DEMUX_CHUNK_MB", "0")
        import frender_b200.cli as cli
        monkeypatch.setattr(cli, "MIN_CHUNK", 50_000, raising=False)
    run_cli(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "out"), str(p1), str(p2)], tmp_path)
    assert sorted(os.listdir(tmp_path / "out")) == sorted(case["sinks"])
    members = 0
    for fname, want in case["sinks"].items():
        path = tmp_path / "out" / fname
        raw = gzip.open(path, "rb").read()
        assert len(raw) == want["bytes"], fname
        assert hashlib.sha256(raw).hexdigest() == want["sha256"], fname
        members = max(members, path.read_bytes().count(bytes.fromhex("1f8b0800000000000003")))
    assert members > (1 if chunk_mb == "0" else 0)


def test_cli_demux_gpu_gzip_empty_sink(tmp_path, monkeypatch):
    """A sink that receives no record is the 20-byte empty member, a valid gzip file."""
    rows = ("idx1,idx2,reads,matched_idx1,matched_idx2,read_type,sample_name,demux_ok\r\n"
            "AAAA,CCCC,1,AAAA,CCCC,demuxable,S1,True\r\nGGGG,TTTT,1,GGGG,TTTT,demuxable,S2,True\r\n")
    (tmp_path / "r.csv").write_text(rows)
    rec = lambda k, n: f"@r:1 {n}:N:0:{k}\nACGT\n+\nFFFF\n".encode()
    (tmp_path / "x_R1_001.fastq.gz").write_bytes(gzip.compress(rec("AAAA+CCCC", 1) * 3))
    (tmp_path / "x_R2_001.fastq.gz").write_bytes(gzip.compress(rec("AAAA+CCCC", 2) * 3))
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", "gpu")
    run_cli(["demux", "-r", str(tmp_path / "r.csv"), "-d", str(tmp_path / "o"),
             str(tmp_path / "x_R1_001.fastq.gz"), str(tmp_path / "x_R2_001.fastq.gz")], tmp_path)
    assert gzip.open(tmp_path / "o" / "S1_frender-demux_R2.fq.gz", "rb").read() == rec("AAAA+CCCC", 2) * 3
    empty = (tmp_path / "o" / "S2_frender-demux_R1.fq.gz").read_bytes()
    assert len(empty) == 20 and gzip.decompress(empty) == b""


def test_cli_demux_gpu_gzip_pairs_on_two_gpus(golden, tmp_path, monkeypatch):
    """FRENDER_GPUS=2 with three lane pairs in gpu mode: every sink decompresses to the one-GPU run's bytes."""
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
    monkeypatch.setenv("FRENDER_GZIP_LEVEL", "gpu")
    run_cli(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "one")] + files, tmp_path)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    run_cli(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "two")] + files, tmp_path)
    names = sorted(os.listdir(tmp_path / "one"))
    assert names == sorted(os.listdir(tmp_path / "two")) == sorted(case["sinks"])
    for name in names:
        assert gzip.open(tmp_path / "one" / name, "rb").read() == gzip.open(tmp_path / "two" / name, "rb").read(), name
