"""Wide (128-bit) keys on the GPU: narrow inputs give the golden outputs, index fields longer than 10+10 give the
oracle's outputs."""
import dataclasses
import gzip
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def wctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=18, wide=True)
    yield c
    c.close()


@pytest.mark.parametrize("name", ["c1", "c2", "c2n0", "c3", "multi", "sampled", "c2_384"])
def test_wide_context_golden_scan(wctx, golden, golden_dir, name):
    """A wide context on narrow inputs: tally with order, both passes, rc calls, oriented sheet."""
    from frender_b200.engine import tally_barcodes
    case = golden["scan"][name]
    files = [os.path.join(golden_dir, f"{name}__{f}") for f in case["files"]]
    counter = tally_barcodes(1, files, case["sample"], ctx=wctx)
    assert wctx.wide
    counter = {k.split("__", 1)[-1]: v for k, v in counter.items()}
    assert {k: [list(x) for x in v.items()] for k, v in counter.items()} == case["tally"]
    assert list(counter) == list(case["tally"])
    first, _ = wctx.process(None, case["indexes"], case["n"], case["rc"])
    assert [[k, v] for k, v in first.items()] == case["first_pass"]
    results, calls, oriented = wctx.analyze(case["indexes"], case["n"], case["rc"])
    if case["rc"]:
        assert [[k, v] for k, v in calls.items()] == case["rc_calls"]
        assert oriented == case["oriented_idx2"]
    want = [[k, {f: v for f, v in rec.items() if f != "demux_ok"}] for k, rec in case["final"]]
    assert [[k, v] for k, v in results.items()] == want


def run_cli(argv, cwd):
    from frender_b200.cli import main
    old = os.getcwd()
    os.chdir(cwd)
    try:
        main(argv)
    finally:
        os.chdir(old)


def test_wide_cli_csv_equals_narrow(golden, golden_dir, tmp_path, monkeypatch):
    """frender scan with 128-bit keys writes the same bytes as with 64-bit keys (c2_384)."""
    import frender_b200.cli as cli
    from frender_b200.engine import Context
    case = golden["scan"]["c2_384"]
    (fname, _), = case["files"].items()
    (tmp_path / fname).write_bytes(open(os.path.join(golden_dir, f"c2_384__{fname}"), "rb").read())
    (tmp_path / "SampleSheet.csv").write_text(case["sheet_csv"])
    argv = ["scan", "-n", str(case["n"]), "-b", str(tmp_path / "SampleSheet.csv")] + (["-rc"] if case["rc"] else [])
    out = tmp_path / f"frender-scan-results_{case['n']}-mismatches_{fname}.csv"
    run_cli(argv + [str(tmp_path / fname)], tmp_path)
    narrow = out.read_bytes()
    out.unlink()
    ctx = Context(0, table_log2=16, wide=True)
    old = os.getcwd()
    os.chdir(tmp_path)
    try:
        cli.frender_scan(cli.build_parser().parse_args(argv + [str(tmp_path / fname)]), ctx=ctx)
    finally:
        os.chdir(old)
        ctx.close()
    assert out.read_bytes() == narrow


def test_wide_header_kats_padded(wctx, golden):
    """Header KATs of both rules with the key padded to 22..42 symbols."""
    import frender_b200._lib as L
    from frender_b200.engine import FrbError
    for case in golden["headers"]:
        line = case["line"].rstrip("\n")
        for rule, want in ((L.RULE_SCAN, case["scan"]), (L.RULE_DEMUX, case["demux"])):
            if not want or not line.endswith(want):
                continue
            for pad in (22 - len(want), 30 - len(want), 42 - len(want)):
                if pad <= 0:
                    continue
                key = want + "ACGTN" * 9
                key = key[:len(want) + pad]
                rec = (line[:len(line) - len(want)] + key + "\nACGT\n+\nFFFF\n").encode()
                wctx.reset()
                if all(ch in "ACGTN+" for ch in key):
                    assert wctx.scan_bytes(rec * 3, rule=rule) == (3, 1)
                    assert wctx.counter()["total"] == {key: 3}, (case, rule, pad)
                else:
                    with pytest.raises(FrbError):
                        wctx.scan_bytes(rec * 3, rule=rule)


def spec_12x12(n_rows=384):
    from frender_b200.synth import _index_set, make_spec
    base = make_spec("C2", seed=99)
    rng = np.random.default_rng(1212)
    return dataclasses.replace(base, l1=12, l2=12, sheet_i7=_index_set(rng, n_rows, 12),
                               sheet_i5=_index_set(rng, n_rows, 12))


@pytest.fixture(scope="module")
def lane_12x12(tmp_path_factory):
    from frender_b200.synth import generate_big
    spec = spec_12x12()
    d = tmp_path_factory.mktemp("lane12")
    text = generate_big(spec, 0, 200_000)
    path = d / "Undetermined_S0_L001_R1_001.fastq.gz"
    path.write_bytes(gzip.compress(text, compresslevel=1))
    (d / "SampleSheet.csv").write_text(spec.sheet_csv())
    return spec, path, text


def test_12x12_lane_cli_vs_oracle(lane_12x12, tmp_path):
    from oracle import frender_oracle as O
    spec, path, _ = lane_12x12
    dst = tmp_path / path.name
    dst.write_bytes(path.read_bytes())
    run_cli(["scan", "-n", "1", "-rc", "-b", str(path.parent / "SampleSheet.csv"), str(dst)], tmp_path)
    counter = O.tally_barcodes(1, [str(dst)])
    results, calls, _ = O.scan_analysis(1, counter, spec.indexes(), 1, True)
    results, _ = O.demux_ok(counter, results)
    out = tmp_path / f"frender-scan-results_1-mismatches_{path.name}.csv"
    assert out.read_bytes() == O.scan_csv_bytes(results)
    calls_csv = [f for f in os.listdir(tmp_path) if "index-2-calls" in f]
    assert len(calls_csv) == 1
    assert (tmp_path / calls_csv[0]).read_bytes() == O.rc_calls_csv_bytes(calls, spec.indexes())


def test_12x12_lane_chunks(wctx, lane_12x12):
    """Several chunk sizes through scan_bytes give the same totals, equal to the oracle's tally."""
    from oracle import frender_oracle as O
    _, _, text = lane_12x12
    want, _ = O.tally_text(text.decode().splitlines())
    for chunk in (None, 1 << 20, 123_457):
        wctx.reset()
        wctx.scan_bytes(text, chunk=chunk)
        got = wctx.counter()["total"]
        assert list(got.items()) == list(want.items()), chunk


def test_mixed_lengths_and_switch(wctx, tmp_path):
    """10+10, 12+12, 20+20, 21+20 and a 42-symbol key without '+' in one file, in first-appearance order; a narrow
    context switches itself to wide keys."""
    from oracle import frender_oracle as O
    from frender_b200.engine import Context, tally_barcodes
    rng = random.Random(5)
    seq = lambda n: "".join(rng.choice("ACGTN") for _ in range(n))
    pool = [seq(10) + "+" + seq(10), seq(12) + "+" + seq(12), seq(20) + "+" + seq(20), seq(21) + "+" + seq(20),
            seq(42), seq(8) + "+" + seq(8)]
    lines = []
    for i in range(5000):
        key = rng.choice(pool) if i % 3 else seq(12) + "+" + seq(12)
        lines += [f"@M:1:FC:1:1:{i}:{i} 1:N:0:{key}", "ACGT", "+", "FFFF"]
    path = tmp_path / "mixed_R1.fastq.gz"
    path.write_bytes(gzip.compress(("\n".join(lines) + "\n").encode()))
    want = O.tally_barcodes(1, [str(path)])
    got = tally_barcodes(1, [path], ctx=wctx)
    assert list(got["total"].items()) == list(want["total"].items())
    narrow = Context(0, table_log2=16)
    try:
        got = tally_barcodes(1, [path], ctx=narrow)
        assert narrow.wide
        assert list(got["total"].items()) == list(want["total"].items())
    finally:
        narrow.close()


@pytest.mark.parametrize("length", [11, 12, 16, 20])
def test_wide_matcher_random_sheets_vs_oracle(wctx, length):
    """Random sheets with duplicated rows and N, n = 0..4, rc mode, against the oracle's process()."""
    from oracle import frender_oracle as O
    rng = random.Random(length)
    seq = lambda n, alpha="ACGT": "".join(rng.choice(alpha) for _ in range(n))
    rows = 40
    idx1 = [seq(length) for _ in range(rows)]
    idx2 = [seq(length) for _ in range(rows)]
    idx1[5], idx2[5] = idx1[3], idx2[3]                       # duplicated row
    idx1[7] = idx1[7][:-1] + "N"
    ids = [f"S{r % 30}" for r in range(rows)]
    indexes = {"id": ids, "idx1": idx1, "idx2": idx2}
    counter = {}
    for _ in range(3000):
        r = rng.randrange(rows)
        a, b = list(idx1[r]), list(rng.choice([idx2[r], O.reverse_complement(idx2[r])]))
        for _ in range(rng.randrange(4)):
            (a if rng.random() < 0.5 else b)[rng.randrange(length)] = rng.choice("ACGTN")
        if rng.random() < 0.2:
            a, b = list(seq(length, "ACGTN")), list(seq(length, "ACGTN"))
        key = "".join(a) + "+" + "".join(b)
        counter[key] = counter.get(key, 0) + rng.randrange(1, 9)
    for n in range(5):
        for rc in (False, True):
            got, _ = wctx.process(counter, indexes, n, rc)
            want = O.process(1, counter, indexes, n, rc)
            assert got == want, (length, n, rc)


def wide_pair(rng, n, r2_records=None, crop_tail=0):
    """R1/R2 texts whose keys are 12+12, 21+20, 10+10 and 42 symbols long, and a results table over them."""
    seq = lambda k: "".join(rng.choice("ACGTN") for _ in range(k))
    keys = [seq(12) + "+" + seq(12) for _ in range(30)] + [seq(21) + "+" + seq(20) for _ in range(5)]
    keys += [seq(10) + "+" + seq(10) for _ in range(5)] + [seq(42)]
    r1, r2 = [], []
    for i in range(n):
        k = rng.choice(keys)
        l1, l2 = rng.randint(1, 300), rng.randint(1, 300)
        name = f"@M0:{i}:FC:1:{rng.randint(1, 99999)}:{rng.randint(1, 99999)}"
        r1.append(f"{name} 1:N:0:{k}\n{'A' * l1}\n+\n{'F' * l1}\n")
        r2.append(f"{name} 2:N:0:{k}\n{'C' * l2}\n+\n{'#' * l2}\n")
    if r2_records is not None:
        r2 = r2[:r2_records]
    t1, t2 = "".join(r1), "".join(r2)
    if crop_tail:
        t2 = t2[:-crop_tail]
    kinds = ["demuxable", "index_hop", "ambiguous", "undetermined"]
    table = {k: (kinds[j % 4], f"S{j % 7}" if j % 4 == 0 else "") for j, k in enumerate(keys)}
    return t1, t2, table


def wide_stream(ctx, t1, t2, table, roles, cut1, cut2):
    """The demux stream of a wide context, two chunks in flight; returns {sink: (R1, R2)}."""
    from frender_b200.engine import pack_keys2
    names = sorted({n for n in roles.values() if n})
    sid = {n: i for i, n in enumerate(names)}
    role_of = {"index_hop": "#hop", "ambiguous": "#amb", "undetermined": "#und"}
    keys = list(table)
    routes = np.array([sid[roles[table[k][1]] if table[k][0] == "demuxable" else roles[role_of[table[k][0]]]]
                       for k in keys], np.uint32)
    lo, hi = pack_keys2(keys)
    ctx.route_load(lo, routes, len(names), keys_hi=hi)
    ctx.route_reset()
    out = {n: (bytearray(), bytearray()) for n in names}
    b1, b2 = t1.encode(), t2.encode()
    p1 = p2 = queued = 0

    def take():
        o1, o2, off1, off2 = ctx.route_pop()[:4]
        for n, i in sid.items():
            out[n][0].extend(o1[off1[i]:off1[i + 1]].tobytes())
            out[n][1].extend(o2[off2[i]:off2[i + 1]].tobytes())

    while True:
        d1, d2 = b1[p1:p1 + cut1()], b2[p2:p2 + cut2()]
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
    return {n: (bytes(a), bytes(b)) for n, (a, b) in out.items()}


@pytest.mark.parametrize("case", ["even", "r2_short", "r2_partial_tail", "tiny_cuts"])
def test_wide_demux_stream_vs_oracle(wctx, case):
    """Random cuts, a short mate, a trailing partial record: the same sinks as the oracle's route_pairs."""
    from oracle import frender_oracle as O
    rng = random.Random(sum(case.encode()) + 42)
    n = 5000
    t1, t2, table = wide_pair(rng, n, r2_records=n - 1200 if case == "r2_short" else None,
                              crop_tail=3 if case == "r2_partial_tail" else 0)
    roles = O.sink_names(table)
    want = O.route_pairs(t1.splitlines(keepends=True), t2.splitlines(keepends=True), table, roles)
    if case == "tiny_cuts":
        cut1, cut2 = (lambda: rng.randint(1, 3000)), (lambda: rng.randint(1, 3000))
    else:
        cut1, cut2 = (lambda: rng.randint(100_000, 400_000)), (lambda: rng.randint(50_000, 500_000))
    got = wide_stream(wctx, t1, t2, table, roles, cut1, cut2)
    for name, (w1, w2) in want.items():
        assert got[name] == (w1, w2), f"{case}: sink {name}"


def test_wide_demux_unknown_key(wctx):
    from oracle import frender_oracle as O
    import frender_b200._lib as L
    from frender_b200.engine import FrbError
    rng = random.Random(9)
    t1, t2, table = wide_pair(rng, 500)
    lost = next(k for k in (line.rsplit(":", 1)[1] for line in t2.splitlines()[::4]) if len(k) == 25)
    del table[lost]
    with pytest.raises(FrbError) as err:
        wide_stream(wctx, t1, t2, table, O.sink_names(table), lambda: 1 << 20, lambda: 1 << 20)
    assert err.value.code == L.ERR_KEY_NOT_FOUND and f"Couldn't find barcode {lost} " in err.value.message
    wctx.route_reset()


def test_12x12_lane_scan_then_demux_cli_vs_oracle(tmp_path):
    """frender scan, then frender demux on the scan's own CSV: the decompressed sinks equal the oracle's."""
    import csv
    from oracle import frender_oracle as O
    from frender_b200.synth import generate_big
    spec = spec_12x12()
    p1 = tmp_path / "Undetermined_S0_L001_R1_001.fastq.gz"
    p2 = tmp_path / "Undetermined_S0_L001_R2_001.fastq.gz"
    p1.write_bytes(gzip.compress(generate_big(spec, 0, 30_000, 1), 1))
    p2.write_bytes(gzip.compress(generate_big(spec, 0, 30_000, 2), 1))
    (tmp_path / "SampleSheet.csv").write_text(spec.sheet_csv())
    run_cli(["scan", "-n", "1", "-rc", "-b", str(tmp_path / "SampleSheet.csv"), str(p1)], tmp_path)
    res = tmp_path / f"frender-scan-results_1-mismatches_{p1.name}.csv"
    with open(res, newline="") as fh:
        table = {r["idx1"] + "+" + r["idx2"]: (r["read_type"], r["sample_name"]) for r in csv.DictReader(fh)}
    assert any(len(k) == 25 for k in table)
    run_cli(["demux", "-r", str(res), "-d", str(tmp_path / "out"), str(p1), str(p2)], tmp_path)
    roles = O.sink_names(table)
    want = O.demux_files(str(p1), str(p2), table, roles)
    got = sorted(os.listdir(tmp_path / "out"))
    assert got == sorted(f"{n}_frender-demux_{r}.fq.gz" for n in want for r in ("R1", "R2"))
    for name, (w1, w2) in want.items():
        assert gzip.open(tmp_path / "out" / f"{name}_frender-demux_R1.fq.gz", "rb").read() == w1, name
        assert gzip.open(tmp_path / "out" / f"{name}_frender-demux_R2.fq.gz", "rb").read() == w2, name


def test_cli_scan_switches_to_wide_and_asserts_on_a_short_sheet(lane_12x12, tmp_path, capsys):
    """A 10+10 sheet over a 12+12 lane: the narrow tally hits KEY_TOO_LONG, the CLI tallies again with 128-bit keys,
    and the matcher ends in the reference's AssertionError (F:227)."""
    spec, path, _ = lane_12x12
    dst = tmp_path / path.name
    dst.write_bytes(path.read_bytes())
    short = dataclasses.replace(spec, l1=10, l2=10, sheet_i7=spec.sheet_i7[:, :10], sheet_i5=spec.sheet_i5[:, :10])
    (tmp_path / "SampleSheet.csv").write_text(short.sheet_csv())
    with pytest.raises(AssertionError):
        run_cli(["scan", "-n", "1", "-b", str(tmp_path / "SampleSheet.csv"), str(dst)], tmp_path)
    assert "tallying again with 128-bit keys" in capsys.readouterr().out


def test_cli_wide_scan_takes_one_gpu(lane_12x12, tmp_path, monkeypatch, capsys):
    """FRENDER_GPUS=2 and -c 4 over two 12+12 files: the wide run takes the one-GPU, one-stream branch."""
    import frender_b200.cli as cli
    spec, path, _ = lane_12x12
    files = []
    for lane in (1, 2):
        dst = tmp_path / f"Undetermined_S0_L00{lane}_R1_001.fastq.gz"
        dst.write_bytes(path.read_bytes())
        files.append(str(dst))

    def no_multi_gpu(*a, **k):
        raise AssertionError("a wide run must not start GPU workers")
    monkeypatch.setattr(cli, "scan_files_multi_gpu", no_multi_gpu)
    monkeypatch.setattr(cli, "scan_files_concurrent", no_multi_gpu)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    run_cli(["scan", "-n", "1", "-c", "4", "-b", str(path.parent / "SampleSheet.csv")] + files, tmp_path)
    assert "one GPU, one inflate stream" in capsys.readouterr().out


def test_cli_narrow_multi_gpu_worker_too_long_goes_wide(lane_12x12, tmp_path, monkeypatch, capsys):
    """A multi-GPU worker that reports KEY_TOO_LONG (as text) sends the CLI to 128-bit keys on one GPU."""
    import frender_b200.cli as cli
    spec, path, _ = lane_12x12
    short = dataclasses.replace(spec, l1=10, l2=10, sheet_i7=spec.sheet_i7[:, :10], sheet_i5=spec.sheet_i5[:, :10])
    (tmp_path / "SampleSheet.csv").write_text(short.sheet_csv())
    files = []
    for lane in (1, 2):
        dst = tmp_path / f"Undetermined_S0_L00{lane}_R1_001.fastq.gz"
        dst.write_bytes(path.read_bytes())
        files.append(str(dst))

    def worker_fails(*a, **k):
        raise SystemExit("GPU worker 0 failed: FrbError('frender_b200 error -5: read 0: index field longer than 21 "
                         "symbols')")
    monkeypatch.setattr(cli, "scan_files_multi_gpu", worker_fails)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    with pytest.raises(AssertionError):      # the 10+10 sheet against 12+12 keys, F:227
        run_cli(["scan", "-n", "1", "-b", str(tmp_path / "SampleSheet.csv")] + files, tmp_path)
    out = capsys.readouterr().out
    assert "tallying again with 128-bit keys" in out and "one GPU, one inflate stream" in out


def test_set_key_width_drops_the_sheet():
    """A sheet packed for one width is not matched on the other: frb_match asks for a new one."""
    import frender_b200._lib as L
    from frender_b200.engine import Context, FrbError
    c = Context(0, table_log2=12)
    try:
        c.load_sheet({"id": ["S1"], "idx1": ["ACGTACGTAC"], "idx2": ["TTTTTGGGGG"]})
        c._ck(L.lib.frb_set_key_width(c._h, 128))
        keys = np.zeros(1, np.uint64)
        counts = np.ones(1, np.uint64)
        c._ck(L.lib.frb_total_load(c._h, keys.ctypes.data_as(L.vp), counts.ctypes.data_as(L.vp), 1))
        with pytest.raises(FrbError) as e:
            c._ck(L.lib.frb_match(c._h, 1, 0, None, None, None, None, None, None, None, None, None, None))
        assert e.value.code == L.ERR_STATE
    finally:
        c.close()
