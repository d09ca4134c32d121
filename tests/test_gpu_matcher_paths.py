"""Every matcher kernel against the C oracle, at the shapes where the choice between them changes.

frb_match takes one of three pairs of kernels (candidate tables, sweep, wide; matcher_cases.py names the pair each case
must take, test_matcher_paths_host.py checks those names against the host's selection rule).  Each case goes through
Context.load_sheet / load_total / match and is compared array by array with the C oracle: the rc pass (m1, m2, type,
srow, m2rc, type_rc, srow_rc and the per-sample sums behind the orientation call), then the oriented pass that reuses
its idx1 verdicts, as `frender scan -rc` runs them, and that pass once more without reuse."""
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import matcher_cases as MC

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
ROW_COLS = ("m1", "m2", "type", "srow", "m2rc", "type_rc", "srow_rc")


@pytest.fixture(scope="module")
def ctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=19)
    yield c
    c.close()


@pytest.fixture(scope="module")
def wctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=19, wide=True)
    yield c
    c.close()


@pytest.fixture(scope="module")
def grid_threads():
    """Threads of the largest grid a matcher kernel takes on this device (sm_count x 8 blocks of 256)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return sms * MC.GRID_BLOCKS_PER_SM * MC.GRID_THREADS_PER_BLOCK


def total_names(ctx):
    keys, counts, _ = ctx.total_arrays()
    return ctx.key_strings(keys, ctx.total_keys_hi() if ctx.wide else None), counts


def expect_sums(sheet, ref, counts):
    """Per sample name (PackedSheet.group_names order): reads whose forward / rc verdict is demuxable to it."""
    f = np.zeros(max(len(sheet.ids), 1), np.uint64)
    r = np.zeros_like(f)
    gid = {name: g for g, name in enumerate(sheet.group_names)}
    for rec, c in zip(ref.tolist(), counts.tolist()):
        if rec[3] >= 0:
            f[gid[sheet.ids[rec[3]]]] += c
        if rec[6] >= 0:
            r[gid[sheet.ids[rec[6]]]] += c
    return f, r


def assert_rows(got, ref, cols, label):
    for j, name in enumerate(cols):
        g = got[name].astype(np.int64)
        bad = np.flatnonzero(g != ref[:, j])
        assert bad.size == 0, (label, name, bad[:5].tolist(), g[bad[:5]].tolist(), ref[bad[:5], j].tolist())


def oracle_rc(names, idx, n):
    import c_oracle
    return np.array(c_oracle.classify_all_rc(names, idx, n), np.int64).reshape(-1, 7)


def oracle_fwd(names, idx, n):
    import c_oracle
    return np.array(c_oracle.classify_all(names, idx, n), np.int64).reshape(-1, 4)


def both_passes(ctx, idx, counter, n, label, fresh=True):
    """rc pass, orientation call from the device's sums, oriented pass reusing the rc pass (and, with `fresh`, the
    same oriented pass after a sheet reload, which runs kernel 1 again): all against the C oracle.  Returns the
    device's outputs of both passes."""
    from frender_b200.engine import reverse_complement
    sheet = ctx.load_sheet(idx)
    ctx.load_total(counter)
    names, counts = total_names(ctx)
    assert names == list(counter)
    res = ctx.match(n, True)
    ref = oracle_rc(names, idx, n)
    assert_rows(res, ref, ROW_COLS, (label, "rc pass"))
    f, r = expect_sums(sheet, ref, counts)
    assert (res["f_sum"] == f).all() and (res["rc_sum"] == r).all(), (label, "sums")
    calls = ctx.rc_calls(res)
    use = np.array([calls[name]["call"] for name in sheet.ids], np.uint8)
    oriented = dict(idx, idx2=[reverse_complement(s) if u else s for s, u in zip(idx["idx2"], use)])
    res2 = ctx.match(n, False, use)
    ref2 = oracle_fwd(names, oriented, n)
    assert_rows(res2, ref2, ROW_COLS[:4], (label, "oriented pass, reused"))
    if fresh:
        ctx.load_sheet(idx)
        res3 = ctx.match(n, False, use)
        for k in ROW_COLS[:4]:
            assert (res3[k] == res2[k]).all(), (label, "oriented pass without reuse", k)
    return res, res2


# ---- shapes: equal, unequal and long index lengths, every n ------------------------------------------------------
@pytest.mark.parametrize("shape", list(MC.SHAPES))
def test_shapes_vs_oracle(ctx, shape):
    l1, l2, _ = MC.SHAPES[shape]
    for n in MC.n_values(l1, l2):
        label = f"shape {shape} n={n}"
        rnd = MC.rng_for(label)
        idx = MC.make_sheet(rnd, l1, l2, MC.SHAPE_ROWS)
        counter = MC.edge_keys(rnd, idx, n, 600)
        res, _ = both_passes(ctx, idx, counter, n, label)
        if n >= max(l1, l2):     # every row matches both indexes (a row's 'x' is one more mismatch, still <= n)
            assert (res["m1"] == 0).all() and (res["m2"] == 0).all() and (res["m2rc"] == 0).all(), label


@pytest.mark.parametrize("l1", MC.SINGLE_L1)
def test_single_index_vs_oracle(ctx, l1):
    """Single-index sheets (l2 = 0, the sweep): the Python oracle's match_single_index, row by row."""
    import frender_oracle as O
    for n in (0, 1, 2, l1):
        label = f"single {l1} n={n}"
        rnd = MC.rng_for(label)
        idx = MC.make_sheet(rnd, l1, 0, MC.SHAPE_ROWS)
        counter = MC.edge_keys(rnd, idx, n, 300)
        ctx.load_sheet(idx)
        ctx.load_total(counter, single=True)
        names, _ = total_names(ctx)
        assert names == list(counter)
        res = ctx.match(n, False)
        for i, key in enumerate(names):
            rows = O.approx_match_rows(key, idx["idx1"], n)
            want = O.match_single_index(key, idx["idx1"], idx["id"], n)
            m1, t, s = int(res["m1"][i]), int(res["type"][i]), int(res["srow"][i])
            assert m1 == (rows[0] if rows else -1), (label, key)
            assert t == (0 if not rows else 2 if len(rows) == 1 else 3), (label, key)
            assert (idx["id"][s] if s >= 0 else "") == want["sample_name"] and (s == rows[0] if s >= 0 else True)


# ---- rows at every boundary between 2048 slots, 4096 slots and the sweep; 1 and 5000 rows ------------------------
@pytest.mark.parametrize("n,rows,path,slots", MC.BOUNDARY, ids=[f"n{b[0]}-rows{b[1]}" for b in MC.BOUNDARY])
def test_boundary_rows_vs_oracle(ctx, n, rows, path, slots):
    label = f"boundary n={n} rows={rows}"
    rnd = MC.rng_for(label)
    idx = MC.make_sheet(rnd, 10, 10, rows)
    counter = MC.edge_keys(rnd, idx, n, 1000 if rows < 2000 else 400)
    both_passes(ctx, idx, counter, n, label, fresh=rows < 5000)


def test_sheet_refusals_keep_the_loaded_sheet(ctx, wctx):
    """5001 rows and every unsupported length are refused with FRB_ERR_ARG before anything is freed: the sheet
    loaded before still matches as the oracle says."""
    import frender_b200._lib as L
    from frender_b200.engine import C, FrbError
    rnd = MC.rng_for("refusals")
    idx = MC.make_sheet(rnd, 8, 8, 32)
    counter = MC.edge_keys(rnd, idx, 1, 200)
    both_passes(ctx, idx, counter, 1, "before refusals", fresh=False)
    big = MC.make_sheet(rnd, 8, 8, MC.MAX_ROWS + 1, odd=False)
    with pytest.raises(FrbError) as e:
        ctx.load_sheet(big)
    assert e.value.code == L.ERR_ARG and "5000-row" in str(e.value)
    z = np.zeros(64, np.uint64)
    g = np.zeros(64, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for l1, l2 in ((12, 9), (0, 8), (22, 0), (10, 11), (22, 1)):       # narrow: l1 + 1 + l2 > 21, l1 = 0, l1 > 21
        assert L.lib.frb_sheet_load(ctx._h, p(z), p(z), p(g), 4, l1, l2) == L.ERR_ARG, (l1, l2)
    for l1, l2 in ((21, 21), (0, 8), (22, 0), (22, 19)):                # wide: 21+21 (43 symbols), l1 = 0, l1 > 21
        assert L.lib.frb_sheet_load2(wctx._h, p(z), p(z), p(z), p(z), p(g), 4, l1, l2) == L.ERR_ARG, (l1, l2)
    res, names = ctx.match(1, True), total_names(ctx)[0]
    assert_rows(res, oracle_rc(names, idx, 1), ROW_COLS, "after refusals")


# ---- scale: more keys than twice each kernel's grid ---------------------------------------------------------------
@pytest.mark.parametrize("which", list(MC.SCALE))
def test_scale_past_two_grids(ctx, wctx, grid_threads, which):
    """More unique keys than twice the largest matcher grid on this device, more than one grid of them with an idx1
    row: kernel 1's grid-stride loop, the work list and kernel 2's loop over it all go round more than once."""
    l1, l2, n, wide, _ = MC.SCALE[which]
    c = wctx if wide else ctx
    rnd = MC.rng_for(f"scale {which}")
    idx = MC.make_sheet(rnd, l1, l2, MC.SHAPE_ROWS, odd=False)
    counter = MC.scale_keys(zlib.crc32(which.encode()), idx, n, int(2.2 * grid_threads))
    assert len(counter) > 2 * grid_threads
    assert MC.idx1_hits(list(counter), idx["idx1"], n) > grid_threads
    both_passes(c, idx, counter, n, f"scale {which}", fresh=False)


# ---- wide contexts --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", list(MC.WIDE_SHAPES))
def test_wide_shapes_vs_oracle(wctx, shape):
    l1, l2 = MC.WIDE_SHAPES[shape]
    for n in (0, 1, 3):
        label = f"wide {shape} n={n}"
        rnd = MC.rng_for(label)
        idx = MC.make_sheet(rnd, l1, l2, MC.SHAPE_ROWS)
        both_passes(wctx, idx, MC.edge_keys(rnd, idx, n, 600), n, label)


def test_wide_5000_rows_vs_oracle(wctx):
    """5000 rows on a wide context: match_wide_kernel's largest launch (5000 x 44 + 16 = 220,016 B)."""
    label = "wide rows=5000"
    rnd = MC.rng_for(label)
    idx = MC.make_sheet(rnd, 10, 10, MC.MAX_ROWS)
    both_passes(wctx, idx, MC.edge_keys(rnd, idx, 1, 400), 1, label, fresh=False)


# ---- the reuse path and its guards ----------------------------------------------------------------------------------
REUSE_SHAPES = {"cand": (10, 10, False), "sweep": (12, 8, False), "wide": (12, 12, True)}


@pytest.mark.parametrize("which", list(REUSE_SHAPES))
def test_reuse_guards(ctx, wctx, which):
    """An rc pass followed by a non-rc pass over a different n, a new total of the same size or a new sheet must
    not reuse the rc pass's idx1 verdicts: each equals the oracle at the new inputs."""
    l1, l2, wide = REUSE_SHAPES[which]
    c = wctx if wide else ctx
    rnd = MC.rng_for(f"reuse {which}")
    idx = MC.make_sheet(rnd, l1, l2, 40)
    counter = MC.edge_keys(rnd, idx, 1, 400)
    use = np.array([rnd.random() < 0.5 for _ in idx["id"]], np.uint8)
    oriented = lambda sh: dict(sh, idx2=[MC.revcomp(s) if u else s for s, u in zip(sh["idx2"], use)])
    names = list(counter)

    def rc_then(n2, change):
        c.load_sheet(idx)
        c.load_total(counter)
        c.match(1, True)
        sheet, keys = change()
        got = c.match(n2, False, use)
        assert_rows(got, oracle_fwd(keys, oriented(sheet), n2), ROW_COLS[:4], (which, n2, change.__name__))

    def same():
        return idx, names

    def new_total():                  # same size, other keys
        other = MC.edge_keys(MC.rng_for(f"reuse {which} other"), idx, 2, 800)
        other = dict(list(other.items())[:len(counter)])
        assert len(other) == len(counter)
        c.load_total(other)
        return idx, list(other)

    idx_b = MC.make_sheet(MC.rng_for(f"reuse {which} sheet b"), l1, l2, 40)

    def new_sheet():                  # same shape, other rows
        c.load_sheet(idx_b)
        return idx_b, names

    rc_then(1, same)
    for n2 in (0, 2):
        rc_then(n2, same)
    rc_then(1, new_total)
    rc_then(1, new_sheet)


@pytest.mark.parametrize("which", ["cand", "sweep"])
def test_failed_pass_is_not_reused(ctx, which):
    """An rc pass over a total with one key of the wrong length raises; the non-rc pass that follows must raise too
    (it used to take the failed pass's verdicts and return them), and frb_demux_ok refuses until a match succeeds."""
    import frender_b200._lib as L
    from frender_b200.engine import FrbError
    l1, l2 = (10, 10) if which == "cand" else (12, 8)
    rnd = MC.rng_for(f"failure {which}")
    idx = MC.make_sheet(rnd, l1, l2, 40)
    good = MC.edge_keys(rnd, idx, 1, 300)
    bad = dict(good)
    bad["A" * (l1 - 1) + "+" + "C" * l2] = 3                # idx1 one symbol short
    ctx.load_sheet(idx)
    m = np.ones((4 + len(idx["id"]), 1), np.uint8)
    for _ in range(2):
        ctx.load_total(bad)
        with pytest.raises(AssertionError):
            ctx.match(1, True)
        with pytest.raises(AssertionError):
            ctx.match(1, False, np.zeros(len(idx["id"]), np.uint8))
        for _ in range(2):
            keys, counts, _ = ctx.total_arrays()
            with pytest.raises(FrbError) as e:
                ctx.demux_ok(m, [(keys, counts)])
            assert e.value.code == L.ERR_STATE
    ctx.load_total(good)
    both_passes(ctx, idx, good, 1, f"after failure {which}", fresh=False)
    keys, counts, _ = ctx.total_arrays()
    ok, bad_files, err = ctx.demux_ok(m, [(keys, counts)])
    assert ok.all() and not bad_files.any() and err is None


# ---- candidate tables against the sweep on the same inputs ----------------------------------------------------------
def cand_cases():
    out = [(f"shape {s} n={n}", l1, l2, n, MC.SHAPE_ROWS) for s, (l1, l2, cand) in MC.SHAPES.items() for n in sorted(cand)]
    out += [(f"boundary n={n} rows={r}", 10, 10, n, r) for n, r, path, _ in MC.BOUNDARY if path == "cand"]
    return out


def cand_arrays(ctx, cases):
    """Both passes of every case as {"<case> <pass> <array>": array}."""
    out = {}
    for label, l1, l2, n, rows in cases:
        rnd = MC.rng_for("cmp " + label)
        idx = MC.make_sheet(rnd, l1, l2, rows)
        sheet = ctx.load_sheet(idx)
        ctx.load_total(MC.edge_keys(rnd, idx, n, 500))
        res = ctx.match(n, True)
        calls = ctx.rc_calls(res)
        use = np.array([calls[name]["call"] for name in sheet.ids], np.uint8)
        res2 = ctx.match(n, False, use)
        for p, r in (("rc", res), ("oriented", res2)):
            for k, v in r.items():
                out[f"{label}|{p}|{k}"] = v
    return out


CHILD = """
import sys
sys.path[:0] = [{root!r}, {oracle!r}, {tests!r}]
import numpy as np
from frender_b200.engine import Context
import test_gpu_matcher_paths as T
ctx = Context(0, table_log2=16)
np.savez({out!r}, **T.cand_arrays(ctx, T.cand_cases()))
ctx.close()
"""


def test_cand_equals_sweep(ctx, tmp_path):
    """FRB_MATCH=sweep (read once per process) in a child: the candidate-eligible cases through the sweep kernels
    give bit for bit what the candidate kernels give here."""
    assert os.environ.get("FRB_MATCH") != "sweep"
    out = tmp_path / "sweep.npz"
    env = dict(os.environ, FRB_MATCH="sweep")
    code = CHILD.format(root=ROOT, oracle=os.path.join(ROOT, "oracle"), tests=HERE, out=str(out))
    proc = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-3000:]
    got = cand_arrays(ctx, cand_cases())
    with np.load(out) as sweep:
        assert sorted(sweep.files) == sorted(got)
        for k, v in got.items():
            assert np.array_equal(v, sweep[k]), k


# ---- frb_demux_ok at size -------------------------------------------------------------------------------------------
FILES = ["Undetermined_S0_L001_R1_001.fastq.gz", "index-hop_L001_R1_001.fastq.gz", "ambiguous_L001_R1_001.fastq.gz",
         "S1_L001_R1_001.fastq.gz", "S2_L001_R1_001.fastq.gz", "S3_L001_R1_001.fastq.gz", "S5_L001_R1_001.fastq.gz",
         "S8_L001_R1_001.fastq.gz", "S12_L001_R1_001.fastq.gz", "S13_L001_R1_001.fastq.gz", "S21_L001_R1_001.fastq.gz",
         "S30_L002_R1_001.fastq.gz", "S34_L002_R1_001.fastq.gz", "lane2_L002_R1_001.fastq.gz",
         "S7-S9_L002_R1_001.fastq.gz", "Undetermined_S0_L002_R1_001.fastq.gz"]
PREFIX = "pfx_"


def demux_case(c, l1, l2, n_keys, seed):
    """16 files of reads over n_keys unique keys, most in the file their class belongs in, a few anywhere.
    Returns (sheet, per-file {key: reads}, classification rows of every key of the total, in total order)."""
    import re

    import c_oracle
    rnd = MC.rng_for(f"demux {seed}")
    idx = MC.make_sheet(rnd, l1, l2, 40, odd=False)
    idx["id"] = [f"{PREFIX}S{r}" for r in range(40)]            # S1 also fits S12_, S13_; S3 also S30_, S34_
    keys = list(MC.edge_keys(rnd, idx, 1, n_keys // 5))
    keys += MC.random_keys(seed, l1, l2, n_keys - len(keys))
    keys += [k[:-1] + e for k in keys[:200] for e in "TN"]      # keys ending in T / N: bit 62 of the low word is set
    keys = list(dict.fromkeys(keys))
    cls = c_oracle.classify_all(keys, idx, 1)
    home = {0: [0, 15], 1: [1, 0], 3: [2, 15]}
    per_file = [dict() for _ in FILES]
    for k, (_, _, t, s) in zip(keys, cls):
        if t == 2:
            want = [f for f, name in enumerate(FILES) if re.search(f"S{s}", name, re.I)] or [13]
        else:
            want = home[t]
        f = rnd.choice(want) if rnd.random() > 0.001 else rnd.randrange(10)
        per_file[f][k] = rnd.randrange(1, 4)
        if rnd.random() < 0.05:
            per_file[rnd.choice(want)][k] = 1
    c.reset()
    for i, name in enumerate(FILES):
        text = "".join(f"@r{j} 1:N:0:{k}\nACGT\n+\nFFFF\n" for k, cnt in per_file[i].items() for j in range(cnt))
        c.scan_bytes(text.encode(), ordinal=i, name=name)
    names, counts = total_names(c)
    assert sorted(names) == sorted(keys)
    c.load_sheet(idx)
    res = c.match(1, False)
    ref = oracle_fwd(names, idx, 1)
    assert_rows(res, ref, ROW_COLS[:4], "demux case")
    return idx, per_file, names, ref


def oracle_demux(idx, per_file, names, ref):
    import frender_oracle as O
    from frender_b200._lib import READ_TYPES
    counter = {"total": {k: 1 for k in names}, **{name: d for name, d in zip(FILES, per_file)}}
    results = {k: {"read_type": READ_TYPES[t], "sample_name": idx["id"][s] if s >= 0 else ""}
               for k, (_, _, t, s) in zip(names, ref.tolist())}
    results, bad = O.demux_ok(counter, results, PREFIX)
    return [results[k]["demux_ok"] for k in names], bad


@pytest.mark.parametrize("wide", [False, True], ids=["narrow", "wide"])
def test_demux_ok_at_size(ctx, wctx, wide):
    """frb_demux_ok over ~200 k unique keys (12+12 on a wide context) in 16 files, from the context's own lists and
    (narrow) from host lists, against the oracle's demux_ok; then with one sample name that is not a valid pattern."""
    import re

    import frender_b200.cli as cli
    c = wctx if wide else ctx
    l = 12 if wide else 10
    idx, per_file, names, ref = demux_case(c, l, l, 100_000 if wide else 200_000, 7 + wide)
    assert sum(k.endswith(("T", "N")) for k in names) > 1000
    m = cli.class_file_matrix(FILES, idx["id"], PREFIX)
    want_ok, want_bad = oracle_demux(idx, per_file, names, ref)
    assert 0 < len(want_bad) < len(FILES) and not all(want_ok) and any(want_ok)
    runs = [c.demux_ok(m, None)]
    if not wide:
        tables = cli.ScanTables.from_ctx(c, FILES)
        runs.append(c.demux_ok(m, tables.files))
    for ok, bad, err in runs:
        assert err is None and ok.tolist() == want_ok
        assert {FILES[f] for f in np.flatnonzero(bad)} == want_bad
    # a sample name that is not a valid pattern, for a row with demuxable keys in the files
    row = int(ref[np.flatnonzero(ref[:, 2] == 2)[0], 3])
    idx_bad = dict(idx, id=[f"{PREFIX}S[{r}" if r == row else x for r, x in enumerate(idx["id"])])
    m_bad = cli.class_file_matrix(FILES, idx_bad["id"], PREFIX)
    assert (m_bad[4 + row] == 2).all()
    with pytest.raises(re.error):
        oracle_demux(idx_bad, per_file, names, ref)
    assert c.demux_ok(m_bad, None)[2] == row
