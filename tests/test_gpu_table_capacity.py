"""Unique-key tables at and past capacity.

Every count passes through the open-addressing table of common.cuh (linear probing, kMaxProbe probes).  The keys here
are aimed at chosen home slots of a 2^10 table, so that probe chains are long, wrap from the last slot to slot 0, or
fill every slot: each insert path must still give the oracle's tally in the oracle's order, raise TABLE_FULL as soon as
one key more than the table holds arrives, and keep reporting that error instead of a partial total until the context
is reset.  The CLI's answer to a full table (larger tables, tally again) must give the oracle's CSV.

Inputs past capacity stay small: a read whose key finds no slot costs kMaxProbe (2^15) probe loads before the error.
"""
import ctypes
import gzip
import os
import re
import shutil
import subprocess
from functools import lru_cache

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "frender_b200", "csrc")

LOG2 = 10
CAP = 1 << LOG2
SHAPES = {"8+8": (8, 8), "10+10": (10, 10), "12+12": (12, 12), "21+20": (21, 20)}
MAX_SYMS = 21
WIDE_MIX = 0x9E3779B97F4A7C15          # a wide key (lo, hi) hashes as hash64(lo ^ hi * WIDE_MIX)
_DEC = np.frombuffer(b"\0ACGTN+", np.uint8)
_SHIFTS = np.arange(MAX_SYMS, dtype=np.uint64) * np.uint64(3)


# ---- host side: where a key lands ------------------------------------------------------------------------------
def hash64(k):
    """murmur3 fmix64, as hash64() in csrc/common.cuh, over a uint64 array."""
    k = np.array(k, dtype=np.uint64, copy=True, ndmin=1)
    with np.errstate(over="ignore"):
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xFF51AFD7ED558CCD)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xC4CEB9FE1A85EC53)
        k ^= k >> np.uint64(33)
    return k


def key_hash(lo, hi):
    """The table's hash of packed keys: hash64(lo) for a narrow key, the wide mix for (lo, hi); hi = 0 gives the
    narrow key's hash."""
    lo, hi = np.asarray(lo, np.uint64), np.asarray(hi, np.uint64)
    with np.errstate(over="ignore"):
        return hash64(lo ^ (hi * np.uint64(WIDE_MIX)))


def home_slots(lo, hi, log2):
    return key_hash(lo, hi) & np.uint64((1 << log2) - 1)


def pack_codes(codes):
    """Symbol codes (rows of 1..6 = ACGTN+) -> (lo, hi) as pack_keys2 packs the strings."""
    codes = codes.astype(np.uint64)
    lo = (codes[:, :MAX_SYMS] << _SHIFTS[:min(codes.shape[1], MAX_SYMS)]).sum(axis=1, dtype=np.uint64)
    hi = np.zeros(len(codes), np.uint64)
    if codes.shape[1] > MAX_SYMS:
        rest = codes[:, MAX_SYMS:]
        hi = (rest << _SHIFTS[:rest.shape[1]]).sum(axis=1, dtype=np.uint64)
    return lo, hi


def window(kind, log2=LOG2):
    """Home slots keys are aimed at: the last 8 slots (chains wrap to slot 0) or one slot (one cluster as long as the
    table)."""
    cap = 1 << log2
    return np.arange(cap - 8, cap, dtype=np.uint64) if kind == "wrap" else np.array([cap // 3], np.uint64)


def aimed_keys(shape, n, slots, log2=LOG2, seed=0):
    """n distinct random index pairs of `shape` (ACGTN symbols) whose home slots in a 2^log2 table are in `slots`,
    by rejection sampling."""
    l1, l2 = SHAPES[shape]
    width = l1 + 1 + l2
    rng = np.random.default_rng(seed)
    got = {}
    while len(got) < n:
        codes = rng.integers(1, 6, size=(1 << 16, width), dtype=np.uint8)
        codes[:, l1] = 6
        lo, hi = pack_codes(codes)
        hit = np.isin(home_slots(lo, hi, log2), slots)
        for s in _DEC[codes[hit]].view(f"S{width}").ravel().tolist():
            got.setdefault(s.decode(), None)
    return list(got)[:n]


@lru_cache(maxsize=None)
def keyset(shape, kind, n, seed=0):
    return tuple(aimed_keys(shape, n, window(kind), seed=seed))


# ---- FASTQ text and the oracle --------------------------------------------------------------------------------------
def fastq(keys, seed=0, short=False, reps=(1, 5)):
    """Reads of every key, 1..4 each, in random order: a key's reads are spread over the file."""
    rng = np.random.default_rng(seed + 17)
    seq = np.repeat(np.arange(len(keys)), rng.integers(*reps, size=len(keys)))
    rng.shuffle(seq)
    if short:   # lines shorter than 24 bytes on average: scan_redo_kernel
        return "".join(f"@r 1:N:0:{keys[i]}\nA\n+\nF\n" for i in seq.tolist()).encode()
    return "".join(f"@r{j} 1:N:0:{keys[i]}\n{'ACGT' * 8}\n+\n{'F' * 32}\n" for j, i in enumerate(seq.tolist())).encode()


def oracle(texts):
    """The reference's barcode_counter for these file texts (names f0, f1, ...), as {name: [(key, reads), ...]}."""
    import frender_oracle as O
    total, out = {}, {}
    for i, t in enumerate(texts):
        counter, _ = O.tally_text(t.decode().splitlines(keepends=True))
        out[f"f{i}"] = list(counter.items())
        for k, v in counter.items():
            total[k] = total.get(k, 0) + v
    return {"total": list(total.items()), **out}


def device(ctx):
    return {name: list(c.items()) for name, c in ctx.counter().items()}


def split_files(keys, n_files, seed=0):
    """Texts of n_files files whose key sets overlap, each about half of `keys`, together all of them."""
    rng = np.random.default_rng(seed + 5)
    owner = rng.integers(0, n_files, size=len(keys))
    extra = rng.integers(0, n_files, size=len(keys))
    return [fastq([k for k, a, b in zip(keys, owner, extra) if f in (a, b)], seed=seed + f) for f in range(n_files)]


def assert_table_full(exc_info):
    import frender_b200._lib as L
    assert exc_info.value.code == L.ERR_TABLE_FULL, exc_info.value
    assert f"unique-key table full (2^{LOG2} slots)" in str(exc_info.value)


LOADS = {"half": CAP // 2, "0.9": int(0.9 * CAP), "0.99": int(0.99 * CAP), "full": CAP}


# ---- A. the host-side hash against the C++ one (no GPU) --------------------------------------------------------------
PIN_KEYS = [0, 1, 0x2A, 0xFFFFFFFFFFFFFFFE, 0x123456789ABCDEF0, 0x0DB6DB6DB6DB6DB6]


def test_hash64_matches_common_cuh(tmp_path):
    """The numpy hash64 gives the C++ hash64 of common.cuh, and the wide mix is the one KeyWidth<true> uses:
    otherwise the keys below would not cluster where they are aimed and the tests would prove nothing."""
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cxx = shutil.which("g++") or shutil.which("nvcc") or (os.path.join(cuda, "bin", "nvcc")
                                                           if os.path.exists(os.path.join(cuda, "bin", "nvcc")) else None)
    if cxx is None or not os.path.exists(os.path.join(cuda, "include", "cuda_runtime.h")):
        pytest.skip("no host compiler / CUDA headers")
    src = tmp_path / "pin.cpp"
    src.write_text('#include <cstdio>\n#include "common.cuh"\nint main() {\n'
                   + "".join(f"    std::printf(\"%llu\\n\", frb::hash64({k}ULL));\n" for k in PIN_KEYS)
                   + "    return 0;\n}\n")
    exe = tmp_path / "pin"
    lang = ["-x", "cu"] if os.path.basename(cxx).startswith("nvcc") else ["-x", "c++"]
    subprocess.run([cxx, "-std=c++17", f"-I{CSRC}", f"-I{os.path.join(cuda, 'include')}", *lang, str(src), "-o",
                    str(exe)], check=True, capture_output=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == hash64(np.array(PIN_KEYS, np.uint64)).tolist()
    text = open(os.path.join(CSRC, "common.cuh")).read()
    mix = re.search(r"hash\(Key k\) \{ return hash64\(k\.lo \^ \(k\.hi \* (0x[0-9A-Fa-f]+)ULL\)\); \}", text)
    assert mix and int(mix.group(1), 16) == WIDE_MIX


def test_aimed_keys_land_in_their_window():
    """The generator's packing is pack_keys / pack_keys2's, and every key it returns has its home slot in the
    window it was aimed at."""
    from frender_b200.engine import pack_keys, pack_keys2
    for shape in SHAPES:
        for kind in ("wrap", "cluster"):
            keys = aimed_keys(shape, 40, window(kind), seed=3)
            assert len(set(keys)) == 40 and all(len(k) == sum(SHAPES[shape]) + 1 for k in keys)
            lo, hi = pack_keys2(keys)
            if sum(SHAPES[shape]) + 1 <= MAX_SYMS:
                assert (pack_keys(keys) == lo).all() and (hi == 0).all()
            assert np.isin(home_slots(lo, hi, LOG2), window(kind)).all()


# ---- B. exact tallies under heavy probing (GPU) ------------------------------------------------------------------
@pytest.fixture(scope="module")
def nctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=LOG2)
    yield c
    c.close()


@pytest.fixture(scope="module")
def wctx():
    from frender_b200.engine import Context
    c = Context(0, table_log2=LOG2, wide=True)
    yield c
    c.close()


def scan(ctx, texts, **kw):
    ctx.reset()
    for i, t in enumerate(texts):
        ctx.scan_bytes(t, ordinal=i, name=f"f{i}", **kw)
    return device(ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("load", list(LOADS))
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
@pytest.mark.parametrize("shape", ["8+8", "10+10"])
@pytest.mark.parametrize("chunk", [None, 6000])
def test_spec_scan_exact(nctx, shape, kind, load, chunk):
    """The speculative whole-file scan (deferred probe steps, then table_add), whole and in many chunks."""
    text = fastq(keyset(shape, kind, LOADS[load]))
    assert scan(nctx, [text], chunk=chunk) == oracle([text])


@pytest.mark.gpu
@pytest.mark.parametrize("load", list(LOADS))
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
@pytest.mark.parametrize("how", ["demux_rule", "sample"])
def test_ws_scan_narrow_exact(nctx, how, kind, load):
    """The general scan kernel on a narrow context (the demux rule and -s both rule out the speculative scan; the
    keys here read the same under both rules)."""
    import frender_b200._lib as L
    text = fastq(keyset("10+10", kind, LOADS[load]))
    kw = {"rule": L.RULE_DEMUX} if how == "demux_rule" else {"sample": text.count(b"\n") // 4}
    assert scan(nctx, [text], **kw) == oracle([text])


@pytest.mark.gpu
@pytest.mark.parametrize("load", list(LOADS))
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
@pytest.mark.parametrize("shape", ["12+12", "21+20", "8+8"])
def test_ws_scan_wide_exact(wctx, shape, kind, load):
    """The general scan kernel on a wide context: 128-bit compare-and-swap claims, wide probe loop."""
    text = fastq(keyset(shape, kind, LOADS[load]))
    assert scan(wctx, [text], chunk=50_000) == oracle([text])


@pytest.mark.gpu
@pytest.mark.parametrize("load", list(LOADS))
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
def test_redo_short_records_exact(nctx, kind, load):
    """Records shorter than 24 bytes: every tile goes to scan_redo_kernel."""
    text = fastq(keyset("8+8", kind, LOADS[load]), short=True)
    for chunk in (None, 7000):
        assert scan(nctx, [text], chunk=chunk) == oracle([text])


def shifted_text(guessed, true, seed=0):
    """A file whose line phase shifts half way: the speculative scan guesses the '@s' lines (keys `guessed`) as
    headers, the count says the '@t' lines (keys `true`), so the guessed keys go in, are taken out again by the
    negate pass (their slots stay, with count 0) and the tiles are redone by count."""
    rng = np.random.default_rng(seed)
    head = fastq(true[: len(true) // 4], seed=seed)
    g = rng.integers(0, len(guessed), size=2 * len(true))
    t = np.concatenate([np.arange(len(true)), rng.integers(0, len(true), size=len(true))])
    rng.shuffle(t)
    body = "".join(f"@s{i} 1:N:0:{guessed[a]}\n{'ACGT' * 8}\n+\n@t{i} 1:N:0:{true[b]}\n"
                   for i, (a, b) in enumerate(zip(g.tolist(), t.tolist())))
    return head + f"@x 1:N:0:{true[0]}\n".encode() + body.encode()


@pytest.mark.gpu
@pytest.mark.parametrize("load", list(LOADS))
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
def test_redo_after_negate_same_keys_exact(nctx, kind, load):
    """A mis-guessed file whose guessed and true keys are the same set: the negate pass and the redo run on a
    table that the set fills up to every slot, and the tally is exact."""
    keys = list(keyset("8+8", kind, LOADS[load]))
    text = shifted_text(keys, keys)
    assert scan(nctx, [text]) == oracle([text])


@pytest.mark.gpu
@pytest.mark.parametrize("n_true,n_guessed", [(CAP // 4, CAP // 2), (CAP // 2, CAP // 2), (CAP // 2, CAP // 2 + 200)])
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
def test_redo_after_negate_other_keys(nctx, kind, n_true, n_guessed):
    """Guessed keys other than the true ones keep their slots (count 0) after the negate pass.  Exact while guessed
    and true keys together fit the table; past that the table may fill up before the redo, and TABLE_FULL is the
    only other acceptable answer."""
    from frender_b200.engine import FrbError
    keys = list(keyset("8+8", kind, CAP + 200))
    true, guessed = keys[:n_true], keys[n_true:n_true + n_guessed]
    text = shifted_text(guessed, true, seed=1)
    want = oracle([text])
    assert len(want["total"]) == n_true <= CAP // 2
    if n_true + n_guessed <= CAP:
        assert scan(nctx, [text]) == want
        return
    try:
        got = scan(nctx, [text])
    except FrbError as exc:
        assert "unique-key table full" in str(exc)
    else:
        assert got == want


@pytest.mark.gpu
@pytest.mark.parametrize("load", ["0.99", "full"])
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_merge_pending_files_exact(nctx, wctx, width, kind, load):
    """Four files, each about half of the keys, together 0.99 of the table or every slot: the per-file lists are
    folded into the total table (merge_pending_files)."""
    ctx, shape = (nctx, "10+10") if width == "narrow" else (wctx, "12+12")
    texts = split_files(list(keyset(shape, kind, LOADS[load])), 4)
    assert scan(ctx, texts) == oracle(texts)


def file_lists(texts):
    """(keys, counts, first) of every text, each tallied on a context of its own."""
    from frender_b200.engine import Context
    w = Context(0, table_log2=LOG2)
    try:
        out = []
        for t in texts:
            w.reset()
            w.scan_bytes(t)
            out.append(w.file_arrays(0))
        return out
    finally:
        w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("load", ["0.99", "full"])
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
def test_total_merge_exact(nctx, kind, load):
    """Lists of other contexts folded into one total (frb_total_merge, the `-c` fold)."""
    from frender_b200.engine import unpack_keys
    texts = split_files(list(keyset("10+10", kind, LOADS[load])), 4)
    nctx.reset()
    for i, (k, c, f) in enumerate(file_lists(texts)):
        nctx.merge_list(k, c, f + (np.uint64(i) << np.uint64(40)))
    keys, counts, _ = nctx.total_arrays()
    assert list(zip(unpack_keys(keys), counts.tolist())) == oracle(texts)["total"]


def write_gz(tmp_path, texts, tag=""):
    paths = []
    for i, t in enumerate(texts):
        p = tmp_path / f"f{i}{tag}_R1_001.fastq.gz"
        p.write_bytes(gzip.compress(t, 1))
        paths.append(p)
    return paths


@pytest.mark.gpu
@pytest.mark.parametrize("load", ["0.99", "full"])
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_gz_batch_exact(nctx, wctx, tmp_path, width, kind, load):
    """A run of small .gz files through the device as one stream (frb_scan_gz_batch), tallied per file and in total."""
    import frender_oracle as O
    ctx, shape = (nctx, "8+8") if width == "narrow" else (wctx, "21+20")
    paths = write_gz(tmp_path, split_files(list(keyset(shape, kind, LOADS[load])), 5))
    ctx.reset()
    assert ctx.scan_gz_batch(paths, 0) is not None, "the library declined the run"
    want = O.tally_barcodes(1, paths)
    assert device(ctx) == {k: list(v.items()) for k, v in want.items()}


# ---- C. TABLE_FULL, and the context after it (GPU) ---------------------------------------------------------------
OVER = [1, 300]


@pytest.mark.gpu
@pytest.mark.parametrize("extra", OVER)
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
@pytest.mark.parametrize("path", ["spec", "spec_chunks", "ws_demux", "ws_sample", "wide", "redo"])
def test_one_file_past_capacity_raises(nctx, wctx, path, kind, extra):
    """cap + 1 and cap + 300 unique keys in one file: TABLE_FULL from the scan, never a tally."""
    import frender_b200._lib as L
    from frender_b200.engine import FrbError
    shape = {"wide": "12+12"}.get(path, "8+8")
    text = fastq(keyset(shape, kind, CAP + extra), short=path == "redo", reps=(1, 3))
    kw = {"spec_chunks": {"chunk": 6000}, "ws_demux": {"rule": L.RULE_DEMUX},
          "ws_sample": {"sample": text.count(b"\n") // 4}}.get(path, {})
    ctx = wctx if path == "wide" else nctx
    with pytest.raises(FrbError) as e:
        scan(ctx, [text], **kw)
    assert_table_full(e)
    fits = fastq(keyset(shape, kind, LOADS["0.9"]))          # the context goes on as before
    assert scan(ctx, [fits]) == oracle([fits])


@pytest.mark.gpu
@pytest.mark.parametrize("extra", OVER)
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
def test_gz_batch_past_capacity(nctx, tmp_path, kind, extra):
    """A batch whose files fit but whose union does not: the files are tallied, the total raises.  A batch with one
    file that does not fit is declined as a whole, and that file raises on its own."""
    from frender_b200.engine import FrbError
    keys = list(keyset("8+8", kind, CAP + extra))
    paths = write_gz(tmp_path, [fastq(keys[i::3], seed=i, reps=(1, 3)) for i in range(3)], "u")
    nctx.reset()
    assert nctx.scan_gz_batch(paths, 0) is not None
    with pytest.raises(FrbError) as e:
        nctx.total_arrays()
    assert_table_full(e)
    big = write_gz(tmp_path, [fastq(keys[:40], seed=3), fastq(keys, seed=4, reps=(1, 3))], "b")
    nctx.reset()
    assert nctx.scan_gz_batch(big, 0) is None
    assert nctx.counter() == {"total": {}}
    with pytest.raises(FrbError) as e:
        nctx.scan_gz(big[1], 1)
    assert_table_full(e)


def overflow_union(shape, kind, extra):
    """Three files that each fit, whose union is cap + extra unique keys."""
    keys = list(keyset(shape, kind, CAP + extra))
    return [fastq(keys[i::3], seed=i, reps=(1, 3)) for i in range(3)]


@pytest.mark.gpu
@pytest.mark.parametrize("extra", OVER)
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_total_error_stays_until_reset(width, kind, extra):
    """Files that fit, a union that does not: building the total raises TABLE_FULL -- and keeps raising it (the
    total table holds part of the union) until reset() or resize_tables().  Then the same context tallies a fitting
    input, and after resize_tables(12) the input that overflowed, exactly."""
    from frender_b200.engine import Context, FrbError
    shape = "10+10" if width == "narrow" else "21+20"
    texts = overflow_union(shape, kind, extra)
    ctx = Context(0, table_log2=LOG2, wide=width == "wide")
    try:
        ctx.reset()
        for i, t in enumerate(texts):
            ctx.scan_bytes(t, ordinal=i, name=f"f{i}")          # every file fits
        for call in (ctx.total_arrays, ctx.total_arrays, ctx.counter, ctx.total_arrays):
            with pytest.raises(FrbError) as e:
                call()
            assert_table_full(e)
        fits = split_files(list(keyset(shape, kind, LOADS["0.9"])), 3)
        assert scan(ctx, fits) == oracle(fits)
        ctx.resize_tables(LOG2 + 2)
        assert scan(ctx, texts) == oracle(texts)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("extra", OVER)
@pytest.mark.parametrize("kind", ["wrap", "cluster"])
def test_total_merge_error_stays_until_reset(kind, extra):
    """Lists folded in with merge_list (the `-c` path) whose union does not fit: TABLE_FULL, and again on every later
    merge_list / total_arrays / counter until reset() or resize_tables()."""
    from frender_b200.engine import Context, FrbError, unpack_keys
    texts = overflow_union("10+10", kind, extra)
    lists = file_lists(texts)
    ctx = Context(0, table_log2=LOG2)

    def fold():
        ctx.reset()
        for i, (k, c, f) in enumerate(lists):
            ctx.merge_list(k, c, f + (np.uint64(i) << np.uint64(40)))
        keys, counts, _ = ctx.total_arrays()
        return list(zip(unpack_keys(keys), counts.tolist()))
    try:
        with pytest.raises(FrbError) as e:
            fold()
        assert_table_full(e)
        for call in (ctx.total_arrays, ctx.counter, ctx.total_arrays, lambda: ctx.merge_list(*lists[0])):
            with pytest.raises(FrbError) as e:
                call()
            assert_table_full(e)
        ctx.reset()
        ctx.merge_list(*lists[0])
        assert list(zip(unpack_keys(ctx.total_arrays()[0]), ctx.total_arrays()[1].tolist())) == \
            list(zip(unpack_keys(lists[0][0]), lists[0][1].tolist()))
        ctx.resize_tables(LOG2 + 2)
        assert fold() == oracle(texts)["total"]
    finally:
        ctx.close()


# ---- D. the CLI's regrow loop (GPU) ------------------------------------------------------------------------------
def run_cli(argv, cwd):
    from frender_b200.cli import main
    old = os.getcwd()
    os.chdir(cwd)
    try:
        main(argv)
    finally:
        os.chdir(old)


def rc(s):
    return s.translate(str.maketrans("ACGTN", "TGCAN"))[::-1]


def lane(shape, n_random, n_files=1, seed=0, sheet_rows=16):
    """(sheet CSV text, file texts): sheet pairs read forward for half of the samples and with idx2 reverse-
    complemented for the other half (30 reads each, in every file), plus n_random random pairs with 1-2 reads,
    spread over the files without repeats."""
    from frender_b200.synth import _index_set
    l1, l2 = SHAPES[shape]
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    i7 = [acgt[r].tobytes().decode() for r in _index_set(rng, sheet_rows, l1)]
    i5 = [acgt[r].tobytes().decode() for r in _index_set(rng, sheet_rows, l2)]
    sheet = "Sample_ID,index,index2\n" + "".join(f"S{r},{a},{b}\n" for r, (a, b) in enumerate(zip(i7, i5)))
    hot = [f"{a}+{b if r % 2 else rc(b)}" for r, (a, b) in enumerate(zip(i7, i5))]
    rand = aimed_keys(shape, n_random, np.arange(1 << LOG2, dtype=np.uint64), seed=seed + 1)
    texts = []
    for f in range(n_files):
        keys = rand[f::n_files]
        reads = hot * 30 + [k for k, n in zip(keys, rng.integers(1, 3, size=len(keys))) for _ in range(n)]
        order = rng.permutation(len(reads))
        texts.append("".join(f"@r{j} 1:N:0:{reads[i]}\n{'ACGT' * 8}\n+\n{'F' * 32}\n"
                             for j, i in enumerate(order.tolist())).encode())
    return sheet, texts


def write_lane(d, sheet, texts):
    d.mkdir()
    (d / "SampleSheet.csv").write_text(sheet)
    paths = []
    for i, t in enumerate(texts):
        p = d / f"Undetermined_S0_L00{i + 1}_R1_001.fastq.gz"
        p.write_bytes(gzip.compress(t, 1))
        paths.append(str(p))
    return paths


def scan_outputs(d):
    out = {}
    for f in os.listdir(d):
        if f.startswith("frender-scan-results_"):
            out["scan"] = (d / f).read_bytes()
        elif f.startswith("frender-index-2-calls_"):
            out["calls"] = (d / f).read_bytes()
    return out


def oracle_outputs(paths, sheet_path):
    import frender_oracle as O
    indexes = O.read_sheet(sheet_path)
    counter = O.tally_barcodes(1, paths)
    results, calls, _ = O.scan_analysis(1, counter, indexes, 1, True)
    results, _ = O.demux_ok(counter, results)
    return {"scan": O.scan_csv_bytes(results), "calls": O.rc_calls_csv_bytes(calls, indexes)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["one_file", "union", "streams", "wide"])
def test_cli_regrows_full_tables(tmp_path, monkeypatch, capsys, case):
    """frender scan from 2^10-slot tables over a lane of about 5,000 unique index pairs: the tables are full twice
    (the tally goes again with 2^12, then 2^14 slots) and the CSVs are byte for byte those of a run with the default
    tables and the oracle's.  union: six files that each fit and together do not (a run of small files, the total
    overflows); streams: the same through `-c 2` (contexts per file, folded with merge_list); wide: 12+12 pairs."""
    shape, n_files = {"one_file": ("8+8", 1), "union": ("10+10", 6), "streams": ("10+10", 6),
                      "wide": ("12+12", 1)}[case]
    sheet, texts = lane(shape, 5000, n_files)
    argv = ["scan", "-n", "1", "-rc"]
    if case == "streams":
        argv += ["-c", "2"]
        monkeypatch.setenv("FRB_GZ_DEVICE", "0")       # the -c policy: two zlib streams on contexts of their own
    outs = {}
    for run in ("default", "small"):
        d = tmp_path / run
        paths = write_lane(d, sheet, texts)
        if run == "small":
            monkeypatch.setenv("FRENDER_TABLE_LOG2", str(LOG2))
        capsys.readouterr()
        run_cli(argv + ["-b", str(d / "SampleSheet.csv")] + paths, d)
        printed = capsys.readouterr().out
        outs[run] = scan_outputs(d)
    assert "tallying again with 2^12" in printed and "tallying again with 2^14" in printed
    want = oracle_outputs(paths, d / "SampleSheet.csv")
    assert outs["small"] == outs["default"] == want


@pytest.mark.gpu
def test_cli_goes_wide_then_grows(tmp_path, monkeypatch, capsys):
    """12+12 pairs under a 10+10 sheet from 2^10-slot tables: both retries in one run (128-bit keys, then larger
    tables twice), and then the matcher's length assertion (F:227), as the reference asserts."""
    sheet, texts = lane("12+12", 5000)
    sheet = "Sample_ID,index,index2\n" + "".join(
        f"{s},{a[:10]},{b[:10]}\n" for s, a, b in (row.split(",") for row in sheet.splitlines()[1:]))
    d = tmp_path / "lane"
    paths = write_lane(d, sheet, texts)
    monkeypatch.setenv("FRENDER_TABLE_LOG2", str(LOG2))
    with pytest.raises(AssertionError):
        run_cli(["scan", "-n", "1", "-b", str(d / "SampleSheet.csv")] + paths, d)
    out = capsys.readouterr().out
    assert "tallying again with 128-bit keys" in out
    assert out.index("128-bit keys") < out.index("tallying again with 2^12") < out.index("tallying again with 2^14")


@pytest.mark.gpu
def test_cli_two_gpus_one_rank_overflows(tmp_path, monkeypatch, capsys):
    """FRENDER_GPUS=2 from 2^10-slot tables: rank 0's files together overflow, rank 1's fit.  The overflow is
    reported before any rank enters a collective, the tally goes again with 2^12 slots, and the CSVs are the
    oracle's."""
    from frender_b200._lib import lib
    n = ctypes.c_int()
    lib.frb_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs")
    sheet, texts = lane("8+8", 0, 4)
    keys = aimed_keys("8+8", 1500, np.arange(CAP, dtype=np.uint64), seed=9)
    extra = {0: keys[:700], 2: keys[700:1400], 1: keys[1400:1450], 3: keys[1450:]}   # file i goes to rank i % 2
    texts = [t + fastq(extra[i], seed=i) for i, t in enumerate(texts)]
    d = tmp_path / "lane"
    paths = write_lane(d, sheet, texts)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    monkeypatch.setenv("FRENDER_TABLE_LOG2", str(LOG2))
    run_cli(["scan", "-n", "1", "-rc", "-b", str(d / "SampleSheet.csv")] + paths, d)
    out = capsys.readouterr().out
    assert "tallying again with 2^12" in out and "2^14" not in out
    assert scan_outputs(d) == oracle_outputs(paths, d / "SampleSheet.csv")
