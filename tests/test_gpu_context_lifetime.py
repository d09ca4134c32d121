"""Ownership of a context's CUDA resources: a failed allocation leaves the context usable with no stale error, and
contexts that come and go with every kind of buffer, event and stream in use give the same results every time."""
import ctypes as C
import gzip
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KINDS = ["demuxable", "index_hop", "ambiguous", "undetermined"]


def make_lane(rng, n, n_keys=40):
    """n read pairs keyed by 8+8 index pairs, and a results table over the keys."""
    bases = "ACGTN"
    keys = ["".join(rng.choice(bases) for _ in range(8)) + "+" + "".join(rng.choice(bases) for _ in range(8))
            for _ in range(n_keys)]
    r1, r2 = [], []
    for i in range(n):
        k = rng.choice(keys)
        l1, l2 = rng.randint(1, 300), rng.randint(1, 300)
        name = f"@M0:{i}:FC:1:{rng.randint(1, 99999)}:{rng.randint(1, 99999)}"
        r1.append(f"{name} 1:N:0:{k}\n{'A' * l1}\n+\n{'F' * l1}\n")
        r2.append(f"{name} 2:N:0:{k}\n{'C' * l2}\n+\n{'#' * l2}\n")
    table = {k: (KINDS[j % 4], f"S{j % 7}" if j % 4 == 0 else "") for j, k in enumerate(keys)}
    return "".join(r1).encode(), "".join(r2).encode(), table


def load_routes(ctx, table):
    """The results table on the device; returns the sink names in sink-id order."""
    import frender_oracle as O
    from frender_b200.engine import pack_keys
    roles = O.sink_names(table)
    names = sorted({n for n in roles.values() if n})
    sid = {n: i for i, n in enumerate(names)}
    role_of = {"index_hop": "#hop", "ambiguous": "#amb", "undetermined": "#und"}
    routes = np.array([sid[roles[v[1]] if v[0] == "demuxable" else roles[role_of[v[0]]]] for v in table.values()],
                      np.uint32)
    ctx.route_load(pack_keys(list(table)), routes, len(names))
    return names


def want_sinks(r1, r2, table):
    import frender_oracle as O
    return O.route_pairs(r1.decode().splitlines(keepends=True), r2.decode().splitlines(keepends=True), table,
                         O.sink_names(table))


def stream(ctx, names, r1, r2, mode="plain", single=False, cut=100_000):
    """r1 (and r2) through the demux stream in chunks of `cut` bytes, two in flight; returns ({sink: (R1, R2)}, pairs)
    with gzip / BGZF members inflated."""
    ctx.route_gzip(mode != "plain", bgzf=mode == "bgzf")
    ctx.route_mates(1 if single else 2)
    ctx.route_reset()
    out = {n: (bytearray(), bytearray()) for n in names}
    pos, queued, total = 0, 0, 0
    unpack = gzip.decompress if mode != "plain" else bytes

    def take():
        nonlocal total
        o1, o2, off1, off2, pairs, _, _ = ctx.route_pop()
        total += pairs
        for i, n in enumerate(names):
            out[n][0].extend(unpack(o1[off1[i]:off1[i + 1]].tobytes()))
            if not single:
                out[n][1].extend(unpack(o2[off2[i]:off2[i + 1]].tobytes()))

    try:
        while True:
            a, b = r1[pos:pos + cut], r2[pos:pos + cut]
            pos += cut
            done = pos >= max(len(r1), len(r2))
            if single:
                ctx.route_push(a, None, 1 if done else 0)
            else:
                ctx.route_push(a, b, 3 if done else (1 if pos >= len(r1) else 0) | (2 if pos >= len(r2) else 0))
            queued += 1
            if queued == 2:
                take()
                queued -= 1
            if done:
                break
        while queued:
            take()
            queued -= 1
    finally:
        ctx.route_reset()
        ctx.route_gzip(False)
        ctx.route_mates(2)
    return {n: (bytes(a), bytes(b)) for n, (a, b) in out.items()}, total


@pytest.fixture(scope="module")
def lane(tmp_path_factory):
    """A small paired lane, its R1 as .gz files (one whole, and in three parts for a batch), and its sample sheet."""
    from frender_b200 import synth
    d = tmp_path_factory.mktemp("lifetime")
    spec = synth.make_spec("C1", n_samples=24)
    text = synth.generate(spec, 0, 6000)
    path = str(d / "Undetermined_S0_L001_R1_001.fastq.gz")
    with gzip.open(path, "wb", compresslevel=1) as fh:
        fh.write(text)
    parts = []
    for i, (g0, g1) in enumerate([(0, 1000), (1000, 2500), (2500, 4000)]):
        p = str(d / f"part{i}_S0_L001_R1_001.fastq.gz")
        with gzip.open(p, "wb", compresslevel=1) as fh:
            fh.write(synth.generate(spec, g0, g1))
        parts.append(p)
    r1, r2, table = make_lane(random.Random(7), 3000)
    return dict(spec=spec, text=text, path=path, parts=parts, r1=r1, r2=r2, table=table)


def scan_and_match(ctx, lane):
    """Tally of the lane's R1 and both matcher passes, against the oracle."""
    import frender_oracle as O
    ctx.reset()
    reads, uniq, raw = ctx.scan_gz(lane["path"], 0)
    assert reads == 6000 and raw == len(lane["text"])
    want = O.tally_barcodes(1, [lane["path"]])
    got = ctx.counter()
    assert list(got["total"].items()) == list(want["total"].items())
    indexes = lane["spec"].indexes()
    res, calls, oriented = ctx.analyze(indexes, 1, True)
    want_res, want_calls, used = O.scan_analysis(1, want, dict(indexes), 1, True)
    assert res == want_res and calls == want_calls and oriented == used["idx2"]
    return res


def test_failed_reserve_leaves_the_context_usable(lane):
    from frender_b200._lib import ERR_CUDA, FrbError
    from frender_b200.engine import Context
    ctx = Context(0, table_log2=16)
    try:
        names = load_routes(ctx, lane["table"])
        with pytest.raises(FrbError) as e:
            ctx.route_reset(1 << 44)  # no device holds buffers for 16 TiB chunks
        assert e.value.code == ERR_CUDA
        want = want_sinks(lane["r1"], lane["r2"], lane["table"])
        for mode in ("plain", "bgzf"):
            got, pairs = stream(ctx, names, lane["r1"], lane["r2"], mode)
            assert pairs == 3000 and got == want, mode
        scan_and_match(ctx, lane)
    finally:
        ctx.close()


def mem_free(ctx):
    import frender_b200._lib as L
    free, total = C.c_uint64(), C.c_uint64()
    ctx._ck(L.lib.frb_mem_info(ctx._h, C.byref(free), C.byref(total)))
    return free.value


def synth_lane(ctx, spec, n):
    """n reads of the device generator, back on the host."""
    import frender_b200._lib as L
    h, lib = ctx._h, L.lib
    pk = lambda rows: np.array([sum(int(c) << (2 * p) for p, c in enumerate(r)) for r in rows], np.uint32)
    i7, i5, cdf = pk(spec.sheet_i7), pk(spec.emit_i5()), np.ascontiguousarray(spec.cdf, np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    ctx._ck(lib.frb_synth_load(h, spec.seed, spec.l1, spec.l2, spec.n_samples, vp(i7), vp(i5), vp(cdf), spec.lane,
                               spec.read_len, spec.sub_t, spec.n_t, spec.rand_t, spec.hop_t))
    dbuf, nb, cap = C.c_void_p(), C.c_uint64(), n * 400 + 4096
    ctx._ck(lib.frb_dev_alloc(h, cap, C.byref(dbuf)))
    try:
        ctx._ck(lib.frb_synth_generate(h, 0, n, 1, dbuf, cap, C.byref(nb)))
        got = np.empty(nb.value, np.uint8)
        ctx._ck(lib.frb_d2h(h, vp(got), dbuf, nb.value))
    finally:
        ctx._ck(lib.frb_dev_free(h, dbuf))
    return got.tobytes()


def cycle(device, lane):
    """One context from creation to close, through every path that owns device memory, events or streams."""
    from frender_b200.engine import Context
    ctx = Context(device, table_log2=16)
    try:
        out = {}
        ctx.reset()
        out["scan_gz"] = ctx.scan_gz(lane["path"], 0)
        out["batch"] = ctx.scan_gz_batch(lane["parts"], 1)
        ctx.gz_open(0, lane["path"])
        spans = []
        while True:
            s = ctx.gz_read(0, 1 << 16, copy=True)
            spans.append(s.data)
            if s.eof or not len(s):
                break
        ctx.gz_close(0)
        out["spans"] = b"".join(spans)
        names = load_routes(ctx, lane["table"])
        out["gzip_stream"] = stream(ctx, names, lane["r1"], lane["r2"], "gzip")
        out["single_end"] = stream(ctx, names, lane["r1"], b"", "bgzf", single=True)
        out["deflate"] = [gzip.decompress(ctx.gz_deflate(lane["text"], bgzf=b)) for b in (False, True)]
        out["synth"] = synth_lane(ctx, lane["spec"], 2000)
        out["match"] = scan_and_match(ctx, lane)
        ok, bad, err = ctx.demux_ok(np.ones((4 + len(ctx.sheet.ids), 1), np.uint8))
        out["demux_ok"] = (ok.tolist(), bad.tolist(), err)
        return out, mem_free(ctx)
    finally:
        ctx.close()


def test_contexts_come_and_go(lane):
    import frender_b200._lib as L
    n = C.c_int()
    L.lib.frb_device_count(C.byref(n))
    for device in range(n.value):
        first, free_1 = cycle(device, lane)
        assert first["spans"] == lane["text"]
        assert all(d == lane["text"] for d in first["deflate"])
        assert first["gzip_stream"][1] == 3000 and first["single_end"][1] == 3000
        for k in range(2, 21):
            got, free_k = cycle(device, lane)
            assert got == first, f"device {device}, cycle {k}"
        print(f"device {device}: free bytes after cycle 1 {free_1}, after cycle 20 {free_k} "
              f"({(free_1 - free_k) / 2**20:+.1f} MiB)")
