"""Narrow (64-bit) against wide (128-bit) keys on one GPU.

1. The same device-generated C2 lane (10+10, frb_synth_*) scanned and matched by a narrow and a wide context,
   alternating, step after step: per-phase time (frb_prof_read: scan, export, match) and whether the exported
   totals and the matcher outputs agree.
2. A host-generated 12+12 lane as .fastq.gz, tallied and analysed end to end on a wide context (reads/s).

Writes one JSON object (stdout and --out) with the card's name and power limit."""
import argparse
import ctypes as C
import dataclasses
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import frender_b200._lib as L  # noqa: E402
from frender_b200._lib import lib  # noqa: E402
from frender_b200.engine import Context  # noqa: E402
from frender_b200.synth import _index_set, generate_big, make_spec  # noqa: E402

GEN_CHUNK = 1 << 24


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = out[0].split(", ")
        return name, power
    except Exception as exc:  # noqa: BLE001
        return f"unknown ({exc})", "unknown"


def step(ctx, dbuf, bounds, spec):
    ck = ctx._ck
    for k in (L.K_SCAN, L.K_EXPORT, L.K_MATCH):
        ctx.prof_read(k)
    t0 = time.perf_counter()
    ck(lib.frb_scan_begin(ctx._h, 0, 0))
    ck(lib.frb_scan_chunk_dev(ctx._h, dbuf, bounds[-1], 0, L.RULE_SCAN, None, None))  # the lane as one chunk
    reads, uniq = C.c_uint64(), C.c_uint64()
    ck(lib.frb_scan_end(ctx._h, C.byref(reads), C.byref(uniq)))
    keys, counts, first = ctx.total_arrays()
    first_pass = ctx.match(1, True)
    calls = ctx.rc_calls(first_pass)
    use = np.array([calls[n]["call"] for n in ctx.sheet.ids], np.uint8)
    second = ctx.match(1, False, use)
    ctx._ck(lib.frb_sync(ctx._h))
    wall = time.perf_counter() - t0
    phases = {name: ctx.prof_read(k)[0] for name, k in (("scan", L.K_SCAN), ("export", L.K_EXPORT), ("match", L.K_MATCH))}
    hi = ctx.total_keys_hi()
    return wall, phases, (keys, hi, counts, first, first_pass, second), reads.value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=100_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--reads12", type=int, default=4_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = card()
    spec = make_spec("C2")
    narrow, wide = Context(0, table_log2=25), Context(0, table_log2=25, wide=True)
    for c in (narrow, wide):
        c.prof(True)
        c.load_sheet(spec.indexes())
    h = narrow._h
    emit_i7 = np.array([sum(int(c) << (2 * p) for p, c in enumerate(row)) for row in spec.sheet_i7], np.uint32)
    emit_i5 = np.array([sum(int(c) << (2 * p) for p, c in enumerate(row)) for row in spec.emit_i5()], np.uint32)
    cdf = np.ascontiguousarray(spec.cdf, np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    narrow._ck(lib.frb_synth_load(h, spec.seed, spec.l1, spec.l2, spec.n_samples, vp(emit_i7), vp(emit_i5), vp(cdf),
                                  spec.lane, spec.read_len, spec.sub_t, spec.n_t, spec.rand_t, spec.hop_t))
    cap = args.reads * (2 * spec.read_len + 80)
    dbuf = C.c_void_p()
    narrow._ck(lib.frb_dev_alloc(h, cap, C.byref(dbuf)))
    bounds, off = [0], 0
    for g in range(0, args.reads, GEN_CHUNK):
        n = C.c_uint64()
        narrow._ck(lib.frb_synth_generate(h, g, min(g + GEN_CHUNK, args.reads), 1, C.c_void_p(dbuf.value + off), cap - off,
                                          C.byref(n)))
        off += n.value
        bounds.append(off)
    res = {"narrow": [], "wide": []}
    equal = True
    for s in range(args.steps + 1):                      # step 0 warms up both
        out = {}
        for tag, c in (("narrow", narrow), ("wide", wide)) if s % 2 == 0 else (("wide", wide), ("narrow", narrow)):
            wall, phases, arrays, reads = step(c, dbuf, bounds, spec)
            out[tag] = arrays
            if s:
                res[tag].append({"wall_s": wall, "ms": phases, "reads": reads})
        a, b = out["narrow"], out["wide"]
        same = all(np.array_equal(x, y) for x, y in zip(a[:4], b[:4])) and not a[1].any()
        for pa, pb in zip(a[4:], b[4:]):
            same &= all(np.array_equal(pa[k], pb[k]) for k in pa)
        equal &= bool(same)
    lib.frb_dev_free(h, dbuf)
    narrow.close()

    # ---- 12+12 lane end to end -------------------------------------------------------------------------------
    base = make_spec("C2", seed=99)
    rng = np.random.default_rng(1212)
    s12 = dataclasses.replace(base, l1=12, l2=12, sheet_i7=_index_set(rng, 384, 12), sheet_i5=_index_set(rng, 384, 12))
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "Undetermined_S0_L001_R1_001.fastq.gz")
        with open(path, "wb") as fh:
            fh.write(gzip.compress(generate_big(s12, 0, args.reads12), compresslevel=1))
        wide.reset()
        wide.scan_gz(path, 0)                            # warm-up
        times = []
        for _ in range(2):
            t0 = time.perf_counter()
            wide.reset()
            wide.scan_gz(path, 0)
            wide.analyze(s12.indexes(), 1, True)
            times.append(time.perf_counter() - t0)
        gz_bytes = os.path.getsize(path)
    wide.close()
    med = lambda xs: float(np.median(xs))
    report = {
        "card": name, "power_limit": power,
        "c2_lane": {"reads": args.reads, "text_bytes": int(bounds[-1]), "steps": args.steps, "outputs_equal": equal,
                    **{tag: {"wall_s_median": med([r["wall_s"] for r in rs]),
                             **{f"{k}_ms_median": med([r["ms"][k] for r in rs]) for k in ("scan", "export", "match")},
                             "scan_GBps": bounds[-1] / 1e6 / med([r["ms"]["scan"] for r in rs]),
                             "per_step": rs} for tag, rs in res.items()}},
        "lane_12x12_e2e": {"reads": args.reads12, "gz_bytes": gz_bytes, "wall_s": times,
                           "reads_per_s": args.reads12 / min(times)},
    }
    txt = json.dumps(report, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
