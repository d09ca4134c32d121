"""Single-end demux stream against the paired one: python tools/bench_demux_single_end.py [reads] [chunk_mb] [steps]
[--out=path]

R1/R2 of a C4-shaped lane are device-generated (frb_synth_*, as tools/bench_demux.py does) and pulled to pinned host
memory; the results table comes from a scan of R1 and both matcher passes.  Two streams go through
frb_route_push / frb_route_pop in chunks of chunk_mb, two in flight, alternating step by step:
  * single: R1 alone (frb_route_set_mates(ctx, 1)), every record routed by its own header;
  * paired: R1 + R2, keys from the R2 headers.
Reported per stream: device time (the library's per-class events, parser K_SCAN + router K_ROUTE), records/s host
-> host (pinned buffers in, pinned buffers out), GB/s of input host -> host, and GB/s on the algorithmic bytes
(2 x R1, or 2 x (R1 + R2)) over the device time.  Checked first, in plain and in BGZF format: every single-end sink
holds exactly the bytes of the paired run's R1 sink (synthetic R1 and R2 headers carry the same index field).  The
card's name and power limit are read in the same run."""
import gzip
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def measure(reads=4_000_000, chunk_mb=64, steps=5, device=0):
    from frender_b200 import _lib as L
    from frender_b200 import synth
    from frender_b200.engine import C, Context
    ctx = Context(device, table_log2=22)
    h, lib, ck = ctx._h, L.lib, ctx._ck
    spec = synth.make_spec("C4")
    pk = lambda rows: np.array([sum(int(c) << (2 * p) for p, c in enumerate(r)) for r in rows], np.uint32)  # noqa: E731
    i7, i5, cdf = pk(spec.sheet_i7), pk(spec.emit_i5()), np.ascontiguousarray(spec.cdf, np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    ck(lib.frb_synth_load(h, spec.seed, spec.l1, spec.l2, spec.n_samples, vp(i7), vp(i5), vp(cdf), spec.lane,
                          spec.read_len, spec.sub_t, spec.n_t, spec.rand_t, spec.hop_t))
    cap = reads * 376 + (1 << 20)
    dbuf = C.c_void_p()
    ck(lib.frb_dev_alloc(h, cap, C.byref(dbuf)))
    mates = []
    try:
        for mate in (1, 2):
            nb = C.c_uint64()
            ck(lib.frb_synth_generate(h, 0, reads, mate, dbuf, cap, C.byref(nb)))
            host = C.c_void_p()
            ck(lib.frb_host_alloc(C.byref(host), nb.value))
            ck(lib.frb_d2h(h, host, dbuf, nb.value))
            mates.append((host, nb.value))
        ck(lib.frb_synth_generate(h, 0, reads, 1, dbuf, cap, C.byref(C.c_uint64())))
        ctx.reset()
        ck(lib.frb_scan_begin(h, 0, 0))
        ck(lib.frb_scan_chunk_dev(h, dbuf, mates[0][1], 0, L.RULE_SCAN, None, None))
        r, u = C.c_uint64(), C.c_uint64()
        ck(lib.frb_scan_end(h, C.byref(r), C.byref(u)))
    finally:
        ck(lib.frb_dev_free(h, dbuf))
    keys, counts, _ = ctx.total_arrays()
    sheet = ctx.load_sheet(spec.indexes())
    first = ctx.match(1, True, None, want_outputs=False)
    use = np.array([first["f_sum"][g] < first["rc_sum"][g] for g in sheet.group], np.uint8)
    res = ctx.match(1, False, use)
    S = spec.n_samples
    sink = np.where(res["type"] == 2, res["srow"], S + np.where(res["type"] == 1, 0, np.where(res["type"] == 3, 1, 2)))
    n_sinks = S + 3
    ctx.route_load(keys, sink.astype(np.uint32), n_sinks)

    chunk = chunk_mb << 20
    o1, o2 = C.c_void_p(), C.c_void_p()
    off1, off2 = np.zeros(n_sinks + 1, np.uint64), np.zeros(n_sinks + 1, np.uint64)
    nrec, c1, c2, bad = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
    (h1, n1), (h2, n2) = mates

    def stream(single, digests=None, packed=False):
        """One pass through the router; digests: one sha256 per sink, continued over the R1 bytes it receives
        (packed: the cells are BGZF blocks, digested decompressed)."""
        ck(lib.frb_route_set_mates(h, 1 if single else 2))
        ck(lib.frb_route_reset(h))
        total, in_flight = 0, 0
        n_chunks = (n1 + chunk - 1) // chunk if single else max((n1 + chunk - 1) // chunk, (n2 + chunk - 1) // chunk)

        def pop():
            nonlocal total
            ck(lib.frb_route_pop(h, C.byref(o1), C.byref(o2), vp(off1), vp(off2), C.byref(nrec), C.byref(c1),
                                 C.byref(c2), C.byref(bad)))
            total += nrec.value
            if digests is not None and off1[-1]:
                out = np.ctypeslib.as_array((C.c_uint8 * int(off1[-1])).from_address(o1.value))
                for s in range(n_sinks):
                    cell = out[int(off1[s]):int(off1[s + 1])].tobytes()
                    digests[s].update(gzip.decompress(cell) if packed and cell else cell)

        for k in range(n_chunks):
            a0, b0 = min(k * chunk, n1), min(k * chunk, n2)
            a1, b1 = min(a0 + chunk, n1), min(b0 + chunk, n2)
            if single:
                ck(lib.frb_route_push(h, C.c_void_p(h1.value + a0), a1 - a0, None, 0, 1 if a1 >= n1 else 0))
            else:
                final = (1 if a1 >= n1 else 0) | (2 if b1 >= n2 else 0)
                ck(lib.frb_route_push(h, C.c_void_p(h1.value + a0), a1 - a0, C.c_void_p(h2.value + b0), b1 - b0, final))
            in_flight += 1
            if in_flight == 2:
                pop()
                in_flight -= 1
        while in_flight:
            pop()
            in_flight -= 1
        return total

    checked = {}
    for fmt in ("plain", "bgzf"):
        ck(lib.frb_route_set_gz_format(h, L.GZ_FORMAT_BGZF if fmt == "bgzf" else L.GZ_FORMAT_PLAIN))
        sums = {}
        for name, single in (("single", True), ("paired", False)):
            sums[name] = [hashlib.sha256() for _ in range(n_sinks)]
            assert stream(single, sums[name], fmt == "bgzf") == reads, name
        same = [a.digest() == b.digest() for a, b in zip(sums["single"], sums["paired"])]
        assert all(same), f"{fmt}: single-end sinks differ from the paired R1 sinks: {same}"
        checked[fmt] = f"all {n_sinks} single-end sinks == paired R1 sinks (sha256 of the bytes)"
    ck(lib.frb_route_set_gz_format(h, L.GZ_FORMAT_PLAIN))

    for single in (True, False):                      # warm-up of both streams
        stream(single)
    ctx.prof(True)
    for k in range(L.K_NUM):
        ctx.prof_read(k)
    runs = {"single": [], "paired": []}
    for _ in range(steps):                            # alternating, step by step
        for name, single in (("single", True), ("paired", False)):
            t0 = time.perf_counter()
            stream(single)
            dt = time.perf_counter() - t0
            scan_ms, _ = ctx.prof_read(L.K_SCAN)
            route_ms, _ = ctx.prof_read(L.K_ROUTE)
            runs[name].append((dt, scan_ms + route_ms, scan_ms, route_ms))
    ctx.prof(False)
    ck(lib.frb_route_set_mates(h, 2))
    ck(lib.frb_route_reset(h))
    for host, _ in mates:
        lib.frb_host_free(host)
    ctx.close()

    out = {"tool": "tools/bench_demux_single_end.py", "card": card(), "reads": reads, "chunk_mb": chunk_mb,
           "steps": steps, "sinks": int(n_sinks), "r1_bytes": int(n1), "r2_bytes": int(n2), "checked": checked}
    for name, rows in runs.items():
        wall = float(np.median([r[0] for r in rows]))
        dev_ms = float(np.median([r[1] for r in rows]))
        inp = n1 if name == "single" else n1 + n2
        out[name] = {"records_per_s_host_to_host": reads / wall, "ms_per_pass_host_to_host": wall * 1e3,
                     "input_gbs_host_to_host": inp / wall / 1e9, "device_ms": dev_ms,
                     "parser_ms": float(np.median([r[2] for r in rows])),
                     "router_ms": float(np.median([r[3] for r in rows])),
                     "records_per_s_device": reads / (dev_ms / 1e3), "algorithmic_bytes": 2 * inp,
                     "device_gbs_algorithmic": 2 * inp / (dev_ms / 1e3) / 1e9,
                     "wall_ms_all_steps": [r[0] * 1e3 for r in rows], "device_ms_all_steps": [r[1] for r in rows]}
    out["single_over_paired_records_per_s"] = (out["single"]["records_per_s_host_to_host"]
                                               / out["paired"]["records_per_s_host_to_host"])
    return out


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if not a.startswith("--out")]
    dest = next((a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--out=")), None)
    result = measure(int(args[0]) if args else 4_000_000, int(args[1]) if len(args) > 1 else 64,
                     int(args[2]) if len(args) > 2 else 5)
    line = json.dumps(result)
    print(line)
    if dest:
        os.makedirs(os.path.dirname(os.path.abspath(dest)), exist_ok=True)
        with open(dest, "w") as fh:
            fh.write(json.dumps(result, indent=1) + "\n")
