"""Demux stream with index reads against the paired one: python tools/bench_demux_index_reads.py [reads] [chunk_mb]
[steps] [--out=path]

R1/R2 of a C4-shaped lane are device-generated (frb_synth_*, as tools/bench_demux.py does) and pulled to pinned host
memory; its I1/I2 (10 bp each) are generated on the host (synth.generate(..., index_read=1 / 2)).  The results table
comes from a scan of R1 and both matcher passes.  Two streams go through the library in chunks of chunk_mb, two in
flight, alternating step by step:
  * paired:  R1 + R2 (frb_route_push / frb_route_pop), keys from the R2 headers;
  * indexed: R1 + R2 + I1 + I2 (frb_route_set_mates2(ctx, 4, 1), frb_route_pushv / frb_route_popv).  An index mate
    reads only what keeps its bytes not yet routed, the chunk in flight included, within the chunk (as frender demux
    does), since its records are several times shorter than the reads'.
Reported per stream: device time (the library's per-class events, parser K_SCAN + router K_ROUTE), records/s host
-> host (pinned buffers in, pinned buffers out), GB/s of input host -> host, and GB/s on the algorithmic bytes
(2 x the input of every mate) over the device time.  Checked first: every sink of every mate of the indexed stream
holds exactly the bytes the N-mate route (tests/index_reads_oracle.py: record i of every mate goes to the sink of
record i's R2 key) gives, restated with numpy over the record offsets (sha256 per sink and mate).  The card's name
and power limit are read in the same run."""
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


def expected_digests(texts, sink_of, n_sinks):
    """sha256 of every sink of every mate under the N-mate route: record i of each text goes to sink sink_of[i], in
    record order."""
    order = np.argsort(sink_of, kind="stable")
    bounds = np.searchsorted(sink_of[order], np.arange(n_sinks + 1))
    out = []
    for text in texts:
        nl = np.flatnonzero(text == 10)
        ends = nl[3::4] + 1
        ends = ends[:len(sink_of)]
        starts = np.concatenate([[0], ends[:-1]])
        digests = []
        for s in range(n_sinks):
            recs = order[bounds[s]:bounds[s + 1]]
            h = hashlib.sha256()
            if len(recs):
                lens = ends[recs] - starts[recs]
                first = np.repeat(starts[recs] - (np.cumsum(lens) - lens), lens)
                h.update(text[first + np.arange(int(lens.sum()))].tobytes())
            digests.append(h.hexdigest())
        out.append(digests)
    return out


def measure(reads=4_000_000, chunk_mb=64, steps=5, device=0):
    from frender_b200 import _lib as L
    from frender_b200 import synth
    from frender_b200.engine import C, Context, unpack_keys
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
    hosts = []
    try:
        for mate in (1, 2):
            nb = C.c_uint64()
            ck(lib.frb_synth_generate(h, 0, reads, mate, dbuf, cap, C.byref(nb)))
            host = C.c_void_p()
            ck(lib.frb_host_alloc(C.byref(host), nb.value))
            ck(lib.frb_d2h(h, host, dbuf, nb.value))
            hosts.append((host, nb.value))
        ck(lib.frb_synth_generate(h, 0, reads, 1, dbuf, cap, C.byref(C.c_uint64())))
        ctx.reset()
        ck(lib.frb_scan_begin(h, 0, 0))
        ck(lib.frb_scan_chunk_dev(h, dbuf, hosts[0][1], 0, L.RULE_SCAN, None, None))
        r, u = C.c_uint64(), C.c_uint64()
        ck(lib.frb_scan_end(h, C.byref(r), C.byref(u)))
    finally:
        ck(lib.frb_dev_free(h, dbuf))
    for k in (1, 2):                                  # I1 / I2 in pinned memory too
        data = synth.generate_big(spec, 0, reads, 1, index_read=k)
        host = C.c_void_p()
        ck(lib.frb_host_alloc(C.byref(host), len(data)))
        C.memmove(host.value, data, len(data))
        hosts.append((host, len(data)))
    keys, counts, _ = ctx.total_arrays()
    sheet = ctx.load_sheet(spec.indexes())
    first = ctx.match(1, True, None, want_outputs=False)
    use = np.array([first["f_sum"][g] < first["rc_sum"][g] for g in sheet.group], np.uint8)
    res = ctx.match(1, False, use)
    S = spec.n_samples
    sink = np.where(res["type"] == 2, res["srow"], S + np.where(res["type"] == 1, 0, np.where(res["type"] == 3, 1, 2)))
    n_sinks = S + 3
    ctx.route_load(keys, sink.astype(np.uint32), n_sinks)
    sink_by_key = dict(zip(unpack_keys(keys), sink.tolist()))
    sink_of = np.array([sink_by_key[k] for k in synth.keys_of(spec, 0, reads)], np.int64)

    chunk = chunk_mb << 20
    sizes = [n for _, n in hosts]
    texts = [np.ctypeslib.as_array((C.c_uint8 * n).from_address(p.value)) for p, n in hosts]
    outs = (C.c_void_p * 4)()
    offs = np.zeros((4, n_sinks + 1), np.uint64)
    carry = np.zeros(4, np.uint64)
    o1, o2 = C.c_void_p(), C.c_void_p()
    nrec, c1, c2, bad = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()

    def stream(mates, digests=None):
        """One pass through the router with 2 or 4 mates; digests[m][s]: sha256 continued over the bytes sink s of
        mate m receives."""
        if mates == 4:
            ck(lib.frb_route_set_mates2(h, 4, 1))
        else:
            ck(lib.frb_route_set_mates(h, 2))
        ck(lib.frb_route_reset(h))
        total, flags, pushed, pos, left = 0, [], [], [0] * mates, [0] * mates
        n_chunks = max((sizes[m] + chunk - 1) // chunk for m in range(2))

        def pop():
            nonlocal total, left
            if mates == 4:
                ck(lib.frb_route_popv(h, outs, vp(offs), C.byref(nrec), vp(carry), C.byref(bad)))
                views, off = [outs[m] for m in range(4)], offs
                left = [int(c) for c in carry]
            else:
                ck(lib.frb_route_pop(h, C.byref(o1), C.byref(o2), vp(offs[0]), vp(offs[1]), C.byref(nrec),
                                     C.byref(c1), C.byref(c2), C.byref(bad)))
                views, off = [o1.value, o2.value], offs
            total += nrec.value
            if digests is not None:
                for m in range(mates):
                    n = int(off[m][-1])
                    if n:
                        out = np.ctypeslib.as_array((C.c_uint8 * n).from_address(views[m]))
                        for s in range(n_sinks):
                            digests[m][s].update(out[int(off[m][s]):int(off[m][s + 1])].tobytes())

        for k in range(n_chunks):
            want = []
            for m in range(mates):
                if m < 2:                               # the reads: chunk k of the file
                    want.append(min((k + 1) * chunk, sizes[m]) - pos[m])
                else:                                   # an index mate: up to the window, the chunk in flight included
                    ahead = sum(p[m] for p in pushed)
                    want.append(max(min(chunk - left[m] - ahead, sizes[m] - pos[m]), 0))
            ptrs = (C.c_void_p * mates)(*[hosts[m][0].value + pos[m] for m in range(mates)])
            n = np.array(want, np.uint64)
            for m in range(mates):
                pos[m] += want[m]
            final = sum(1 << m for m in range(mates) if pos[m] >= sizes[m])
            if mates == 4:
                ck(lib.frb_route_pushv(h, ptrs, vp(n), final))
            else:
                ck(lib.frb_route_push(h, ptrs[0], want[0], ptrs[1], want[1], final))
            flags.append(final)
            pushed.append(want)
            if len(flags) == 2:
                pop()
                flags.pop(0)
                pushed.pop(0)
        while flags:
            pop()
            flags.pop(0)
        return total

    ck(lib.frb_route_set_gz_format(h, L.GZ_FORMAT_PLAIN))
    sums = [[hashlib.sha256() for _ in range(n_sinks)] for _ in range(4)]
    assert stream(4, sums) == reads
    want = expected_digests(texts, sink_of, n_sinks)
    got = [[d.hexdigest() for d in mate] for mate in sums]
    bad_sinks = [(m, s) for m in range(4) for s in range(n_sinks) if got[m][s] != want[m][s]]
    assert not bad_sinks, f"sinks that differ from the N-mate route: {bad_sinks[:10]}"
    checked = f"all {n_sinks} sinks of all 4 mates == the N-mate route restated over the record offsets (sha256)"

    for mates in (2, 4):                              # warm-up of both streams
        stream(mates)
    ctx.prof(True)
    for k in range(L.K_NUM):
        ctx.prof_read(k)
    runs = {"paired": [], "indexed": []}
    for _ in range(steps):                            # alternating, step by step
        for name, mates in (("paired", 2), ("indexed", 4)):
            t0 = time.perf_counter()
            assert stream(mates) == reads
            dt = time.perf_counter() - t0
            scan_ms, _ = ctx.prof_read(L.K_SCAN)
            route_ms, _ = ctx.prof_read(L.K_ROUTE)
            runs[name].append((dt, scan_ms + route_ms, scan_ms, route_ms))
    ctx.prof(False)
    ck(lib.frb_route_set_mates(h, 2))
    ck(lib.frb_route_reset(h))
    for host, _ in hosts:
        lib.frb_host_free(host)
    ctx.close()

    out = {"tool": "tools/bench_demux_index_reads.py", "card": card(), "reads": reads, "chunk_mb": chunk_mb,
           "steps": steps, "sinks": int(n_sinks), "r1_bytes": sizes[0], "r2_bytes": sizes[1], "i1_bytes": sizes[2],
           "i2_bytes": sizes[3], "checked": checked}
    for name, rows in runs.items():
        wall = float(np.median([r[0] for r in rows]))
        dev_ms = float(np.median([r[1] for r in rows]))
        inp = sum(sizes[:2 if name == "paired" else 4])
        out[name] = {"records_per_s_host_to_host": reads / wall, "ms_per_pass_host_to_host": wall * 1e3,
                     "input_gbs_host_to_host": inp / wall / 1e9, "device_ms": dev_ms,
                     "parser_ms": float(np.median([r[2] for r in rows])),
                     "router_ms": float(np.median([r[3] for r in rows])),
                     "records_per_s_device": reads / (dev_ms / 1e3), "algorithmic_bytes": 2 * inp,
                     "device_gbs_algorithmic": 2 * inp / (dev_ms / 1e3) / 1e9,
                     "wall_ms_all_steps": [r[0] * 1e3 for r in rows], "device_ms_all_steps": [r[1] for r in rows]}
    out["indexed_over_paired_records_per_s"] = (out["indexed"]["records_per_s_host_to_host"]
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
