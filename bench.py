#!/usr/bin/env python
"""Benchmark of the scan hot path: read-names/s scanned + matched (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--reads R] [--workload scan|demux]
                    [--dump-outputs DIR]

One step = one pass of the whole scan path over one synthetic NovaSeq-lane shaped input
(config C2: 10+10 bp UDI, 384-sample sheet, `scan -n 1 -rc`): fused parse+pack+count kernel ->
sorted unique list -> matcher pass 1 (forward + reverse-complement) -> per-sample orientation
call -> matcher pass 2.
  value   kernel-only: the lane resident in HBM, results left on the device.
  e2e     what a user runs: one `.fastq.gz` of the lane through frb_scan_gz (the compressed bytes go host ->
          device, are inflated there, scanned where they lie) + both matcher passes + D2H of keys, counts and
          per-key results, wall clock.  `e2e_pcie` is the round-1 leg (decompressed text in pinned host
          memory through frb_scan_chunk_host) beside a plain pinned-memcpy measurement of the link.
N > 1: one process per GPU (torchrun), each rank owns one lane (weak scaling); inside the step the per-rank
unique tables are merged over NCCL so that every key ends on one rank (frb_shardmerge), each rank matches its
share, and the per-sample orientation sums are all-reduced (the call of F:354-388 is over all reads of the job).
`--impl reference` times the reference itself (baseline/_ref/frender.py, copied there by
__graft_entry__.build(); the oracle port when it is absent) with all host cores on a bounded sample of the same
lane: the first reads of the stream the e2e leg uses.
After the timed loop the result is CHECKED: counts sum to the reads, shares of the ranks are disjoint, and the
first 3 M reads of the lane -- tally, both matcher passes, orientation calls -- equal the C oracle's.
`--scaling strong` (N > 1) deals the record chunks of ONE lane to the ranks instead of one lane each.
`--dump-outputs DIR` (N = 1) writes what the last timed step computed as .npy files (see dump_outputs).
At N = 1 the line also carries a `demux` object: BASELINE configs[3] through the record router as a stream
(tools/bench_demux.py: 4 M pairs, 64 MB chunks cut anywhere, two in flight, every sink's byte stream compared with
the C oracle's demux loop); `--workload demux` makes that the line, with the reference's frender_demux beside it.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIG = "C2"
N_SUBS = 1
GEN_CHUNK = 8_000_000          # reads per generator call
CPU_SAMPLE_READS = 200_000     # bounded sample for the CPU arm (about 3 s of the reference per step)
E2E_MAX_BYTES = 6 << 30        # host-resident sample for the pinned-text leg (e2e_pcie)
E2E_GZ_READS = 4_000_000       # reads in the .fastq.gz of the end-to-end leg
CHECK_READS = 3_000_000        # prefix of the lane compared with the C oracle after the timed loop
DUMP_ROWS = 1 << 19            # unique keys sampled by --dump-outputs (13 M at the default lane; 29 MB of .npy)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU (default: 400M or what HBM holds)")
    ap.add_argument("--table-log2", type=int, default=0, help="slots of the unique-key tables (default: by input size)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-demux", action="store_true")
    ap.add_argument("--workload", default="scan", choices=["scan", "demux"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: one lane per GPU; strong: ONE lane, its record chunks dealt to the GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (float32/float64; "
                         "a fixed, seeded sample of the unique keys) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl == "reference" or args.workload != "scan"):
        ap.error("--dump-outputs writes the outputs of the scan workload on the GPU (--workload scan, no --impl reference)")
    return args


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference on a bounded sample (shared by cpu_baseline and
# --impl reference).  This is the one place outside tests/ that executes oracle/.
# ------------------------------------------------------------------------------------------------
def cpu_sample(tmpdir, reads=CPU_SAMPLE_READS):
    """The first `reads` reads of the lane (the stream the e2e leg compresses) as one .fastq.gz + its sheet."""
    import gzip

    from frender_b200 import synth
    spec = synth.make_spec(CONFIG)
    data = synth.generate_big(spec, 0, reads)
    path = os.path.join(tmpdir, "Undetermined_S0_L001_R1_001.fastq.gz")
    with gzip.open(path, "wb", compresslevel=1) as fh:
        fh.write(data)
    return spec, path, len(data)


def load_reference():
    """The reference itself (baseline/_ref/frender.py, an unmodified copy made by __graft_entry__.build()), or
    None when it is not there."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "frender.py")):
        return None
    import importlib
    import warnings
    warnings.simplefilter("ignore")
    # under its own module name: its process pools pickle their work functions by reference (frender.scan_file)
    sys.path.insert(0, ref_dir)
    sys.modules.pop("frender", None)
    mod = importlib.import_module("frender")
    assert os.path.dirname(os.path.abspath(mod.__file__)) == ref_dir, mod.__file__
    return mod


def cpu_step(spec, path, cores, ref=None):
    """scan -n 1 -rc on one file, host only: tally + both matcher passes.  ref: the reference module; None: the
    oracle port.  Returns (total s, tally s, matcher s, unique keys)."""
    import contextlib
    import io
    indexes = spec.indexes()
    t0 = time.perf_counter()
    if ref is not None:
        with contextlib.redirect_stdout(io.StringIO()):
            counter = ref.tally_barcodes(cores, [path], None)                       # F:183-207
            t1 = time.perf_counter()
            first = ref.process(cores, counter["total"], indexes, N_SUBS, True)   # F:391-426
            calls = ref.call_rc_mode_per_id(ref.flatten_results(first), indexes["id"])      # F:354-388
            oriented = dict(indexes)
            oriented["idx2"] = [ref.reverse_complement(b) if calls[i]["call"] else b
                                for b, i in zip(indexes["idx2"], indexes["id"])]     # F:618-623
            results = ref.process(cores, counter["total"], oriented, N_SUBS, False)  # F:628-630
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import frender_oracle as O
        counter = O.tally_barcodes(cores, [path])
        t1 = time.perf_counter()
        results, calls, _ = O.scan_analysis(cores, counter, indexes, N_SUBS, True)
    t2 = time.perf_counter()
    return t2 - t0, t1 - t0, t2 - t1, len(results)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    ref = load_reference()
    kind = "reference" if ref is not None else "port"
    with tempfile.TemporaryDirectory() as d:
        spec, path, nbytes = cpu_sample(d)
        times, parts = [], []
        for i in range(args.warmup + args.steps):
            total, t_tally, t_match, uniq = cpu_step(spec, path, cores, ref)
            if i >= args.warmup:
                times.append(total)
                parts.append((t_tally, t_match))
    ms = 1e3 * sum(times) / len(times)
    value = CPU_SAMPLE_READS / (ms / 1e3)
    what = ("/root/reference/frender.py (unmodified copy in baseline/_ref): tally_barcodes + process(rc) + "
            "call_rc_mode_per_id + process" if ref is not None else "oracle port of the reference")
    sample = (f"{what}; the first {CPU_SAMPLE_READS} reads of the {CONFIG} lane ({nbytes} B decompressed) from one "
              f".fastq.gz per step: gzip inflate + tally (1 core: one file) + matcher both passes on {cores} cores; "
              f"{uniq} unique keys")
    line = {
        "impl": "reference", "metric": "read_names_per_s_scanned_matched", "value": value, "unit": "reads/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u64",
        "data": "synthetic", "config": workload_config(args.reads or 400_000_000, args.gpus),
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": kind, "sample": sample,
                         "tally_s": sum(p[0] for p in parts) / len(parts),
                         "match_s": sum(p[1] for p in parts) / len(parts)},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# Demux workload (configs[3]): the record router as a stream, and the reference's demux beside it
# ------------------------------------------------------------------------------------------------
DEMUX_PAIRS = 4_000_000         # pairs per GPU and pass (1.5 GB per mate; chunks of 64 MB, two in flight)
DEMUX_CPU_PAIRS = 50_000        # bounded sample for the reference's demux (gz in -> 387 gz sinks out)


def demux_cpu_sample(tmpdir, pairs=DEMUX_CPU_PAIRS):
    """R1/R2 .fastq.gz of the first `pairs` pairs of the C4 lane and the scan-results CSV of R1 (made by this repo's
    scan; the reference's parse_results_file wants the columns in the order its demux asserts, F:645-664)."""
    import contextlib
    import csv
    import gzip
    import io

    from frender_b200 import cli, synth
    spec = synth.make_spec("C4")
    paths = []
    for mate in (1, 2):
        path = os.path.join(tmpdir, f"Undetermined_S0_L001_R{mate}_001.fastq.gz")
        with gzip.open(path, "wb", compresslevel=1) as fh:
            fh.write(synth.generate_big(spec, 0, pairs, mate))
        paths.append(path)
    sheet = os.path.join(tmpdir, "SampleSheet.csv")
    idx = spec.indexes()
    with open(sheet, "w", newline="") as fh:
        w = csv.writer(fh)
        w.writerow(["Sample_ID", "index", "index2"])
        w.writerows(zip(idx["id"], idx["idx1"], idx["idx2"]))
    cwd = os.getcwd()
    os.chdir(tmpdir)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            cli.main(["scan", "-n", str(N_SUBS), "-rc", "-b", sheet, "-o", "bench", paths[0]])
        made = [f for f in os.listdir(tmpdir) if f.startswith("frender-scan-results_")][0]
    finally:
        os.chdir(cwd)
    rows = list(csv.reader(open(os.path.join(tmpdir, made), newline="")))
    head = rows[0]
    order = [head.index(c) for c in ["idx1", "idx2", "reads", "matched_idx1", "matched_idx2", "read_type", "sample_name",
                                     "demux_ok"]]
    res = os.path.join(tmpdir, "results.csv")
    with open(res, "w", newline="") as fh:
        csv.writer(fh).writerows([[r[i] for i in order] for r in rows])
    return paths, res


def demux_cpu_step(paths, res, outdir, ref):
    """The reference's frender_demux (F:733-814) on the sample files, or -- without baseline/_ref -- this repo's
    oracle port of it with the same gzip sinks.  Returns seconds."""
    import argparse
    import contextlib
    import gzip
    import io
    t0 = time.perf_counter()
    if ref is not None:
        ns = argparse.Namespace(no_index_hop=False, no_ambiguous=False, no_undeter=False, no_samples=False, o=None,
                                d=outdir, r=res, files=list(paths))
        ref.args = ns                                                    # open_files reads a global (F:672)
        with contextlib.redirect_stdout(io.StringIO()):
            ref.frender_demux(ns)
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import frender_oracle as O
        table = O.parse_results_file(res)
        os.makedirs(outdir, exist_ok=True)
        for name, (a, b) in O.demux_files(paths[0], paths[1], table, O.sink_names(table)).items():
            for mate, data in (("R1", a), ("R2", b)):
                with gzip.open(os.path.join(outdir, f"{name}_{mate}.fastq.gz"), "wb") as fh:
                    fh.write(data)
    return time.perf_counter() - t0


def demux_cli_step(paths, res, outdir):
    """This repo's `demux` on the same files: host inflate -> device router -> host deflate.  Returns seconds."""
    import contextlib
    import io

    from frender_b200 import cli
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        cli.main(["demux", "-r", res, "-d", outdir] + list(paths))
    return time.perf_counter() - t0


def demux_files_equal(dir_a, dir_b):
    import gzip
    import hashlib
    names = sorted(os.listdir(dir_a))
    if names != sorted(os.listdir(dir_b)):
        return False
    digest = lambda p: hashlib.sha256(gzip.open(p, "rb").read()).hexdigest()
    return all(digest(os.path.join(dir_a, n)) == digest(os.path.join(dir_b, n)) for n in names)


def demux_cpu_baseline(with_cli=True, steps=1, warmup=0):
    """The reference's demux on the sample files: `warmup` untimed runs, then the mean of `steps` timed ones (each
    into a directory of its own, as the reference writes into an empty one)."""
    cores = len(os.sched_getaffinity(0))
    ref = load_reference()
    with tempfile.TemporaryDirectory() as d:
        paths, res = demux_cpu_sample(d)
        times = [demux_cpu_step(paths, res, os.path.join(d, f"out_ref{i}"), ref) for i in range(warmup + steps)]
        t_ref = sum(times[warmup:]) / steps
        out = {"value": DEMUX_CPU_PAIRS / t_ref, "unit": "pairs/s", "cores": 1,
               "kind": "reference" if ref is not None else "port",
               "sample": f"frender_demux on the first {DEMUX_CPU_PAIRS} pairs of the C4 lane: R1/R2 .fastq.gz in, 387 "
                         f".fastq.gz sinks out (gzip level 9, as the reference opens them), one process as the "
                         f"reference runs it ({cores} cores on the box)"}
        if with_cli:
            t_cli = demux_cli_step(paths, res, os.path.join(d, "out_b200"))
            out["same_files_through_this_repo"] = {
                "pairs_per_s": DEMUX_CPU_PAIRS / t_cli, "threads": cores,
                "what": "frender_b200 demux on the same files (host inflate threads, device router stream, host deflate threads at the CLI's default level 6; includes creating the CUDA context)",
                "sinks_identical_after_gunzip": demux_files_equal(os.path.join(d, f"out_ref{warmup + steps - 1}"),
                                                                  os.path.join(d, "out_b200"))}
    return out


def run_demux(args):
    """--workload demux: configs[3] through the record router.  value = pairs/s by the device's own time (parser of
    both mates + router), e2e = the same stream from pinned host buffers to pinned host buffers."""
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            cpu = demux_cpu_baseline(with_cli=False, steps=args.steps, warmup=args.warmup)
            print(json.dumps({"impl": "reference", "metric": "record_pairs_per_s_demuxed", "value": cpu["value"],
                              "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                              "ms_per_step": 1e3 * DEMUX_CPU_PAIRS / cpu["value"], "higher_is_better": True,
                              "scaling": "weak", "vs_baseline": None, "dtype": "u8/u64", "data": "synthetic",
                              "config": demux_config(args.reads or DEMUX_PAIRS, args.gpus), "cpu_baseline": cpu,
                              "e2e": {"value": cpu["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0,
                                      "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from bench_demux import measure
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo", rank=rank, world_size=world)
    pairs = args.reads or DEMUX_PAIRS
    sampler = Clocks(local) if rank == 0 else None
    if dist:
        dist.barrier()
    m = measure(local, pairs, 64, args.steps, args.warmup)
    clk = sampler.stop() if sampler else None
    parts = [m]
    if dist:
        parts = [None] * world
        dist.all_gather_object(parts, m)
    if rank == 0:
        kernel_ms = max(p["kernel_ms"] for p in parts)
        pass_ms = max(p["ms_per_pass_host_to_host"] for p in parts)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peaks = {"sustained": json.load(open(peaks_path))["hbm_gbs"], "source": "MEASURED_PEAKS.json hbm_gbs (measured copy)"}
        else:
            peaks = {"sustained": 6650.0, "source": "fallback of B200_PROFILING.md"}
        moved = sum(p["algorithmic_bytes"] for p in parts)
        ach = m["algorithmic_bytes"] / (m["kernel_ms"] * 1e-3) / 1e9
        line = {"metric": "record_pairs_per_s_demuxed", "value": world * pairs / (kernel_ms * 1e-3), "unit": "pairs/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": kernel_ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u64",
                "data": "synthetic (device-generated R1/R2 of the C4 lane, pulled to pinned host memory)",
                "config": demux_config(pairs, world), "clocks": clk,
                "e2e": {"value": world * pairs / (pass_ms * 1e-3), "unit": "pairs/s",
                        "h2d_bytes_per_step": moved // 2, "d2h_bytes_per_step": moved // 2,
                        "what": "frb_route_push / frb_route_pop from pinned host buffers to pinned host buffers, "
                                "64 MB chunks cut at fixed byte counts, two in flight; no gzip on either side",
                        "gbs_in_plus_out_per_gpu": m["host_to_host_gbs_in_plus_out"]},
                "gpu_launches": m["gpu_launches_per_pass"],
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["sustained"], "unit": "GB/s",
                             "frac": ach / peaks["sustained"], "traffic": None,
                             "what": "parser (both mates) + router kernels together: algorithmic bytes 2 x (R1 + R2) "
                                     "per pass over their summed event time (rank 0); launched per 64 MB chunk, so "
                                     "launch tails count", "peak_source": peaks["source"]},
                "checked": m["checked"], "parser_ms": m["parser_ms"], "router_ms": m["router_ms"],
                "cpu_baseline": None if args.no_cpu or world > 1 else demux_cpu_baseline()}
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


def demux_config(pairs_per_gpu, n_gpus):
    return {"workload": "demux -r of a paired R1/R2 synthetic NovaSeq lane (10+10 bp UDI, 384-sample sheet) into 384 "
                        "sample sinks + Index-hop + Ambiguous + Undetermined (BASELINE.json configs[3], bounded to what a "
                        "few seconds of PCIe traffic hold)", "pairs_per_gpu": pairs_per_gpu,
            "pairs_total": pairs_per_gpu * n_gpus, "sharding": "one lane per GPU, outputs rank-local",
            "l2": "inputs far larger than L2 (1.5 GB per mate)"}


def workload_config(reads_per_gpu, n_gpus):
    return {"workload": "scan -n 1 -rc, synthetic NovaSeq-lane Undetermined R1, 10+10 bp UDI, 384-sample sheet "
                        "(BASELINE configs[1])",
            "reads_per_gpu": reads_per_gpu, "reads_total": reads_per_gpu * n_gpus, "read_len": 151,
            "index": "10+10", "samples": 384, "n_mismatches": N_SUBS, "rc": True,
            "l2_policy": "inputs larger than L2 (no flush needed)" if reads_per_gpu * 373 > (256 << 20)
            else "input smaller than L2"}


# ------------------------------------------------------------------------------------------------
class Clocks:
    """SM clock and throttle-reason sampler for the timed region (the counters of B200_PROFILING.md's
    nvidia-smi line; every 50 ms through NVML, every 200 ms through the nvidia-smi child).  Read through NVML in-process when pynvml is importable: an
    `nvidia-smi -lms` child re-queries the whole device each period and was seen to hold up the sampled
    rank's CUDA calls for 10-600 ms at a time; falls back to that child otherwise."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, device):
        self.proc = self.thread = None
        self.sm, self.mx, self.reasons = [], 0, set()
        try:
            if os.environ.get("FRB_BENCH_NO_CLOCKS"):
                raise RuntimeError("clock sampling disabled")
            import threading

            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [v for v in vis.split(",") if v.strip()]
            index = int(ids[device]) if ids and all(v.strip().isdigit() for v in ids) else device
            handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
            self.stop_flag = threading.Event()

            def loop():
                while not self.stop_flag.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)))
                        mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                        self.reasons.update(name for name, bit in self.BITS.items() if mask & bit)
                    except pynvml.NVMLError:
                        pass
                    self.stop_flag.wait(0.05)

            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.source = "nvml"
            return
        except Exception:
            self.thread = None
        self.source = "nvidia-smi"
        self.path = tempfile.mktemp(suffix=".csv")
        self.fh = open(self.path, "w")
        try:
            if os.environ.get("FRB_BENCH_NO_CLOCKS"):
                raise OSError("clock sampling disabled")
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={device}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=self.fh, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.thread:
            self.stop_flag.set()
            self.thread.join()
        else:
            if self.proc:
                self.proc.terminate()
                self.proc.wait()
            self.fh.close()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for row in open(self.path):
                f = [x.strip() for x in row.split(",")]
                if len(f) < 9:
                    continue
                try:
                    self.sm.append(float(f[1]))
                    self.mx = max(self.mx, float(f[2]))
                except ValueError:
                    continue
                for name, flag in zip(names, f[5:9]):
                    if flag.lower().startswith("active"):
                        self.reasons.add(name)
            os.unlink(self.path)
        sm = self.sm
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": self.mx or None,
                "reasons": sorted(self.reasons), "samples": len(sm), "source": self.source}


def dump_outputs(out_dir, ctx, n_reads, res, last):
    """--dump-outputs: what the last timed step computed, as a caller of the scan path receives it -- the unique-key
    list (key, reads, first read) with each key's oriented-pass match (F:618-630), reads per read type and per sample
    row over all keys, and the per-sample orientation sums and calls (F:354-388).  Per-key arrays hold a fixed, seeded
    sample of DUMP_ROWS keys (rows of the first-appearance list, `key_row`); packed keys are split into 32-bit halves
    so that float64 holds them exactly.  res: the matcher part of the step run once more with its per-key outputs
    copied to the host (inside the timed loop they stay on the device); last: its orientation sums and calls."""
    keys, counts, first = ctx.total_arrays()
    n = len(keys)
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    weights = counts.astype(np.float64)
    demuxable = res["srow"] >= 0
    arrays = {
        "totals": np.array([n_reads, n], np.float64),
        "key_row": rows.astype(np.float64),
        "key_hi": (keys[rows] >> np.uint64(32)).astype(np.float64),
        "key_lo": (keys[rows] & np.uint64(0xFFFFFFFF)).astype(np.float64),
        "reads": counts[rows].astype(np.float64),
        "first_read": first[rows].astype(np.float64),
        "matched_idx1_row": res["m1"][rows].astype(np.float32),
        "matched_idx2_row": res["m2"][rows].astype(np.float32),
        "read_type": res["type"][rows].astype(np.float32),
        "sample_row": res["srow"][rows].astype(np.float32),
        "reads_per_read_type": np.bincount(res["type"], weights, minlength=4),
        "reads_per_sample_row": np.bincount(res["srow"][demuxable], weights[demuxable], minlength=len(ctx.sheet.ids)),
        "orientation_reads_f": last["f_sum"].astype(np.float64),
        "orientation_reads_rc": last["rc_sum"].astype(np.float64),
        "orientation_rc_call": last["use"].astype(np.float32),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def run_b200(args):
    from frender_b200 import _lib as L
    from frender_b200 import synth
    from frender_b200.engine import C, Context, PackedSheet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one process (--gpus 1)")
    dist = None
    if world > 1:
        import torch.distributed as dist  # host-side rendezvous only (gloo); the data path is NCCL in the .so
        dist.init_process_group("gloo", rank=rank, world_size=world)

    spec = synth.make_spec(CONFIG, lane=1 if args.scaling == "strong" else 1 + rank % 8)
    lib = L.lib
    probe = Context(local, table_log2=10)
    free_b, total_b = C.c_uint64(), C.c_uint64()
    probe._ck(lib.frb_mem_info(probe._h, C.byref(free_b), C.byref(total_b)))
    probe.close()
    strong = args.scaling == "strong" and world > 1
    reads = args.reads or 400_000_000
    if strong:          # one lane for the whole job: rank r scans the reads [r * reads, (r + 1) * reads) of it
        reads = -(-reads // world)
    bytes_per_read = 375.0
    table_log2 = args.table_log2 or (26 if reads > 100_000_000 else (24 if reads > 8_000_000 else 21))
    overhead = 2 * (32 << table_log2) + (8 << 30)
    # sized by the device's total memory, not by what is free at the moment: the same arguments on the same GPU model
    # give the same lane, so that two runs (and two builds) compute on identical inputs
    fit = int((total_b.value - overhead) / bytes_per_read)
    if reads > fit:
        reads = max(1_000_000, fit // 1_000_000 * 1_000_000)
    cap = int(reads * 374.6) + (64 << 20)
    need = cap + 2 * (32 << table_log2)           # the resident lane + the two unique-key tables
    if need > free_b.value:                       # memory held by other processes on this GPU
        raise SystemExit(f"bench.py: the {reads}-read lane needs {need / 1e9:.1f} GB of device memory, but only "
                         f"{free_b.value / 1e9:.1f} GB of {total_b.value / 1e9:.1f} GB is free on GPU {local}; "
                         f"free the GPU or pass a smaller --reads")
    ctx = Context(local, table_log2=table_log2)
    h = ctx._h
    ck = ctx._ck

    # ---- synthetic lane, generated on the device, resident in HBM -------------------------------
    emit_i7 = np.array([sum(int(c) << (2 * p) for p, c in enumerate(row)) for row in spec.sheet_i7], np.uint32)
    emit_i5 = np.array([sum(int(c) << (2 * p) for p, c in enumerate(row)) for row in spec.emit_i5()], np.uint32)
    cdf = np.ascontiguousarray(spec.cdf, np.uint64)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    ck(lib.frb_synth_load(h, spec.seed, spec.l1, spec.l2, spec.n_samples, vp(emit_i7), vp(emit_i5), vp(cdf),
                          spec.lane, spec.read_len, spec.sub_t, spec.n_t, spec.rand_t, spec.hop_t))
    dbuf = C.c_void_p()
    ck(lib.frb_dev_alloc(h, cap, C.byref(dbuf)))
    g_base = rank * reads
    off, bounds = 0, [0]
    t_gen = time.perf_counter()
    for g in range(0, reads, GEN_CHUNK):
        n = C.c_uint64()
        ck(lib.frb_synth_generate(h, g_base + g, g_base + min(g + GEN_CHUNK, reads), 1,
                                  C.c_void_p(dbuf.value + off), cap - off, C.byref(n)))
        off += n.value
        bounds.append(off)
    nbytes = off
    t_gen = time.perf_counter() - t_gen

    sheet = ctx.load_sheet(PackedSheet(spec.indexes()))
    if world > 1:
        ident = (C.c_char * 128)()
        if rank == 0:
            ck(lib.frb_nccl_unique_id(ident))
        box = [bytes(ident)]
        dist.broadcast_object_list(box, src=0)
        ck(lib.frb_nccl_init(h, box[0], rank, world))

    def barrier():
        if dist:
            dist.barrier()

    last = {}       # orientation sums and calls of the latest step (--dump-outputs)

    def analyze(want_outputs):
        """matcher pass 1 (rc) -> orientation call -> pass 2; returns unique count"""
        r = ctx.match(N_SUBS, True, None, want_outputs=False)
        f_sum, rc_sum = r["f_sum"], r["rc_sum"]
        if world > 1:   # every rank matched its share of the merged keys: the call is over the whole job
            f_sum, rc_sum = ctx.allreduce(f_sum), ctx.allreduce(rc_sum)
        use = np.array([f_sum[g] < rc_sum[g] for g in sheet.group], np.uint8)               # F:376
        last.update(f_sum=f_sum, rc_sum=rc_sum, use=use)
        out = ctx.match(N_SUBS, False, use, want_outputs=want_outputs)
        return out

    def step_resident():
        ck(lib.frb_reset(h))
        # weak: every rank its own file (ordinal = rank).  strong: the ranks hold consecutive chunks of ONE file: same
        # ordinal, and the chunk's global line number makes `first` the read ordinal within the whole file
        ck(lib.frb_scan_begin(h, 0 if strong else rank, 0))
        ck(lib.frb_scan_chunk_dev(h, dbuf, nbytes, 4 * g_base if strong else 0, L.RULE_SCAN, None, None))
        n_reads, n_uniq = C.c_uint64(), C.c_uint64()
        ck(lib.frb_scan_end(h, C.byref(n_reads), C.byref(n_uniq)))
        if world > 1:
            ck(lib.frb_shardmerge(h, C.byref(n_uniq)))
        analyze(False)
        return n_reads.value

    def timed(fn, steps, warmup, after_warmup=None):
        for _ in range(warmup):
            fn()
        ck(lib.frb_sync(h))
        if after_warmup:
            after_warmup()
        barrier()
        ms_all = []
        t_wall = time.perf_counter()
        for _ in range(steps):
            ck(lib.frb_timer_start(h))
            got = fn()
            ms = C.c_float()
            ck(lib.frb_timer_stop(h, C.byref(ms)))
            ms_all.append(ms.value)
            if os.environ.get("FRB_BENCH_VERBOSE"):
                print(f"[rank {rank}] step {len(ms_all)}: {ms.value:.2f} ms", file=sys.stderr)
        ck(lib.frb_sync(h))
        t_wall = time.perf_counter() - t_wall
        barrier()
        return sum(ms_all), t_wall, got

    ctx.prof(True)
    mark = {}

    def start_counting():      # the timed steps only: per-class device time and launch count start after warm-up
        for k in range(L.K_NUM):
            ctx.prof_read(k, reset=True)
        mark["launches"] = ctx.launches()

    clocks = Clocks(local)
    ms_total, wall_s, got_reads = timed(step_resident, args.steps, args.warmup, start_counting)
    clk = clocks.stop()
    launches = ctx.launches() - mark["launches"]
    assert got_reads == reads, (got_reads, reads)
    prof = {k: ctx.prof_read(k, reset=True) for k in range(L.K_NUM)}
    n_uniq = C.c_uint64()
    ck(lib.frb_total_finish(h, C.byref(n_uniq)))
    if args.dump_outputs:
        # the step's own matcher sequence on the list the last timed step left resident: rc pass -> orientation call
        # -> oriented pass, which reuses the rc pass's idx1 verdicts exactly as inside the step
        dump_outputs(args.dump_outputs, ctx, got_reads, analyze(True), last)
    if dist:    # the shares are disjoint: the job's unique keys are their sum
        box = [None] * world
        dist.all_gather_object(box, n_uniq.value)
        n_uniq = C.c_uint64(sum(box))

    # device time of the step, max over ranks
    ms_step = ms_total / args.steps
    if dist:
        box = [None] * world
        dist.all_gather_object(box, ms_step)
        ms_step = max(box)
    value = reads * world / (ms_step / 1e3)

    # ---- roofline of the dominant kernel (parse+pack+count), live CUDA events -------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy)"
    else:
        peak, peak_src = 6650.0, "fallback of B200_PROFILING.md"
    scan_ms, scan_n = prof[L.K_SCAN]
    scan_ms_per = scan_ms / max(scan_n, 1)
    achieved = nbytes / (scan_ms_per * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_scan_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = nbytes * tj["traffic_per_algorithmic_byte"]
        traffic_src = ("dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture (%s), scaled "
                       "from %d to %d algorithmic bytes" % (tj["source"], tj["algorithmic_bytes"], nbytes))
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "scan_spec_kernel (parse+pack+count, warp-specialised, speculative line phase)",
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": scan_ms_per,
                "step_share": {name: prof[k][0] / args.steps for name, k in
                               (("scan_ms", L.K_SCAN), ("export_sort_merge_ms", L.K_EXPORT),
                                ("match_ms", L.K_MATCH), ("clear_ms", L.K_OTHER), ("verify_ms", L.K_VERIFY))}}

    # ---- end to end, as a user runs it: one .fastq.gz -> frb_scan_gz (compressed bytes host -> device, inflated
    #      there, scanned where they lie) -> both matcher passes -> D2H of keys, counts and per-key results ----
    e2e = e2e_pcie = None
    if not args.no_e2e:
        import zlib
        g_reads = min(E2E_GZ_READS, reads)
        raw = np.empty(int(g_reads * 376), np.uint8)
        n_raw = C.c_uint64()
        tmpbuf = C.c_void_p()
        ck(lib.frb_dev_alloc(h, raw.size, C.byref(tmpbuf)))
        ck(lib.frb_synth_generate(h, g_base, g_base + g_reads, 1, tmpbuf, raw.size, C.byref(n_raw)))
        ck(lib.frb_d2h(h, vp(raw), tmpbuf, n_raw.value))
        ck(lib.frb_dev_free(h, tmpbuf))
        with tempfile.TemporaryDirectory() as d:
            gz_path = os.path.join(d, "Undetermined_S0_L001_R1_001.fastq.gz")
            z = zlib.compressobj(1, zlib.DEFLATED, 31)       # ONE gzip member, as a sequencer's fastq.gz
            with open(gz_path, "wb") as fh:
                view = memoryview(raw)[:n_raw.value]
                for off in range(0, n_raw.value, 64 << 20):
                    fh.write(z.compress(view[off:off + (64 << 20)]))
                fh.write(z.flush())
            gz_size = os.path.getsize(gz_path)
            d2h = [0]

            def step_gz():
                ctx.reset()
                got_r, _, got_raw = ctx.scan_gz(gz_path, rank)
                if world > 1:
                    n_u = C.c_uint64()
                    ck(lib.frb_shardmerge(h, C.byref(n_u)))
                keys, counts, _ = ctx.total_arrays()
                out = analyze(True)
                d2h[0] = keys.nbytes + counts.nbytes + sum(v.nbytes for v in out.values())
                assert got_raw == n_raw.value
                return got_r

            e_steps, e_warm = max(2, min(args.steps, 5)), max(1, min(args.warmup, 3))
            _, e_wall, e_got = timed(step_gz, e_steps, e_warm)
            assert e_got == g_reads, (e_got, g_reads)
            e_s = e_wall / e_steps
            if dist:
                box = [None] * world
                dist.all_gather_object(box, e_s)
                e_s = max(box)
            e2e = {"value": g_reads * world / e_s, "unit": "reads/s", "h2d_bytes_per_step": gz_size,
                   "d2h_bytes_per_step": d2h[0], "reads_per_step_per_gpu": g_reads, "ms_per_step": e_s * 1e3,
                   "gz_bytes": gz_size, "raw_bytes": n_raw.value, "inflate_gbs": n_raw.value / e_s / 1e9,
                   "sample": "one single-member .fastq.gz (zlib level 1) of the first %d reads of the lane through "
                             "frb_scan_gz (device-side inflate) + both matcher passes + D2H of keys, counts and "
                             "per-key results; wall clock, sync both sides" % g_reads}
            if rank == 0 and world == 1:
                # the same file with zlib on a host thread (round 1's path, FRB_GZ_DEVICE=0 in a child process)
                code = ("import sys, time; sys.path.insert(0, %r)\n"
                        "from frender_b200.engine import Context\n"
                        "ctx = Context(%d, table_log2=22); ctx.scan_gz(%r, 0); ctx.reset()\n"
                        "t0 = time.perf_counter(); r, u, raw = ctx.scan_gz(%r, 0); print(r / (time.perf_counter() - t0))"
                        % (ROOT, local, gz_path, gz_path))
                res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                                     env=dict(os.environ, FRB_GZ_DEVICE="0"))
                if res.returncode == 0:
                    e2e["host_zlib_reads_per_s"] = float(res.stdout.strip().splitlines()[-1])

        # ---- round 1's leg: decompressed text in pinned host memory -> H2D -> kernels -> D2H, and what the
        #      link alone does (one pinned cudaMemcpy of the same bytes) -----------------------------------
        k = max(1, sum(1 for b in bounds[1:] if b <= E2E_MAX_BYTES))
        e_bytes = bounds[k]
        e_reads = min(k * GEN_CHUNK, reads)
        hbuf = C.c_void_p()
        ck(lib.frb_host_alloc(C.byref(hbuf), e_bytes))
        ck(lib.frb_d2h(h, hbuf, dbuf, e_bytes))
        d2h = [0]

        def step_host():
            ck(lib.frb_reset(h))
            ck(lib.frb_scan_begin(h, rank, 0))
            ck(lib.frb_scan_chunk_host(h, hbuf, e_bytes, 0, L.RULE_SCAN))
            n_reads, n_uniq = C.c_uint64(), C.c_uint64()
            ck(lib.frb_scan_end(h, C.byref(n_reads), C.byref(n_uniq)))
            if world > 1:
                ck(lib.frb_shardmerge(h, C.byref(n_uniq)))
            keys, counts, _ = ctx.total_arrays()
            out = analyze(True)
            d2h[0] = keys.nbytes + counts.nbytes + sum(v.nbytes for v in out.values())
            return n_reads.value

        _, p_wall, p_got = timed(step_host, 2, 1)
        assert p_got == e_reads, (p_got, e_reads)
        p_s = p_wall / 2
        scratch = C.c_void_p()
        ck(lib.frb_dev_alloc(h, e_bytes, C.byref(scratch)))
        ck(lib.frb_h2d(h, scratch, hbuf, e_bytes))
        t0 = time.perf_counter()
        ck(lib.frb_h2d(h, scratch, hbuf, e_bytes))
        link_s = time.perf_counter() - t0
        ck(lib.frb_dev_free(h, scratch))
        ck(lib.frb_host_free(hbuf))
        if dist:
            box = [None] * world
            dist.all_gather_object(box, (p_s, link_s))
            p_s, link_s = max(b[0] for b in box), max(b[1] for b in box)
        e2e_pcie = {"value": e_reads * world / p_s, "unit": "reads/s", "h2d_bytes_per_step": e_bytes,
                    "d2h_bytes_per_step": d2h[0], "h2d_gbs": e_bytes / p_s / 1e9,
                    "pinned_memcpy_gbs": e_bytes / link_s / 1e9, "pcie_frac": (e_bytes / p_s) / (e_bytes / link_s),
                    "sample": "host-pinned decompressed FASTQ (first %d reads of the lane) through "
                              "frb_scan_chunk_host; pcie_frac = its H2D rate / a plain pinned cudaMemcpy of the "
                              "same bytes on the same GPU at the same time on every rank" % e_reads}

    # ---- the result itself: conservation, disjoint shares, and the lane's first reads against the C oracle -----
    checked = None
    if not args.no_check:
        step_resident()
        keys, counts, first = ctx.total_arrays()
        total_reads = int(counts.sum())
        if dist:
            box = [None] * world
            dist.all_gather_object(box, (total_reads, keys))
            total_reads = sum(b[0] for b in box)
            allk = np.concatenate([b[1] for b in box])
            assert len(np.unique(allk)) == len(allk), "shares of the ranks overlap"
        assert total_reads == reads * world, (total_reads, reads * world)
        assert (np.diff(first.astype(np.int64)) > 0).all(), "total list is not in first-appearance order"
        checked = {"conservation": True, "shares_disjoint": True if dist else None}
        if rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import c_oracle
            from frender_b200.engine import reverse_complement, unpack_keys
            c_reads = min(CHECK_READS, reads)
            c_bytes = bounds[1] if GEN_CHUNK <= c_reads else None
            sub = np.empty(int(c_reads * 376), np.uint8)
            n_sub, tmpbuf = C.c_uint64(), C.c_void_p()
            ck(lib.frb_dev_alloc(h, sub.size, C.byref(tmpbuf)))
            ck(lib.frb_synth_generate(h, g_base, g_base + c_reads, 1, tmpbuf, sub.size, C.byref(n_sub)))
            ck(lib.frb_d2h(h, vp(sub), tmpbuf, n_sub.value))
            cctx = Context(local, table_log2=21)
            ck2 = cctx._ck
            ck2(lib.frb_scan_begin(cctx._h, 0, 0))
            ck2(lib.frb_scan_chunk_dev(cctx._h, tmpbuf, n_sub.value, 0, L.RULE_SCAN, None, None))
            r_, u_ = C.c_uint64(), C.c_uint64()
            ck2(lib.frb_scan_end(cctx._h, C.byref(r_), C.byref(u_)))
            want, want_reads = c_oracle.tally(sub[:n_sub.value].tobytes())
            k2, c2, _ = cctx.total_arrays()
            names = unpack_keys(k2)
            assert r_.value == want_reads == c_reads and names == list(want) and c2.tolist() == list(want.values()), \
                "tally of the lane's first reads differs from the C oracle"
            idx = spec.indexes()
            cctx.load_sheet(idx)
            res = cctx.match(N_SUBS, True)
            ref = np.array(c_oracle.classify_all_rc(names, idx, N_SUBS), np.int32)
            for col, name in enumerate(("m1", "m2", "type", "srow", "m2rc", "type_rc", "srow_rc")):
                assert (res[name].astype(np.int32) == ref[:, col]).all(), "first pass differs from the C oracle: " + name
            calls = c_oracle.rc_calls(names, c2.tolist(), ref.tolist(), idx)
            got_calls = cctx.rc_calls(res)
            assert {k: (v["call"], v["reads_f"], v["reads_rc"]) for k, v in got_calls.items()} == calls
            use = np.array([calls[name][0] for name in idx["id"]], np.uint8)
            oriented = dict(idx, idx2=[reverse_complement(b) if u else b for b, u in zip(idx["idx2"], use)])
            res2 = cctx.match(N_SUBS, False, use)
            ref2 = np.array(c_oracle.classify_all(names, oriented, N_SUBS), np.int32)
            for col, name in enumerate(("m1", "m2", "type", "srow")):
                assert (res2[name].astype(np.int32) == ref2[:, col]).all(), "second pass differs from the C oracle: " + name
            cctx.close()
            ck(lib.frb_dev_free(h, tmpbuf))
            checked["c_oracle"] = {"reads": c_reads, "unique_keys": len(names), "tally": True, "pass_rc": True,
                                   "orientation_calls": True, "pass_oriented": True}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = len(os.sched_getaffinity(0))
        ref = load_reference()
        with tempfile.TemporaryDirectory() as d:
            cspec, path, cbytes = cpu_sample(d)
            total, t_tally, t_match, uniq = cpu_step(cspec, path, cores, ref)
        cpu = {"value": CPU_SAMPLE_READS / total, "unit": "reads/s", "cores": cores,
               "kind": "reference" if ref is not None else "port",
               "sample": f"the first {CPU_SAMPLE_READS} reads of the same lane from one .fastq.gz: inflate+tally "
                         f"{t_tally:.2f}s (1 core, one file) + matcher both passes {t_match:.2f}s on {cores} cores"}

    if rank == 0:
        line = {
            "metric": "read_names_per_s_scanned_matched", "value": value, "unit": "reads/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "u8/u64", "data": "synthetic (device-generated, "
            "counter-based; byte-identical to frender_b200/synth.py)",
            "config": workload_config(reads, world), "clocks": clk, "e2e": e2e, "e2e_pcie": e2e_pcie,
            "checked": checked,
            "gpu_launches": launches,
            "roofline": roofline, "cpu_baseline": cpu,
            "unique_keys": n_uniq.value, "input_bytes_per_gpu": nbytes, "gen_s": t_gen,
            "kernel_only_reads_per_s_per_gpu": reads / (scan_ms_per * 1e-3),
        }
    ck(lib.frb_dev_free(h, dbuf))
    ctx.close()
    if rank == 0:
        if world == 1 and not args.no_demux:
            # configs[3] beside the headline: the record router as a stream (python bench.py --workload demux is
            # the full line for it, with the reference's demux timed beside)
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from bench_demux import measure
            line["demux"] = measure(local, DEMUX_PAIRS, 64, 2, 1)
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


def main():
    # stdout carries the one JSON line: NCCL's version/warning banner (NCCL_DEBUG=VERSION|WARN in some
    # environments) goes to stderr, or away
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        del os.environ["NCCL_DEBUG"]
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    args = parse_args()
    if args.workload == "demux":
        run_demux(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
