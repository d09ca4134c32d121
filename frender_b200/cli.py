"""Drop-in command line of frender (`frender.py scan ...`, `frender.py demux ...`).

Flags, sample-sheet parsing, file discovery, output names, the scan-results CSV layout, the
index-2-calls CSV, stdout messages and the per-sample fastq.gz outputs follow the reference
(/root/reference/frender.py, "F:").  The per-read and per-unique-key work (read-name parse,
unique-combination count, mismatch matching with reverse-complement orientation, record routing)
runs in the CUDA library; this module is the host shell around it.
"""
import argparse
import csv
import gzip
import os
import re
import zlib
from datetime import datetime, timezone
from math import floor
from pathlib import Path

import numpy as np

from . import _lib
from .engine import (Context, FrbError, MAX_SYMS as _MAX_SYMS, READ_TYPES, pack_keys, pack_keys2, reverse_complement,
                     unpack_keys)

STAMP = "%Y-%M-%d_%H%M_%Z"          # sic: minutes where the month should be (F:599, F:912)
MIN_CHUNK = 1 << 20                  # smallest demux window (bytes per mate)


# ---------------------------------------------------------------------------------------------
# host, cold: cores, sample sheet, file discovery (F:9-151, F:685-716)
# ---------------------------------------------------------------------------------------------
def get_cores(cores):
    """F:9-22.  The value now sizes host-side (de)compression helpers; the GPU does the rest."""
    assert cores >= 0, "Number of cores is negative... what does that mean?"
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count()
    if cores == 0:
        return avail
    if 0 < cores < 1:
        return max(floor(cores * avail), 1)
    return int(cores)


def find_barcode_file(directory):
    """Newest-sorting csv/txt whose path looks like a barcode table (F:25-49)."""
    directory = Path(directory)
    assert directory.is_dir(), "The specified directory does not exist"
    hits = [p for p in directory.rglob("**/*")
            if re.search("barcode.*association", str(p), re.I) or re.search("sample.*sheet", str(p), re.I)]
    hits = sorted((p for p in hits if re.search(r"\.csv$|\.txt$", str(p), re.I)), reverse=True)
    if not hits:
        raise SystemExit(
            "I couldn't find a barcode table in that directory. Please either specify one with the argment -b "
            "or specify a directory including a barcode table. File names matching '.*barcode.*association.*' "
            "or '.*sample.*sheet.*' (case insensitive) are accepted.")
    print(f"Found barcode association file {os.path.basename(hits[0])}")
    return hits[0]


def get_indexes(barcode_file):
    """{"id", "idx1", "idx2"} column lists of the sample sheet (F:52-116): an Illumina
    [Header]..[Data] preamble is skipped, columns are found by regex on the header row.
    Extension: a sheet without an index2 column yields idx2 = None (single index)."""
    with open(barcode_file, "r") as handle:
        rows = csv.reader(handle)
        header = next(rows)
        if re.search(r"\[Header\]", header[0]):
            while not re.search(r"\[Data\]", next(rows)[0]):     # a blank row raises IndexError as in F:58
                pass
            header = next(rows)

        def col(pattern, veto=None):
            for i, name in enumerate(header):
                if re.search(pattern, name, re.I) and not (veto and re.search(veto, name, re.I)):
                    return i
            raise ValueError(
                f"""Couldn't find column matching "{pattern}"{' but not "' + veto + '"' if veto else ''} """
                f"in csv header {header}")

        try:
            c_id, c_1 = col("id|name"), col("index", "id|2")
        except ValueError as exc:
            print("Error finding columns in provided barcode file:")
            raise SystemExit(exc)
        try:
            c_2 = col("index.*2")
        except ValueError as exc:
            if os.environ.get("FRENDER_SINGLE_INDEX"):
                c_2 = None
            else:
                print("Error finding columns in provided barcode file:")
                raise SystemExit(exc)
        out = {"id": [], "idx1": [], "idx2": [] if c_2 is not None else None}
        for row in rows:
            out["id"].append(row[c_id])
            out["idx1"].append(row[c_1])
            if c_2 is not None:
                out["idx2"].append(row[c_2])
        return out


def parse_files(file_dict, just_r1):
    """fastq.gz paths of a directory (optionally R1 only) or of an explicit list (F:119-151)."""
    kind = list(file_dict.keys())[0]
    paths = []
    if kind == "dir":
        print(f"Scanning {file_dict['dir']} for fastq files. "
              f"{'Using read 1 files only for speed...' if just_r1 else ''}")
        paths = [p for p in Path(file_dict["dir"]).rglob("**/*") if p.is_file()]
    elif kind == "file":
        given = file_dict["file"]
        paths = [Path(a) for a in given if Path(a).is_file()] if isinstance(given, list) else [given]
    keep = []
    for p in paths:
        if re.search(r"\.f[ast]*q\.gz$", str(p), re.I):
            keep.append(p)
        else:
            print(f"Ignoring non-fastq file {os.path.basename(p)}")
    if kind == "dir" and just_r1:
        keep = [p for p in keep if re.search("R1", os.path.basename(p), re.I)]
    return keep


def is_read_mate(a, b):
    """F:685-693: names differ in exactly one character and carry _R1_ / _R2_."""
    if sum(1 for x, y in zip(a, b) if x != y) != 1:
        return False
    r = {int(re.search("_R[12]_", s)[0].strip("_").replace("R", "")) for s in (a, b)}
    return r == {1, 2}


def get_paired_files(files):
    """[(R1, R2)] (F:696-716)."""
    pairs = []
    for r1 in (p for p in files if re.search("_R1_", str(p), re.I)):
        mates = [q for q in files if is_read_mate(str(r1), str(q))]
        if len(mates) > 1:
            raise SystemExit(f"Found more than one potential read 2 file for {r1}")
        if not mates:
            raise SystemExit(f"Couldn't find a read 2 file for {r1}")
        pairs.append((r1, mates[0]))
    return pairs


# ---------------------------------------------------------------------------------------------
# scan (F:567-642)
# ---------------------------------------------------------------------------------------------
class ScanTables:
    """Results of the tally as arrays: total list + per-file lists (dict semantics of
    barcode_counter: a repeated basename keeps its first position and the last file's counts)."""

    def __init__(self, names, total, per_file, keys_hi=None):
        self.keys, self.counts = total
        self.keys_hi = keys_hi          # upper words of a wide context's keys, else None
        self.names = list(names)
        slot = {}
        for i, name in enumerate(names):
            slot.setdefault(name, len(slot))
        self.file_names = list(slot)
        latest = {name: i for i, name in enumerate(names)}
        self.files = [per_file[latest[name]] for name in self.file_names]

    @classmethod
    def from_ctx(cls, ctx, names):
        keys, counts, _ = ctx.total_arrays()
        keys_hi = ctx.total_keys_hi() if ctx.wide else None
        return cls(names, (keys, counts), [ctx.file_arrays(i)[:2] for i in range(len(names))], keys_hi)


def _scan_worker(rank, n_ranks, device, ident, jobs, sample, table_log2, conn):
    """One process per GPU (FRENDER_GPUS > 1): scan this rank's files, report, and -- once the parent has heard
    from every rank that its scans went through -- merge the per-rank tables over NCCL and send the per-file
    lists (and, from rank 0, the merged total) to the parent.  A rank that fails never enters the collective,
    and neither does anybody else: the parent only says "go" when all ranks are ready for it."""
    try:
        ctx = Context(device, table_log2=table_log2)
        ctx.nccl_init(ident, rank, n_ranks)
        ctx.reset()
        out = []
        k = 0
        while k < len(jobs):                    # runs of small files as one stream, like the one-GPU path
            paths = [path for _, path in jobs]
            run = small_file_run(paths, k) if not sample else 1
            done = ctx.scan_gz_batch(paths[k:k + run], [o for o, _ in jobs[k:k + run]]) if run > 1 else None
            if done is None:
                done = [ctx.scan_gz(jobs[k][1], jobs[k][0], sample)[:2]]
            for j, (reads, uniq, *_) in enumerate(done):
                fk, fc, _ = ctx.file_arrays(k + j)
                out.append((jobs[k + j][0], reads, uniq, fk, fc))
            k += len(done)
        conn.send(("scanned", None, None))
        if not conn.recv():                     # another rank failed: no collective
            return
        ctx.allmerge()
        total = ctx.total_arrays()[:2] if rank == 0 else None
        conn.send(("ok", out, total))
        ctx.close()
    except BaseException as exc:            # forwarded: the parent re-raises
        try:
            conn.send(("error", repr(exc), None))
        except OSError:
            pass
    finally:
        conn.close()


def scan_files_concurrent(files, sample, streams, device, table_log2, main_ctx):
    """`-c N` on one GPU: N files are inflated and scanned at the same time, each on its own context
    (own tables, streams and zlib thread; ctypes releases the GIL), which is the reference's file-level
    pool (F:189-193) with the GPU behind it.  The per-file lists are folded into main_ctx's total on
    the device (F:199-203)."""
    import queue
    import threading
    jobs = queue.Queue()
    for item in enumerate(files):
        jobs.put(item)
    per_file, errors = {}, []

    def worker():
        try:
            ctx = Context(device, table_log2=table_log2)
            while True:
                try:
                    ordinal, path = jobs.get_nowait()
                except queue.Empty:
                    break
                ctx.reset()
                reads, uniq, _ = ctx.scan_gz(path, ordinal, sample)
                fk, fc, ff = ctx.file_arrays(0)
                per_file[ordinal] = (reads, uniq, fk, fc, ff)
            ctx.close()
        except BaseException as exc:
            errors.append(exc)

    # a stream that falls back to its zlib thread is bound by it (≈ 0.5 GB/s), so small staging buffers are enough
    # there and make the per-context set-up (pinned ring, device stages) cheap; streams that inflate on the device
    # size their buffers from the file (a few GB each for files of 128 MB and more -- hence at most 4 streams by
    # default: one device-inflated stream already does what twenty zlib threads do)
    had = os.environ.get("FRB_STAGE_MB")
    if had is None:
        os.environ["FRB_STAGE_MB"] = "16"
    threads = [threading.Thread(target=worker) for _ in range(streams)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if had is None:
        del os.environ["FRB_STAGE_MB"]
    if errors:
        raise errors[0]
    main_ctx.reset()
    for ordinal in range(len(files)):
        _, _, fk, fc, ff = per_file[ordinal]
        main_ctx.merge_list(fk, fc, ff + (np.uint64(ordinal) << np.uint64(40)))
    return per_file, main_ctx.total_arrays()[:2]


def scan_files_multi_gpu(files, sample, n_gpus, table_log2, worker=_scan_worker):
    """File-level sharding over n_gpus GPUs (SURVEY 8e): file i goes to rank i % n_gpus.  The parent listens to
    all ranks at once (and to their exit): the first failure, or a rank that dies, ends the job with that rank's
    error instead of leaving the others in a collective that can never complete."""
    import multiprocessing as mp
    from multiprocessing.connection import wait

    from .shard import assign
    mpc = mp.get_context("spawn")
    ident = Context.nccl_unique_id()
    jobs = list(enumerate(files))
    procs, pipes = [], []
    for rank in range(n_gpus):
        parent, child = mpc.Pipe(duplex=True)
        p = mpc.Process(target=worker, args=(rank, n_gpus, rank, ident, assign(jobs, rank, n_gpus), sample,
                                             table_log2, child))
        p.start()
        child.close()
        procs.append(p)
        pipes.append(parent)

    def stop_all(message):
        for conn in pipes:
            try:
                conn.send(False)
            except OSError:
                pass
        for p in procs:
            p.join(timeout=5)
            if p.is_alive():
                p.terminate()
        raise SystemExit(message)

    def collect(expect):
        """one message of kind `expect` from every rank"""
        got = {}
        while len(got) < n_gpus:
            pending = [r for r in range(n_gpus) if r not in got]
            ready = wait([pipes[r] for r in pending] + [procs[r].sentinel for r in pending])
            for r in pending:
                if pipes[r] in ready:
                    try:
                        status, payload, tot = pipes[r].recv()
                    except EOFError:
                        stop_all(f"GPU worker {r} exited without a result")
                    if status != expect:
                        stop_all(f"GPU worker {r} failed: {payload}")
                    got[r] = (payload, tot)
                elif procs[r].sentinel in ready and not pipes[r].poll():
                    stop_all(f"GPU worker {r} exited without a result")
        return got

    collect("scanned")
    for conn in pipes:
        conn.send(True)
    results = collect("ok")
    per_file, total = {}, None
    for rank in range(n_gpus):
        payload, tot = results[rank]
        for ordinal, reads, uniq, fk, fc in payload:
            per_file[ordinal] = (reads, uniq, fk, fc)
        if tot is not None:
            total = tot
    for p in procs:
        p.join()
    return per_file, total


def class_file_matrix(files, sheet_ids, prefix):
    """uint8 [(4 + sheet rows), files]: does the NAME of file f fit keys of class c (read type 0/1/3, or 4 + sample
    row for demuxable keys)?  The reference's own regexes (sample name as a pattern, F:521-550), evaluated once per
    class and file; 2 = the sample name is not a valid pattern."""
    fixed = {0: re.compile("undetermined", re.I), 1: re.compile("undetermined|index-hop", re.I),
             3: re.compile("undetermined|ambiguous", re.I)}
    match = np.zeros((4 + len(sheet_ids), len(files)), np.uint8)
    patterns = {}
    for f, fname in enumerate(files):
        for t, pat in fixed.items():
            match[t, f] = bool(pat.search(fname))
        for row, name in enumerate(sheet_ids):
            if name not in patterns:
                try:
                    patterns[name] = re.compile(name.removeprefix(prefix), re.I)
                except re.error:
                    patterns[name] = None                  # only an error if such a key really sits in a file
            pat = patterns[name]
            match[4 + row, f] = 2 if pat is None else bool(pat.search(fname))
    return match


def demux_ok_flags(ctx, tables, sheet_ids, prefix):
    """demux_ok per unique key and the set of files holding a key they should not (F:504-564): the class x file
    matrix from the host, the reduction over the unique keys of every file on the device (frb_demux_ok) against
    the last classification."""
    files = tables.file_names
    if not files:
        return np.ones(len(tables.keys), bool), set()
    if ctx.wide:
        # the context's own per-file lists, one per file scanned; a file whose basename a later file repeats is not
        # part of barcode_counter (F:205) and fits every class
        files = tables.names
        match = class_file_matrix(files, sheet_ids, prefix)
        last = {name: i for i, name in enumerate(files)}
        for i, name in enumerate(files):
            if last[name] != i:
                match[:, i] = 1
        ok, bad, err_row = ctx.demux_ok(match)
    else:
        ok, bad, err_row = ctx.demux_ok(class_file_matrix(files, sheet_ids, prefix), tables.files)
    if err_row is not None:
        re.compile(sheet_ids[err_row].removeprefix(prefix), re.I)   # raises what the reference's re.search raises
    return ok, {files[f] for f in np.flatnonzero(bad)}


def report_rc_call_info(rc_calls, indexes, out_csv_name):
    """stdout table + index-2-calls CSV (F:429-479)."""
    name = out_csv_name.replace("frender-scan-results_", "frender-index-2-calls_")
    print("Based on the barcodes in the supplied fastq file, the following index 2 sequences will be used\n"
          f"(also recorded in {name}):\n")
    print("Sample Name", "Supplied Index 2", "Reads supporting (forward)", "Reverse complement Index 2",
          "Reads supporting (rev comp)", "Final call", sep="\t")
    rows = []
    for sample, call in rc_calls.items():
        supplied = indexes["idx2"][indexes["id"].index(sample)]
        flipped = reverse_complement(supplied)
        print(sample, supplied, call["reads_f"], flipped, call["reads_rc"],
              "reverse complement" if call["call"] else "forward", sep="\t")
        rows.append([sample, supplied, call["reads_f"], flipped, call["reads_rc"],
                     "TRUE" if call["call"] else "FALSE"])
    with open(name, "w", newline="") as fh:
        w = csv.writer(fh)
        w.writerow(["sample_name", "supplied_index_2", "reads_supplied_index_2", "rc_index_2",
                    "reads_rc_index_2", "use_rc"])
        w.writerows(rows)


def initial_table_log2(files):
    """Slots of the unique-key tables for these inputs: FRENDER_TABLE_LOG2, or from the compressed size (about
    70 bytes of .fastq.gz per read; a lane's unique index pairs are a few percent of its reads; load <= 1/4)."""
    env = os.environ.get("FRENDER_TABLE_LOG2")
    if env:
        return int(env)
    biggest = max((os.path.getsize(str(f)) for f in files), default=0)
    total = sum(os.path.getsize(str(f)) for f in files)
    expected_unique = max(biggest, total // 2) // 70 // 12
    log2 = 16
    while (1 << log2) < 4 * expected_unique and log2 < 28:
        log2 += 1
    return log2


SMALL_FILE = 32 << 20           # a .fastq.gz below this keeps the GPU a tenth busy on its own
SMALL_RUN_BYTES = 96 << 20      # compressed bytes of one run (one piece of the device inflate)


def small_file_run(files, start):
    """How many files from files[start] on go through the device as one stream (1: the file on its own)."""
    total, n = 0, 0
    for path in files[start:start + 256]:
        size = os.path.getsize(str(path))
        if size >= SMALL_FILE or size < 18 or total + size > SMALL_RUN_BYTES:
            break
        total += size
        n += 1
    return max(n, 1)


def concurrent_streams(cores, files):
    """Files scanned at the same time on one GPU for `-c N` (one context per stream).  FRENDER_MAX_STREAMS
    overrides.  With host zlib (FRB_GZ_DEVICE=0) every stream is a zlib thread and N of them are N times as fast.
    With the inflate on the device one stream does what twenty zlib threads do on a large file, a second context
    only adds its buffers (a few GB), and runs of small files are inflated together as one stream
    (small_file_run): the files go one after the other."""
    n_files = len(files)
    env = os.environ.get("FRENDER_MAX_STREAMS")
    if env:
        return max(1, min(cores, n_files, int(env)))
    if os.environ.get("FRB_GZ_DEVICE", "1") == "0":
        return max(1, min(cores, n_files, 16))
    return 1


def tally_files(ctx, files, names, sample, cores, n_gpus):
    """tally_barcodes (F:183-207) over the three ways of spreading the files: ranks, `-c` streams, one by one."""
    if ctx.wide and (n_gpus > 1 or cores > 1):
        print("Index fields longer than 21 symbols: one GPU, one inflate stream "
              "(FRENDER_GPUS / -c over 128-bit keys are not supported yet).")
        return tally_files(ctx, files, names, sample, 1, 1)
    if n_gpus > 1:
        per_file, total = scan_files_multi_gpu(files, sample, n_gpus, ctx.table_log2)
        for ordinal, name in enumerate(names):
            reads, uniq = per_file[ordinal][:2]
            print(f"Tallying barcodes from {name}...found {uniq} new barcode{'' if uniq == 1 else 's'} "
                  f"in {reads} reads.")
        tables = ScanTables(names, total, [per_file[i][2:] for i in range(len(names))])
        ctx.load_total_arrays(*total)
    elif cores > 1 and len(files) > 1 and concurrent_streams(cores, files) > 1:
        streams = concurrent_streams(cores, files)
        per_file, total = scan_files_concurrent(files, sample, streams, ctx.device, ctx.table_log2, ctx)
        for ordinal, name in enumerate(names):
            reads, uniq = per_file[ordinal][:2]
            print(f"Tallying barcodes from {name}...found {uniq} new barcode{'' if uniq == 1 else 's'} "
                  f"in {reads} reads.")
        tables = ScanTables(names, total, [per_file[i][2:4] for i in range(len(names))])
    else:
        ordinal = 0
        while ordinal < len(files):
            # a run of small files goes through the device as ONE gzip stream of several members
            run = small_file_run(files, ordinal) if not sample else 1
            done = ctx.scan_gz_batch(files[ordinal:ordinal + run], ordinal) if run > 1 else None
            if done is None:
                done = [ctx.scan_gz(files[ordinal], ordinal, sample)[:2]]
            for k, (reads, uniq, *_) in enumerate(done):
                print(f"Tallying barcodes from {names[ordinal + k]}...found {uniq} new barcode{'' if uniq == 1 else 's'} "
                      f"in {reads} reads.")
            ordinal += len(done)
        tables = ScanTables.from_ctx(ctx, names)
    return tables


def frender_scan(args, ctx=None):
    num_subs, rc_mode = args.n, args.rc
    cores = get_cores(args.c)
    sample = args.s
    infix = args.o if args.o else ""
    prefix = args.p if args.p else ""
    if args.b is None:
        if len(args.files) != 1:
            raise SystemExit("You have not specified a barcode table. Please either specify one with the argment -b "
                             "or specify a directory including a barcode table")
        barcode_file = find_barcode_file(Path(args.files[0]))
    else:
        barcode_file = Path(args.b)
    indexes = get_indexes(barcode_file)

    if len(args.files) == 1:                                                    # F:587-601
        target = Path(args.files[0])
        if target.is_dir():
            files = {"dir": target}
            out_csv_name = f"frender-scan-results_{num_subs}-mismatches_{infix}_{target.parts[-1]}.csv"
        elif target.is_file():
            files = {"file": target}
            out_csv_name = f"frender-scan-results_{num_subs}-mismatches_{infix}_{target.name}.csv"
        else:
            raise SystemExit("Specified directory or file path doesn't seem to exist!")
    else:
        files = {"file": [Path(f) for f in args.files]}
        stamp = datetime.strftime(datetime.now(timezone.utc), STAMP)
        out_csv_name = f"frender-scan-results_{num_subs}-mismatches_{infix}_{stamp}.csv"
    out_csv_name = out_csv_name.replace("__", "_")
    files = parse_files(files, just_r1=True)

    own_ctx = ctx is None
    ctx = ctx or Context(int(os.environ.get("FRENDER_DEVICE", "0")), table_log2=initial_table_log2(files))
    try:
        # ---- tally (F:183-207) -----------------------------------------------------------------
        print(f"Scanning {len(files)} files on GPU {ctx.device} with {cores} inflate stream{'' if cores == 1 else 's'}...")
        if sample:
            assert sample >= 1, "Number of reads to sample must be ≥ 1!"
            print(f"Sampling {sample} reads from the head of each file...")
        names = [os.path.basename(str(path)) for path in files]
        n_gpus = min(int(os.environ.get("FRENDER_GPUS", "1")), max(len(files), 1))
        l1 = len(indexes["idx1"][0]) if len(indexes["idx1"]) else 0
        l2 = len(indexes["idx2"][0]) if indexes.get("idx2") is not None and len(indexes["idx2"]) else 0
        if l1 + (1 + l2 if l2 else 0) > _MAX_SYMS and not ctx.wide:
            ctx.set_wide()        # the sheet's own keys need 128-bit keys
        while True:
            # A dict never refuses a key (F:172-177): when the unique-key tables turn out too small for the
            # input they are re-created four times as large and the tally starts over.
            try:
                ctx.reset()
                tables = tally_files(ctx, files, names, sample, cores, n_gpus)
                break
            except (FrbError, SystemExit) as exc:
                # a GPU worker of a multi-GPU run reports its error as text (SystemExit)
                too_long = (isinstance(exc, FrbError) and exc.code == _lib.ERR_KEY_TOO_LONG) or (
                    isinstance(exc, SystemExit) and "index field longer than 21 symbols" in str(exc))
                if too_long and not ctx.wide:
                    print("\nindex fields longer than 21 symbols: tallying again with 128-bit keys")
                    ctx.set_wide()
                    continue
                full = (isinstance(exc, FrbError) and exc.code == _lib.ERR_TABLE_FULL) or "unique-key table full" in str(exc)
                if not full or ctx.table_log2 + 2 > 32:
                    raise
                print(f"\nunique-key tables of 2^{ctx.table_log2} slots are full: tallying again with "
                      f"2^{ctx.table_log2 + 2}")
                ctx.resize_tables(ctx.table_log2 + 2)
        print("Scanning complete! Analyzing barcodes...")

        # ---- matcher (F:610-630) ---------------------------------------------------------------
        sheet = ctx.load_sheet(indexes)
        if sheet.single and rc_mode:
            raise SystemExit("-rc needs a dual-index sample sheet")
        use = None
        idx2_used = sheet.idx2
        if rc_mode:
            first = ctx.match(num_subs, True, None, want_outputs=False)
            rc_calls = ctx.rc_calls(first)
            print("First round of analysis complete.")
            report_rc_call_info(rc_calls, indexes, out_csv_name)
            use = np.array([rc_calls[name]["call"] for name in sheet.ids], np.uint8)
            idx2_used = [b if u else a for a, b, u in zip(sheet.idx2, sheet.rc_idx2, use)]
            print("\nRe-analyzing barcodes with corrected index 2 sequences...")
        res = ctx.match(num_subs, False, use)

        # ---- demux_ok + CSV (F:632-642) --------------------------------------------------------
        ok, bad_files = demux_ok_flags(ctx, tables, sheet.ids, prefix)
        if bad_files:
            print("Incorrectly demultiplexed barcodes found! Affected files:")
            for f in sorted(bad_files):
                print(f)
        else:
            print("It appears that all files are already correctly demultiplexed.")
        print(f"Analysis complete! Writing results to {out_csv_name}")
        write_scan_csv(out_csv_name, tables, res, sheet, idx2_used, ok)
    finally:
        if own_ctx:
            ctx.close()
    return out_csv_name


def write_scan_csv(path, tables, res, sheet, idx2_used, ok):
    """idx1,idx2,matched_idx1,matched_idx2,read_type,sample_name,reads,demux_ok -- the layout the
    reference actually writes (dict insertion order, F:286-291, F:311, F:556; csv.DictWriter F:499).
    Formatted by the library (frb_write_scan_csv): a lane has ~10^7 unique keys."""
    import ctypes as C
    n = len(tables.keys)

    def strings(items):
        arr = (C.c_char_p * max(len(items), 1))()
        for i, item in enumerate(items):
            arr[i] = item.encode()
        return arr

    hi = None if tables.keys_hi is None else np.ascontiguousarray(tables.keys_hi, np.uint64)
    arrays = [np.ascontiguousarray(tables.keys, np.uint64), np.ascontiguousarray(tables.counts, np.uint64),
              np.ascontiguousarray(res["m1"], np.int32), np.ascontiguousarray(res["m2"], np.int32),
              np.ascontiguousarray(res["type"], np.uint8), np.ascontiguousarray(res["srow"], np.int32),
              np.ascontiguousarray(ok, np.uint8)]
    ptrs = [a.ctypes.data_as(C.c_void_p) for a in arrays]
    rc = _lib.lib.frb_write_scan_csv2(os.fsencode(str(path)), ptrs[0], None if hi is None else hi.ctypes.data_as(C.c_void_p),
                                      *ptrs[1:], n, strings(sheet.idx1), strings(idx2_used), strings(sheet.ids),
                                      len(sheet.ids), 1 if sheet.single else 0)
    _lib.check(None, rc)


# ---------------------------------------------------------------------------------------------
# demux (F:645-814)
# ---------------------------------------------------------------------------------------------
SCAN_LAYOUT = ["idx1", "idx2", "matched_idx1", "matched_idx2", "read_type", "sample_name", "reads", "demux_ok"]
DEMUX_LAYOUT = ["idx1", "idx2", "reads", "matched_idx1", "matched_idx2", "read_type", "sample_name"]


def parse_results_file(result_file):
    """{key: (read_type, sample_id)}.  The reference reads columns 0, 1, 5, 6 after asserting the readme's column
    order (F:649-664) -- an order its own `scan` does not write (SURVEY finding 1), so the reference's demux refuses
    the reference's scan output.  EXTENSION: the layout `scan` actually writes is accepted as well, by column
    name; every other header fails with the reference's assertion."""
    with open(result_file, newline="") as fh:
        rows = csv.reader(fh)
        header = next(rows)
        if header[0:8] == SCAN_LAYOUT:
            kind, sid = header.index("read_type"), header.index("sample_name")
            return {r[0] + "+" + r[1]: (r[kind], r[sid]) for r in rows}
        assert header[0:7] == DEMUX_LAYOUT, f"${result_file} does not appear to be a valid frender result file!"
        return {r[0] + "+" + r[1]: (r[5], r[6]) for r in rows}


class GzSink:
    """One output file: gzip member stream fed with raw record bytes."""

    def __init__(self, path, level):
        self.fh = open(path, "wb")
        self.z = zlib.compressobj(level, zlib.DEFLATED, 31)

    def write(self, data):
        if len(data):
            self.fh.write(self.z.compress(data))

    def close(self):
        self.fh.write(self.z.flush())
        self.fh.close()


class TextChunks:
    """Decompressed bytes of a fastq.gz with the newline translation of text mode (F:776), piece by piece."""

    def __init__(self, path):
        self.fh = gzip.open(path, "rb")
        self.eof = False
        self.held = b""            # a trailing "\r": the next byte decides whether it is half of "\r\n"

    def read(self, size):
        """About `size` bytes (all that is left at the end of the file, where self.eof turns True)."""
        piece = self.fh.read(max(size - len(self.held), 1))
        if not piece:
            self.eof = True
            out, self.held = self.held.replace(b"\r", b"\n"), b""
            return out
        if self.held or b"\r" in piece:
            piece = self.held + piece
            self.held = b""
            if piece.endswith(b"\r"):
                piece, self.held = piece[:-1], b"\r"
            piece = piece.replace(b"\r\n", b"\n").replace(b"\r", b"\n")
        return piece


def _demux_worker(rank, device, jobs, opts, out_dir, threads, conn):
    """One process per GPU: the file pairs `jobs` = [(ordinal, r1, r2)], each into its own part directory."""
    try:
        os.environ["FRENDER_DEVICE"] = str(device)
        os.environ["FRENDER_GPUS"] = "1"
        os.environ["FRENDER_DEMUX_THREADS"] = str(threads)
        ctx = Context(device, table_log2=12)
        try:
            for ordinal, r1, r2 in jobs:
                ns = argparse.Namespace(**opts, files=[str(r1), str(r2)], d=f"{out_dir}.part{ordinal}")
                frender_demux(ns, ctx=ctx)
        finally:
            ctx.close()
        conn.send(("ok", None))
    except SystemExit as exc:
        conn.send(("error", str(exc)))
    except BaseException as exc:
        conn.send(("error", repr(exc)))
    finally:
        conn.close()


def demux_pairs_multi_gpu(args, pairs, n_gpus, out_dir, worker=_demux_worker):
    """FRENDER_GPUS=N with several R1/R2 pairs (lanes): pair i is routed on GPU i % N into rank-local part files
    (SURVEY 8e: the demux outputs stay rank-local); the parts of every sink are then appended in pair order --
    gzip members one after the other, so every sink decompresses to exactly what the sequential loop over the
    pairs (F:774) writes."""
    import multiprocessing as mp
    import shutil
    from multiprocessing.connection import wait

    from .shard import assign
    mpc = mp.get_context("spawn")
    opts = {k: getattr(args, k) for k in ("no_index_hop", "no_ambiguous", "no_undeter", "no_samples", "o", "r")}
    jobs = [(i, r1, r2) for i, (r1, r2) in enumerate(pairs)]
    threads = max(2, len(os.sched_getaffinity(0)) // n_gpus)
    procs, pipes = [], []
    for rank in range(n_gpus):
        parent, child = mpc.Pipe(duplex=False)
        p = mpc.Process(target=worker, args=(rank, rank, assign(jobs, rank, n_gpus), opts, out_dir, threads, child))
        p.start()
        child.close()
        procs.append(p)
        pipes.append(parent)
    failure = None
    pending = set(range(n_gpus))
    while pending and failure is None:
        ready = wait([pipes[r] for r in pending] + [procs[r].sentinel for r in pending])
        for r in list(pending):
            if pipes[r] in ready or (procs[r].sentinel in ready and pipes[r].poll()):
                try:
                    status, payload = pipes[r].recv()
                except EOFError:
                    status, payload = "error", "exited without a result"
                if status != "ok":
                    failure = f"GPU worker {r} failed: {payload}"
                pending.discard(r)
            elif procs[r].sentinel in ready:
                failure = f"GPU worker {r} exited without a result"
                pending.discard(r)
    for p in procs:
        if failure is not None and p.is_alive():
            p.terminate()
        p.join()
    if failure is not None:
        raise SystemExit(failure)
    parts = [f"{out_dir}.part{i}" for i in range(len(pairs))]
    for name in sorted(os.listdir(parts[0])):
        with open(out_dir + name, "wb") as out:
            for part in parts:
                with open(os.path.join(part, name), "rb") as src:
                    shutil.copyfileobj(src, out, 1 << 22)
    for part in parts:
        shutil.rmtree(part)


def frender_demux(args, ctx=None):
    index_hop, ambiguous = not args.no_index_hop, not args.no_ambiguous
    undeter, samples = not args.no_undeter, not args.no_samples
    undeter_name = f"Undetermined{'-ambiguous' if ambiguous else ''}{'-index-hop' if index_hop else ''}"
    result_file = Path(args.r)
    if not result_file.is_file():
        raise SystemExit(f"File {result_file} not found")
    table = parse_results_file(result_file)
    ids = list(set(v[1] for v in table.values()) - {""})
    if (not ids) and samples:
        print("Warning: no demuxable sample ids found in the supplied frender result file!")

    if len(args.files) == 1:
        target = Path(args.files[0])
        if target.is_dir():
            files = {"dir": target}
        elif target.is_file():
            files = {"file": target}
        else:
            raise SystemExit("Specified directory or file path doesn't seem to exist!")
    else:
        files = {"file": [Path(f) for f in args.files]}
    pairs = get_paired_files(parse_files(files, just_r1=False))

    out_dir = args.d if args.d.endswith("/") else args.d + "/"
    os.mkdir(args.d)                                                            # FileExistsError as in F:755
    n_gpus = int(os.environ.get("FRENDER_GPUS", "1"))
    if ctx is None and n_gpus > 1 and len(pairs) > 1:
        return demux_pairs_multi_gpu(args, pairs, min(n_gpus, len(pairs)), out_dir)
    level = int(os.environ.get("FRENDER_GZIP_LEVEL", "6"))
    infix = args.o + "_" if args.o else ""
    sink_names = []                                                             # sink id -> name

    def open_sink(name):
        sink_names.append(name)
        return len(sink_names) - 1

    sample_sink = {sid: open_sink(sid) for sid in ids} if samples else {}
    undeter_sink = open_sink(undeter_name) if undeter else None
    hop_sink = open_sink("Index-hop") if index_hop else undeter_sink
    amb_sink = open_sink("Ambiguous") if ambiguous else undeter_sink
    sinks = [{r: GzSink(f"{out_dir}{name}_frender-demux_{infix}{r}.fq.gz", level) for r in ("R1", "R2")}
             for name in sink_names]
    n_sinks = len(sink_names)
    reject = n_sinks                                                            # "Unrecognized read type" bucket

    def route_of(kind, sid):                                                    # F:780-805
        if kind == "demuxable" and sample_sink:
            return sample_sink[sid]
        if kind == "index_hop" and hop_sink is not None:
            return hop_sink
        if kind == "ambiguous" and amb_sink is not None:
            return amb_sink
        if kind == "undetermined" and undeter_sink is not None:
            return undeter_sink
        return reject

    routes = np.array([route_of(*v) for v in table.values()], np.uint32)

    own_ctx = ctx is None
    ctx = ctx or Context(int(os.environ.get("FRENDER_DEVICE", "0")), table_log2=12)
    # keys longer than 21 symbols in the results table: the router takes 128-bit keys
    wide = any(len(k) > _MAX_SYMS for k in table)
    if wide != ctx.wide:
        ctx.set_wide(wide)
    keys, keys_hi = pack_keys2(list(table.keys())) if wide else (pack_keys(list(table.keys())), None)
    chunk = max(int(os.environ.get("FRENDER_DEMUX_CHUNK_MB", "64")) << 20, MIN_CHUNK)
    # Host side of the router: inflate of the two mates and deflate of the sinks run on a thread pool (zlib
    # releases the GIL).  Every sink sees the same sequence of compress() calls as a serial loop would make,
    # so the output files are byte-identical to it; the writes of chunk k overlap the inflate of chunk k+1.
    from concurrent.futures import ThreadPoolExecutor
    workers = max(2, int(os.environ.get("FRENDER_DEMUX_THREADS", str(len(os.sched_getaffinity(0))))))
    pool = ThreadPoolExecutor(max_workers=workers)
    writes = []

    def drain():
        for f in writes:
            f.result()
        writes.clear()

    def write_out(popped):
        o1, o2, off1, off2 = popped[:4]
        if off1[reject + 1] > off1[reject]:
            raise SystemExit("Unrecognized read type found in supplied frender result file!")
        drain()                                     # a sink's compress() calls stay in order
        for s in range(n_sinks):
            if off1[s + 1] > off1[s]:
                writes.append(pool.submit(sinks[s]["R1"].write, o1[off1[s]:off1[s + 1]]))
            if off2[s + 1] > off2[s]:
                writes.append(pool.submit(sinks[s]["R2"].write, o2[off2[s]:off2[s + 1]]))

    try:
        ctx.route_load(keys, routes, n_sinks + 1, keys_hi)
        for r1_path, r2_path in pairs:
            print(f"Demultiplexing {r1_path.name}...")
            # The pair as a STREAM of chunks, two in flight: while chunk k is routed on the device and chunk k-1
            # comes back and is deflated, chunk k+1 is inflated.  Chunks are cut anywhere; records that are not
            # complete yet (and the lead of one mate over the other) are carried on the device.
            a, b = TextChunks(r1_path), TextChunks(r2_path)
            ctx.route_reset(chunk)
            flags, carry, over = [], (0, 0), False
            while not over:
                want = [max(chunk - c, MIN_CHUNK // 4) for c in carry]   # carry + new bytes stay within the window
                fills = [pool.submit(a.read, 0 if a.eof else want[0]), pool.submit(b.read, 0 if b.eof else want[1])]
                da, db = (f.result() for f in fills)
                flags.append((1 if a.eof else 0) | (2 if b.eof else 0))
                ctx.route_push(da, db, flags[-1])
                over = a.eof and b.eof
                if len(flags) == 2:
                    popped, was = ctx.route_pop(), flags.pop(0)
                    write_out(popped)
                    carry = popped[5:7]
                    # zip() ends with the shorter mate (F:777): that file is over and nothing of it is left on
                    # the device (which ignores the chunk that is already queued behind this one)
                    over = over or bool(was & 1 and carry[0] == 0) or bool(was & 2 and carry[1] == 0)
            for _ in flags:
                write_out(ctx.route_pop())
    except FrbError as exc:
        if exc.code == _lib.ERR_KEY_NOT_FOUND:
            raise SystemExit(exc.message)
        raise
    finally:
        try:
            drain()
        finally:
            list(pool.map(lambda s: (s["R1"].close(), s["R2"].close()), sinks))
            pool.shutdown()
        if own_ctx:
            ctx.close()


# ---------------------------------------------------------------------------------------------
def build_parser():
    """The argparse surface of the reference, flag for flag (F:817-926)."""
    parser = argparse.ArgumentParser(prog="frender.py")
    sub = parser.add_subparsers()
    scan = sub.add_parser("scan", help="Scan file(s) or directory and compare to a supplied barcode table")
    scan.add_argument("-n", metavar="[int]", type=int, required=True,
                      help="REQUIRED: Number of mismatches allowed between supplied barcodes and fastq file(s)")
    scan.add_argument("-rc", action="store_true",
                      help="Scan/demultiplex using reverse complement of index 2 as well as forward sequence "
                           "(to check for mistakes with e.g. HiSeq 4000 and other systems)")
    scan.add_argument("-c", metavar="cores", type=float, default=1,
                      help="Number of cores to use for analysis, default = 1. Use 0 for all available, a number "
                           "between 0 and 1 for a fraction of all available cores, or a number >= 1 for a specified "
                           "number of cores")
    scan.add_argument("-s", metavar="sample", type=int,
                      help="If set, sample an absolute number of reads from the head of each file (s >= 1)")
    scan.add_argument("-o", metavar="output_name", help="name infix for output files")
    scan.add_argument("-p", metavar="fix_prefix",
                      help="When matching sample ids to filenames, remove this prefix from the sample id")
    scan.add_argument("-b", metavar="barcode_table",
                      help=".csv formatted file containing barcode associations with ids. REQUIRED unless you "
                           "specify a directory already containing such a file.")
    scan.add_argument("files", nargs="+",
                      help="Fastq file, list of fastq files, or directory path containing fastq files "
                           "(subdirectories will be searched as well)")
    scan.set_defaults(func=frender_scan)

    demux = sub.add_parser("demux", help="Demultiplex reads into sample and undetermined files according to "
                                         "supplied frender scan results file")
    demux.add_argument("-i", "--no-index-hop", action="store_true",
                       help="don't split index hop reads into their own file (will be included in undetermined "
                            "file unless -u is set)")
    demux.add_argument("-a", "--no-ambiguous", action="store_true",
                       help="don't split ambiguous reads into their own file (will be included in undetermined "
                            "file unless -u is set)")
    demux.add_argument("-u", "--no-undeter", action="store_true", help="do NOT produce undetermined files")
    demux.add_argument("-s", "--no-samples", action="store_true", help="do NOT produce individual sample files")
    demux.add_argument("-o", metavar="output_name", help="name infix for output files")
    demux.add_argument("-d", metavar="output_dir",
                       default=f"./frender-demux-output_{datetime.strftime(datetime.now(timezone.utc), STAMP)}/",
                       help="output directory (default: ./frender-demux-output_{date_time}/)")
    demux.add_argument("-r", metavar="result_file", required=True,
                       help="REQUIRED: frender scan result file (typically named "
                            "'frender-scan-result_n-mismatches_{output infix or file/directory name}.csv')")
    demux.add_argument("files", nargs="+",
                       help="Fastq file, list of fastq files, or directory path containing fastq files "
                            "(subdirectories will be searched as well)")
    demux.set_defaults(func=frender_demux)
    return parser


def main(argv=None):
    args = build_parser().parse_args(argv)
    args.func(args)
