"""BGZF written on the device, against the gzip members of FRENDER_GZIP_LEVEL=gpu.
usage: bench_bgzf.py [out.json] [demux pairs] [encoder GB] [parent tree]

Encoder alone: the inputs of bench_gz_deflate.py -- a synthetic C2 lane with all-'F' qualities and with qualities
binned 85/10/4/1 %, >= `encoder GB` (default 2) per style in 256 MiB calls, far above the 126 MB L2.  Per style, one
warm-up call of each format, then gzip (frb_gz_deflate) and BGZF (frb_gz_deflate_bgzf) calls alternated; device time
of the FRB_K_DEFLATE kernels of each (CUDA events).  Output size of each format beside zlib level 1 on the whole call.

Read-back: the two outputs of the last call written to files and inflated on the device (frb_gz_inflate); the
FRB_K_INFLATE kernel time after one warm-up, and whether the device path took the file.

`frender demux` of a C4-shaped lane pair (default 4 M pairs, input at zlib level 1): FRENDER_GZIP_LEVEL=gpu and =bgzf
alternated twice in this one process; pairs/s, output bytes, and whether the decompressed sinks are identical.

Gzip-mode check (with a parent tree built beside this one): sha256 of frb_gz_deflate's output for the two lane styles
and of the sinks of a FRENDER_GZIP_LEVEL=gpu demux of the same files, computed by the parent's library and by this
one on the same seeded input."""
import csv
import gzip
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib
from argparse import Namespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from frender_b200 import _lib, bgzf, synth  # noqa: E402
from frender_b200.cli import frender_demux, frender_scan  # noqa: E402
from frender_b200.engine import Context  # noqa: E402

out_json = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else "bgzf.json")
pairs = int(sys.argv[2]) if len(sys.argv) > 2 else 4_000_000
enc_gb = float(sys.argv[3]) if len(sys.argv) > 3 else 2.0
parent = os.path.abspath(sys.argv[4]) if len(sys.argv) > 4 else None
CALL = 256 << 20

# sha256 of gzip-mode outputs with the package of the tree argv[1]: frb_gz_deflate of the lane files argv[2:4],
# then the sinks of `frender demux` (FRENDER_GZIP_LEVEL=gpu) of argv[4], argv[5] with results argv[6] into argv[7]
GZIP_DIGESTS = r"""
import hashlib, json, os, sys
from argparse import Namespace
sys.path.insert(0, sys.argv[1])
from frender_b200.cli import frender_demux
from frender_b200.engine import Context
out = {}
ctx = Context(0, table_log2=12)
for path in sys.argv[2:4]:
    out[os.path.basename(path)] = hashlib.sha256(ctx.gz_deflate(open(path, "rb").read())).hexdigest()
ctx.close()
os.environ["FRENDER_GZIP_LEVEL"] = "gpu"
frender_demux(Namespace(r=sys.argv[6], d=sys.argv[7], o=None, no_index_hop=False, no_ambiguous=False,
                        no_undeter=False, no_samples=False, files=[sys.argv[4], sys.argv[5]]))
h = hashlib.sha256()
for n in sorted(os.listdir(sys.argv[7])):
    h.update(n.encode())
    h.update(hashlib.sha256(open(os.path.join(sys.argv[7], n), "rb").read()).digest())
out["demux_gpu_sinks"] = h.hexdigest()
print("DIGESTS " + json.dumps(out))
"""


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def lane(style, n_bytes):
    spec = synth.make_spec("C2")
    parts, size, g = [], 0, 0
    while size < n_bytes:
        d = synth.generate(spec, g, g + 200_000)
        parts.append(synth.binned_qualities(d, g) if style == "binned" else d)
        size += len(parts[-1])
        g += 200_000
    return b"".join(parts)[:n_bytes]


def sinks_digest(out, decompress):
    h = hashlib.sha256()
    for n in sorted(os.listdir(out)):
        h.update(n.encode())
        raw = open(os.path.join(out, n), "rb").read()
        h.update(hashlib.sha256(gzip.decompress(raw) if decompress else raw).digest())
    return h.hexdigest()


result = {"card": card(), "tool": "tools/bench_bgzf.py", "encoder": {}, "read_back": {}, "demux": {},
          "gzip_mode_check": {}}
print("card, power limit:", result["card"], flush=True)
work = tempfile.mkdtemp(prefix="bench_bgzf_")
FORMATS = {"gpu": False, "bgzf": True}   # FRENDER_GZIP_LEVEL name -> gz_deflate(bgzf=)
try:
    # ---- encoder alone, and read-back ----------------------------------------------------------------------------
    ctx = Context(0, table_log2=12)
    lane_files = []
    for style in ("allF", "binned"):
        data = lane(style, CALL)
        lane_files.append(os.path.join(work, f"lane_{style}.fastq"))
        with open(lane_files[-1], "wb") as fh:
            fh.write(data)
        z1 = len(zlib.compress(data, 1))
        for b in FORMATS.values():
            ctx.gz_deflate(data, bgzf=b)  # warm-up: module load, buffers
        calls = max(1, int(enc_gb * (1 << 30) / CALL + 0.999))
        ms = {f: 0.0 for f in FORMATS}
        outs = {f: set() for f in FORMATS}
        last = {}
        ctx.prof(True)
        ctx.prof_read(_lib.K_DEFLATE)
        for _ in range(calls):
            for f, b in FORMATS.items():
                last[f] = ctx.gz_deflate(data, bgzf=b)
                ms[f] += ctx.prof_read(_lib.K_DEFLATE)[0]
                outs[f].add(hashlib.sha256(last[f]).hexdigest())
        ctx.prof(False)
        assert zlib.decompress(last["gpu"], 31) == data and gzip.decompress(last["bgzf"]) == data
        blocks = list(bgzf.iter_blocks(last["bgzf"]))
        total = calls * len(data)
        r = {"input_bytes_per_format": total, "calls_per_format": calls, "call_bytes": len(data),
             "zlib1_bytes": z1, "bgzf_blocks": len(blocks) - 1, "max_block_bytes": max(b + 1 for _, b, _ in blocks)}
        for f in FORMATS:
            r[f] = {"kernel_ms": round(ms[f], 3), "encoder_GBps": round(total / (ms[f] * 1e-3) / 1e9, 2),
                    "output_bytes": len(last[f]), "ratio": round(len(data) / len(last[f]), 3),
                    "size_vs_zlib1": round(len(last[f]) / z1, 4), "identical_output_every_call": len(outs[f]) == 1}
        r["bgzf_size_vs_gpu"] = round(len(last["bgzf"]) / len(last["gpu"]), 4)
        result["encoder"][style] = r
        print("encoder", style, json.dumps(r), flush=True)
        # read-back on the device
        rb = {}
        for f, z in last.items():
            path = os.path.join(work, f"{style}_{f}.fastq.gz")
            with open(path, "wb") as fh:
                fh.write(z)
            got = ctx.gz_inflate(path, len(data) + 1)  # warm-up
            ctx.prof(True)
            ctx.prof_read(_lib.K_INFLATE)
            t0 = time.perf_counter()
            got = ctx.gz_inflate(path, len(data) + 1)
            wall = time.perf_counter() - t0
            kms = ctx.prof_read(_lib.K_INFLATE)[0]
            ctx.prof(False)
            rb[f] = {"device_path_taken": got is not None, "text_equal": got == data, "compressed_bytes": len(z),
                     "kernel_ms": round(kms, 3), "inflate_GBps_text": round(len(data) / (kms * 1e-3) / 1e9, 2) if kms else None,
                     "call_wall_GBps_text": round(len(data) / wall / 1e9, 2)}
            os.remove(path)
        result["read_back"][style] = rb
        print("read_back", style, json.dumps(rb), flush=True)
        del data, last
    ctx.close()

    # ---- frender demux end to end ----------------------------------------------------------------------------------
    spec = synth.make_spec("C4")
    r1, r2 = os.path.join(work, "L_R1_001.fastq.gz"), os.path.join(work, "L_R2_001.fastq.gz")
    for path, mate in ((r1, 1), (r2, 2)):
        z = zlib.compressobj(1, zlib.DEFLATED, 31)
        with open(path, "wb") as fh:
            for o in range(0, pairs, 200_000):
                fh.write(z.compress(synth.generate(spec, o, min(o + 200_000, pairs), read_no=mate)))
            fh.write(z.flush())
    os.chdir(work)
    with open("SampleSheet.csv", "w") as fh:
        fh.write(spec.sheet_csv())
    frender_scan(Namespace(n=1, rc=True, c=1, s=None, o="res", p=None, b="SampleSheet.csv", files=[r1]))
    rows = list(csv.reader(open([f for f in os.listdir(work) if f.startswith("frender-scan-results_")][0], newline="")))
    order = [rows[0].index(c) for c in ("idx1", "idx2", "reads", "matched_idx1", "matched_idx2", "read_type",
                                        "sample_name", "demux_ok")]
    results_csv = os.path.join(work, "results.csv")
    with open(results_csv, "w", newline="") as fh:
        csv.writer(fh).writerows([[r[i] for i in order] for r in rows])
    runs = {arm: [] for arm in FORMATS}
    digests, raw_gpu = {}, None
    for rep in range(2):
        for arm in runs:
            out = os.path.join(work, f"out_{arm}_{rep}")
            os.environ["FRENDER_GZIP_LEVEL"] = arm
            t0 = time.perf_counter()
            frender_demux(Namespace(r=results_csv, d=out, o=None, no_index_hop=False, no_ambiguous=False,
                                    no_undeter=False, no_samples=False, files=[r1, r2]))
            dt = time.perf_counter() - t0
            names = sorted(os.listdir(out))
            runs[arm].append({"s": round(dt, 3), "pairs_per_s": round(pairs / dt, 1),
                              "output_bytes": sum(os.path.getsize(os.path.join(out, n)) for n in names),
                              "files": len(names)})
            print("demux", arm, runs[arm][-1], flush=True)
            if rep == 0:
                digests[arm] = sinks_digest(out, True)
                if arm == "bgzf":
                    for n in names:
                        bb = open(os.path.join(out, n), "rb").read()
                        assert bb.endswith(bgzf.EOF_BLOCK) and sum(1 for _ in bgzf.iter_blocks(bb)) >= 1
                else:
                    raw_gpu = sinks_digest(out, False)
            shutil.rmtree(out)
    os.environ.pop("FRENDER_GZIP_LEVEL", None)
    result["demux"] = {
        "pairs": pairs, "shape": "C4", "input": "zlib level 1", "host_threads": len(os.sched_getaffinity(0)),
        "arms": {f"FRENDER_GZIP_LEVEL={a}": v for a, v in runs.items()},
        "decompressed_sinks_identical_across_arms": digests["gpu"] == digests["bgzf"],
    }
    print(json.dumps(result["demux"]), flush=True)

    # ---- gzip mode: the parent's library and this one on the same input --------------------------------------------
    if parent:
        for name, tree in (("parent", parent), ("this", ROOT)):
            out = os.path.join(work, f"digest_{name}")
            p = subprocess.run([sys.executable, "-c", GZIP_DIGESTS, tree, *lane_files, r1, r2, results_csv, out],
                               capture_output=True, text=True, cwd=work)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("DIGESTS ")]
            result["gzip_mode_check"][name] = (json.loads(line[-1][8:]) if line and not p.returncode
                                               else {"error": (p.stderr or p.stdout)[-2000:]})
            shutil.rmtree(out, ignore_errors=True)
        this_run = result["gzip_mode_check"]["this"]
        result["gzip_mode_check"]["equal"] = result["gzip_mode_check"]["parent"] == this_run and "error" not in this_run
        result["gzip_mode_check"]["demux_gpu_sinks_of_the_timed_run"] = raw_gpu
        print(json.dumps(result["gzip_mode_check"]), flush=True)
finally:
    os.chdir(ROOT)
    shutil.rmtree(work, ignore_errors=True)

os.makedirs(os.path.dirname(out_json), exist_ok=True)
with open(out_json, "w") as fh:
    json.dump(result, fh, indent=1)
print("wrote", out_json)
