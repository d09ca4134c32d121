"""The device gzip writer, alone and inside `frender demux`.
usage: bench_gz_deflate.py [out.json] [demux pairs] [encoder GB]

Encoder alone: frb_gz_deflate over a synthetic C2 lane (all-'F' qualities as synth.py writes them, and qualities
binned 85/10/4/1 %), device time of the FRB_K_DEFLATE kernels (CUDA events) after one warm-up call, on >= 2 GB of
input per lane style in 256 MiB calls (the working set is far above the 126 MB L2).  Ratio beside zlib levels 1 and 6
on the first 32 MiB of the same bytes.

`demux` end to end: FRENDER_GZIP_LEVEL=6, =1 and =gpu on a C4-shaped lane pair, the three arms alternated twice
within this one process; pairs/s, output bytes, and whether the decompressed sinks are identical across the arms."""
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

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from frender_b200 import _lib, synth  # noqa: E402
from frender_b200.cli import frender_demux, frender_scan  # noqa: E402
from frender_b200.engine import Context  # noqa: E402

out_json = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else "gz_deflate.json")
pairs = int(sys.argv[2]) if len(sys.argv) > 2 else 4_000_000
enc_gb = float(sys.argv[3]) if len(sys.argv) > 3 else 2.0
CALL = 256 << 20


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


result = {"card": card(), "tool": "tools/bench_gz_deflate.py", "encoder": {}, "demux": {}}
print("card, power limit:", result["card"], flush=True)

# ---- encoder alone ---------------------------------------------------------------------------------------------------
ctx = Context(0, table_log2=12)
for style in ("allF", "binned"):
    data = lane(style, CALL)
    sample = data[:32 << 20]
    z1, z6 = len(zlib.compress(sample, 1)), len(zlib.compress(sample, 6))
    ctx.gz_deflate(data)  # warm-up: module load, buffers
    ctx.prof(True)
    ctx.prof_read(_lib.K_DEFLATE)
    calls = max(1, int(enc_gb * (1 << 30) / CALL + 0.999))
    t0 = time.perf_counter()
    outs = set()
    for _ in range(calls):
        z = ctx.gz_deflate(data)
        outs.add(hashlib.sha256(z).hexdigest())
    wall = time.perf_counter() - t0
    ms, launches = ctx.prof_read(_lib.K_DEFLATE)
    ctx.prof(False)
    zs = ctx.gz_deflate(sample)
    assert zlib.decompress(z, 31) == data and zlib.decompress(zs, 31) == sample
    total = calls * len(data)
    r = {
        "input_bytes": total, "calls": calls, "call_bytes": len(data),
        "kernel_ms": round(ms, 3), "kernel_launches": launches,
        "encoder_GBps": round(total / (ms * 1e-3) / 1e9, 2),
        "call_wall_GBps_incl_pcie": round(total / wall / 1e9, 2),
        "identical_output_every_call": len(outs) == 1,
        "ratio_device": round(len(data) / len(z), 3),
        "ratio_device_32MiB": round(len(sample) / len(zs), 3),
        "ratio_zlib1_32MiB": round(len(sample) / z1, 3),
        "ratio_zlib6_32MiB": round(len(sample) / z6, 3),
        "size_vs_zlib1": round(len(zs) / z1, 3),
    }
    result["encoder"][style] = r
    print(style, json.dumps(r), flush=True)
ctx.close()

# ---- frender demux end to end --------------------------------------------------------------------------------------
spec = synth.make_spec("C4")


def gz_write(path, mate):
    z = zlib.compressobj(1, zlib.DEFLATED, 31)
    with open(path, "wb") as fh:
        for o in range(0, pairs, 200_000):
            fh.write(z.compress(synth.generate(spec, o, min(o + 200_000, pairs), read_no=mate)))
        fh.write(z.flush())


with tempfile.TemporaryDirectory() as d:
    os.chdir(d)
    r1, r2 = os.path.join(d, "L_R1_001.fastq.gz"), os.path.join(d, "L_R2_001.fastq.gz")
    gz_write(r1, 1)
    gz_write(r2, 2)
    with open("SampleSheet.csv", "w") as fh:
        fh.write(spec.sheet_csv())
    frender_scan(Namespace(n=1, rc=True, c=1, s=None, o="res", p=None, b="SampleSheet.csv", files=[r1]))
    rows = list(csv.reader(open([f for f in os.listdir(d) if f.startswith("frender-scan-results_")][0], newline="")))
    order = [rows[0].index(c) for c in ("idx1", "idx2", "reads", "matched_idx1", "matched_idx2", "read_type",
                                        "sample_name", "demux_ok")]
    with open("results.csv", "w", newline="") as fh:
        csv.writer(fh).writerows([[r[i] for i in order] for r in rows])
    runs = {arm: [] for arm in ("6", "1", "gpu")}
    digests = {}
    for rep in range(2):
        for arm in runs:
            out = os.path.join(d, f"out_{arm}_{rep}")
            os.environ["FRENDER_GZIP_LEVEL"] = arm
            t0 = time.perf_counter()
            frender_demux(Namespace(r="results.csv", d=out, o=None, no_index_hop=False, no_ambiguous=False,
                                    no_undeter=False, no_samples=False, files=[r1, r2]))
            dt = time.perf_counter() - t0
            names = sorted(os.listdir(out))
            size = sum(os.path.getsize(os.path.join(out, n)) for n in names)
            runs[arm].append({"s": round(dt, 3), "pairs_per_s": round(pairs / dt, 1), "output_bytes": size,
                              "files": len(names)})
            print(arm, runs[arm][-1], flush=True)
            if rep == 0:
                h = hashlib.sha256()
                for n in names:
                    h.update(n.encode())
                    h.update(hashlib.sha256(gzip.open(os.path.join(out, n), "rb").read()).digest())
                digests[arm] = h.hexdigest()
            shutil.rmtree(out)
    result["demux"] = {
        "pairs": pairs, "shape": "C4", "host_threads": len(os.sched_getaffinity(0)),
        "arms": {f"FRENDER_GZIP_LEVEL={a}": v for a, v in runs.items()},
        "decompressed_sinks_identical_across_arms": len(set(digests.values())) == 1,
    }
    print(json.dumps(result["demux"]), flush=True)

os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
with open(out_json, "w") as fh:
    json.dump(result, fh, indent=1)
print("wrote", out_json)
