"""`frender demux` with the mates inflated on the device against zlib on the host.
usage: bench_demux_gz.py [out.json] [pairs (0: no demux runs)] [parent tree]

Lane: a C4-shaped lane pair of `pairs` pairs (default 4 M), written once with zlib level 1 and once with level 6.
Arms: FRB_GZ_DEVICE in {0, 1} x FRENDER_GZIP_LEVEL in {1, gpu}, the four arms alternated twice within this one process
for each input level.  Per run: wall time and pairs/s, and the FRB_K_INFLATE / FRB_K_ROUTE / FRB_K_DEFLATE kernel time
of the profiled context passed to frender_demux (CUDA events around every kernel class).  The sink files of the two
FRB_GZ_DEVICE arms are compared byte for byte.

Regression check: `bench.py --gpus 1` (scan `value` and `e2e`) of this tree and of a parent tree built beside it
(third argument), alternated twice."""
import csv
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
from frender_b200 import _lib, synth  # noqa: E402
from frender_b200.cli import frender_demux, frender_scan  # noqa: E402
from frender_b200.engine import Context  # noqa: E402

out_json = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else "demux_gz.json")
pairs = int(sys.argv[2]) if len(sys.argv) > 2 else 4_000_000
parent = os.path.abspath(sys.argv[3]) if len(sys.argv) > 3 else None


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


result = {"card": card(), "tool": "tools/bench_demux_gz.py", "pairs": pairs, "shape": "C4",
          "host_threads": len(os.sched_getaffinity(0)), "demux": {}, "bench_py": {}}
print("card, power limit:", result["card"], flush=True)
spec = synth.make_spec("C4")


def gz_write(path, mate, level):
    z = zlib.compressobj(level, zlib.DEFLATED, 31)
    with open(path, "wb") as fh:
        for o in range(0, pairs, 200_000):
            fh.write(z.compress(synth.generate(spec, o, min(o + 200_000, pairs), read_no=mate)))
        fh.write(z.flush())


def sinks_digest(out):
    h = hashlib.sha256()
    for n in sorted(os.listdir(out)):
        h.update(n.encode())
        with open(os.path.join(out, n), "rb") as fh:
            h.update(hashlib.sha256(fh.read()).digest())
    return h.hexdigest()


ARMS = [("0", "1"), ("1", "1"), ("0", "gpu"), ("1", "gpu")]   # (FRB_GZ_DEVICE, FRENDER_GZIP_LEVEL)
CLASSES = {"inflate": _lib.K_INFLATE, "route": _lib.K_ROUTE, "deflate": _lib.K_DEFLATE}
if pairs:                                                      # pairs = 0: the bench.py comparison only
    with tempfile.TemporaryDirectory() as d:
        os.chdir(d)
        with open("SampleSheet.csv", "w") as fh:
            fh.write(spec.sheet_csv())
        ctx = Context(0, table_log2=12)
        for in_level in (1, 6):
            r1, r2 = os.path.join(d, f"L{in_level}_R1_001.fastq.gz"), os.path.join(d, f"L{in_level}_R2_001.fastq.gz")
            gz_write(r1, 1, in_level)
            gz_write(r2, 2, in_level)
            if in_level == 1:
                frender_scan(Namespace(n=1, rc=True, c=1, s=None, o="res", p=None, b="SampleSheet.csv", files=[r1]))
                rows = list(csv.reader(open([f for f in os.listdir(d) if f.startswith("frender-scan-results_")][0],
                                            newline="")))
                order = [rows[0].index(c) for c in ("idx1", "idx2", "reads", "matched_idx1", "matched_idx2", "read_type",
                                                    "sample_name", "demux_ok")]
                with open("results.csv", "w", newline="") as fh:
                    csv.writer(fh).writerows([[r[i] for i in order] for r in rows])
            runs = {a: [] for a in ARMS}
            digests = {}
            for rep in range(2):
                for arm in ARMS:
                    os.environ["FRB_GZ_DEVICE"], os.environ["FRENDER_GZIP_LEVEL"] = arm
                    out = os.path.join(d, f"out_{in_level}_{arm[0]}_{arm[1]}_{rep}")
                    ctx.prof(True)
                    for k in CLASSES.values():
                        ctx.prof_read(k)
                    t0 = time.perf_counter()
                    frender_demux(Namespace(r="results.csv", d=out, o=None, no_index_hop=False, no_ambiguous=False,
                                            no_undeter=False, no_samples=False, files=[r1, r2]), ctx=ctx)
                    dt = time.perf_counter() - t0
                    kms = {name: round(ctx.prof_read(k)[0], 2) for name, k in CLASSES.items()}
                    ctx.prof(False)
                    run = {"s": round(dt, 3), "pairs_per_s": round(pairs / dt, 1), "kernel_ms": kms,
                           "output_bytes": sum(os.path.getsize(os.path.join(out, n)) for n in os.listdir(out))}
                    runs[arm].append(run)
                    print(in_level, arm, run, flush=True)
                    if rep == 0:
                        digests[arm] = sinks_digest(out)
                    shutil.rmtree(out)
            result["demux"][f"input_zlib_level_{in_level}"] = {
                "input_bytes": os.path.getsize(r1) + os.path.getsize(r2),
                "arms": {f"FRB_GZ_DEVICE={a[0]},FRENDER_GZIP_LEVEL={a[1]}": v for a, v in runs.items()},
                "sinks_byte_identical_across_FRB_GZ_DEVICE": {
                    lvl: digests[("0", lvl)] == digests[("1", lvl)] for lvl in ("1", "gpu")},
            }
            os.remove(r1)
            os.remove(r2)
        ctx.close()
        os.environ.pop("FRB_GZ_DEVICE", None)
        os.environ.pop("FRENDER_GZIP_LEVEL", None)

# ---- bench.py of this tree against the parent tree -------------------------------------------------------------------
if parent:
    trees = {"this": ROOT, "parent": parent}
    for rep in range(2):
        for name, tree in trees.items():
            p = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", "5",
                                "--warmup", "2", "--no-cpu", "--no-demux"], capture_output=True, text=True, cwd=tree)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
            if p.returncode or not line:
                result["bench_py"].setdefault(name, []).append({"error": (p.stderr or p.stdout)[-2000:]})
                continue
            j = json.loads(line[-1])
            row = {"value": j.get("value"), "e2e": (j.get("e2e") or {}).get("value")}
            result["bench_py"].setdefault(name, []).append(row)
            print("bench.py", name, row, flush=True)

os.makedirs(os.path.dirname(out_json), exist_ok=True)
with open(out_json, "w") as fh:
    json.dump(result, fh, indent=1)
print("wrote", out_json)
