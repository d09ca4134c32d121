"""Multi-rank paths.  CPU: the rank-count invariance of the merge on gloo, world size 2 (host logic
only, oracle tallies stand in for the device tables).  GPU: NCCL merge against the oracle when the
box has >= 2 GPUs (tests/mgpu_check.py under torchrun)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "oracle"))
import torch.distributed as dist
import frender_oracle as O
from frender_b200 import synth
from frender_b200.shard import assign, merge_lists
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
spec = synth.make_spec("C1", n_samples=12)
chunks = [(i, i * 500, (i + 1) * 500) for i in range(7)]            # (ordinal, g0, g1): 7 chunks, 2 ranks
mine = assign(chunks, rank, world)
local = []
for ordinal, g0, g1 in mine:
    counter, _ = O.tally_text(synth.generate(spec, g0, g1).decode().splitlines(keepends=True))
    firsts = {{}}
    for pos, key in enumerate(synth.keys_of(spec, g0, g1)):
        firsts.setdefault(key, (ordinal << 40) | pos)
    local.append([(k, n, firsts[k]) for k, n in counter.items()])
gathered = [None] * world
dist.all_gather_object(gathered, local)
merged = merge_lists([lst for per_rank in gathered for lst in per_rank])
want, _ = O.tally_text(synth.generate(spec, 0, 3500).decode().splitlines(keepends=True))
assert list(merged.items()) == list(want.items()), "merged tally differs from the single-process oracle"
dist.barrier()
dist.destroy_process_group()
'''


def test_merge_is_rank_count_invariant_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]


SHARD_WORKER = r'''
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "oracle"))
import numpy as np
import torch.distributed as dist
import frender_oracle as O
from frender_b200 import synth
from frender_b200.engine import pack_keys
from frender_b200.shard import assign, fold_share, key_owner, merge_lists, shard_lists
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
spec = synth.make_spec("C1", n_samples=12)
chunks = [(i, i * 500, (i + 1) * 500) for i in range(7)]
local = []
for ordinal, g0, g1 in assign(chunks, rank, world):
    counter, _ = O.tally_text(synth.generate(spec, g0, g1).decode().splitlines(keepends=True))
    firsts = {{}}
    for pos, key in enumerate(synth.keys_of(spec, g0, g1)):
        firsts.setdefault(key, (ordinal << 40) | pos)
    local += [(k, n, firsts[k]) for k, n in counter.items()]
mine = merge_lists([local])                                   # the rank's own total, as before the exchange
entries = [(k, n, min(p for kk, _, p in local if kk == k)) for k, n in mine.items()]
pack = lambda key: int(pack_keys([key])[0])
parts = shard_lists(entries, world, pack)                     # what this rank sends to every peer
everything = [None] * world
dist.all_gather_object(everything, parts)                     # stands in for the grouped send/recv
share = fold_share([everything[src][rank] for src in range(world)])
assert all(key_owner(pack(k), world) == rank for k, _, _ in share)
shares = [None] * world
dist.all_gather_object(shares, share)
union = sorted((pos, k, n) for sh in shares for k, n, pos in sh)
assert len({{k for _, k, _ in union}}) == len(union), "shares overlap"
want, _ = O.tally_text(synth.generate(spec, 0, 3500).decode().splitlines(keepends=True))
assert [(k, n) for _, k, n in union] == list(want.items()), "union of the shares differs from the oracle"
dist.barrier()
dist.destroy_process_group()
'''


def test_sharded_merge_gloo(tmp_path):
    """Host twin of frb_shardmerge on two gloo ranks: owner partition, exchange, fold; the shares are
    disjoint, every key sits on its owner, and their union is the single-process oracle's tally in order."""
    script = tmp_path / "shard_worker.py"
    script.write_text(SHARD_WORKER.format(root=ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29536", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]


def test_assign_covers_everything_once():
    from frender_b200.shard import assign
    items = list(range(23))
    for world in (1, 2, 3, 8):
        parts = [assign(items, r, world) for r in range(world)]
        assert sorted(x for p in parts for x in p) == items


@pytest.mark.gpu
def test_nccl_merge_matches_oracle():
    import ctypes
    n = ctypes.c_int()
    from frender_b200._lib import lib
    lib.frb_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(n.value, 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29534", os.path.join(ROOT, "tests", "mgpu_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "mgpu ok" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


@pytest.mark.gpu
def test_cli_scan_file_sharding_two_gpus(tmp_path, monkeypatch):
    """FRENDER_GPUS=2: files sharded over two GPUs, tables merged over NCCL, CSV byte-identical to the
    reference's output for the same three files."""
    import ctypes
    import json
    from conftest import GOLDEN_DIR, unb64
    from frender_b200._lib import lib
    n = ctypes.c_int()
    lib.frb_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs")
    case = json.load(open(os.path.join(GOLDEN_DIR, "golden.json")))["scan"]["multi"]
    files = []
    for fname in case["files"]:
        dst = tmp_path / fname
        dst.write_bytes(open(os.path.join(GOLDEN_DIR, f"multi__{fname}"), "rb").read())
        files.append(str(dst))
    (tmp_path / "SampleSheet.csv").write_text(case["sheet_csv"])
    monkeypatch.setenv("FRENDER_GPUS", "2")
    monkeypatch.chdir(tmp_path)
    from frender_b200.cli import main
    main(["scan", "-n", "1", "-rc", "-p", case["prefix"], "-o", "m", "-b", str(tmp_path / "SampleSheet.csv")] + files)
    out = [f for f in os.listdir(tmp_path) if f.startswith("frender-scan-results_")][0]
    assert (tmp_path / out).read_bytes() == unb64(case["scan_csv"])


def _failing_worker(rank, n_ranks, device, ident, jobs, sample, table_log2, conn):
    """Stands in for cli._scan_worker on a box without GPUs: rank 1 fails its scan, rank 0 succeeds and must not
    be left waiting for a collective."""
    if rank == 1:
        raise RuntimeError("bad header in file of rank 1")
    conn.send(("scanned", None))
    if not conn.recv():
        return
    conn.send(("ok", ([], None)))


def test_multi_gpu_rank_failure_ends_the_job(monkeypatch):
    """A rank whose scan fails (any rank, not just rank 0) ends the whole job with its message; nobody enters the
    collective (the workers wait for the parent's go)."""
    import frender_b200.cli as cli
    monkeypatch.setattr(cli.Context, "nccl_unique_id", staticmethod(lambda: b"\0" * 128))
    with pytest.raises(SystemExit, match="GPU worker 1 failed: .*bad header"):
        cli.scan_files_multi_gpu(["a", "b", "c"], None, 2, 12, worker=_failing_worker)


def _stub_demux_worker(rank, device, jobs, opts, out_dir, threads, conn):
    """Stands in for cli._demux_worker without a GPU: writes one gzip member per sink and pair."""
    import gzip
    for ordinal, r1, r2 in jobs:
        if "bad" in str(r1):
            raise SystemExit("Couldn't find barcode GGGG+TTTT in supplied frender result file!")
        os.mkdir(f"{out_dir}.part{ordinal}")
        for sink in ("S1_frender-demux_R1.fq.gz", "Undetermined_frender-demux_R1.fq.gz"):
            with open(os.path.join(f"{out_dir}.part{ordinal}", sink), "wb") as fh:
                fh.write(gzip.compress(f"{sink}:{ordinal}:{os.path.basename(str(r1))}\n".encode() if "S1" in sink or ordinal == 1
                                       else b""))
    conn.send(("ok", None))


def test_multi_gpu_demux_joins_the_parts_in_pair_order(tmp_path):
    """Pair i goes to rank i % N; every sink is the parts of all pairs in pair order (gzip members), the part
    directories are gone afterwards; a failing rank ends the job with its message."""
    import argparse
    import gzip
    import frender_b200.cli as cli
    out = str(tmp_path / "out") + "/"
    os.mkdir(out)
    ns = argparse.Namespace(no_index_hop=False, no_ambiguous=False, no_undeter=False, no_samples=False, o=None, r="r.csv")
    pairs = [(f"L00{i}_R1_001.fastq.gz", f"L00{i}_R2_001.fastq.gz") for i in range(1, 6)]
    cli.demux_pairs_multi_gpu(ns, pairs, 2, out, worker=_stub_demux_worker)
    assert sorted(os.listdir(out)) == ["S1_frender-demux_R1.fq.gz", "Undetermined_frender-demux_R1.fq.gz"]
    got = gzip.open(out + "S1_frender-demux_R1.fq.gz", "rb").read().decode().splitlines()
    assert got == [f"S1_frender-demux_R1.fq.gz:{i}:L00{i + 1}_R1_001.fastq.gz" for i in range(5)]
    assert gzip.open(out + "Undetermined_frender-demux_R1.fq.gz", "rb").read() == \
        b"Undetermined_frender-demux_R1.fq.gz:1:L002_R1_001.fastq.gz\n"
    out2 = str(tmp_path / "out2") + "/"
    os.mkdir(out2)
    with pytest.raises(SystemExit, match="GPU worker 1 failed: Couldn't find barcode GGGG\\+TTTT"):
        cli.demux_pairs_multi_gpu(ns, [("a_R1", "a_R2"), ("bad_R1", "bad_R2")], 2, out2, worker=_stub_demux_worker)


@pytest.mark.gpu
def test_cli_demux_pairs_on_two_gpus(tmp_path, monkeypatch):
    """FRENDER_GPUS=2 with three lane pairs: every sink decompresses to what the one-GPU run writes."""
    import ctypes
    import gzip
    import json
    from conftest import GOLDEN_DIR, unb64
    from frender_b200 import synth
    from frender_b200._lib import lib
    from frender_b200.cli import main
    n = ctypes.c_int()
    lib.frb_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs")
    gold = json.load(open(os.path.join(GOLDEN_DIR, "golden.json")))
    case = gold["demux"]["c1"]
    scan = gold["scan"][case["scan_case"]]
    spec = synth.make_spec(scan["config"], n_samples=scan["n_samples"])
    files = []
    for lane, (g0, g1) in enumerate([(0, 1200), (1200, 2100), (2100, 3000)], start=1):
        for mate in (1, 2):
            p = tmp_path / f"Undetermined_S0_L00{lane}_R{mate}_001.fastq.gz"
            p.write_bytes(gzip.compress(synth.generate_big(spec, g0, g1, mate), 1))
            files.append(str(p))
    (tmp_path / "results.csv").write_bytes(unb64(case["results_csv"]))
    main(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "one")] + files)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    main(["demux", "-r", str(tmp_path / "results.csv"), "-d", str(tmp_path / "two")] + files)
    names = sorted(os.listdir(tmp_path / "one"))
    assert names == sorted(os.listdir(tmp_path / "two")) == sorted(case["sinks"])
    for name in names:
        assert gzip.open(tmp_path / "one" / name, "rb").read() == gzip.open(tmp_path / "two" / name, "rb").read(), name
    # the three lanes are the golden case's reads in order: the sinks are the golden sinks
    import hashlib
    for name, want in case["sinks"].items():
        assert hashlib.sha256(gzip.open(tmp_path / "two" / name, "rb").read()).hexdigest() == want["sha256"], name
