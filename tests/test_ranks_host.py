"""The rank supervisor of multi-GPU scan and demux (shard.Ranks) with stub workers, and the scan's retry policy over
WorkerFailed: no GPU, only the library that _lib loads."""
import argparse
import multiprocessing as mp
import os

import pytest

import frender_b200._lib as L
import frender_b200.cli as cli
from frender_b200.engine import FrbError
from frender_b200.shard import WorkerFailed


def _table_full_worker(rank, n_ranks, device, ident, jobs, sample, table_log2, conn):
    """Stands in for cli._scan_worker: rank 1 overflows its table; rank 0 scans and writes down the parent's answer
    to its "scanned" next to its first file."""
    if rank == 1:
        raise FrbError(L.ERR_TABLE_FULL, "unique-key table full")
    conn.send(("scanned", None))
    go = conn.recv()
    with open(jobs[0][1] + ".go", "w") as fh:
        fh.write(repr(go))
    if go:
        conn.send(("ok", ([], None)))


def _vanishing_worker(rank, n_ranks, device, ident, jobs, sample, table_log2, conn):
    """Stands in for cli._scan_worker: rank 0 dies without a word; rank 1 scans and waits for the parent."""
    if rank == 0:
        os._exit(3)
    conn.send(("scanned", None))
    if conn.recv():
        conn.send(("ok", ([], None)))


@pytest.fixture
def no_nccl(monkeypatch):
    monkeypatch.setattr(cli.Context, "nccl_unique_id", staticmethod(lambda: b"\0" * 128))


def test_frb_error_of_a_rank_keeps_its_code(tmp_path, no_nccl):
    files = [str(tmp_path / name) for name in ("a", "b", "c")]
    with pytest.raises(WorkerFailed) as info:
        cli.scan_files_multi_gpu(files, None, 2, 12, worker=_table_full_worker)
    exc = info.value
    assert (exc.rank, exc.frb_code) == (1, L.ERR_TABLE_FULL)
    assert str(exc) == "GPU worker 1 failed: FrbError('frender_b200 error -6: unique-key table full')"
    assert (tmp_path / "a.go").read_text() == "False"          # rank 0 was told not to enter the collective
    assert mp.active_children() == []


def test_rank_that_exits_without_a_message(no_nccl):
    with pytest.raises(WorkerFailed, match="^GPU worker 0 exited without a result$") as info:
        cli.scan_files_multi_gpu(["a", "b", "c"], None, 2, 12, worker=_vanishing_worker)
    assert (info.value.rank, info.value.frb_code) == (0, None)
    assert mp.active_children() == []


def _failing_demux_worker(rank, device, jobs, opts, out_dir, threads, conn):
    """Stands in for cli._demux_worker: every pair gets its part directory; rank 1 fails after writing its part."""
    for ordinal, r1, r2 in jobs:
        os.mkdir(f"{out_dir}.part{ordinal}")
        with open(os.path.join(f"{out_dir}.part{ordinal}", "S1_frender-demux_R1.fq.gz"), "wb") as fh:
            fh.write(b"")
    if rank == 1:
        raise SystemExit("Couldn't find barcode GGGG+TTTT in supplied frender result file!")
    conn.send(("ok", None))


def test_failed_multi_gpu_demux_leaves_no_part_directories(tmp_path):
    out = str(tmp_path / "out") + "/"
    os.mkdir(out)
    ns = argparse.Namespace(no_index_hop=False, no_ambiguous=False, no_undeter=False, no_samples=False, o=None, r="r.csv")
    pairs = [(f"L00{i}_R1_001.fastq.gz", f"L00{i}_R2_001.fastq.gz") for i in range(1, 5)]
    with pytest.raises(WorkerFailed) as info:
        cli.demux_pairs_multi_gpu(ns, pairs, 2, out, worker=_failing_demux_worker)
    assert os.listdir(out) == [] and sorted(os.listdir(tmp_path)) == ["out"]
    assert str(info.value) == "GPU worker 1 failed: Couldn't find barcode GGGG+TTTT in supplied frender result file!"
    assert info.value.frb_code is None
    assert mp.active_children() == []


class _Ctx:
    """What frender_scan asks of its context up to the tally, when scan_files_multi_gpu does the tally."""
    device, wide, table_log2 = 0, False, 12

    def __init__(self):
        self.resized = []

    def reset(self):
        pass

    def resize_tables(self, log2):
        self.resized.append(log2)
        self.table_log2 = log2


def _scan(tmp_path, monkeypatch, errors):
    """frender scan over two files on FRENDER_GPUS=2 whose multi-GPU tally raises `errors` one after the other."""
    files = [tmp_path / f"L00{i}_R1_001.fastq.gz" for i in (1, 2)]
    for f in files:
        f.write_bytes(b"")
    (tmp_path / "SampleSheet.csv").write_text("Sample_ID,index,index2\nS1,ACGTACGT,TTTTGGGG\n")
    calls = []

    def tally(*a, **k):
        calls.append(a)
        raise errors[len(calls) - 1]
    monkeypatch.setattr(cli, "scan_files_multi_gpu", tally)
    monkeypatch.setenv("FRENDER_GPUS", "2")
    monkeypatch.chdir(tmp_path)
    ctx = _Ctx()
    args = cli.build_parser().parse_args(["scan", "-n", "1", "-b", str(tmp_path / "SampleSheet.csv")] +
                                         [str(f) for f in files])
    with pytest.raises(WorkerFailed) as info:
        cli.frender_scan(args, ctx=ctx)
    return info.value, ctx, calls


def test_scan_retries_on_the_code_not_on_the_text(tmp_path, monkeypatch, capsys):
    text = "FrbError('frender_b200 error -6: unique-key table full')"
    err = WorkerFailed(1, text, frb_code=None)
    got, ctx, calls = _scan(tmp_path, monkeypatch, [err])
    assert got is err and len(calls) == 1 and ctx.resized == []
    assert "tallying again" not in capsys.readouterr().out


def test_scan_grows_the_tables_on_a_ranks_table_full(tmp_path, monkeypatch, capsys):
    last = WorkerFailed(0, "RuntimeError('disk on fire')")
    got, ctx, calls = _scan(tmp_path, monkeypatch, [WorkerFailed(1, "full", frb_code=L.ERR_TABLE_FULL), last])
    assert got is last and len(calls) == 2 and ctx.resized == [14]
    assert "unique-key tables of 2^12 slots are full: tallying again with 2^14" in capsys.readouterr().out
