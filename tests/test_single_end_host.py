"""Single-end demux (FRENDER_SINGLE_END=1) without a GPU: the oracle's single-end loop against the reference's own
golden outputs, the selection of the input files and its refusals, the default left as it is, and the multi-GPU
join of (R1, None) jobs."""
import argparse
import gzip
import hashlib
import os
from argparse import Namespace

import pytest

import frender_oracle as O
import single_end_oracle as SE
from conftest import unb64
from frender_b200 import synth


def golden_r1(golden, name):
    """Golden demux case `name` and the R1 text it was made from."""
    case = golden["demux"][name]
    scan = golden["scan"][case["scan_case"]]
    spec = synth.make_spec(scan["config"], n_samples=scan["n_samples"])
    return case, synth.generate_big(spec, 0, case["reads"], 1)


@pytest.mark.parametrize("name", ["c1", "c1_ia", "c4"])
def test_oracle_single_end_equals_the_references_r1_sinks(golden, tmp_path, name):
    """R1 and R2 headers of these cases carry the same key and R2 is not truncated: routing R1 by its own headers
    writes exactly the reference's R1 sinks."""
    case, r1 = golden_r1(golden, name)
    path = tmp_path / "Undetermined_S0_L001_R1_001.fastq.gz"
    path.write_bytes(gzip.compress(r1, 1))
    res = tmp_path / "results.csv"
    res.write_bytes(unb64(case["results_csv"]))
    table = O.parse_results_file(res)
    flags = case["flags"]
    roles = O.sink_names(table, index_hop=not flags.get("i", False), ambiguous=not flags.get("a", False))
    infix = (flags["o"] + "_") if flags.get("o") else ""
    got = {f"{sink}_frender-demux_{infix}R1.fq.gz": data for sink, data in SE.demux_file_single(path, table, roles).items()}
    want = {f: v for f, v in case["sinks"].items() if f.endswith("_R1.fq.gz")}
    assert sorted(got) == sorted(want)
    for fname, w in want.items():
        assert len(got[fname]) == w["bytes"], fname
        assert hashlib.sha256(got[fname]).hexdigest() == w["sha256"], fname


def test_oracle_single_end_pads_a_partial_record_and_refuses_unknown_keys():
    table = {"AC+GT": ("demuxable", "S1"), "TT+AA": ("undetermined", "")}
    roles = O.sink_names(table)
    text = "@a 1:N:0:AC+GT\nAC\n+\nFF\n@b 1:N:0:TT+AA\nTT"
    got = SE.route_single(text.splitlines(keepends=True), table, roles)
    assert got["S1"] == b"@a 1:N:0:AC+GT\nAC\n+\nFF\n"
    assert got[roles["#und"]] == b"@b 1:N:0:TT+AA\nTT"
    with pytest.raises(SystemExit, match="Couldn't find barcode GG\\+CC in supplied frender result file!"):
        SE.route_single(["@d 1:N:0:GG+CC\n", "A\n", "+\n", "F\n"], table, roles)


# ---- file selection ----------------------------------------------------------------------------------------------
def touch(d, *names):
    for n in names:
        (d / n).write_bytes(gzip.compress(b""))
    return [d / n for n in names]


def test_single_end_selection(tmp_path):
    from frender_b200.cli import get_single_end_files, parse_files
    a, b, _ = touch(tmp_path, "A_S1_L001_R1_001.fastq.gz", "B_S2_L001_R1_001.fastq.gz", "B_S2_L001_I1_001.fastq.gz")
    (tmp_path / "notes.txt").write_text("x")
    # a directory of R1 files: the R1s, the other fastq files and non-fastq files ignored
    assert sorted(get_single_end_files(parse_files({"dir": tmp_path}, just_r1=False))) == [a, b]
    # an explicit list
    assert get_single_end_files(parse_files({"file": [a, b]}, just_r1=False)) == [a, b]
    assert get_single_end_files(parse_files({"file": a}, just_r1=False)) == [a]


def test_single_end_refuses_paired_input_and_no_r1(tmp_path):
    from frender_b200.cli import get_single_end_files, parse_files
    r1, r2 = touch(tmp_path, "A_S1_L001_R1_001.fastq.gz", "A_S1_L001_R2_001.fastq.gz")
    with pytest.raises(SystemExit, match="has a read 2 file"):
        get_single_end_files(parse_files({"file": [r1, r2]}, just_r1=False))
    with pytest.raises(SystemExit, match="no read 1 file"):
        get_single_end_files(parse_files({"file": [r2]}, just_r1=False))
    with pytest.raises(SystemExit, match="no read 1 file"):
        get_single_end_files([])


def demux_args(tmp_path, files):
    res = tmp_path / "results.csv"
    res.write_text("idx1,idx2,reads,matched_idx1,matched_idx2,read_type,sample_name\nAC,GT,1,AC,GT,demuxable,S1\n")
    return Namespace(r=str(res), d=str(tmp_path / "out"), o=None, no_index_hop=False, no_ambiguous=False,
                     no_undeter=False, no_samples=False, files=[str(f) for f in files])


@pytest.mark.parametrize("env", [None, "0"])
def test_default_still_wants_a_read_2_file(tmp_path, monkeypatch, env):
    """Without FRENDER_SINGLE_END (or with 0) an R1 without a mate ends the run as before, ahead of any device work
    and of the output directory."""
    from frender_b200.cli import frender_demux
    if env is None:
        monkeypatch.delenv("FRENDER_SINGLE_END", raising=False)
    else:
        monkeypatch.setenv("FRENDER_SINGLE_END", env)
    (r1,) = touch(tmp_path, "A_S1_L001_R1_001.fastq.gz")
    with pytest.raises(SystemExit, match="Couldn't find a read 2 file for"):
        frender_demux(demux_args(tmp_path, [r1]))
    assert not (tmp_path / "out").exists()


def test_single_end_cli_refusals_come_before_any_device_work(tmp_path, monkeypatch):
    from frender_b200.cli import frender_demux
    monkeypatch.setenv("FRENDER_SINGLE_END", "1")
    r1, r2 = touch(tmp_path, "A_S1_L001_R1_001.fastq.gz", "A_S1_L001_R2_001.fastq.gz")
    with pytest.raises(SystemExit, match="has a read 2 file"):
        frender_demux(demux_args(tmp_path, [r1, r2]))
    with pytest.raises(SystemExit, match="no read 1 file"):
        frender_demux(demux_args(tmp_path, [r2]))
    assert not (tmp_path / "out").exists()


# ---- multi-GPU join ----------------------------------------------------------------------------------------------
def _stub_single_end_worker(rank, device, jobs, opts, out_dir, threads, conn):
    """Stands in for cli._demux_worker without a GPU: one gzip member per R1 sink and job; jobs carry no R2."""
    try:
        for ordinal, r1, r2 in jobs:
            assert r2 is None
            os.mkdir(f"{out_dir}.part{ordinal}")
            for sink in ("S1_frender-demux_R1.fq.gz", "Undetermined_frender-demux_R1.fq.gz"):
                with open(os.path.join(f"{out_dir}.part{ordinal}", sink), "wb") as fh:
                    fh.write(gzip.compress(f"{sink}:{ordinal}:{rank}:{os.path.basename(str(r1))}\n".encode()))
        conn.send(("ok", None))
    except BaseException as exc:
        conn.send(("error", repr(exc)))
    finally:
        conn.close()


def test_multi_gpu_single_end_appends_the_parts_in_file_order(tmp_path):
    import frender_b200.cli as cli
    out = str(tmp_path / "out") + "/"
    os.mkdir(out)
    ns = argparse.Namespace(no_index_hop=False, no_ambiguous=False, no_undeter=False, no_samples=False, o=None, r="r.csv")
    units = [(f"L00{i}_R1_001.fastq.gz", None) for i in range(1, 6)]
    cli.demux_pairs_multi_gpu(ns, units, 2, out, worker=_stub_single_end_worker)
    assert sorted(os.listdir(out)) == ["S1_frender-demux_R1.fq.gz", "Undetermined_frender-demux_R1.fq.gz"]
    for sink in os.listdir(out):
        got = gzip.open(out + sink, "rb").read().decode().splitlines()
        assert got == [f"{sink}:{i}:{i % 2}:L00{i + 1}_R1_001.fastq.gz" for i in range(5)]
    assert sorted(os.listdir(tmp_path)) == ["out"]
