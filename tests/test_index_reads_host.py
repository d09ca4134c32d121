"""Demux with index reads (FRENDER_INDEX_READS=1) without a GPU: the discovery of the I1 / I2 files in directory and
explicit-list form, its refusals, the single-end combination, the default left as it is, the N-mate oracle against
the paired oracle, and the index paths reaching the multi-GPU workers."""
import argparse
import gzip
import os
import random
from argparse import Namespace

import pytest

import frender_oracle as O
import index_reads_oracle as IR
from frender_b200 import synth


def touch(d, *names):
    for n in names:
        (d / n).write_bytes(gzip.compress(b""))
    return [d / n for n in names]


def lanes_of(files, single=False, indexed=True):
    from frender_b200.cli import demux_lanes, parse_files
    return demux_lanes(parse_files(files, just_r1=False), single, indexed)


LANE = ["L_S1_L001_R1_001.fastq.gz", "L_S1_L001_R2_001.fastq.gz", "L_S1_L001_I1_001.fastq.gz",
        "L_S1_L001_I2_001.fastq.gz"]


# ---- discovery ---------------------------------------------------------------------------------------------------
def test_discovery_directory_and_list(tmp_path):
    r1, r2, i1, i2 = touch(tmp_path, *LANE)
    s1, s2, j1, j2 = touch(tmp_path, *(n.replace("L001", "L002") for n in LANE))
    (tmp_path / "notes.txt").write_text("x")
    lanes, reads = lanes_of({"dir": tmp_path})
    assert reads == ["R1", "R2", "I1", "I2"]
    assert sorted(lanes) == [(r1, r2, i1, i2), (s1, s2, j1, j2)]
    lanes, reads = lanes_of({"file": [i2, r2, i1, r1]})        # any order of the list
    assert (lanes, reads) == ([(r1, r2, i1, i2)], ["R1", "R2", "I1", "I2"])


@pytest.mark.parametrize("kind", ["I1", "I2"])
def test_discovery_one_kind(tmp_path, kind):
    r1, r2 = touch(tmp_path, LANE[0], LANE[1])
    (ix,) = touch(tmp_path, LANE[0].replace("_R1_", f"_{kind}_"))
    assert lanes_of({"dir": tmp_path}) == ([(r1, r2, ix)], ["R1", "R2", kind])


def test_discovery_single_end(tmp_path):
    r1, i1, i2 = touch(tmp_path, LANE[0], LANE[2], LANE[3])
    assert lanes_of({"dir": tmp_path}, single=True) == ([(r1, None, i1, i2)], ["R1", "I1", "I2"])
    # the index files never count as read 2 files of a single-end run
    assert lanes_of({"file": [r1, i1]}, single=True) == ([(r1, None, i1)], ["R1", "I1"])


def test_discovery_refusals(tmp_path):
    r1, r2, i1, i2 = touch(tmp_path, *LANE)
    s1, s2, j1 = touch(tmp_path, *(n.replace("L001", "L002") for n in LANE[:3]))
    with pytest.raises(SystemExit, match=r"L_S1_L002_R1_001.fastq.gz has no I2 file \(L_S1_L002_I2_001.fastq.gz\)"):
        lanes_of({"dir": tmp_path})
    with pytest.raises(SystemExit, match="index read file .*L_S1_L001_I2_001.fastq.gz has no read 1 file"):
        lanes_of({"file": [s1, s2, j1, i2]})
    with pytest.raises(SystemExit, match="no index read file"):
        lanes_of({"file": [r1, r2]})
    with pytest.raises(SystemExit, match="has no read 1 file"):
        lanes_of({"file": [r2, i1]})


def test_discovery_takes_index_files_by_their_illumina_suffix(tmp_path):
    """A sample name holding _I1_ is part of a read file's name, not an index read: only the _I1_ / _I2_ in front of
    the three-digit number and the suffix marks an index file."""
    names = [n.replace("L_S1", "Lib_I1_x_S1") for n in LANE]
    r1, r2, i1, i2 = touch(tmp_path, *names)
    assert lanes_of({"dir": tmp_path}) == ([(r1, r2, i1, i2)], ["R1", "R2", "I1", "I2"])
    with pytest.raises(SystemExit, match="no index read file"):
        lanes_of({"file": [r1, r2]})


@pytest.mark.parametrize("env", [None, "0"])
def test_default_discovery_is_unchanged(tmp_path, monkeypatch, env):
    """Without FRENDER_INDEX_READS (or with 0): the R1/R2 lanes as before, and an I1 file beside them makes the
    pairing fail as it always did, ahead of any device work and of the output directory."""
    from frender_b200.cli import frender_demux, get_paired_files, parse_files
    if env is None:
        monkeypatch.delenv("FRENDER_INDEX_READS", raising=False)
    else:
        monkeypatch.setenv("FRENDER_INDEX_READS", env)
    d = tmp_path / "in"
    d.mkdir()
    r1, r2 = touch(d, LANE[0], LANE[1])
    assert lanes_of({"dir": d}, indexed=False) == (get_paired_files(parse_files({"dir": d}, False)), ["R1", "R2"])
    touch(d, LANE[2])
    with pytest.raises(TypeError):
        frender_demux(demux_args(tmp_path, [d]))
    assert not (tmp_path / "out").exists()


def demux_args(tmp_path, files):
    res = tmp_path / "results.csv"
    res.write_text("idx1,idx2,reads,matched_idx1,matched_idx2,read_type,sample_name\nAC,GT,1,AC,GT,demuxable,S1\n")
    return Namespace(r=str(res), d=str(tmp_path / "out"), o=None, no_index_hop=False, no_ambiguous=False,
                     no_undeter=False, no_samples=False, files=[str(f) for f in files])


def test_cli_refusals_come_before_any_device_work(tmp_path, monkeypatch):
    from frender_b200.cli import frender_demux
    monkeypatch.setenv("FRENDER_INDEX_READS", "1")
    d = tmp_path / "in"
    d.mkdir()
    r1, r2 = touch(d, LANE[0], LANE[1])
    with pytest.raises(SystemExit, match="no index read file"):
        frender_demux(demux_args(tmp_path, [r1, r2]))
    (orphan,) = touch(d, "X_S9_L001_I1_001.fastq.gz")
    with pytest.raises(SystemExit, match="has no read 1 file"):
        frender_demux(demux_args(tmp_path, [d]))
    assert not (tmp_path / "out").exists()


# ---- oracle ------------------------------------------------------------------------------------------------------
def test_n_mate_oracle_agrees_with_the_paired_oracle():
    spec = synth.make_spec("C1", n_samples=12)
    r1, r2 = synth.generate(spec, 0, 3000, 1).decode(), synth.generate(spec, 0, 3000, 2).decode()
    i1, i2 = (synth.generate(spec, 0, 3000, 1, k).decode() for k in (1, 2))
    keys = sorted(set(synth.keys_of(spec, 0, 3000)))
    kinds = ["demuxable", "index_hop", "ambiguous", "undetermined"]
    table = {k: (kinds[j % 4], f"S{j % 5}" if j % 4 == 0 else "") for j, k in enumerate(keys)}
    roles = O.sink_names(table)
    lines = [t.splitlines(keepends=True) for t in (r1, r2, i1, i2)]
    want = O.route_pairs(lines[0], lines[1], table, roles)
    got = IR.route_mates(lines, 1, table, roles)
    assert {n: v[:2] for n, v in got.items()} == want
    # every index record sits in the sink of its read's R2 key, in read order
    for name, (a, _, c, d) in got.items():
        heads = [ln for ln in a.decode().splitlines()[0::4]]
        assert heads == c.decode().splitlines()[0::4] == d.decode().splitlines()[0::4]
    # a shorter index file ends the zip; a trailing partial record is padded
    cut = lines[2][:4 * 1000 + 2]
    short = IR.route_mates([lines[0], lines[1], cut], 1, table, roles)
    assert sum(v[0].count(b"\n@A00123") + (v[0][:1] == b"@") for v in short.values()) == 1001
    assert sum(len(v[2]) for v in short.values()) == sum(len(x) for x in cut)


def test_n_mate_oracle_single_end_key_from_r1():
    table = {"AC+GT": ("demuxable", "S1"), "TT+AA": ("undetermined", "")}
    roles = O.sink_names(table)
    r1 = "@a 1:N:0:AC+GT\nAC\n+\nFF\n@b 1:N:0:TT+AA\nTT\n+\nFF\n"
    i1 = "@a 1:N:0:AC+GT\nAC\n+\nFF\n@b 1:N:0:TT+AA\nTT\n+\nFF\n"
    got = IR.route_mates([r1.splitlines(True), i1.splitlines(True)], 0, table, roles)
    assert got["S1"] == (b"@a 1:N:0:AC+GT\nAC\n+\nFF\n",) * 2
    with pytest.raises(SystemExit, match="Couldn't find barcode GG\\+CC"):
        IR.route_mates([["@d 1:N:0:GG+CC\n", "A\n", "+\n", "F\n"]] * 2, 0, table, roles)


# ---- multi-GPU ---------------------------------------------------------------------------------------------------
def _stub_index_worker(rank, device, jobs, opts, out_dir, threads, conn):
    """Stands in for cli._demux_worker without a GPU: one gzip member per sink, read and job, naming the job's
    files."""
    for ordinal, r1, r2, *index in jobs:
        assert len(index) == 2
        os.mkdir(f"{out_dir}.part{ordinal}")
        for read, path in zip(("R1", "R2", "I1", "I2"), (r1, r2, *index)):
            with open(os.path.join(f"{out_dir}.part{ordinal}", f"S1_frender-demux_{read}.fq.gz"), "wb") as fh:
                fh.write(gzip.compress(f"{ordinal}:{rank}:{os.path.basename(str(path))}\n".encode()))
    conn.send(("ok", None))


def test_multi_gpu_workers_receive_the_index_paths(tmp_path):
    import frender_b200.cli as cli
    d = tmp_path / "in"
    d.mkdir()
    for lane in range(1, 4):
        touch(d, *(n.replace("L001", f"L00{lane}") for n in LANE))
    lanes, _ = lanes_of({"dir": d})
    lanes.sort()
    out = str(tmp_path / "out") + "/"
    os.mkdir(out)
    ns = argparse.Namespace(no_index_hop=False, no_ambiguous=False, no_undeter=False, no_samples=False, o=None, r="r.csv")
    cli.demux_pairs_multi_gpu(ns, lanes, 2, out, worker=_stub_index_worker)
    assert sorted(os.listdir(out)) == [f"S1_frender-demux_{r}.fq.gz" for r in ("I1", "I2", "R1", "R2")]
    for k, read in enumerate(("R1", "R2", "I1", "I2")):
        got = gzip.open(f"{out}S1_frender-demux_{read}.fq.gz", "rb").read().decode().splitlines()
        assert got == [f"{i}:{i % 2}:{lanes[i][k].name}" for i in range(3)]
    assert sorted(os.listdir(tmp_path)) == ["in", "out"]
