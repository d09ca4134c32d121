"""BGZF on the host (frender_b200.bgzf): the block parser on hand-built blocks and the joining of BGZF parts of a
multi-GPU demux.  No GPU needed."""
import gzip
import struct
import zlib

import pytest

from frender_b200 import bgzf


def block(data, level=6):
    """One BGZF block of `data` as htslib writes it: raw deflate behind the 18-byte header, CRC-32 and ISIZE."""
    z = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = z.compress(data) + z.flush()
    bsize = 18 + len(body) + 8 - 1
    head = bytes.fromhex("1f8b08040000000000ff060042430200") + struct.pack("<H", bsize)
    return head + body + struct.pack("<II", zlib.crc32(data), len(data))


def bgzf_file(pieces):
    return b"".join(block(p) for p in pieces) + bgzf.EOF_BLOCK


PIECES = [b"@r1\nACGT\n+\nFFFF\n" * 300, b"", bytes(range(256)) * 40, b"x"]


def test_eof_block_is_an_empty_block():
    assert len(bgzf.EOF_BLOCK) == 28
    assert list(bgzf.iter_blocks(bgzf.EOF_BLOCK)) == [(0, 27, 0)]
    assert gzip.decompress(bgzf.EOF_BLOCK) == b""
    assert block(b"", 6) == bgzf.EOF_BLOCK


def test_iter_blocks_walks_hand_built_blocks():
    buf = bgzf_file(PIECES)
    blocks = list(bgzf.iter_blocks(buf))
    assert len(blocks) == len(PIECES) + 1
    pos = 0
    for (off, bsize, isize), piece in zip(blocks, PIECES + [b""]):
        assert off == pos and isize == len(piece)
        raw = buf[off + 18:off + bsize + 1 - 8]
        assert zlib.decompressobj(-15).decompress(raw) == piece
        pos = off + bsize + 1
    assert pos == len(buf)
    assert gzip.decompress(buf) == b"".join(PIECES)
    assert list(bgzf.iter_blocks(b"")) == []


def test_iter_blocks_takes_a_memoryview_and_numpy_bytes():
    import numpy as np
    buf = bgzf_file(PIECES[:2])
    want = list(bgzf.iter_blocks(buf))
    assert list(bgzf.iter_blocks(memoryview(buf))) == want
    assert list(bgzf.iter_blocks(np.frombuffer(buf, np.uint8))) == want


@pytest.mark.parametrize("damage", ["magic", "plain_gzip", "no_bc", "xlen", "bsize_past_end", "bsize_small",
                                    "truncated_trailer", "truncated_header"])
def test_iter_blocks_rejects_what_is_not_bgzf(damage):
    good = bgzf_file(PIECES[:1])
    buf = bytearray(good)
    if damage == "magic":
        buf[1] = 0x8c
    elif damage == "plain_gzip":
        buf = bytearray(gzip.compress(PIECES[0]))
    elif damage == "no_bc":
        buf[12:14] = b"XY"
    elif damage == "xlen":
        buf[10] = 8
    elif damage == "bsize_past_end":
        struct.pack_into("<H", buf, 16, len(good))
    elif damage == "bsize_small":
        struct.pack_into("<H", buf, 16, 20)
    elif damage == "truncated_trailer":
        buf = bytearray(block(PIECES[0])[:-3])
    elif damage == "truncated_header":
        buf = buf[:len(good) - 28 + 10]
    with pytest.raises(bgzf.BgzfError):
        list(bgzf.iter_blocks(bytes(buf)))


def test_join_files_keeps_one_eof_block_at_the_end(tmp_path):
    """Parts with blocks and parts that are the EOF block alone join into one file that decompresses to the
    concatenated inputs and is exactly the file of all blocks in a row."""
    parts = [[PIECES[0], PIECES[2]], [], [PIECES[3]], [], [PIECES[0]]]
    paths = []
    for i, p in enumerate(parts):
        path = tmp_path / f"part{i}.fq.gz"
        path.write_bytes(bgzf_file(p))
        paths.append(path)
    out = tmp_path / "joined.fq.gz"
    bgzf.join_files(out, paths, chunk=1000)
    got = out.read_bytes()
    flat = [x for p in parts for x in p]
    assert got == bgzf_file(flat)
    assert got.count(bgzf.EOF_BLOCK) == 1 and got.endswith(bgzf.EOF_BLOCK)
    assert gzip.decompress(got) == b"".join(flat)
    assert [isize for _, _, isize in bgzf.iter_blocks(got)] == [len(x) for x in flat] + [0]


def test_join_files_of_empty_parts_is_the_eof_block(tmp_path):
    paths = []
    for i in range(3):
        paths.append(tmp_path / f"p{i}")
        paths[-1].write_bytes(bgzf.EOF_BLOCK)
    bgzf.join_files(tmp_path / "out", paths)
    assert (tmp_path / "out").read_bytes() == bgzf.EOF_BLOCK
    bgzf.join_files(tmp_path / "none", [])
    assert (tmp_path / "none").read_bytes() == bgzf.EOF_BLOCK


def test_join_files_refuses_a_part_without_eof_block(tmp_path):
    (tmp_path / "a").write_bytes(bgzf_file([PIECES[0]]))
    (tmp_path / "b").write_bytes(block(PIECES[0]))
    with pytest.raises(bgzf.BgzfError):
        bgzf.join_files(tmp_path / "out", [tmp_path / "a", tmp_path / "b"])
    (tmp_path / "c").write_bytes(b"\x1f\x8b")
    with pytest.raises(bgzf.BgzfError):
        bgzf.join_files(tmp_path / "out", [tmp_path / "c"])
