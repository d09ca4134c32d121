"""BGZF, the blocked gzip of htslib and bgzip, on the host: parsing of block headers and joining of BGZF files.

A BGZF file is a run of gzip members ("blocks") of at most 64 KiB each.  Every block has the 18-byte header
1f 8b 08 04 00000000 00 ff 0600 'B' 'C' 0200 BSIZE, where BSIZE (little-endian u16) is the block's length - 1,
then raw deflate data, CRC-32 and ISIZE of its own input.  The file ends with the empty block EOF_BLOCK.  The device
writes the blocks (Context.gz_deflate(bgzf=True), and the demux stream in BGZF format); nothing here compresses.
"""
import struct

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
HEADER = bytes.fromhex("1f8b08040000000000ff06004243")  # the header up to the BC field's length
HEADER_BYTES = 18
TRAILER_BYTES = 8


class BgzfError(ValueError):
    """The bytes are not BGZF."""


def iter_blocks(buf):
    """Yield (offset, bsize, isize) of every block of `buf` (bytes-like), in order: the block is
    buf[offset:offset + bsize + 1], its deflate data buf[offset + 18:offset + bsize - 7].  Raises BgzfError on
    anything that is not a whole number of BGZF blocks: another magic or flag byte, an extra field other than the
    single BC subfield, a BSIZE too small for a block or running past the end, a truncated header or trailer."""
    view = memoryview(buf).cast("B")
    n, pos = len(view), 0
    while pos < n:
        if n - pos < HEADER_BYTES:
            raise BgzfError(f"truncated block header at {pos}")
        head = view[pos:pos + HEADER_BYTES].tobytes()
        if head[:4] != HEADER[:4]:
            raise BgzfError(f"no BGZF block header at {pos}")
        if head[10:14] != HEADER[10:14] or head[14:16] != b"\x02\x00":
            raise BgzfError(f"no BC extra field in the block at {pos}")
        bsize = struct.unpack_from("<H", head, 16)[0]
        if bsize + 1 < HEADER_BYTES + TRAILER_BYTES:
            raise BgzfError(f"BSIZE {bsize} of the block at {pos} is too small for a block")
        if pos + bsize + 1 > n:
            raise BgzfError(f"the block at {pos} (BSIZE {bsize}) runs past the end ({n} bytes)")
        isize = struct.unpack_from("<I", view, pos + bsize + 1 - 4)[0]
        yield pos, bsize, isize
        pos += bsize + 1


def join_files(out_path, part_paths, chunk=1 << 22):
    """Write the BGZF files `part_paths`, in order, as one BGZF file: every part must end with the EOF block, which
    is dropped from every part but the last, so the result holds exactly one EOF block, at its end (no parts: the
    EOF block alone).  Parts are streamed; of each, only the last 28 bytes are checked."""
    with open(out_path, "wb") as out:
        for i, path in enumerate(part_paths):
            with open(path, "rb") as src:
                size = src.seek(0, 2)
                src.seek(max(size - len(EOF_BLOCK), 0))
                if src.read() != EOF_BLOCK:
                    raise BgzfError(f"{path} does not end with the BGZF EOF block")
                src.seek(0)
                left = size if i == len(part_paths) - 1 else size - len(EOF_BLOCK)
                while left:
                    piece = src.read(min(left, chunk))
                    if not piece:
                        raise BgzfError(f"{path} became shorter while it was read")
                    out.write(piece)
                    left -= len(piece)
        if not part_paths:
            out.write(EOF_BLOCK)
