"""BGZF (blocked gzip, as bgzip and htslib write it) -- the compressed FASTA form
MotifSearch.upload_fastn_bgzf takes.

A BGZF file is a series of gzip members of at most 64 KiB each.  Every member's header carries
the extra subfield `BC` with the member's size less one (BSIZE), and its trailer the CRC-32 and
size (ISIZE) of its uncompressed data, so a reader learns where every member's output goes from the
headers alone.  A file ends with an empty member, EOF_BLOCK.
"""
from __future__ import annotations

import struct
import zlib

# the empty member every BGZF file ends with (SAM/BAM format specification, section 4.1.2)
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")

# ID1 ID2 CM FLG(FEXTRA) MTIME XFL OS(unknown) XLEN=6, then SI1 SI2 = "BC", SLEN = 2, BSIZE
_HEAD = bytes.fromhex("1f8b08040000000000ff0600") + b"BC\x02\x00"


def write_bgzf(data, level: int = 6, block: int = 0xff00, strategy: int = zlib.Z_DEFAULT_STRATEGY,
               eof: bool = True) -> bytes:
    """`data` as BGZF: one member per `block` bytes (bgzip's 0xff00 by default), each a raw
    DEFLATE stream at zlib `level` and `strategy`, then EOF_BLOCK unless eof=False.  Raises
    ValueError when a member would exceed 65 536 bytes (incompressible data in blocks of 64 KiB)."""
    data = memoryview(bytes(data))
    if not 1 <= block <= 65536:
        raise ValueError(f"block of {block} bytes: BGZF members hold 1 to 65536")
    out = []
    for o in range(0, len(data), block):
        chunk = data[o:o + block]
        co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        cdata = co.compress(chunk) + co.flush()
        size = len(_HEAD) + 2 + len(cdata) + 8
        if size > 65536:
            raise ValueError(f"member at byte {o} would take {size} bytes; BGZF allows 65536")
        out += [_HEAD, struct.pack("<H", size - 1), cdata, struct.pack("<II", zlib.crc32(chunk), len(chunk))]
    if eof:
        out.append(EOF_BLOCK)
    return b"".join(out)
