"""Reference encoder / decoder of byte format 5 (DESIGN.md section 15, GainedCheckerboardHierarchical; numpy / plain Python, test-only,
the product never imports it).  A format-5 z string is the unsized format-4 string of oracle/rans_checkerboard.py with its header
replaced by <BBHBBHI> = (version 5, arm, M, K, L, q_code, checksum field), the field being the symbol checksum plus
quality_term(L, q_code) mod 2^32; a sized string then sets 0x80 in the version byte, adds section 12's size term to the field and
puts <HH> = (H, W) after the header.  The y string is format 4's."""
from __future__ import annotations

import struct

from . import rans_checkerboard as RC
from .rans import HEADER
from .rans_sized import SIZE, SIZED, mix32, size_term

VERSION = 5
GAINED_HEADER = struct.Struct("<BBHBBHI")


def quality_term(levels, q_code):
    return mix32(0xFFFFFFFE, (levels << 16) | q_code)


def encode_image(y, z, y_table, z_table, header_fields, size=None):
    """header_fields = (arm, M, K, L, q_code, symbol checksum); otherwise rans_checkerboard.encode_image's arguments."""
    arm, M, K, L, q_code, csum = header_fields
    y_string, z4 = RC.encode_image(y, z, y_table, z_table, (arm, M, K, 0))
    field = (csum + quality_term(L, q_code)) % (1 << 32)
    if size is None:
        header = GAINED_HEADER.pack(VERSION, arm, M, K, L, q_code, field)
    else:
        header = GAINED_HEADER.pack(VERSION | SIZED, arm, M, K, L, q_code, (field + size_term(*size)) % (1 << 32)) + SIZE.pack(*size)
    return y_string, header + z4[HEADER.size:]


def decode_image(y_string, z_string, y_table, z_table, m, hz, wz):
    """-> (y, z, (version byte, arm, M, K, L, q_code, symbol checksum, H, W)); an unsized string gives H, W = 64 hz, 64 wz."""
    hdr = GAINED_HEADER.unpack_from(z_string, 0)
    assert hdr[0] & 0x7F == VERSION
    pos, size, field = GAINED_HEADER.size, (64 * hz, 64 * wz), hdr[6]
    if hdr[0] & SIZED:
        size = SIZE.unpack_from(z_string, pos)
        pos += SIZE.size
        field = (field - size_term(*size)) % (1 << 32)
    csum = (field - quality_term(hdr[4], hdr[5])) % (1 << 32)
    z4 = HEADER.pack(RC.VERSION, hdr[1], hdr[2], hdr[3], 0) + z_string[pos:]
    y, z, _ = RC.decode_image(y_string, z4, y_table, z_table, m, hz, wz)
    return y, z, tuple(hdr[:6]) + (csum,) + tuple(size)
