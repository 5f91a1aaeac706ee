"""Reference encoder / decoder of the layered byte format of ScalableImageCoding (DESIGN.md section 10; numpy / plain Python,
test-only, the product never imports it).  It builds on oracle/rans.py, the reference coder of the single-layer format: the same
lane segments, lane order, rANS arithmetic and escapes, with three strings per image (y1, y2, z) and a header of its own.  Like
oracle/rans.py it takes the integer tables as input, so what it pins is the format."""
from __future__ import annotations

import struct

import numpy as np

from .rans import Y_LANES, Z_LANES, LaneDecoder, encode_lane, lane_order, pack, symbol_ops, unpack

SCALABLE_VERSION = 2
SCALABLE_HEADER = struct.Struct("<BBHHBII")      # version, arm, M, M1, K, base checksum, enhancement checksum


def _encode_layer(kind, sym, table, lanes):
    m, h, w = sym.shape
    segs = []
    for lane in range(lanes):
        ops = []
        for c, i, j in lane_order(kind, m, h, w, lane, lanes):
            ops += symbol_ops(int(sym[c, i, j]), *(table(c, i, j) if kind == "y" else table(c)))
        segs.append(encode_lane(ops))
    return segs


def _decode_layer(segs, kind, m, h, w, lanes, table):
    sym = np.zeros((m, h, w), dtype=np.int64)
    for lane in range(lanes):
        dec = LaneDecoder(segs[lane])
        for c, i, j in lane_order(kind, m, h, w, lane, lanes):
            sym[c, i, j] = dec.symbol(*(table(c, i, j) if kind == "y" else table(c)))
    return sym


def encode_scalable_image(y1, y2, z, y1_table, y2_table, z_table, header_fields):
    """y1 [M1, hy, wy], y2 [M2, hy, wy], z [M, hz, wz] integer symbols of one image; y*_table(c, i, j) (c = the head's channel) /
    z_table(c) -> (cdf, lo, n); header_fields = (arm, M, M1, K, base checksum, enhancement checksum) -> (y1, y2, z strings).
    Lanes: min(32, M1) for y1, min(32, M2) for y2, min(4, M) for z."""
    y1s = _encode_layer("y", y1, y1_table, min(Y_LANES, y1.shape[0]))
    y2s = _encode_layer("y", y2, y2_table, min(Y_LANES, y2.shape[0]))
    zs = _encode_layer("z", z, z_table, min(Z_LANES, z.shape[0]))
    return pack(b"", y1s), pack(b"", y2s), pack(SCALABLE_HEADER.pack(SCALABLE_VERSION, *header_fields), zs)


def decode_scalable_image(y1_string, y2_string, z_string, y1_table, y2_table, z_table, hz, wz):
    """-> (y1 [M1, 4 hz, 4 wz], y2 [M2, ...] or None when y2_string is None (the base layer alone), z [M, hz, wz], header tuple);
    M, M1 come from the header."""
    hdr = SCALABLE_HEADER.unpack_from(z_string, 0)
    assert hdr[0] == SCALABLE_VERSION
    M, M1 = hdr[2], hdr[3]
    hy, wy = 4 * hz, 4 * wz
    _, zsegs = unpack(z_string[SCALABLE_HEADER.size:], min(Z_LANES, M), False)
    z = _decode_layer(zsegs, "z", M, hz, wz, min(Z_LANES, M), z_table)
    _, segs = unpack(y1_string, min(Y_LANES, M1), False)
    y1 = _decode_layer(segs, "y", M1, hy, wy, min(Y_LANES, M1), y1_table)
    y2 = None
    if y2_string is not None:
        _, segs = unpack(y2_string, min(Y_LANES, M - M1), False)
        y2 = _decode_layer(segs, "y", M - M1, hy, wy, min(Y_LANES, M - M1), y2_table)
    return y1, y2, z, hdr
