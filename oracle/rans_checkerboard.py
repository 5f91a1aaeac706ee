"""Reference encoder / decoder of byte format 4 (DESIGN.md section 14, JointCheckerboardHierarchical; numpy / plain Python,
test-only, the product never imports it).  Like oracle/rans.py it takes the integer tables as input, so what it pins is the format:
the lane layout of channel classes x row bands, the two-pass order inside a lane, rANS arithmetic, escapes, string layout, and the
size extension of section 12 (written and read here directly, as oracle/rans_sized.py does for formats 1-3)."""
from __future__ import annotations

import struct

import numpy as np

from .rans import HEADER, LaneDecoder, encode_lane, pack, symbol_ops, unpack
from .rans_sized import SIZE, SIZED, size_term

VERSION = 4
Y_CLASSES, Z_LANES, BAND_ROWS = 32, 4, 16


def y_lane_count(m, hy):
    return min(Y_CLASSES, m) * -(-hy // BAND_ROWS)


def y_lane_order(m, h, w, lane):
    """(c, i, j) of y lane `lane` in decode order: lane r * Lc + l holds the channels c = l (mod Lc) of the rows [16 r, 16 r + 16);
    pass 0 = its anchors (i + j even) in raster order, each pixel's channels ascending; pass 1 = its non-anchors likewise."""
    lc = min(Y_CLASSES, m)
    r, l = divmod(lane, lc)
    rows = range(BAND_ROWS * r, min(BAND_ROWS * (r + 1), h))
    return [(c, i, j) for s in (0, 1) for i in rows for j in range(w) if (i + j + s) % 2 == 0 for c in range(l, m, lc)]


def z_lane_order(m, h, w, lane):
    return [(c, i, j) for i in range(h) for j in range(w) for c in range(lane, m, min(Z_LANES, m))]


def encode_image(y, z, y_table, z_table, header_fields, size=None):
    """y [m, hy, wy], z [m, hz, wz] integer symbols of one image; y_table(c, i, j) / z_table(c) -> (cdf, lo, n); header_fields =
    (arm, M, K, symbol checksum); size = (H, W) for a sized string, else None -> (y_string, z_string)."""
    m, hy, wy = y.shape
    ysegs = []
    for lane in range(y_lane_count(m, hy)):
        ops = []
        for c, i, j in y_lane_order(m, hy, wy, lane):
            ops += symbol_ops(int(y[c, i, j]), *y_table(c, i, j))
        ysegs.append(encode_lane(ops))
    zsegs = []
    for lane in range(min(Z_LANES, m)):
        ops = []
        for c, i, j in z_lane_order(m, *z.shape[1:], lane):
            ops += symbol_ops(int(z[c, i, j]), *z_table(c))
        zsegs.append(encode_lane(ops))
    arm, M, K, csum = header_fields
    if size is None:
        header = HEADER.pack(VERSION, arm, M, K, csum)
    else:
        header = HEADER.pack(VERSION | SIZED, arm, M, K, (csum + size_term(*size)) % (1 << 32)) + SIZE.pack(*size)
    return pack(b"", ysegs), pack(header, zsegs)


def decode_image(y_string, z_string, y_table, z_table, m, hz, wz):
    """-> (y [m, 4 hz, 4 wz], z [m, hz, wz] int64, (version byte, arm, M, K, symbol checksum, H, W)); an unsized string gives
    H, W = 64 hz, 64 wz."""
    hy, wy = 4 * hz, 4 * wz
    hdr = HEADER.unpack_from(z_string, 0)
    assert hdr[0] & 0x7F == VERSION
    size, csum = (64 * hz, 64 * wz), hdr[4]
    if hdr[0] & SIZED:
        size = SIZE.unpack_from(z_string, HEADER.size)
        csum = (csum - size_term(*size)) % (1 << 32)
        z_string = HEADER.pack(VERSION, *hdr[1:]) + z_string[HEADER.size + SIZE.size:]
    _, zsegs = unpack(z_string, min(Z_LANES, m), True)
    _, ysegs = unpack(y_string, y_lane_count(m, hy), False)
    z = np.zeros((m, hz, wz), dtype=np.int64)
    for lane, seg in enumerate(zsegs):
        dec = LaneDecoder(seg)
        for c, i, j in z_lane_order(m, hz, wz, lane):
            z[c, i, j] = dec.symbol(*z_table(c))
    y = np.zeros((m, hy, wy), dtype=np.int64)
    for lane, seg in enumerate(ysegs):
        dec = LaneDecoder(seg)
        for c, i, j in y_lane_order(m, hy, wy, lane):
            y[c, i, j] = dec.symbol(*y_table(c, i, j))
    return y, z, (hdr[0],) + tuple(hdr[1:4]) + (csum,) + tuple(size)
