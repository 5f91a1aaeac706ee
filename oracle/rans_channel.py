"""Reference encoder / decoder of byte format 6 (DESIGN.md section 16, ChannelCheckerboardHierarchical; numpy / plain Python,
test-only, the product never imports it).  Like oracle/rans.py it takes the integer tables as input, so what it pins is the format:
the z header <BBHBB> + S <H> slice widths + <I> checksum field (plus section 12's size extension), the y lane table and the
slice-major lanes, each slice laid out as a format-4 latent of its own channels (oracle/rans_checkerboard.py's walk)."""
from __future__ import annotations

import struct

import numpy as np

from . import rans_checkerboard as RC
from .rans import LaneDecoder, encode_lane, pack, symbol_ops, unpack
from .rans_sized import SIZE, SIZED, size_term

VERSION = 6
Z_LANES = 4


def header(S):
    return struct.Struct("<BBHBB" + "H" * S + "I")


def y_lanes(slices, hy):
    """[(slice, offset, lane within the slice)] in string order."""
    out, o = [], 0
    for s, m in enumerate(slices):
        out += [(s, o, lane) for lane in range(RC.y_lane_count(m, hy))]
        o += m
    return out


def encode_image(y, z, y_table, z_table, header_fields, slices, size=None):
    """y [M, hy, wy], z [M, hz, wz] integer symbols of one image; y_table(c, i, j) / z_table(c) -> (cdf, lo, n) with c the channel of
    the full latent; header_fields = (arm, M, K, symbol checksum); size = (H, W) for a sized string, else None."""
    M, hy, wy = y.shape
    ysegs = []
    for s, o, lane in y_lanes(slices, hy):
        ops = []
        for c, i, j in RC.y_lane_order(slices[s], hy, wy, lane):
            ops += symbol_ops(int(y[o + c, i, j]), *y_table(o + c, i, j))
        ysegs.append(encode_lane(ops))
    zsegs = []
    for lane in range(min(Z_LANES, M)):
        ops = []
        for c, i, j in RC.z_lane_order(M, *z.shape[1:], lane):
            ops += symbol_ops(int(z[c, i, j]), *z_table(c))
        zsegs.append(encode_lane(ops))
    arm, M_, K, csum = header_fields
    hdr = header(len(slices))
    if size is None:
        head = hdr.pack(VERSION, arm, M_, K, len(slices), *slices, csum)
    else:
        head = hdr.pack(VERSION | SIZED, arm, M_, K, len(slices), *slices, (csum + size_term(*size)) % (1 << 32)) + SIZE.pack(*size)
    return pack(b"", ysegs), pack(head, zsegs)


def decode_image(y_string, z_string, y_table, z_table, hz, wz):
    """-> (y [M, 4 hz, 4 wz], z [M, hz, wz] int64, (version byte, arm, M, K, slices, symbol checksum, H, W)); an unsized string gives
    H, W = 64 hz, 64 wz."""
    hy, wy = 4 * hz, 4 * wz
    v, arm, M, K, S = struct.unpack_from("<BBHBB", z_string, 0)
    assert v & 0x7F == VERSION
    hdr = header(S).unpack_from(z_string, 0)
    slices, csum = tuple(hdr[5:5 + S]), hdr[-1]
    pos, size = header(S).size, (64 * hz, 64 * wz)
    if v & SIZED:
        size = SIZE.unpack_from(z_string, pos)
        pos += SIZE.size
        csum = (csum - size_term(*size)) % (1 << 32)
    _, zsegs = unpack(z_string[pos:], min(Z_LANES, M), False)
    order = y_lanes(slices, hy)
    _, ysegs = unpack(y_string, len(order), False)
    z = np.zeros((M, hz, wz), dtype=np.int64)
    for lane, seg in enumerate(zsegs):
        dec = LaneDecoder(seg)
        for c, i, j in RC.z_lane_order(M, hz, wz, lane):
            z[c, i, j] = dec.symbol(*z_table(c))
    y = np.zeros((M, hy, wy), dtype=np.int64)
    for (s, o, lane), seg in zip(order, ysegs):
        dec = LaneDecoder(seg)
        for c, i, j in RC.y_lane_order(slices[s], hy, wy, lane):
            y[o + c, i, j] = dec.symbol(*y_table(o + c, i, j))
    return y, z, (v, arm, M, K, slices, csum) + tuple(size)
