"""Reference encoder / decoder of the byte format of DESIGN.md section 9 (numpy / plain Python; test-only, the product never
imports it).  It takes the integer tables as input - CPU erf cannot reproduce the device's floats - so what it pins is the format:
lane assignment, symbol order, rANS arithmetic, escapes, string layout.

A table row is (cdf, lo, n): cdf[0] = 0 < cdf[1] < ... < cdf[n + 1] = 2^16; bin i < n is the symbol lo + i, bin n the escape."""
from __future__ import annotations

import struct

import numpy as np

PREC = 16
RANS_L = 1 << 16
VERSION = 1
Y_LANES, Z_LANES = 32, 4
HEADER = struct.Struct("<BBHBI")


def wavefront(h, w):
    """Steps of the y decode: pixel (i, j) at step 3 i + j; pixels of a step with i ascending."""
    steps = [[] for _ in range(3 * h + w - 3)]
    for i in range(h):
        for j in range(w):
            steps[3 * i + j].append((i, j))
    return [sorted(s) for s in steps]


def lane_order(kind, m, h, w, lane, lanes):
    """(c, i, j) of lane `lane` in decode order; kind "y" (wavefront) or "z" (raster)."""
    pixels = [p for s in wavefront(h, w) for p in s] if kind == "y" else [(i, j) for i in range(h) for j in range(w)]
    return [(c, i, j) for (i, j) in pixels for c in range(lane, m, lanes)]


def symbol_ops(sym, cdf, lo, n):
    """(start, freq) operations of one symbol in decode order: its bin, then for an escape the zigzag value as two raw 16-bit
    words (low half first)."""
    if lo <= sym < lo + n:
        i = sym - lo
        return [(int(cdf[i]), int(cdf[i + 1] - cdf[i]))]
    z = 2 * sym if sym >= 0 else -2 * sym - 1
    return [(int(cdf[n]), int(cdf[n + 1] - cdf[n])), (z & 0xFFFF, 1), (z >> 16, 1)]


def encode_lane(ops):
    """ops in decode order -> lane segment: final state (uint32 LE), then the 16-bit LE words in decode order."""
    x, out = RANS_L, []
    for start, freq in reversed(ops):
        while x >= (freq << 16):
            out.append(x & 0xFFFF)
            x >>= 16
        x = ((x // freq) << PREC) + (x % freq) + start
    return struct.pack("<I", x) + np.array(out[::-1], dtype="<u2").tobytes()


class LaneDecoder:
    def __init__(self, seg: bytes):
        self.x = struct.unpack_from("<I", seg, 0)[0]
        self.words = np.frombuffer(seg[4:], dtype="<u2")
        self.pos = 0

    def _next(self):
        v = int(self.words[self.pos]) if self.pos < len(self.words) else 0
        self.pos += 1
        return v

    def _advance(self, start, freq, slot):
        self.x = freq * (self.x >> PREC) + slot - start
        if self.x < RANS_L:
            self.x = (self.x << 16) | self._next()

    def symbol(self, cdf, lo, n):
        slot = self.x & 0xFFFF
        i = int(np.searchsorted(np.asarray(cdf[:n + 2]), slot, side="right")) - 1
        self._advance(int(cdf[i]), int(cdf[i + 1] - cdf[i]), slot)
        if i < n:
            return lo + i
        zlo = self.x & 0xFFFF
        self._advance(zlo, 1, zlo)
        zhi = self.x & 0xFFFF
        self._advance(zhi, 1, zhi)
        z = zlo | (zhi << 16)
        return -(z >> 1) - 1 if z & 1 else z >> 1


def _varint(n):
    out = bytearray()
    while True:
        b, n = n & 0x7F, n >> 7
        out.append(b | (0x80 if n else 0))
        if not n:
            return bytes(out)


def pack(header: bytes, segs):
    return header + b"".join(_varint((len(s) - 4) // 2) for s in segs) + b"".join(segs)


def unpack(data: bytes, lanes, header: bool):
    pos, hdr = 0, None
    if header:
        hdr = HEADER.unpack_from(data, 0)
        pos = HEADER.size
    lens = []
    for _ in range(lanes):
        n, k = 0, 0
        while True:
            b = data[pos]
            pos += 1
            n |= (b & 0x7F) << (7 * k)
            k += 1
            if not b & 0x80:
                break
        lens.append(n)
    segs = []
    for n in lens:
        segs.append(data[pos:pos + 4 + 2 * n])
        pos += 4 + 2 * n
    assert pos == len(data)
    return hdr, segs


def encode_image(y, z, y_table, z_table, header_fields):
    """y [m, hy, wy], z [m, hz, wz] integer symbols of one image; y_table(c, i, j) / z_table(c) -> (cdf, lo, n);
    header_fields = (arm, M, K, checksum) -> (y_string, z_string)."""
    m = y.shape[0]
    ly, lz = min(Y_LANES, m), min(Z_LANES, m)
    strings = []
    for kind, sym, table, lanes in (("y", y, y_table, ly), ("z", z, z_table, lz)):
        segs = []
        for lane in range(lanes):
            ops = []
            for c, i, j in lane_order(kind, m, sym.shape[1], sym.shape[2], lane, lanes):
                ops += symbol_ops(int(sym[c, i, j]), *(table(c, i, j) if kind == "y" else table(c)))
            segs.append(encode_lane(ops))
        strings.append(segs)
    return pack(b"", strings[0]), pack(HEADER.pack(VERSION, *header_fields), strings[1])


def decode_image(y_string, z_string, y_table, z_table, m, hz, wz):
    """-> (y [m, 4 hz, 4 wz], z [m, hz, wz] int64, header tuple)."""
    hy, wy = 4 * hz, 4 * wz
    ly, lz = min(Y_LANES, m), min(Z_LANES, m)
    out = {}
    hdr, zsegs = unpack(z_string, lz, True)
    _, ysegs = unpack(y_string, ly, False)
    for kind, segs, lanes, (h, w), table in (("z", zsegs, lz, (hz, wz), z_table), ("y", ysegs, ly, (hy, wy), y_table)):
        sym = np.zeros((m, h, w), dtype=np.int64)
        for lane in range(lanes):
            dec = LaneDecoder(segs[lane])
            for c, i, j in lane_order(kind, m, h, w, lane, lanes):
                sym[c, i, j] = dec.symbol(*(table(c, i, j) if kind == "y" else table(c)))
        out[kind] = sym
    return out["y"], out["z"], hdr
