"""Reference encoder / decoder of the size extension of DESIGN.md section 12, shared by the three byte formats (numpy / plain
Python, test-only, the product never imports it).  A sized z string is the unsized one of oracle/rans.py (version 1),
oracle/rans_scalable.py (version 2) or oracle/rans_residual.py (version 3) with three changes: bit 7 of the version byte set, every
checksum field holding the symbol checksum plus size_term(H, W) mod 2^32, and <HH> = (H, W) between the header and the lane table.
y, y1 and y2 strings do not change.  So the coders here write the unsized strings with those coders and apply the three changes,
and read them by undoing the changes."""
from __future__ import annotations

import struct

from .rans import HEADER, decode_image, encode_image
from .rans_residual import decode_residual_image, encode_residual_image
from .rans_scalable import SCALABLE_HEADER, decode_scalable_image, encode_scalable_image

SIZED = 0x80
SIZE = struct.Struct("<HH")
CHECKSUM_FIELDS = {1: (HEADER, (4,)), 2: (SCALABLE_HEADER, (5, 6)), 3: (HEADER, (4,))}    # header, checksum field indices


def mix32(idx, v):
    """The 32-bit mix of the product's symbol checksum (csrc/codec.cu), on Python ints."""
    m = 0xFFFFFFFF
    h = ((idx * 0x9E3779B1) & m) ^ ((v + 0x7F4A7C15) & m)
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & m
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & m
    return h ^ (h >> 16)


def size_term(h, w):
    return mix32(0xFFFFFFFF, (h << 16) | w)


def to_sized(z_string, size):
    """An unsized z string of any of the three formats -> the sized string of an image of size = (H, W)."""
    header, fields = CHECKSUM_FIELDS[z_string[0]]
    hdr = list(header.unpack_from(z_string, 0))
    hdr[0] |= SIZED
    for i in fields:
        hdr[i] = (hdr[i] + size_term(*size)) % (1 << 32)
    return header.pack(*hdr) + SIZE.pack(*size) + z_string[header.size:]


def from_sized(z_string):
    """A sized z string -> (the unsized string, (H, W))."""
    assert z_string[0] & SIZED
    header, fields = CHECKSUM_FIELDS[z_string[0] & 0x7F]
    hdr = list(header.unpack_from(z_string, 0))
    size = SIZE.unpack_from(z_string, header.size)
    hdr[0] &= 0x7F
    for i in fields:
        hdr[i] = (hdr[i] - size_term(*size)) % (1 << 32)
    return header.pack(*hdr) + z_string[header.size + SIZE.size:], size


def encode_sized_image(version, size, *args):
    """encode_image (version 1), encode_scalable_image (2) or encode_residual_image (3) with the same arguments (header fields with
    the symbol checksums), the z string (the last) written for an image of size = (H, W)."""
    enc = {1: encode_image, 2: encode_scalable_image, 3: encode_residual_image}[version]
    strings = enc(*args)
    return strings[:-1] + (to_sized(strings[-1], size),)


def decode_sized_image(version, *args):
    """decode_image (version 1), decode_scalable_image (2) or decode_residual_image (3) of sized strings, with the same arguments ->
    their results, the header tuple as stored (version byte with bit 7) but with the symbol checksums, followed by (H, W)."""
    strings = list(args)
    at = 2 if version == 2 else 1                                # the z string
    stored = strings[at][0]
    strings[at], size = from_sized(strings[at])
    dec = {1: decode_image, 2: decode_scalable_image, 3: decode_residual_image}[version]
    out = dec(*strings)
    return out[:-1] + ((stored,) + tuple(out[-1][1:]) + tuple(size),)
