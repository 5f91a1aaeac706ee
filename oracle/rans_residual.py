"""Reference encoder / decoder of the byte format of HierarchicalMixtureResidual's coder (DESIGN.md section 11; numpy / plain Python,
test-only, the product never imports it).  The format is the single-layer one of oracle/rans.py with version byte 3, so this builds
on it (and on the per-layer lane coding of oracle/rans_scalable.py): the same lane segments, lane order, rANS arithmetic, escapes
and string layout.  Like oracle/rans.py it takes the integer tables as input, so what it pins is the format."""
from __future__ import annotations

from .rans import HEADER, Y_LANES, Z_LANES, pack, unpack
from .rans_scalable import _decode_layer, _encode_layer

RESIDUAL_VERSION = 3


def encode_residual_image(y, z, y_table, z_table, header_fields):
    """y [M, hy, wy], z [M, hz, wz] integer symbols of one image; y_table(c, i, j) / z_table(c) -> (cdf, lo, n); header_fields =
    (arm, M, K, checksum) -> (y string, z string).  Lanes: min(32, M) for y, min(4, M) for z."""
    m = y.shape[0]
    ys = _encode_layer("y", y, y_table, min(Y_LANES, m))
    zs = _encode_layer("z", z, z_table, min(Z_LANES, m))
    return pack(b"", ys), pack(HEADER.pack(RESIDUAL_VERSION, *header_fields), zs)


def decode_residual_image(y_string, z_string, y_table, z_table, hz, wz):
    """-> (y [M, 4 hz, 4 wz], z [M, hz, wz] int64, header tuple); M comes from the header."""
    hdr = HEADER.unpack_from(z_string, 0)
    assert hdr[0] == RESIDUAL_VERSION
    m = hdr[2]
    ly, lz = min(Y_LANES, m), min(Z_LANES, m)
    _, zsegs = unpack(z_string, lz, True)
    _, ysegs = unpack(y_string, ly, False)
    z = _decode_layer(zsegs, "z", m, hz, wz, lz, z_table)
    y = _decode_layer(ysegs, "y", m, 4 * hz, 4 * wz, ly, y_table)
    return y, z, hdr
