"""GPU: the bf16-pair epilogue of conv_tc_kernel through per-warp staging slices (epilogue_block_slices, the default) writes
exactly what the CTA-wide staging rounds of epilogue_block (NIC_TC_EPI_SLICES=0) write - bit for bit, in the one-CTA and the
CTA-pair form, at ragged shapes: odd tile counts, partial last tiles, widths that are not a multiple of 16, batch 1."""
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

T = nn.ConvTranspose2d
# name: (conv, epilogue, batch, h_in, w_in, out_c_total, out_c_offset); epilogue "gdn" runs the conv with a bias epilogue into
# a bf16-pair scratch and then the GDN kernel (g_a layers 2 and 3 as the bf16x3 arm runs them)
CASES = {
    "gs3": (lambda: T(128, 128, 5, 2, 2, output_padding=1), "bias", 3, 61, 101, 0, 0),       # g_s layer 3, 4 phases, 101 px per phase row
    "gs3_b1": (lambda: T(128, 128, 5, 2, 2, output_padding=1), "bias", 1, 128, 190, 0, 0),
    "ga2": (lambda: nn.Conv2d(128, 128, 5, 2, 2), "gdn", 5, 250, 382, 0, 0),                 # 125 x 191 outputs
    "ga2_b1": (lambda: nn.Conv2d(128, 128, 5, 2, 2), "gdn", 1, 256, 330, 0, 0),
    "ga3": (lambda: nn.Conv2d(128, 128, 5, 2, 2), "gdn", 7, 122, 190, 0, 0),                 # 61 x 95 outputs
    "ga3_b1": (lambda: nn.Conv2d(128, 128, 5, 2, 2), "bias", 1, 124, 186, 0, 0),
    "lrelu_192": (lambda: nn.Conv2d(128, 192, 5, 2, 2), "lrelu", 3, 90, 134, 0, 0),          # two N tiles, the second half empty
    "window": (lambda: nn.Conv2d(128, 128, 5, 2, 2), "bias", 2, 98, 150, 256, 64),           # channel window of a wider tensor
}


def _run(name, conv, x, pair, slices, monkeypatch):
    from neural_image_compression_b200 import engine, _lib
    from neural_image_compression_b200._lib import EPI_BIAS, EPI_GDN, EPI_LRELU
    from neural_image_compression_b200.gdn import GDN
    _, epi, b, h, w, ctot, coff = CASES[name]
    dev = x.device
    if epi == "gdn":
        torch.manual_seed(5)
        op = engine.ConvOp(conv, EPI_GDN, gdn=GDN(128).to(dev))
    else:
        op = engine.ConvOp(conv, EPI_LRELU if epi == "lrelu" else EPI_BIAS)
    ho, wo = engine.conv_out_hw(conv, h, w)
    c = ctot or conv.out_channels
    out = torch.full((b, ho, wo, 2 * c), -7, dtype=torch.int16, device=dev).view(torch.bfloat16)   # a pattern no kernel writes
    monkeypatch.setenv("NIC_TC_PAIR", pair)
    monkeypatch.setenv("NIC_TC_EPI_SLICES", slices)
    op.run(x, b, h, w, "bf16x3", out=out, out_c_total=ctot, out_c_offset=coff)
    torch.cuda.synchronize()
    assert _lib.load().nic_pipeline_status() == 0
    return out.view(torch.int16)


@pytest.mark.parametrize("pair", ["0", "1"])
@pytest.mark.parametrize("name", list(CASES))
def test_slices_are_bit_identical_to_the_staging_rounds(name, pair, monkeypatch):
    from neural_image_compression_b200 import engine
    dev = torch.device("cuda:0")
    torch.manual_seed(11)
    make, epi, b, h, w, ctot, coff = CASES[name]
    conv = make().to(dev)
    x = engine.to_pair(torch.randn(b, h, w, 128, device=dev))
    ref = _run(name, conv, x, pair, "0", monkeypatch)
    got = _run(name, conv, x, pair, "1", monkeypatch)
    c = conv.out_channels
    if ctot:    # the window is written, hi and lo, and nothing outside it
        for base in (coff, ctot + coff):
            assert not (ref[..., base:base + c] == -7).all()
        untouched = torch.ones(2 * ctot, dtype=torch.bool, device=dev)
        untouched[coff:coff + c] = False
        untouched[ctot + coff:ctot + coff + c] = False
        assert (got[..., untouched] == -7).all()
    else:
        assert not (ref == -7).any()
    assert torch.equal(ref, got)
