"""Any-size coder benchmark (DESIGN.md section 12): the three models at 1080 x 1920 (B = 1 and B = 8) and 3024 x 4032 (B = 1).

Per model and size: encode and decode time per call (host clock around calls that end in a device synchronise - compress and
decompress synchronise themselves for their device-to-host copies; one warm-up call first), coded bits per original pixel next to
the model's bits per padded pixel (rd_terms of the eval forward on the edge-padded image), and the extra bytes of a sized header.
The window kernel (nic_image_window) is timed with CUDA events over --window-reps launches for the encoder's pad and the decoder's
crop at each size; its bytes (source read once + destination written) over that time are reported as a share of the device-to-device
copy bandwidth measured in the same run (torch copy of a 2 GiB buffer, far larger than L2).  Models: JointAutoregressiveHierarchical
(128, K=3), ScalableImageCoding(192, 128, K=1) and HierarchicalMixtureResidual(192, K=1), bf16x3, calib-style weights; inputs are
seeded uniform noise.  Prints one JSON line and writes it to --out.

    python tools/any_size_codec_bench.py --out profiles/r6_any_size_codec_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SIZES = ((1, 1080, 1920), (8, 1080, 1920), (1, 3024, 4032))
RESIDUAL_GAINS = (17.98, 141.28)


def models():
    from tests import helpers as Hl
    return {
        "JointAutoregressiveHierarchical(128, K=3)": lambda: Hl.seeded_model(128, 3, "calib", precision="bf16x3"),
        "ScalableImageCoding(192, 128, K=1)": lambda: Hl.seeded_scalable_model(192, 128, 1, "calib", precision="bf16x3"),
        "HierarchicalMixtureResidual(192, K=1)": lambda: Hl.seeded_residual_model(192, 1, *RESIDUAL_GAINS, precision="bf16x3"),
    }


def timed(fn, reps):
    import torch
    fn()                                                       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps, out


def event_ms(fn, reps):
    import torch
    fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / reps


def copy_bandwidth():
    """Bytes per second of a device-to-device copy of 2 GiB (read + write)."""
    import torch
    a = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    ms = event_ms(lambda: b.copy_(a), 20)
    return 2 * a.numel() * 4 / (ms * 1e-3)


def window_case(B, H, W, reps, bw):
    import torch
    from neural_image_compression_b200 import codec
    torch.manual_seed(0)
    x = torch.rand((B, 3, H, W), device="cuda")
    hp, wp = 64 * (-(-H // 64)), 64 * (-(-W // 64))
    xp = codec.window(x, hp, wp)
    out = {}
    for what, src, h, w in (("pad", x, hp, wp), ("crop", xp, H, W)):
        ms = event_ms(lambda: codec.window(src, h, w), reps)
        nbytes = 4 * B * 3 * (H * W + hp * wp)
        out[what] = {"ms": ms, "bytes": nbytes, "share_of_copy_bandwidth": nbytes / (ms * 1e-3) / bw}
    return out


def coder_case(model, B, H, W, reps):
    import torch
    import torch.nn.functional as F
    from neural_image_compression_b200 import codec, scalable_codec
    from neural_image_compression_b200.RateDistortionLoss import rd_terms
    from tests import helpers as Hl
    x = Hl.seeded_input((B, 3, H, W)).cuda()
    hp, wp = 64 * (-(-H // 64)), 64 * (-(-W // 64))
    xp = F.pad(x, (0, wp - W, 0, hp - H), mode="replicate")
    with torch.no_grad():
        out = model(xp, training=False)
    model_bits = 0.0
    for key in ("logp_y1", "logp_y2") if "logp_y1" in out else ("logp_y",):
        per_image, _ = rd_terms({"x_hat": out["x_hat"], "logp_y": out[key], "logp_z": out["logp_z"]}, xp, 0.005)
        model_bits += float(per_image[0].double().sum())
    model_bits += float(per_image[1].double().sum())
    t_enc, enc = timed(lambda: model.compress(x), reps)
    t_dec, dec = timed(lambda: model.decompress(**enc), reps)
    assert torch.equal(dec["y_hat"], out["y_in"]) and torch.equal(dec["x_hat"], out["x_hat"][..., :H, :W])
    coded = 8 * sum(len(s) for layer in enc["strings"] for s in layer)
    header = scalable_codec.HEADER if "logp_y1" in out else codec.HEADER
    return {"batch": B, "size": f"{W}x{H}", "padded": f"{wp}x{hp}", "encode_ms": 1e3 * t_enc, "decode_ms": 1e3 * t_dec,
            "coded_bits_per_original_pixel": coded / (B * H * W), "model_bits_per_padded_pixel": model_bits / (B * hp * wp),
            "sized_header_extra_bytes": codec.SIZE.size, "z_header_bytes": header.size + codec.SIZE.size}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--window-reps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from codec_bench import card
    if not torch.cuda.is_available():
        raise SystemExit("any_size_codec_bench needs a B200")
    bw = copy_bandwidth()
    res = {**card(), "copy_bandwidth_GBps": bw / 1e9,
           "window": {f"{W}x{H}x{B}": window_case(B, H, W, args.window_reps, bw) for B, H, W in SIZES}, "models": {}}
    for name, make in models().items():
        model = make().cuda()
        res["models"][name] = [coder_case(model, B, H, W, args.reps) for B, H, W in SIZES]
        del model
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
