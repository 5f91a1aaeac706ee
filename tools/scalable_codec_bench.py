"""Layered-coder benchmark: compress() / decompress() / decompress(base_only=True) of ScalableImageCoding(192, 128, K=1), bf16x3
arm, calib weights (BASELINE configs[4]), at 2048 x 1536 with B = 1 and at 768 x 512 with B = 8.

Per size: encode, full decode and base-only decode time per call (host clock around calls that end in a device synchronise;
compress and decompress synchronise themselves for their device-to-host copies; one warm-up call first), coded bpp per layer
against vision_rd_loss's bpp_y1 + bpp_z, bpp_y2 and bpp_total of the same images, the fixed bytes per image (header, lane-length
tables, final rANS states), and the time of one decode step's nic_codec_params call (CUDA events, a middle step) against one
full-latent pass of the same head on the engine (context conv + the three 1x1 convs, as the eval forward runs them).  Prints one
JSON line and writes it to --out.  Inputs are seeded uniform noise images.

    python tools/scalable_codec_bench.py --out profiles/r4_scalable_codec_bench_1gpu.json
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


def fixed_bytes(strings, model):
    """Per image: header + lane-length tables + 4 state bytes per lane."""
    from neural_image_compression_b200 import codec, scalable_codec as sc
    y1s, y2s, zs = strings
    ln = [codec.lanes(codec.Y_LANES, model.M1), codec.lanes(codec.Y_LANES, model.M2), codec.lanes(codec.Z_LANES, model.M)]
    out = []
    for parts in zip(y1s, y2s, zs):
        n = sc.HEADER.size
        for s, lanes, skip in zip(parts, ln, (0, 0, sc.HEADER.size)):
            offs, _ = codec.parse_string(s[skip:], lanes, False)[1:]
            n += offs[0] + 4 * lanes                           # the lane table ends where the first segment starts
        out.append(n)
    return out


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps, r


def event_ms(fn, reps):
    import torch
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def step_kernel_vs_engine(model, out, reps):
    """ms per call: nic_codec_params at a middle step (head 1 alone, both heads) vs one full-latent engine pass of head 1 / head 2."""
    import torch
    from neural_image_compression_b200 import scalable_codec as sc
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    B, M, hy, wy = y.shape
    M1 = model.M1
    yn = y.permute(0, 2, 3, 1)
    parts = [yn[..., :M1].contiguous(), yn[..., M1:].contiguous()]
    psi = sc.psi_nhwc(model, z.permute(0, 2, 3, 1).contiguous())
    t = (3 * hy + wy - 3) // 2
    one = sc.ParamHeads(model, parts[:1], psi, all_pixels=False)
    both = sc.ParamHeads(model, parts, psi, all_pixels=False)
    allpix = sc.ParamHeads(model, parts, psi, all_pixels=True)
    res = {"step": t, "step_params_head1_ms": event_ms(lambda: one.run(t), reps),
           "step_params_both_heads_ms": event_ms(lambda: both.run(t), reps),
           "all_pixels_params_both_heads_ms": event_ms(lambda: allpix.run(-1), max(3, reps // 10))}
    yp = torch.cat([parts[0], torch.zeros_like(parts[0])], dim=-1).to(torch.bfloat16).contiguous()      # symbols: exact in bf16
    yp2 = torch.cat([parts[1], torch.zeros_like(parts[1])], dim=-1).to(torch.bfloat16).contiguous()
    for i, (ctx, ep, m, ypair) in enumerate(((model.context_model_1, model.entropy_parameters_1, M1, yp),
                                             (model.context_model_2, model.entropy_parameters_2, model.M2, yp2)), start=1):
        c = 2 * m + 2 * M
        comb = torch.zeros((B, hy, wy, 2 * c), dtype=torch.bfloat16, device=y.device)

        def engine_pass():
            ctx.masked._op.run(ypair, B, hy, wy, "bf16x3", out=comb, out_c_total=c, out_c_offset=0)
            a = ep.ops[0].run(comb, B, hy, wy, "bf16x3")
            a = ep.ops[1].run(a, B, hy, wy, "bf16x3")
            return ep.ops[2].run(a, B, hy, wy, "bf16x3", out_layout=0, out_dtype=torch.float32)
        res[f"engine_full_latent_head{i}_ms"] = event_ms(engine_pass, reps)
    return res


def run_case(model, B, H, W, reps, step_reps):
    import torch
    from neural_image_compression_b200.RateDistortionLoss import vision_rd_loss
    from tests import helpers as Hl
    x = Hl.seeded_input((B, 3, H, W)).cuda()
    with torch.no_grad():
        out = model(x, training=False)
        rd = vision_rd_loss(out, x, 0.005)
    t_enc, enc = timed(lambda: model.compress(x), reps)
    t_dec, dec = timed(lambda: model.decompress(**enc), reps)
    t_base, _ = timed(lambda: model.decompress([enc["strings"][0], None, enc["strings"][2]], enc["shape"], base_only=True), reps)
    assert torch.equal(dec["y_hat"], out["y_in"]) and torch.equal(dec["x_hat"], out["x_hat"])
    y1s, y2s, zs = enc["strings"]
    px = B * H * W
    steps = 3 * (H // 16) + W // 16 - 3
    fb = fixed_bytes(enc["strings"], model)
    return {
        "size": f"{W}x{H}", "batch": B, "decode_steps": steps,
        "encode_ms": 1e3 * t_enc, "decode_ms": 1e3 * t_dec, "decode_base_only_ms": 1e3 * t_base,
        "decode_ms_per_step": 1e3 * t_dec / steps, "decode_base_only_ms_per_step": 1e3 * t_base / steps,
        "coded_bpp_base": 8 * sum(len(a) + len(b) for a, b in zip(y1s, zs)) / px,
        "coded_bpp_y2": 8 * sum(len(s) for s in y2s) / px,
        "coded_bpp_total": 8 * sum(len(a) + len(b) + len(c) for a, b, c in zip(y1s, y2s, zs)) / px,
        "model_bpp_y1_plus_z": float(rd["bpp_y1"] + rd["bpp_z"]), "model_bpp_y2": float(rd["bpp_y2"]),
        "model_bpp_total": float(rd["bpp_total"]),
        "fixed_bytes_per_image": fb[0],
        **step_kernel_vs_engine(model, out, step_reps),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--step-reps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from codec_bench import card
    from tests import helpers as Hl
    if not torch.cuda.is_available():
        raise SystemExit("scalable_codec_bench needs a B200")
    model = Hl.seeded_scalable_model(192, 128, 1, "calib", precision="bf16x3").cuda()
    res = {"model": "ScalableImageCoding(192, 128, K=1), bf16x3, calib weights", **card(),
           "cases": [run_case(model, 1, 1536, 2048, args.reps, args.step_reps), run_case(model, 8, 512, 768, args.reps, args.step_reps)]}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
