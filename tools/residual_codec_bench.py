"""Coder benchmark of HierarchicalMixtureResidual(192, K=1), bf16x3 arm, calib-style weights (the g_a / h_a gains of the residual
parity cases), at 768 x 512 with B = 1 and B = 16 and at 2048 x 1536 with B = 1.

Per size: encode and decode time per call (host clock around calls that end in a device synchronise; compress and decompress
synchronise themselves for their device-to-host copies; one warm-up call first), decode time per wavefront step, split into the
step's nic_codec_params call and its nic_codec_decode_step call (CUDA events, a middle step), coded bpp against rd_loss's
bpp_total of the same images, and the fixed bytes per image (header, lane-length tables, final rANS states).

Head-to-head at the same middle step: nic_codec_decode_step against the nic_codec_tables(TABLES) + nic_codec_decode pair it
replaces, CUDA events over --step-reps launches each, the two alternated --rounds times in this one run.  Both start every launch
from the lanes' first state (init = 1) on the same raw parameters, so they decode the same symbols.  Prints one JSON line and
writes it to --out.  Inputs are seeded uniform noise images.

    python tools/residual_codec_bench.py --out profiles/r5_residual_codec_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

GAINS = (17.98, 141.28)


def fixed_bytes(strings, M):
    """Per image: header + lane-length tables + 4 state bytes per lane."""
    from neural_image_compression_b200 import codec
    out = []
    for y, z in zip(*strings):
        n = 0
        for s, lanes, skip in ((y, codec.lanes(codec.Y_LANES, M), 0), (z, codec.lanes(codec.Z_LANES, M), codec.HEADER.size)):
            _, offs, _ = codec.parse_string(s[skip:], lanes, False)
            n += skip + offs[0] + 4 * lanes                   # the lane table ends where the first segment starts
        out.append(n)
    return out


def step_head_to_head(model, out, enc, step_reps, rounds):
    """ms per launch at a middle step: the step's parameters, the one-launch step decode, and the table + decode pair."""
    import numpy as np
    import torch
    from neural_image_compression_b200 import _lib, codec, residual_codec as rc, scalable_codec as sc
    from neural_image_compression_b200._lib import CODEC_GM, check, current_stream, ptr
    from scalable_codec_bench import event_ms
    lib = _lib.load()
    y, z = out["y_in"] + 0.0, out["z_in"] + 0.0
    B, M, hy, wy = y.shape
    K = model.K
    lanes = codec.lanes(codec.Y_LANES, M)
    t = (3 * hy + wy - 3) // 2
    psi = sc.psi_nhwc(model, z.permute(0, 2, 3, 1).contiguous())
    y_nhwc = y.permute(0, 2, 3, 1).contiguous()
    step = sc.ParamHeads(model, [y_nhwc], psi, all_pixels=False)
    allpix = sc.ParamHeads(model, [y_nhwc], psi, all_pixels=True)
    allpix.run(-1)
    raw = allpix.raw[0]
    y_strings, z_strings, _, y_lanes, _ = rc._parse_all(model, enc["strings"], enc["shape"])
    start = np.cumsum([0] + [len(s) for s in y_strings])
    dev = y.device
    blob = torch.frombuffer(bytearray(b"".join(y_strings)), dtype=torch.uint8).to(dev)
    off = torch.tensor([start[b] + o for b in range(B) for o in y_lanes[b][0]], dtype=torch.int64, device=dev)
    nw = torch.tensor([n for b in range(B) for n in y_lanes[b][1]], dtype=torch.int32, device=dev)
    res = [torch.zeros((B, hy, wy, M), device=dev) for _ in range(2)]
    state = [torch.empty(B * lanes, dtype=torch.int32, device=dev) for _ in range(2)]
    pos = [torch.empty(B * lanes, dtype=torch.int32, device=dev) for _ in range(2)]
    tabs = codec.step_tables(raw, M, K, t)
    st = current_stream()

    def one():
        check(lib.nic_codec_decode_step(ptr(blob), ptr(off), ptr(nw), ptr(state[0]), ptr(pos[0]), 1, ptr(raw), B, M, K, hy, wy, lanes, t,
                                        ptr(res[0]), st), "nic_codec_decode_step")

    def pair():
        codec.step_tables(raw, M, K, t, tabs)
        check(lib.nic_codec_decode(CODEC_GM, ptr(blob), ptr(off), ptr(nw), ptr(state[1]), ptr(pos[1]), 1, ptr(tabs[0]), ptr(tabs[1]),
                                   ptr(tabs[2]), B, M, hy, wy, lanes, t, ptr(res[1]), st), "nic_codec_decode")
    one_ms, pair_ms = [], []
    for _ in range(rounds):
        one_ms.append(event_ms(one, step_reps))
        pair_ms.append(event_ms(pair, step_reps))
    assert torch.equal(res[0], res[1]) and torch.equal(state[0], state[1]) and torch.equal(pos[0], pos[1])
    return {"step": t, "step_params_ms": event_ms(lambda: step.run(t), step_reps),
            "step_decode_one_launch_ms": one_ms, "step_decode_table_pair_ms": pair_ms}


def run_case(model, B, H, W, reps, step_reps, rounds):
    import torch
    from neural_image_compression_b200.RateDistortionLoss import rd_loss
    from scalable_codec_bench import timed
    from tests import helpers as Hl
    x = Hl.seeded_input((B, 3, H, W)).cuda()
    with torch.no_grad():
        out = model(x, training=False)
        rd = rd_loss(out, x, 0.005)
    t_enc, enc = timed(lambda: model.compress(x), reps)
    t_dec, dec = timed(lambda: model.decompress(**enc), reps)
    assert torch.equal(dec["y_hat"], out["y_in"]) and torch.equal(dec["x_hat"], out["x_hat"])
    px = B * H * W
    steps = 3 * (H // 16) + W // 16 - 3
    return {
        "size": f"{W}x{H}", "batch": B, "decode_steps": steps,
        "encode_ms": 1e3 * t_enc, "decode_ms": 1e3 * t_dec, "decode_ms_per_step": 1e3 * t_dec / steps,
        "coded_bpp": 8 * sum(len(a) + len(b) for a, b in zip(*enc["strings"])) / px,
        "model_bpp_total": float(rd["bpp_total"]),
        "fixed_bytes_per_image": fixed_bytes(enc["strings"], model.M)[0],
        **step_head_to_head(model, out, enc, step_reps, rounds),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--step-reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from codec_bench import card
    from tests import helpers as Hl
    if not torch.cuda.is_available():
        raise SystemExit("residual_codec_bench needs a B200")
    model = Hl.seeded_residual_model(192, 1, *GAINS, precision="bf16x3").cuda()
    res = {"model": f"HierarchicalMixtureResidual(192, K=1), bf16x3, g_a / h_a gains {GAINS}", **card(),
           "cases": [run_case(model, B, H, W, args.reps, args.step_reps, args.rounds)
                     for B, H, W in ((1, 512, 768), (16, 512, 768), (1, 1536, 2048))]}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
