"""Space-channel coder benchmark (DESIGN.md section 16): ChannelCheckerboardHierarchical (64-channel slices) against
JointCheckerboardHierarchical at M = 128 and 192, K = 3, bf16x3, calib-style weights (the same seeded trunk; the sigma biases of every
slice head raised as the parent's), alternated call by call in one run.

Per M: the graph-replayed eval forward at 16 x 3 x 512 x 768 (CUDA events over --graph-reps replays, lean outputs), the graphed
training step at 8 x 3 x 256 x 256 (parallel.ShardedTrainer(graph=True), CUDA events over --train-steps steps), and per size
(768 x 512 at B = 1 and 16, 1080 x 1920 and 3024 x 4032 at B = 1) encode and decode time per call (host clock around calls that end in
a device synchronise; one warm-up call each, then the median of --reps alternated calls), coded bits over model bits (rd_terms of the
eval forward on the padded image), and one decode parameter pass and one decode-pass launch of the channel model timed alone with CUDA
events (slice 1's parameters: hand-off + two context convs + 1x1 stack; slice 1's pass-1 kernel).  Inputs are seeded uniform noise.
The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line and writes it to --out.

    python tools/channel_codec_bench.py --out profiles/r9_channel_codec_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SIZES = ((1, 512, 768), (16, 512, 768), (1, 1080, 1920), (1, 3024, 4032))


def models(M: int = 128):
    """{name: constructor} of the two models at M (calib weights for 128, calib192 for 192)."""
    import torch
    from neural_image_compression_b200.Models import ChannelCheckerboardHierarchical, JointCheckerboardHierarchical
    from tests import helpers as Hl
    from tests.test_channel_host import apply_channel_init
    init = "calib" if M == 128 else "calib192"

    def cb():
        torch.manual_seed(0)
        m = JointCheckerboardHierarchical(M, K=3, precision="bf16x3")
        m.load_state_dict(Hl.apply_init({k: v.clone() for k, v in m.state_dict().items()}, init))
        return m

    def ch():
        torch.manual_seed(0)
        m = ChannelCheckerboardHierarchical(M, K=3, precision="bf16x3")
        m.load_state_dict(apply_channel_init({k: v.clone() for k, v in m.state_dict().items()}, init))
        return m
    return {"JointCheckerboardHierarchical": cb, "ChannelCheckerboardHierarchical": ch}


def decode_parts(model, x, reps):
    """(parameter pass ms, decode-pass kernel ms) of slice 1 of the channel decoder at x's size."""
    import numpy as np
    import torch
    from checkerboard_codec_bench import event_ms
    from neural_image_compression_b200 import _lib, channel_codec
    from neural_image_compression_b200._lib import current_stream, ptr
    enc = model.compress(x)
    _, _, _, y_lanes, _, _ = channel_codec._parse_sized(model, enc["strings"], enc["shape"])
    with torch.no_grad():
        out = model(x, training=False)
    B, M, hy, wy = out["y_in"].shape
    ys = enc["strings"][0]
    sl = channel_codec.slice_lanes(model.slices, hy)
    first = sl[0][1]
    lc, ln = sl[1]
    start = np.cumsum([0] + [len(s) for s in ys])
    blob = torch.frombuffer(bytearray(b"".join(ys)), dtype=torch.uint8).cuda()
    off = torch.tensor([start[b] + y_lanes[b][0][first + l] for b in range(B) for l in range(ln)], dtype=torch.int64).cuda()
    nw = torch.tensor([y_lanes[b][1][first + l] for b in range(B) for l in range(ln)], dtype=torch.int32).cuda()
    path = channel_codec.SlicePath(model, B, hy, wy, x.device)
    path.hyper(out["z_in"].permute(0, 2, 3, 1).contiguous())
    y_nhwc = out["y_in"].permute(0, 2, 3, 1).contiguous()
    raw = path.raw(1, path.symbols(y_nhwc))
    state, pos = torch.zeros(B * ln, dtype=torch.int32).cuda(), torch.zeros(B * ln, dtype=torch.int32).cuda()
    scratch = torch.zeros_like(y_nhwc)
    lib = _lib.load()
    o, m = model.offsets[1], model.slices[1]
    t_param = event_ms(lambda: path.raw(1, path.symbols(y_nhwc)), reps)
    t_pass = event_ms(lambda: lib.nic_codec_decode_pass_slice(ptr(blob), ptr(off), ptr(nw), ptr(state), ptr(pos), ptr(raw), B, M, o, m, 3,
                                                              hy, wy, lc, channel_codec.BAND_ROWS, 1, ptr(scratch), current_stream()), reps)
    return t_param, t_pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--part-reps", type=int, default=20)
    ap.add_argument("--graph-reps", type=int, default=30)
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ms", default="128,192")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    from checkerboard_codec_bench import wall
    from codec_bench import card
    from gained_bench import graphed_forward_ms
    from neural_image_compression_b200 import parallel
    from neural_image_compression_b200.RateDistortionLoss import rd_terms
    from tests import helpers as Hl
    if not torch.cuda.is_available():
        raise SystemExit("channel_codec_bench needs a B200")
    res = {**card(), "config": "K=3, bf16x3, calib weights (calib192 at M = 192), 64-channel slices", "by_M": {}}
    for M in [int(v) for v in args.ms.split(",")]:
        ms = {name: make().cuda() for name, make in models(M).items()}
        r = {}
        x = Hl.seeded_input((16, 3, 512, 768)).cuda()
        fwd = {k: [] for k in ms}
        for _ in range(args.rounds):
            for k, m in ms.items():
                fwd[k].append(graphed_forward_ms(m, x, args.graph_reps))
        r["eval_forward_graphed_16x3x512x768_ms"] = {k: {"median": statistics.median(v), "all": v} for k, v in fwd.items()}
        del x
        xt = Hl.seeded_input((8, 3, 256, 256)).cuda()
        trainers = {k: parallel.ShardedTrainer(make().cuda(), lambda_rd=0.0067, graph=True) for k, make in models(M).items()}
        for tr in trainers.values():
            for _ in range(3):
                tr.step(xt)
        torch.cuda.synchronize()
        step = {k: [] for k in trainers}
        for _ in range(args.rounds):
            for k, tr in trainers.items():
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for _ in range(args.train_steps):
                    tr.step(xt)
                e.record()
                e.synchronize()
                step[k].append(s.elapsed_time(e) / args.train_steps)
        r["train_step_graphed_8x3x256x256_ms"] = {k: {"median": statistics.median(v), "all": v} for k, v in step.items()}
        del trainers, xt
        torch.cuda.empty_cache()
        r["sizes"] = []
        for B, H, W in SIZES:
            x = Hl.seeded_input((B, 3, H, W)).cuda()
            hp, wp = 64 * (-(-H // 64)), 64 * (-(-W // 64))
            xp = F.pad(x, (0, wp - W, 0, hp - H), mode="replicate")
            row = {"batch": B, "size": f"{W}x{H}"}
            encs = {name: m.compress(x) for name, m in ms.items()}            # warm-up
            for name, m in ms.items():
                m.decompress(**encs[name])
            times = {name: {"encode": [], "decode": []} for name in ms}
            for _ in range(args.reps):                                        # alternated
                for name, m in ms.items():
                    t, encs[name] = wall(lambda: m.compress(x))
                    times[name]["encode"].append(t)
                    t, _ = wall(lambda: m.decompress(**encs[name]))
                    times[name]["decode"].append(t)
            for name, m in ms.items():
                with torch.no_grad():
                    out = m(xp, training=False)
                per_image, _ = rd_terms(out, xp, 0.005)
                model_bits = float((per_image[0] + per_image[1]).double().sum())
                coded = 8 * sum(len(s) for layer in encs[name]["strings"] for s in layer)
                row[name] = {"encode_ms": 1e3 * statistics.median(times[name]["encode"]),
                             "decode_ms": 1e3 * statistics.median(times[name]["decode"]),
                             "coded_bits": coded, "model_bits": model_bits, "coded_over_model_bits": coded / model_bits}
                del out
            t_param, t_pass = decode_parts(ms["ChannelCheckerboardHierarchical"], xp, args.part_reps)
            row["channel_parameter_pass_ms"], row["channel_decode_pass_kernel_ms"] = t_param, t_pass
            r["sizes"].append(row)
            print(json.dumps({"M": M, **row}), flush=True)
            del x, xp, encs
            torch.cuda.empty_cache()
        res["by_M"][str(M)] = r
        del ms
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
