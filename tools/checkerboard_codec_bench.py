"""Checkerboard coder benchmark (DESIGN.md section 14): JointCheckerboardHierarchical against JointAutoregressiveHierarchical, both
at M = 128, K = 3, bf16x3, calib-style weights (the same seeded draw), alternated call by call in one run.

Per size (768 x 512 at B = 1 and 16, 1080 x 1920 and 3024 x 4032 at B = 1): encode and decode time per call of both models (host
clock around calls that end in a device synchronise - compress and decompress synchronise themselves for their device-to-host copies;
one warm-up call of each first; the median of --reps alternated calls), the checkerboard model's coded bits against its model bits
(rd_terms of the eval forward on the padded image), and the two parts of a checkerboard decode pass timed alone with CUDA events:
the parameter pass (codec.ParamPath.raw: hand-off + context conv + anchor zeroing + 1x1 stack) and the decode-pass kernel
(nic_codec_decode_pass, pass 1).  Last, the graph-replayed eval forward of both models at 16 x 3 x 512 x 768 (CUDA events over
--graph-reps replays), whose difference is what the anchor-zeroing launch costs.  Inputs are seeded uniform noise.  Prints one JSON
line and writes it to --out.

    python tools/checkerboard_codec_bench.py --out profiles/r7_checkerboard_codec_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SIZES = ((1, 512, 768), (16, 512, 768), (1, 1080, 1920), (1, 3024, 4032))


def models():
    import torch
    from neural_image_compression_b200.Models import JointCheckerboardHierarchical
    from tests import helpers as Hl

    def cb():
        torch.manual_seed(0)
        m = JointCheckerboardHierarchical(128, K=3, precision="bf16x3")
        m.load_state_dict(Hl.apply_init({k: v.clone() for k, v in m.state_dict().items()}, "calib"))
        return m
    return {"JointAutoregressiveHierarchical": lambda: Hl.seeded_model(128, 3, "calib", precision="bf16x3"),
            "JointCheckerboardHierarchical": cb}


def wall(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


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


def pass_parts(model, x, reps):
    """(parameter pass ms, decode-pass kernel ms) of the checkerboard decoder at x's size."""
    import torch
    from neural_image_compression_b200 import _lib, checkerboard_codec, codec
    from neural_image_compression_b200._lib import current_stream, ptr
    enc = model.compress(x)
    (_, _, _, y_lanes, _, _) = checkerboard_codec._parse_sized(model, enc["strings"], enc["shape"])
    with torch.no_grad():
        out = model(x, training=False)
    B, M, hy, wy = out["y_in"].shape
    ys = enc["strings"][0]
    blob = torch.frombuffer(bytearray(b"".join(ys)), dtype=torch.uint8).cuda()
    import numpy as np
    start = np.cumsum([0] + [len(s) for s in ys])
    off = torch.tensor([start[b] + o for b in range(B) for o in y_lanes[b][0]], dtype=torch.int64).cuda()
    nw = torch.tensor([n for b in range(B) for n in y_lanes[b][1]], dtype=torch.int32).cuda()
    path = codec.ParamPath(model, B, hy, wy, x.device)
    _, comb = path.hyper(out["z_in"].permute(0, 2, 3, 1).contiguous())
    y_nhwc = out["y_in"].permute(0, 2, 3, 1).contiguous()
    raw = path.raw(y_nhwc, comb)
    lc, lr = checkerboard_codec.y_lanes(M, hy)
    state, pos = torch.zeros(B * lc * lr, dtype=torch.int32).cuda(), torch.zeros(B * lc * lr, dtype=torch.int32).cuda()
    scratch = torch.zeros_like(y_nhwc)
    lib = _lib.load()
    t_param = event_ms(lambda: path.raw(y_nhwc, comb), reps)
    t_pass = event_ms(lambda: lib.nic_codec_decode_pass(ptr(blob), ptr(off), ptr(nw), ptr(state), ptr(pos), ptr(raw), B, M, 3, hy, wy, lc,
                                                        checkerboard_codec.BAND_ROWS, 1, ptr(scratch), current_stream()), reps)
    return t_param, t_pass


def graph_forward_ms(model, reps):
    import torch
    from tests import helpers as Hl
    x = Hl.seeded_input((16, 3, 512, 768)).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        for _ in range(2):
            model(x, training=False)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g), torch.no_grad():
        model(x, training=False)
    return event_ms(g.replay, reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--part-reps", type=int, default=20)
    ap.add_argument("--graph-reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    from codec_bench import card
    from neural_image_compression_b200.RateDistortionLoss import rd_terms
    from tests import helpers as Hl
    if not torch.cuda.is_available():
        raise SystemExit("checkerboard_codec_bench needs a B200")
    ms = {name: make().cuda() for name, make in models().items()}
    res = {**card(), "config": "M=128, K=3, bf16x3, calib weights", "sizes": []}
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
                t, dec = wall(lambda: m.decompress(**encs[name]))
                times[name]["decode"].append(t)
        for name, m in ms.items():
            with torch.no_grad():
                out = m(xp, training=False)
            per_image, _ = rd_terms(out, xp, 0.005)
            model_bits = float((per_image[0] + per_image[1]).double().sum())
            coded = 8 * sum(len(s) for layer in encs[name]["strings"] for s in layer)
            row[name] = {"encode_ms": 1e3 * statistics.median(times[name]["encode"]), "decode_ms": 1e3 * statistics.median(times[name]["decode"]),
                         "coded_bits": coded, "model_bits": model_bits, "coded_over_model_bits": coded / model_bits}
        cb = ms["JointCheckerboardHierarchical"]
        row["decode_speedup"] = row["JointAutoregressiveHierarchical"]["decode_ms"] / row["JointCheckerboardHierarchical"]["decode_ms"]
        t_param, t_pass = pass_parts(cb, xp, args.part_reps)
        row["checkerboard_parameter_pass_ms"], row["checkerboard_decode_pass_kernel_ms"] = t_param, t_pass
        res["sizes"].append(row)
        print(json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    res["graph_forward_16x3x512x768_ms"] = {}
    for _ in range(2):                                                    # alternated
        for name, m in ms.items():
            res["graph_forward_16x3x512x768_ms"].setdefault(name, []).append(graph_forward_ms(m, args.graph_reps))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
