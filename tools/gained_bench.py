"""Gain-unit benchmark (DESIGN.md section 15): GainedCheckerboardHierarchical against JointCheckerboardHierarchical, both at M = 128,
K = 3, bf16x3, calib-style weights (the same seeded draw; the gained model's log-gain rows set to linspace(log 0.25, log 4) for g and
its negation for ginv, so that the rate moves with q), alternated in one run.

Measures: the graph-replayed eval forward at 16 x 3 x 512 x 768 (CUDA events over --graph-reps replays, the two models alternated
--rounds times), the graphed training step at 8 x 3 x 256 x 256 (parallel.ShardedTrainer(graph=True); the gained one with lambdas,
alternated likewise), and encode / decode time (host clock around calls that end in a device synchronise; median of --reps calls
after a warm-up) with the coded bpp at q in {0, (L - 1) / 2, L - 1}, at 768 x 512 with B = 16 and at 1080 x 1920.  Inputs are seeded
uniform noise.  The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line and writes it to --out.

    python tools/gained_bench.py --out profiles/r8_gained_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

LAMBDAS = [0.0018, 0.0035, 0.0067, 0.013, 0.025, 0.0483]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def models():
    import torch
    from neural_image_compression_b200.Models import GainedCheckerboardHierarchical
    from checkerboard_codec_bench import models as cb_models
    parent = cb_models()["JointCheckerboardHierarchical"]()
    gained = GainedCheckerboardHierarchical(128, K=3, levels=len(LAMBDAS), precision="bf16x3")
    gained.load_state_dict(parent.state_dict(), strict=False)
    with torch.no_grad():
        for t in gained.gain_units.tables():
            t.copy_(torch.linspace(math.log(0.25), math.log(4.0), gained.levels)[:, None].expand_as(t))
        gained.gain_units.y_log_inv_gain.neg_()
        gained.gain_units.z_log_inv_gain.neg_()
    return {"JointCheckerboardHierarchical": parent, "GainedCheckerboardHierarchical": gained}


def graphed_forward_ms(model, x, reps):
    import torch
    # the gained model at its top quality, given as a device tensor: host values would be copied to the device inside the capture
    kw = {"quality": torch.full((x.shape[0],), float(model.levels - 1), device=x.device)} if hasattr(model, "levels") else {}
    with torch.no_grad():
        for _ in range(2):
            model(x, training=False, lean=True, **kw)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            model(x, training=False, lean=True, **kw)
    g.replay()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        g.replay()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_gained_bench_1gpu.json"))
    ap.add_argument("--graph-reps", type=int, default=50)
    ap.add_argument("--train-steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    from checkerboard_codec_bench import wall
    from neural_image_compression_b200 import parallel
    from neural_image_compression_b200.RateDistortionLoss import rd_terms
    from tests import helpers as Hl
    if not torch.cuda.is_available():
        raise SystemExit("tools/gained_bench.py measures on a GPU; none is visible")
    dev = "cuda:0"
    res = {"card": card(), "torch": torch.__version__}
    ms = {k: m.to(dev) for k, m in models().items()}
    # graph-replayed eval forward, alternated
    x = Hl.seeded_input((16, 3, 512, 768)).to(dev)
    fwd = {k: [] for k in ms}
    for _ in range(args.rounds):
        for k, m in ms.items():
            fwd[k].append(graphed_forward_ms(m, x, args.graph_reps))
    res["eval_forward_graphed_16x3x512x768_ms"] = {k: {"median": statistics.median(v), "all": v} for k, v in fwd.items()}
    del x
    torch.cuda.empty_cache()
    # graphed training step, alternated (each trainer keeps its own graph)
    xt = Hl.seeded_input((8, 3, 256, 256)).to(dev)
    trainers = {k: parallel.ShardedTrainer(models()[k].to(dev), **({"lambdas": LAMBDAS} if k.startswith("Gained") else {"lambda_rd": 0.0067}),
                                           graph=True) for k in ms}
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
    res["train_step_graphed_8x3x256x256_ms"] = {k: {"median": statistics.median(v), "all": v} for k, v in step.items()}
    del trainers, xt
    torch.cuda.empty_cache()
    # codec at three qualities
    gm = ms["GainedCheckerboardHierarchical"]
    L = gm.levels
    codec_res = []
    for B, H, W in ((16, 512, 768), (1, 1080, 1920)):
        x = Hl.seeded_input((B, 3, H, W)).to(dev)
        for q in (0.0, (L - 1) / 2, float(L - 1)):
            enc_t, dec_t = [], []
            for _ in range(args.reps + 1):
                t, enc = wall(lambda: gm.compress(x, quality=q))
                enc_t.append(t)
                t, _ = wall(lambda: gm.decompress(**enc))
                dec_t.append(t)
            nbytes = sum(len(a) + len(b) for a, b in zip(*enc["strings"]))
            codec_res.append({"B": B, "H": H, "W": W, "q": q, "encode_ms": 1e3 * statistics.median(enc_t[1:]),
                              "decode_ms": 1e3 * statistics.median(dec_t[1:]), "coded_bpp": 8 * nbytes / (B * H * W)})
        del x
        torch.cuda.empty_cache()
    res["codec"] = codec_res
    # coded bpp against q (768 x 512, B = 4) with the model's rate beside it
    x = Hl.seeded_input((4, 3, 512, 768)).to(dev)
    curve = []
    for q in [i * (L - 1) / 10 for i in range(11)]:
        enc = gm.compress(x, quality=q)
        with torch.no_grad():
            per_image, scal = rd_terms(gm(x, training=False, quality=q), x, 0.0)
        nbytes = sum(len(a) + len(b) for a, b in zip(*enc["strings"]))
        curve.append({"q": q, "coded_bpp": 8 * nbytes / (4 * 512 * 768), "model_bpp": float(scal[2]), "psnr": float(scal[4])})
    res["bpp_vs_q_4x512x768"] = curve
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
