"""Entropy-coder benchmark: compress() / decompress() of JointAutoregressiveHierarchical(128, K=3), bf16x3 arm, calib weights.

Per batch size (768x512 images, B = 1 and B = 16): encode and decode time per call (host clock around calls that end in a device
synchronise; compress and decompress synchronise themselves for their device-to-host copies), images/s, coded bpp against
rd_loss's bpp_total of the same images, and the fixed per-image bytes (header, lane-length table, final rANS states) - also at
256x256.  Prints one JSON line (and writes it to --out).  Inputs are seeded uniform noise images.

    python tools/codec_bench.py --reps 3 --out profiles/r3_codec_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def fixed_bytes(strings):
    from neural_image_compression_b200 import codec
    ys, zs = strings
    out = []
    for y, z in zip(ys, zs):
        n = 0
        for s, lanes, hdr in ((y, codec.Y_LANES, False), (z, codec.Z_LANES, True)):
            _, offs, _ = codec.parse_string(s, lanes, hdr)
            n += offs[0] + 4 * lanes                       # header + lane-length table, then one 4-byte state per lane
        out.append(n)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from neural_image_compression_b200.RateDistortionLoss import rd_loss
    from tests import helpers as H
    assert torch.cuda.is_available(), "codec_bench needs a B200"
    dev = "cuda:0"
    model = H.seeded_model(128, 3, "calib", precision="bf16x3").to(dev)
    res = {"model": "JointAutoregressiveHierarchical(128, K=3) bf16x3, calib weights", **card(), "runs": []}
    for B, H_, W_ in ((1, 512, 768), (16, 512, 768), (2, 256, 256)):
        x = H.seeded_input((B, 3, H_, W_)).to(dev)
        with torch.no_grad():
            rd = rd_loss(model(x, training=False), x, 0.005)
        enc = model.compress(x)                           # warm-up of every shape the timed calls use
        model.decompress(**enc)
        torch.cuda.synchronize()
        te, td = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            enc = model.compress(x)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            model.decompress(**enc)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            te.append(t1 - t0)
            td.append(t2 - t1)
        nbytes = [len(a) + len(b) for a, b in zip(*enc["strings"])]
        fixed = fixed_bytes(enc["strings"])
        e, d = min(te), min(td)
        res["runs"].append({
            "batch": B, "size": f"{W_}x{H_}", "encode_ms": round(1e3 * e, 2), "decode_ms": round(1e3 * d, 2),
            "encode_images_per_s": round(B / e, 2), "decode_images_per_s": round(B / d, 2),
            "encode_ms_all": [round(1e3 * v, 2) for v in te], "decode_ms_all": [round(1e3 * v, 2) for v in td],
            "coded_bpp": round(8 * sum(nbytes) / (B * H_ * W_), 5), "rd_loss_bpp_total": round(float(rd["bpp_total"]), 5),
            "bytes_per_image": nbytes, "fixed_bytes_per_image": fixed,
            "fixed_share": round(max(f / n for f, n in zip(fixed, nbytes)), 5),
        })
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
