"""MS-SSIM training benchmark: the backward kernel nic_ms_ssim_bwd alone, and the graphed training step with the MS-SSIM loss
against the MSE step.

Kernel: nic_ms_ssim_bwd (five tile launches, one per level) at 8 x 3 x 256 x 256 (the training crop) and 16 x 3 x 768 x 512, CUDA
events over --reps calls after a warm-up, inputs are seeded uniform images and x_hat = x + 5 % noise.  The FLOPs and bytes are
counted from the shapes (the work the algorithm needs, not the halo the tiles recompute): per pixel of a level, six moment maps
and three transposed maps, each a separable 11-tap filter (2 x 11 FMAs = 44 FLOPs), plus about 40 FLOPs for the derivative and
the gather; bytes = x, y read and the gradient written once per level pixel, the coarser gradient read once per pixel.  The fp32
CUDA-core bound is 148 SMs x 128 FMA lanes x 2 FLOPs x the max SM clock read in this run; the memory bound 7.7 TB/s.  The
working set of the small case fits in L2.

Step: parallel.ShardedTrainer(graph=True) at BASELINE configs[3] (JointAutoregressiveHierarchical(128, K=3), bf16x3, 8 x 3 x 256 x
256), distortion "mse" against "ms-ssim", --steps replays each, CUDA events, the two alternated --rounds times in this run.

    python tools/ms_ssim_train_bench.py --out profiles/r7_ms_ssim_train_bench_1gpu.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1]), "max_sm_clock_mhz": float(q[2])}


def levels(h, w):
    out = [(h, w)]
    for _ in range(4):
        h, w = (h + h % 2) // 2, (w + w % 2) // 2
        out.append((h, w))
    return out


def counts(planes, h, w):
    flops = bytes_ = 0
    for i, (lh, lw) in enumerate(levels(h, w)):
        px = planes * lh * lw
        flops += px * (9 * 44 + 40)
        bytes_ += px * 12 + (planes * levels(h, w)[i + 1][0] * levels(h, w)[i + 1][1] * 4 if i < 4 else 0)
    return flops, bytes_


def kernel_ms(shape, reps):
    import torch
    from neural_image_compression_b200 import _lib
    from neural_image_compression_b200.Evaluator import combine_levels, ms_ssim_levels, term_grads
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(3)
    y = torch.rand(shape, device="cuda", generator=g)
    x = y + 0.05 * torch.randn(shape, device="cuda", generator=g)
    b, c, h, w = shape
    ws = torch.empty(lib.nic_ms_ssim_bwd_workspace_bytes(b * c, h, w), dtype=torch.uint8, device="cuda")
    terms, val = combine_levels(ms_ssim_levels(x, y, workspace=ws))
    coef = term_grads(terms, val) / (b * c)
    gx = torch.empty_like(x)

    def call():
        _lib.check(lib.nic_ms_ssim_bwd(_lib.ptr(x), _lib.ptr(y), b * c, h, w, 1.0, _lib.ptr(coef), _lib.ptr(gx), _lib.ptr(ws),
                                       ws.numel(), _lib.current_stream()), "nic_ms_ssim_bwd")
    for _ in range(10):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from neural_image_compression_b200 import parallel
    from tests import helpers as H
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card()}
    fp32_peak = 148 * 128 * 2 * res["card"]["max_sm_clock_mhz"] * 1e6
    res["kernel"] = []
    for shape in [(8, 3, 256, 256), (16, 3, 768, 512)]:
        ms = kernel_ms(shape, a.reps)
        flops, nbytes = counts(shape[0] * shape[1], shape[2], shape[3])
        t_c, t_m = flops / fp32_peak, nbytes / 7.7e12
        res["kernel"].append({"shape": shape, "ms": ms, "gflop": flops / 1e9, "mbytes": nbytes / 1e6,
                              "tflops": flops / ms / 1e9, "gbytes_s": nbytes / ms / 1e6,
                              "bound": "compute (fp32 CUDA cores)" if t_c > t_m else "memory",
                              "share_of_bound": max(t_c, t_m) * 1e3 / ms})
        print(res["kernel"][-1], flush=True)
    x = H.seeded_input((8, 3, 256, 256)).cuda()
    trainers = {}
    for dist in ("mse", "ms-ssim"):
        model = H.seeded_model(128, 3, "calib", precision="bf16x3").cuda()
        model.train_precision = "bf16x3"
        trainers[dist] = parallel.ShardedTrainer(model, 0.005 if dist == "mse" else 8.0, lr=1e-5, graph=True, distortion=dist)
        for _ in range(3):
            trainers[dist].step(x)
    torch.cuda.synchronize()
    step = {"mse": [], "ms-ssim": []}
    for _ in range(a.rounds):
        for dist, tr in trainers.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                tr.step(x)
            e1.record()
            torch.cuda.synchronize()
            step[dist].append(e0.elapsed_time(e1) / a.steps)
    res["step_ms"] = step
    mse, msssim = sorted(step["mse"]), sorted(step["ms-ssim"])
    res["step_median_ms"] = {"mse": mse[len(mse) // 2], "ms-ssim": msssim[len(msssim) // 2]}
    res["step_overhead"] = res["step_median_ms"]["ms-ssim"] / res["step_median_ms"]["mse"] - 1
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
