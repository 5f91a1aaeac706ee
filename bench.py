#!/usr/bin/env python
"""Headline benchmark: 768x512 images/s of forward + likelihood + rate-distortion terms (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision bf16x3|bf16|fp32|mixed] [--dump-outputs DIR]

The default arm is precision="bf16x3": every transform on the tcgen05 tensor cores with hi/lo-split bf16 operands (fp32 grade) -
the arm that meets the parity bar of BASELINE.json (symbols, likelihoods 1e-4, bpp / PSNR 1e-3; tests/test_gpu_model.py).  The
single-pass bf16 arm (2.6x faster, NOT parity grade: ~0.7 % symbol flips) is timed beside it and reported as "throughput_arm".

Workload (config.workload): BASELINE.json configs[1] - JointAutoregressiveHierarchical(128, K=3), lambda 0.005,
eval forward + rd_loss terms on a synthetic 16 x 3 x 512 x 768 batch PER GPU (weak scaling; ranks hold disjoint
images; the only collective is the all-gather of per-image (bits_y, bits_z, mse)).
One "step" = model(x, training=False) + the rd terms on one batch.

  value   : whole-job images/s with the inputs already resident in HBM (4 rotating batches = 302 MB > 126 MB L2)
  e2e     : the same through the public module API with pinned HOST inputs: H2D copy of the batch, forward,
            rd_loss(...) whose Python floats force the D2H read - all inside the timed region
  roofline: dominant kernel = conv_tc_kernel on the 128->128 5x5 stride-2 conv of g_a layer 2 (SURVEY.md §2.2 k2),
            ALGORITHMIC FLOPs / its CUDA-event duration, against the measured bf16 peak of MEASURED_PEAKS.json; in the
            bf16x3 arm the kernel issues 3x the algorithmic MMA work (roofline.tensor_pipe_frac counts the issued FLOPs)
  cpu_baseline: the oracle (torch CPU port of the reference's path) on the box's host cores, bounded sample
  residual_variant : (extra) the 3x3 residual family (HierarchicalMixtureResidual, SURVEY.md section 8 row f4), batch 4 per GPU
  strong_scaling   : (extra) the same 16-image batch split over the ranks (graph replay and collective timed apart)
  config3_context_entropy : (extra) BASELINE.json configs[2] isolated: context conv + entropy-parameter stack (+ likelihood)
  scalable_variant : (extra) BASELINE.json configs[4] - ScalableImageCoding(192, 128) on one 2048 x 1536 image per GPU, bf16x3 arm
  train_step  : (extra, not the headline) BASELINE.json configs[3] - the reference's training step (Trainer.py:79-86: forward with
            noise, rd_loss, backward, Adam) on 8 x 3 x 256 x 256 crops PER GPU through ShardedTrainer (hand-written backward
            kernels, bucketed NCCL gradient all-reduce), CUDA-event timed, max over ranks; the oracle's autograd step on the
            host cores beside it (rank 0, bounded sample)

--impl reference runs only that CPU arm (rank 0) and prints the same line shape with "impl": "reference".

--dump-outputs DIR writes what the last timed step returned on rank 0 (the model's output dict and the rd terms) as DIR/<name>.npy,
float32, so that two builds can be compared output for output on the same seeded inputs (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it (it may be read-only)

M, K, LAMBDA = 128, 3, 0.005
H_IMG, W_IMG, B_PER_GPU = 512, 768, 16
WORKLOAD = "GM K=3 capacity-128 hyperprior+context model, lambda=0.005, eval forward + likelihood + rd terms, " \
           "synthetic 768x512, batch 16 per GPU (BASELINE.json configs[1])"
FLOPS_PER_IMAGE = 73.572e9                      # SURVEY.md §8d, algorithmic (masked taps skipped)
# dominant kernel: g_a layer 2, Conv2d(128,128,5,s2,p2) on 256x384 -> 128x192 (SURVEY §2.2 k2); the GDN contraction that follows
# is fused into the same kernel in the bf16 arm and a separate HBM-bound kernel (gdn_x3_kernel) in the bf16x3 arm
K2_CONV_FLOPS_PER_IMAGE = 2.0 * 128 * 192 * 128 * 128 * 25
K2_GDN_FLOPS_PER_IMAGE = 2.0 * 128 * 192 * 128 * 128


# seeded weights of the benchmark model: the reference's default init under torch.manual_seed(0), re-scaled so that the symbols are
# non-trivial and the likelihoods well conditioned (the "calib" set of oracle/make_golden.py: last g_a conv x34, last h_a conv
# x3.86, +3 on the sigma biases of the entropy-parameter head)
def bench_model(precision="fp32", device=None):
    import torch
    from neural_image_compression_b200.Models import JointAutoregressiveHierarchical
    torch.manual_seed(0)
    model = JointAutoregressiveHierarchical(M, K=K, precision=precision)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    for k in ("encoder.net.6.weight", "encoder.net.6.bias"):
        sd[k] = sd[k] * 34.0
    for k in ("hyper_encoder.net.4.weight", "hyper_encoder.net.4.bias"):
        sd[k] = sd[k] * 3.86
    b = sd["entropy_parameters.net.4.bias"].clone()
    b[2 * b.numel() // 3:] += 3.0
    sd["entropy_parameters.net.4.bias"] = b
    model.load_state_dict(sd)
    return model if device is None else model.to(device)


def bench_scalable_model(device):
    import torch
    from neural_image_compression_b200.Models import ScalableImageCoding
    torch.manual_seed(0)
    model = ScalableImageCoding(192, 128, K=1, precision="bf16x3")
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    for k in ("encoder.net.6.weight", "encoder.net.6.bias"):
        sd[k] = sd[k] * 34.0
    for k in ("hyper_encoder.net.4.weight", "hyper_encoder.net.4.bias"):
        sd[k] = sd[k] * 3.86
    for head in ("entropy_parameters_1", "entropy_parameters_2"):
        b = sd[f"{head}.net.4.bias"].clone()
        b[b.numel() // 2:] += 3.0
        sd[f"{head}.net.4.bias"] = b
    model.load_state_dict(sd)
    return model.to(device)


def seeded_input(shape, seed=1):
    import torch
    g = torch.Generator(device="cpu"); g.manual_seed(seed)
    return torch.rand(*shape, generator=g)


DUMP_MAX_ELEMS = 1 << 20        # per array: the outputs of one 16-image step then come to ~35 MB, inside the 64 MB budget
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(arrays: dict, out_dir: str) -> None:
    """Write every floating-point tensor of `arrays` as out_dir/<name>.npy in float32 (float64 stays float64); other entries (flags,
    None) are skipped.  An array of more than DUMP_MAX_ELEMS elements is reduced to a fixed sample of its flattened elements:
    DUMP_MAX_ELEMS distinct indices in ascending order, drawn from a generator seeded with 0, so arrays of equal size share one index
    set, from run to run and from build to build."""
    import numpy as np
    import torch
    picked, index = {}, {}
    for name, t in arrays.items():
        if not isinstance(t, torch.Tensor) or not t.is_floating_point():
            continue
        t = t.detach().double() if t.dtype == torch.float64 else t.detach().float()
        n = t.numel()
        if n > DUMP_MAX_ELEMS:
            if n not in index:
                g = torch.Generator(device="cpu"); g.manual_seed(0)
                index[n] = torch.randperm(n, generator=g)[:DUMP_MAX_ELEMS].sort().values
            t = t.reshape(-1)[index[n].to(t.device)]
        picked[name] = t.cpu().numpy()
    total = sum(a.nbytes for a in picked.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in picked.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"bf16_burst": p["bf16_tflops"], "bf16_sustained": p["bf16_tflops_sustained"], "hbm": p["hbm_gbs"], "src": "measured"}
    except Exception:
        return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:6]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set(); self.join(timeout=3)
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_reference_arm(images: int, iters: int, warmup: int = 1):
    """The reference's CPU path (oracle port, torch CPU fp32, all host threads): `warmup` untimed + `iters` timed passes over
    `images` images of the workload."""
    import torch
    from oracle import forward as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = bench_model()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = seeded_input((images, 3, H_IMG, W_IMG))
    with torch.no_grad():
        for _ in range(max(1, warmup)):
            O.rd_loss(O.forward(sd, x, M, K), x, LAMBDA)              # warm-up passes (thread pool, allocator), untimed
        times = []
        for _ in range(iters):
            t0 = time.perf_counter()
            rd = O.rd_loss(O.forward(sd, x, M, K), x, LAMBDA)
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return {"value": images / t, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{iters} timed passes over {images} x 3x512x768 images after {max(1, warmup)} warm-up pass(es), torch CPU "
                      f"fp32 ({torch.get_num_threads()} threads)", "bpp_total": rd["bpp_total"], "psnr": rd["psnr"], "s_per_pass": t,
            "total_s": sum(times)}


def cpu_train_step(images: int = 2):
    """The reference's training step on the host cores: autograd over the oracle port + restated Adam, one pass (bounded sample)."""
    import torch
    from oracle import backward as OB
    torch.set_num_threads(os.cpu_count() or 1)
    model = bench_model()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    x = seeded_input((images, 3, 256, 256))
    torch.manual_seed(5)
    nz, ny = torch.rand(images, M, 4, 4) - 0.5, torch.rand(images, M, 16, 16) - 0.5
    t0 = time.perf_counter()
    _, grads, _ = OB.loss_and_grads(sd, x, M, K, nz, ny, LAMBDA)
    OB.adam_step(sd, grads)
    t = time.perf_counter() - t0
    return {"value": images / t, "unit": "images/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": f"one step on {images} x 3x256x256 crops (forward + rd_loss + autograd backward + Adam), torch CPU fp32"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("NIC_BENCH_PRECISION", "bf16x3"),
                    choices=["bf16x3", "bf16", "fp32", "mixed"],
                    help="bf16x3 = tcgen05 arm with hi/lo-split operands, fp32 grade (headline: meets the parity bar); bf16 = single-pass "
                         "tcgen05 throughput arm; fp32 = CUDA-core parity arm; mixed = g_a/h_a fp32, rest bf16")
    ap.add_argument("--batch", type=int, default=B_PER_GPU, help="images per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-max-seconds", type=float, default=150.0, help="--impl reference: bound on the timed region (the step count is cut, and reported, if needed)")
    ap.add_argument("--no-residual", action="store_true", help="skip the 3x3 residual-family line item (HierarchicalMixtureResidual, SURVEY.md 8 f4)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling line item (global batch 16 split over the ranks)")
    ap.add_argument("--no-config3", action="store_true", help="skip the isolated context + entropy-parameter (+ likelihood) line item (BASELINE.json configs[2])")
    ap.add_argument("--no-other-arms", action="store_true", help="skip the short runs of the other precision arms reported beside the headline")
    ap.add_argument("--no-scalable", action="store_true", help="skip the scalable-coding line item (BASELINE.json configs[4])")
    ap.add_argument("--no-train-step", action="store_true", help="skip the training-step line item (BASELINE.json configs[3])")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy, float32; "
                                                          "arrays over 2^20 elements as a fixed seeded sample (dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        # every step is ONE pass over the full 16-image batch of the workload (1.7 s on 16 host threads): exactly `steps` timed
        # passes after `warmup` warm-up passes, like the GPU arm; --ref-max-seconds bounds the run (fewer timed steps, reported)
        images = args.batch
        est = 2.0 * images / 10.0                                  # ~10 images/s on a 16-thread host
        steps = max(1, min(args.steps, int(args.ref_max_seconds / max(est, 1e-3))))
        base = cpu_reference_arm(images, steps, warmup=args.warmup)
        line = {"impl": "reference", "metric": "768x512 images/s (fwd+likelihood+rd terms)", "value": base["value"], "unit": "images/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": base["s_per_pass"] * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "global_batch": images, "parallelism": "host cores (rank 0)", "precision": "f32",
                           "steps_requested": args.steps,
                           "reference": "the reference's CPU path = oracle port (torch CPU fp32, same ops in the same order; the reference "
                                        "itself is 14 loose scripts that cannot be installed or travel to the GPU box, DESIGN.md section 2)"},
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": base["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # keep stdout clean for the ONE JSON line: anything libraries print (e.g. "NCCL version ...") goes to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)
    json_out = os.fdopen(json_fd, "w")

    import torch
    import torch.distributed as dist
    from neural_image_compression_b200 import _lib, engine, parallel
    from neural_image_compression_b200.RateDistortionLoss import rd_loss, rd_terms

    assert torch.cuda.is_available(), "bench.py needs a B200"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.nic_check_device(), "nic_check_device")
    peaks = load_peaks()

    B = args.batch
    model = bench_model(args.precision, dev)
    nbuf = 4
    gen = torch.Generator(device="cpu"); gen.manual_seed(1000 + rank)
    host_batches = [torch.rand((B, 3, H_IMG, W_IMG), generator=gen).pin_memory() for _ in range(nbuf)]
    dev_batches = [hb.to(dev) for hb in host_batches]
    use_graph = not args.no_graph
    evaluator = parallel.ShardedEvaluator(model, LAMBDA, lean=False, graph=use_graph)

    def step(i):
        return evaluator.step(dev_batches[i % nbuf])

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    sync_all()
    sampler = ClockSampler(local_rank); sampler.start()
    l0 = lib.nic_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out, terms = step(i)
    e1.record()
    sync_all()
    launches = lib.nic_launch_count() - l0
    if use_graph and evaluator.launches_per_step:
        launches = evaluator.launches_per_step * args.steps          # kernels replayed from the captured graph
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = B * world * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:
        # now, before later steps overwrite them: a graphed step returns the static buffers of its CUDA graph
        dump_outputs({**out, **{k: v for k, v in terms.items() if k != "scalars"}}, args.dump_outputs)

    # ---- e2e: pinned host input -> H2D -> forward -> rd_loss floats (D2H) every step -----------------
    # public API: ShardedEvaluator.evaluate_host_batches - per batch: pinned-host -> device copy (on a copy stream, overlapping
    # the previous batch's kernels), the forward + rd terms, and the device -> host read of the 8 result scalars
    def host_stream(n):
        for i in range(n):
            yield host_batches[i % nbuf]
    for vals in evaluator.evaluate_host_batches(host_stream(min(3, max(2, args.warmup)))):
        pass
    sync_all()
    e0.record()
    for vals in evaluator.evaluate_host_batches(host_stream(args.steps)):
        res = {"bpp_total": vals[2], "psnr": vals[4]}
    e1.record()
    sync_all()
    ms_e2e = max(e0.elapsed_time(e1), 0.0)
    te = torch.tensor([ms_e2e], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = B * world * args.steps / (float(te.item()) / 1e3)
    h2d = B * 3 * H_IMG * W_IMG * 4
    d2h = 8 * 4

    _, terms = evaluator.step(dev_batches[0])
    terms = {k: float(terms[k]) for k in ("bpp_total", "psnr")}

    # ---- strong scaling (SURVEY.md section 8d): BASELINE configs[1] is "batch=16" - the SAME 16 images split over the ranks
    # (16 / world per GPU), with the local graph replay and the all-gather + fold of the per-image terms broken out ------------
    strong = None
    if not args.no_strong and 16 % world == 0:
        bs = 16 // world
        ev_s = evaluator if bs == B else parallel.ShardedEvaluator(model, LAMBDA, lean=False, graph=use_graph)
        xs = [db[:bs].contiguous() for db in dev_batches]
        ns = max(20, args.steps)

        def timed(fn, n):
            for i in range(3):
                fn(i)
            sync_all()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n):
                fn(i)
            b.record()
            sync_all()
            tt = torch.tensor([a.elapsed_time(b)], device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()) / n
        ms_step = timed(lambda i: ev_s.step(xs[i % nbuf]), ns)
        ms_local = timed(lambda i: (ev_s._graphed_local(xs[i % nbuf]) if use_graph else ev_s._local(xs[i % nbuf])), ns)
        per_img = torch.rand((3, bs), device=dev)
        ms_coll = timed(lambda i: parallel.rd_terms_on_device(parallel.gather_per_image(per_img), H_IMG * W_IMG, LAMBDA), ns) if world > 1 else 0.0
        strong = {"scaling": "strong", "global_batch": bs * world, "images_per_gpu": bs, "value": bs * world / (ms_step / 1e3), "unit": "images/s",
                  "ms_per_step": ms_step, "local_step_ms": ms_local, "allgather_and_fold_ms": ms_coll, "steps": ns,
                  "note": "the same 16-image batch split over the ranks; per-GPU work shrinks with N, so launch latency and the "
                          "collective's latency (a 3 x B_local float all-gather + one fold kernel) weigh in"}
        if ev_s is not evaluator:
            del ev_s

    # ---- BASELINE configs[2] isolated (SURVEY.md section 8d "Config 3"): masked 5x5 context conv + entropy-parameter 1x1 stack
    # (+ the GM likelihood kernel) on y_in [B,128,32,48], psi [B,256,32,48]: 5.74 GFLOP / image algorithmic (12 live taps) --------
    config3 = None
    if not args.no_config3 and args.precision in ("bf16x3", "bf16"):
        from neural_image_compression_b200._lib import Q_PASSTHRU as _QP
        pair = args.precision == "bf16x3"
        cw = 2 if pair else 1
        hy, wy = H_IMG // 16, W_IMG // 16
        yq = torch.round(4 * torch.randn((B, hy, wy, M), device=dev))
        y_in_nhwc = engine.to_pair(yq) if pair else yq.to(torch.bfloat16)
        y_in_nchw = yq.permute(0, 3, 1, 2).contiguous()
        psi = torch.randn((B, hy, wy, 2 * M), device=dev)
        combined = torch.zeros((B, hy, wy, cw * 4 * M), dtype=torch.bfloat16, device=dev)
        if pair:
            pp = engine.to_pair(psi)
            combined[..., 2 * M:4 * M] = pp[..., :2 * M]; combined[..., 6 * M:8 * M] = pp[..., 2 * M:]
        else:
            combined[..., 2 * M:] = psi.to(torch.bfloat16)
        ep = model.entropy_parameters.ops
        model.context_model.masked.apply_mask_()

        c3_plan = engine.CtxEpPlan(model.context_model.masked._op, ep, B, hy, wy, args.precision, M, K, dev, full=True)

        def ctx_ep(i, with_lik=True):
            # ONE C-ABI call (nic_ctx_ep_fwd): context conv, the three 1x1 layers and - with_lik - the likelihood kernel
            c3_plan.run(y_in_nhwc, combined, y_in=y_in_nchw if with_lik else None, qmode=_QP)

        def time_c3(with_lik):
            for i in range(3):
                ctx_ep(i, with_lik)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n3 = max(20, args.steps)
            a.record()
            for i in range(n3):
                ctx_ep(i, with_lik)
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n3
        with torch.no_grad():
            ms_c3, ms_c3l = time_c3(False), time_c3(True)
        c3_flops = 5.7378e9 * B
        config3 = {"workload": "BASELINE.json configs[2] isolated: masked 5x5 context conv (12 live taps) + entropy-parameter 1x1 stack "
                               "512->640->640->1152 on y_in [B,128,32,48], psi [B,256,32,48]; + GM-K3 likelihood kernel (full dict)",
                   "batch": B, "ms_context_plus_stack": ms_c3, "ms_with_likelihood": ms_c3l, "algorithmic_gflop": c3_flops / 1e9,
                   "tflops": c3_flops / (ms_c3 / 1e3) / 1e12, "frac_of_bf16_peak": c3_flops / (ms_c3 / 1e3) / 1e12 / peaks["bf16_burst"],
                   "images_per_s": B / (ms_c3l / 1e3),
                   "launch": "one nic_ctx_ep_fwd call per pass = 4 (5) kernel launches back to back, inputs L2-resident as in the model"}
        del combined, psi, yq
    # ---- the other precision arms on the same workload (short runs), reported beside the headline arm -----------------
    other_arms = {}
    if not args.no_other_arms:
        for arm in ("bf16x3", "bf16", "fp32"):
            if arm == args.precision:
                continue
            m2 = bench_model(arm, dev)
            ev2 = parallel.ShardedEvaluator(m2, LAMBDA, lean=False, graph=use_graph and arm != "fp32")
            n2 = 3 if arm == "fp32" else max(5, args.steps)
            for i in range(3):
                ev2.step(dev_batches[i % nbuf])
            torch.cuda.synchronize()
            a0, a1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for i in range(n2):
                _, t2 = ev2.step(dev_batches[i % nbuf])
            a1e.record()
            torch.cuda.synchronize()
            _, t2 = ev2.step(dev_batches[0])                    # rd terms of every arm are reported on the same batch
            other_arms[arm] = {"images_per_s_per_gpu": B * n2 / (a0.elapsed_time(a1e) / 1e3), "ms_per_step": a0.elapsed_time(a1e) / n2,
                               "bpp_total": float(t2["bpp_total"]), "psnr": float(t2["psnr"]),
                               "parity_grade": arm != "bf16"}
            del m2, ev2
        torch.cuda.empty_cache()

    # ---- dominant kernel, timed per launch with CUDA events on the launching stream ------------------
    kern_prec = {"bf16": "bf16", "fp32": "fp32", "mixed": "fp32", "bf16x3": "bf16x3"}[args.precision]   # g_a layer 2 timed alone
    if kern_prec == "bf16x3":
        # conv_tc_kernel alone, exactly as the model launches it (bias epilogue, bf16-pair output that gdn_x3_kernel then reads):
        # the GDN of this layer is a separate kernel in this arm
        op = engine.ConvOp(model.encoder.net[2], _lib.EPI_BIAS)
        a1 = engine.to_pair(torch.randn((B, H_IMG // 2, W_IMG // 2, M), device=dev))
        k2_kwargs, k2_flops, k2_kernel = {}, K2_CONV_FLOPS_PER_IMAGE, \
            "conv_tc_kernel, g_a layer 2: conv 128->128 5x5 s2 with hi/lo-split operands (3 MMA passes), 16x256x384 input"
    else:
        op = model.encoder.ops[1]
        a1 = torch.randn((B, H_IMG // 2, W_IMG // 2, M), device=dev).to(engine.act_dtype(kern_prec))
        k2_kwargs, k2_flops, k2_kernel = {}, K2_CONV_FLOPS_PER_IMAGE + K2_GDN_FLOPS_PER_IMAGE, \
            "g_a layer 2: conv 128->128 5x5 s2 + fused GDN, 16x256x384 input"
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    durs = []
    for i in range(3 + max(5, args.steps)):
        flush.zero_()                                        # > L2: the layer input is re-fetched from HBM each time
        ks, ke = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ks.record()
        op.run(a1, B, H_IMG // 2, W_IMG // 2, kern_prec, **k2_kwargs)
        ke.record()
        torch.cuda.synchronize()
        if i >= 3:
            durs.append(ks.elapsed_time(ke))
    k2_ms = statistics.mean(durs)
    achieved = k2_flops * B / (k2_ms / 1e3) / 1e12
    peak = peaks["bf16_burst"]
    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this shape from the ncu --set full captures
    # (bf16x3: 908.2 MB + 179.4 MB, profiles/r2_ncu_full_k2.txt; algorithmic: 805.3 MB of pair input + 201.3 MB of output +
    #  2.5 MB of weights - the hi patches are fetched twice per tile, a tenth of the second fetches reach DRAM;
    #  bf16: 403.8 MB + 83.3 MB, profiles/r1_ncu_full_v6_k2_bf16.txt)
    k2_traffic = {"bf16": 487.1e6, "bf16x3": 1087.6e6}.get(kern_prec) if B == 16 else None
    passes = 3 if kern_prec == "bf16x3" else 1
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": k2_traffic,
                "kernel": k2_kernel, "ms_per_launch": k2_ms, "mma_passes": passes, "tensor_pipe_frac": passes * achieved / peak,
                "peak_source": f"{peaks['src']} bf16 burst (kernel timed alone)",
                "whole_step_tflops": FLOPS_PER_IMAGE * B * args.steps / (ms_total / 1e3) / 1e12}

    # ---- the HBM-bound kernel north_star names: quantise + GM-K3 likelihood + log + bit sums, full (dict) variant -------
    from neural_image_compression_b200.EntropyModels import gm_likelihood
    from neural_image_compression_b200._lib import Q_ROUND
    lik = {}
    for lb in (B, 16 * B):
        yl = 5 * torch.randn((lb, M, H_IMG // 16, W_IMG // 16), device=dev)
        rawl = torch.randn((lb, 3 * K * M, H_IMG // 16, W_IMG // 16), device=dev)
        ld = []
        lout = gm_likelihood(yl, rawl, M, K, Q_ROUND, full=True)          # output tensors reused below: no allocator calls between
        for i in range(23):                                               # the two events, only the C-ABI launch
            flush.zero_()
            ks, ke = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ks.record(); gm_likelihood(yl, rawl, M, K, Q_ROUND, full=True, out=lout); ke.record()
            torch.cuda.synchronize()
            if i >= 3:
                ld.append(ks.elapsed_time(ke))
        del lout
        lms = statistics.mean(ld)
        nbytes = yl.numel() * 88                                  # SURVEY.md §8d: 52 B/elem + 36 B/elem for weights/mus/sigmas
        lik[f"batch{lb}"] = {"ms": lms, "GB/s": nbytes / (lms / 1e3) / 1e9, "frac_of_hbm_peak": nbytes / (lms / 1e3) / 1e9 / peaks["hbm"]}
        del yl, rawl
    roofline_lik = {"bound": "hbm", "kernel": "gm_likelihood_flat_kernel<K=3, full>", "unit": "GB/s", "peak": peaks["hbm"],
                    "bytes_per_y_element": 88, "peak_source": f"{peaks['src']} copy bandwidth", **lik}

    # ---- the training step (BASELINE.json configs[3]) - extra line item, every rank takes part (gradient all-reduce) ----------
    train = None
    if not args.no_train_step:
        try:                                     # an extra line item must never cost the headline line
            del evaluator, flush
            torch.cuda.empty_cache()
            tb = 8
            tmodel = bench_model(args.precision, dev)
            trainer = parallel.ShardedTrainer(tmodel, LAMBDA, lr=1e-4, graph=use_graph)
            tgen = torch.Generator(device="cpu"); tgen.manual_seed(2000 + rank)
            crops = [torch.rand((tb, 3, 256, 256), generator=tgen).to(dev) for _ in range(4)]
            for i in range(3):
                trainer.step(crops[i % 4])
            sync_all()
            ts, te = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nt = max(5, args.steps)
            ts.record()
            for i in range(nt):
                trd = trainer.step(crops[i % 4])
            te.record()
            sync_all()
            tt_ms = torch.tensor([ts.elapsed_time(te)], device=dev)
            if world > 1:
                dist.all_reduce(tt_ms, op=dist.ReduceOp.MAX)
            from neural_image_compression_b200.training import train_precision
            train = {"workload": "rate-distortion training step, 256x256 crops, batch 8 per GPU (BASELINE.json configs[3]): forward with noise, "
                                 "rd_loss, backward, gradient all-reduce, Adam(lr 1e-4)",
                     "value": tb * world * nt / (float(tt_ms.item()) / 1e3), "unit": "images/s", "ms_per_step": float(tt_ms.item()) / nt,
                     "steps": nt, "arm": train_precision(tmodel),
                     "launch": "forward + loss + backward (+ Adam on one rank) replayed from one CUDA graph" if use_graph else "per-kernel launches",
                     "loss_last": float(trd["loss"].detach()), "scaling": "weak"}
            del trainer, tmodel, crops
        except Exception as e:               # noqa: BLE001
            train = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- the scalable-coding variant (BASELINE.json configs[4]): one 2048 x 1536 image per GPU, forward + vision_rd_loss ---------
    scalable = None
    if not args.no_scalable:
        try:
            from neural_image_compression_b200.RateDistortionLoss import vision_rd_loss
            smodel = bench_scalable_model(dev)
            sgen = torch.Generator(device="cpu"); sgen.manual_seed(3000 + rank)
            simgs = [torch.rand((1, 3, 1536, 2048), generator=sgen).to(dev) for _ in range(2)]
            sfwd = parallel.GraphedForward(smodel) if use_graph else (lambda t: smodel(t, training=False))
            with torch.no_grad():
                for i in range(3):
                    vision_rd_loss(sfwd(simgs[i % 2]), simgs[i % 2], LAMBDA)
                sync_all()
                ss, se = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ns = 10
                ss.record()
                for i in range(ns):
                    srd = vision_rd_loss(sfwd(simgs[i % 2]), simgs[i % 2], LAMBDA)       # forward = one graph replay; the loss reads its scalars back
                se.record()
                sync_all()
            st_ms = torch.tensor([ss.elapsed_time(se)], device=dev)
            if world > 1:
                dist.all_reduce(st_ms, op=dist.ReduceOp.MAX)
            scalable = {"workload": "ScalableImageCoding(192, 128, K=1) eval forward + vision_rd_loss, synthetic 2048x1536, one image per GPU "
                                    "(BASELINE.json configs[4]; the reference's forward with the four repairs of SURVEY.md 2.4, no LST)",
                        "value": world * ns / (float(st_ms.item()) / 1e3), "unit": "images/s", "ms_per_image": float(st_ms.item()) / ns,
                        "precision": "bf16x3", "algorithmic_tflops": 1.2547 * world * ns / (float(st_ms.item()) / 1e3),
                        "bpp_total": float(srd["bpp_total"]), "psnr": float(srd["psnr"]), "scaling": "weak"}
            del smodel, simgs
            torch.cuda.empty_cache()
        except Exception as e:               # noqa: BLE001
            scalable = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- the 3x3 residual family (SURVEY.md section 8 row f4): HierarchicalMixtureResidual(128, K=3), same workload shape -------------
    residual = None
    if not args.no_residual:
        try:
            from neural_image_compression_b200.Models import HierarchicalMixtureResidual
            torch.manual_seed(0)
            rmodel = HierarchicalMixtureResidual(M, K=K, precision="bf16x3").to(dev)
            rfwd = parallel.GraphedForward(rmodel, lean=True) if use_graph else (lambda t: rmodel(t, training=False, lean=True))
            rb = 4
            rx = [db[:rb].contiguous() for db in dev_batches[:2]]
            with torch.no_grad():
                for i in range(3):
                    rd_loss(rfwd(rx[i % 2]), rx[i % 2], LAMBDA)
                sync_all()
                rs, re_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                nr = 10
                rs.record()
                for i in range(nr):
                    rrd = rd_loss(rfwd(rx[i % 2]), rx[i % 2], LAMBDA)
                re_.record()
                sync_all()
            rt_ms = torch.tensor([rs.elapsed_time(re_)], device=dev)
            if world > 1:
                dist.all_reduce(rt_ms, op=dist.ReduceOp.MAX)
            residual = {"workload": "HierarchicalMixtureResidual(128, K=3) (3x3 residual transforms, Models.py:109-205) eval forward + rd_loss, synthetic "
                                    "768x512, batch 4 per GPU, layer-by-layer on the conv engine (random-init weights)",
                        "value": rb * world * nr / (float(rt_ms.item()) / 1e3), "unit": "images/s", "ms_per_step": float(rt_ms.item()) / nr,
                        "precision": "bf16x3", "bpp_total": float(rrd["bpp_total"]), "scaling": "weak"}
            del rfwd, rx
            torch.cuda.empty_cache()
            if not args.no_train_step:
                # its training step (training.Tape over the residual graphs): 8 crops of 256 x 256 per GPU, as configs[3]
                rtr = parallel.ShardedTrainer(rmodel, LAMBDA, lr=1e-4, graph=use_graph)
                rgen = torch.Generator(device="cpu"); rgen.manual_seed(3000 + rank)
                rcrops = [torch.rand((8, 3, 256, 256), generator=rgen).to(dev) for _ in range(2)]
                for i in range(3):
                    rtr.step(rcrops[i % 2])
                sync_all()
                rs, re_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                rs.record()
                for i in range(nr):
                    rtl = rtr.step(rcrops[i % 2])
                re_.record()
                sync_all()
                rtt = torch.tensor([rs.elapsed_time(re_)], device=dev)
                if world > 1:
                    dist.all_reduce(rtt, op=dist.ReduceOp.MAX)
                residual["train_step"] = {"workload": "forward with noise + rd_loss + backward + gradient all-reduce + Adam, 8 x 3x256x256 crops per GPU",
                                          "value": 8 * world * nr / (float(rtt.item()) / 1e3), "unit": "images/s",
                                          "ms_per_step": float(rtt.item()) / nr, "loss_last": float(rtl["loss"].detach())}
                del rtr, rcrops
            del rmodel
            torch.cuda.empty_cache()
        except Exception as e:               # noqa: BLE001
            residual = dict(residual or {}, error=f"{type(e).__name__}: {e}"[:300])

    assert lib.nic_pipeline_status() == 0, "a tensor-core kernel aborted on an expired pipeline wait: numbers invalid"
    if rank == 0:
        cpu = None if args.no_cpu_baseline else cpu_reference_arm(B_PER_GPU, 6, warmup=1)
        line = {
            "metric": "768x512 images/s (fwd+likelihood+rd terms)", "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "bf16": "bf16", "mixed": "f32(g_a,h_a)+bf16", "bf16x3": "bf16x3 (bf16 hi+lo operands, f32 accumulate)"}[args.precision],
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": B * world, "parallelism": f"dp{world}", "precision": args.precision,
                       "l2": "4 rotating input batches (302 MB) + >400 MB of per-step intermediates exceed the 126 MB L2",
                       "launch": "one CUDA-graph replay per step" if use_graph else "per-kernel launches from Python"},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_likelihood": roofline_lik,
            "rd": {"bpp_total": float(terms["bpp_total"]), "psnr": float(terms["psnr"]), "e2e_bpp_total": res["bpp_total"]},
        }
        if other_arms:
            line["other_arms"] = other_arms
            if "bf16" in other_arms:
                line["throughput_arm"] = {"precision": "bf16", "value": other_arms["bf16"]["images_per_s_per_gpu"] * world, "unit": "images/s",
                                          "note": "single-pass bf16 tcgen05 arm; NOT parity grade (symbols flip at bf16 precision)"}
        if cpu is not None:
            line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
            line["rd"]["cpu_sample_bpp_total"] = cpu["bpp_total"]
        if train is not None:
            if not args.no_cpu_baseline and "error" not in train:
                train["cpu_baseline"] = cpu_train_step(2)
            line["train_step"] = train
        if scalable is not None:
            line["scalable_variant"] = scalable
        if residual is not None:
            line["residual_variant"] = residual
        if strong is not None:
            line["strong_scaling"] = strong
        if config3 is not None:
            line["config3_context_entropy"] = config3
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
