"""Data-parallel evaluation and training: the images of a batch are sharded across ranks (one process per GPU).

The forward pass has no cross-image operation (no batch norm; GDN is per pixel), so there is no
data-path collective.  The only exchange is the one the rate-distortion terms need
(RateDistortionLoss.py:19-31 take means over the WHOLE batch, and PSNR is the log of the batch-mean
MSE): each rank contributes its per-image (bits_y, bits_z, mse) and one all-gather over
NCCL / NVLink rebuilds the global vectors, after which every rank evaluates the same formulas in
the same order.  Works with any torch.distributed backend (gloo on CPU in the tests).
"""
from __future__ import annotations

import math
import os
from typing import Optional

import torch
import torch.distributed as dist


def gather_per_image(per_image_local: torch.Tensor, group=None) -> torch.Tensor:
    """[3, B_local] on every rank -> [3, B_global] (rank-major image order) on every rank."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return per_image_local
    world = dist.get_world_size(group)
    local = per_image_local.contiguous()
    out = torch.empty(world * local.numel(), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, local.reshape(-1), group=group)
    return out.reshape(world, local.shape[0], -1).permute(1, 0, 2).reshape(local.shape[0], -1)


def rd_terms_from_per_image(per_image: torch.Tensor, num_pixels: int, lambda_rd: float) -> dict:
    """RateDistortionLoss.py:19-34 from per-image (bits_y, bits_z, mse) rows; tensors stay on device."""
    bits_y, bits_z, mse_i = per_image[0].double(), per_image[1].double(), per_image[2].double()
    bpp_y, bpp_z = (bits_y / num_pixels).mean(), (bits_z / num_pixels).mean()
    mse = mse_i.mean()
    bpp_total = bpp_y + bpp_z
    return {
        "loss": (bpp_total + lambda_rd * (255 ** 2) * mse).float(),
        "bpp_y": bpp_y.float(), "bpp_z": bpp_z.float(), "bpp_total": bpp_total.float(), "mse": mse.float(),
        "psnr": (-10 * torch.log10(mse + 1e-8)).float(),
        "mse_per_image": per_image[2], "psnr_per_image": -10 * torch.log10(per_image[2] + 1e-8),
        "bits_y": bits_y.mean().float(), "bits_z": bits_z.mean().float(), "bits_total": (bits_y + bits_z).mean().float(),
    }


def shard_batch(x: torch.Tensor, rank: int, world: int) -> torch.Tensor:
    """Contiguous shard of the batch for `rank`; the batch must divide evenly ("replicas only" otherwise)."""
    b = x.shape[0]
    if b % world:
        raise ValueError(f"batch {b} does not divide over {world} ranks")
    per = b // world
    return x[rank * per:(rank + 1) * per]


SCALAR_KEYS = ("bpp_y", "bpp_z", "bpp_total", "mse", "psnr", "loss", "bits_y", "bits_z")


def rd_terms_on_device(per_image: torch.Tensor, num_pixels: int, lambda_rd: float) -> dict:
    """Same terms as rd_terms_from_per_image, folded by ONE kernel (nic_rd_reduce) - used on the GPU path."""
    from . import _lib
    lib = _lib.load()
    per_image = per_image.contiguous().float()
    scalars = torch.empty(8, dtype=torch.float32, device=per_image.device)
    _lib.check(lib.nic_rd_reduce(_lib.ptr(per_image), per_image.shape[1], num_pixels, float(lambda_rd), _lib.ptr(scalars),
                                 _lib.current_stream()), "nic_rd_reduce")
    return scalars_to_terms(scalars, per_image)


def scalars_to_terms(scalars: torch.Tensor, per_image: torch.Tensor) -> dict:
    out = {k: scalars[i] for i, k in enumerate(SCALAR_KEYS)}
    out["bits_total"] = None                      # = bits_y + bits_z; formed lazily by the caller if wanted
    out["mse_per_image"] = per_image[2]
    out["scalars"] = scalars
    return out


class GraphedForward:
    """``model(x, training=False)`` replayed from a CUDA graph per input shape (any of the model classes: the forward pass issues no
    host synchronisation).  The captured pass has its parallel branches (g_s beside the entropy side, Models._branch_stream); the
    graph is re-captured when a parameter or buffer changed.  The returned dict holds STATIC tensors that the next call overwrites."""

    def __init__(self, model, **forward_kwargs):
        self.model, self.kw, self._graphs = model, forward_kwargs, {}

    def _params_key(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.model.parameters()) + list(self.model.buffers()))

    @torch.no_grad()
    def __call__(self, x: torch.Tensor) -> dict:
        key = (tuple(x.shape), x.device)
        ent = self._graphs.get(key)
        if ent is not None and ent[3] != self._params_key():
            ent = None
        if ent is None:
            static_x = x.clone()
            side = torch.cuda.Stream(device=x.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    self.model(static_x, training=False, **self.kw)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self.model(static_x, training=False, **self.kw)
            ent = (g, static_x, out, self._params_key())
            self._graphs[key] = ent
        g, static_x, out, _ = ent
        if static_x.data_ptr() != x.data_ptr():
            static_x.copy_(x, non_blocking=True)
        g.replay()
        return out


class ShardedEvaluator:
    """model(x_local) + rd terms on this rank's images, then one all-gather for the global terms.

    graph=True captures the whole local step (every kernel of the forward pass and of the rd terms, ~45 launches) in
    a CUDA graph per input shape and replays it: the host then issues one graph launch per batch instead of ~45
    kernel launches plus their tensor-map encodes.  Outputs of a graphed step live in static buffers that the next
    step overwrites (copy what you want to keep).
    """

    def __init__(self, model, lambda_rd: float, group=None, lean: bool = True, graph: bool = False):
        self.model, self.lambda_rd, self.group, self.lean, self.graph = model, lambda_rd, group, lean, graph
        self._graphs = {}
        self.launches_per_step = None

    def _local(self, x_local):
        from .RateDistortionLoss import rd_terms
        out = self.model(x_local, training=False, lean=self.lean)
        per_image, scalars = rd_terms(out, x_local, self.lambda_rd)
        return out, per_image, scalars

    def _params_key(self):
        """(storage, version) of every parameter and buffer: a captured graph is valid for exactly these weights."""
        return tuple((t.data_ptr(), t._version) for t in list(self.model.parameters()) + list(self.model.buffers()))

    def _graphed_local(self, x_local, slot: int = 0):
        key = (tuple(x_local.shape), x_local.device, slot)
        ent = self._graphs.get(key)
        if ent is not None and ent[3] != self._params_key():
            # the weights changed since the capture (optimizer step, load_state_dict, .to()): the graph holds pointers to packed
            # weights / GDN parameters / the factorized table derived from the OLD values - drop it and capture again
            ent = None
            self._graphs.pop(key)
        if ent is None:
            static_x = torch.empty_like(x_local)
            static_x.copy_(x_local)
            side = torch.cuda.Stream(device=x_local.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                     # warm-up: weight packing, attribute setting, allocations
                for _ in range(2):
                    self._local(static_x)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            from . import _lib
            lib = _lib.load()
            g = torch.cuda.CUDAGraph()
            n0 = lib.nic_launch_count()
            with torch.cuda.graph(g):
                res = self._local(static_x)
            self.launches_per_step = int(lib.nic_launch_count() - n0)      # kernels of this library inside one replay
            # the key is taken AFTER the warm-up (the masked conv zeroes its dead taps in place on the first forward, which
            # bumps that parameter's version once); the packed caches the graph reads stay alive in the ConvOps until a
            # weight changes, and a changed weight changes this key before the next replay
            ent = (g, static_x, res, self._params_key())
            self._graphs[key] = ent
        g, static_x, res, _ = ent
        if static_x.data_ptr() != x_local.data_ptr():
            static_x.copy_(x_local, non_blocking=True)
        g.replay()
        return res

    def static_input(self, shape, device, slot: int = 0):
        """The input buffer of graph `slot` for `shape` (fill it directly, e.g. with a pinned-host copy, to skip one device copy).
        Two slots = two captured instances of the step with their own input and intermediate buffers: the host -> device copy
        into one slot's input overlaps the replay of the other."""
        ent = self._graphs.get((tuple(shape), device, slot))
        return None if ent is None else ent[1]

    @torch.no_grad()
    def evaluate_host_batches(self, host_batches):
        """Evaluate an iterable of pinned HOST batches [B,3,H,W]; yields the 8 rd scalars (Python floats) per batch.

        The upload of batch i+1 (pinned host -> device, on a copy stream) overlaps the kernels of batch i; every batch
        still pays its own host->device copy and its own device->host read of the result.
        """
        dev = next(self.model.parameters()).device
        copy_stream = torch.cuda.Stream(device=dev)
        it = iter(host_batches)
        staging, ready = [None, None], [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [None, None]                          # recorded on the compute stream once a step has been queued on the slot

        def upload(slot, hb):
            if self.graph:
                # the copy lands in the INPUT BUFFER of this slot's captured graph (captured on first use): no device -> device hop
                tgt = self.static_input(hb.shape, dev, slot)
                if tgt is None:
                    self._graphed_local(hb.to(dev), slot)
                    tgt = self.static_input(hb.shape, dev, slot)
                staging[slot] = tgt
            elif staging[slot] is None or staging[slot].shape != hb.shape:
                staging[slot] = torch.empty(hb.shape, dtype=torch.float32, device=dev)
            with torch.cuda.stream(copy_stream):
                if consumed[slot] is not None:
                    copy_stream.wait_event(consumed[slot])       # the step that read this slot may still be running
                staging[slot].copy_(hb, non_blocking=True)
                ready[slot].record(copy_stream)

        nxt = next(it, None)
        if nxt is None:
            return
        upload(0, nxt)
        # results come back through two pinned buffers: the device -> host copy of batch i is queued behind its kernels and
        # read one iteration later, so the host queues batch i + 1 before it blocks on batch i (the device never idles
        # between batches; every batch still pays its own host -> device copy and device -> host read)
        res_host = [torch.empty(8, dtype=torch.float32).pin_memory() for _ in range(2)]
        res_done = [torch.cuda.Event(), torch.cuda.Event()]
        pending = None
        i = 0
        while nxt is not None:
            cur = i & 1
            nxt = next(it, None)
            if nxt is not None:
                upload(cur ^ 1, nxt)                    # overlaps the step below; slot cur^1 was consumed two steps ago
            torch.cuda.current_stream().wait_event(ready[cur])
            _, terms = self.step(staging[cur], slot=cur)
            if consumed[cur] is None:
                consumed[cur] = torch.cuda.Event()
            consumed[cur].record()
            res_host[cur].copy_(terms["scalars"], non_blocking=True)
            res_done[cur].record()
            if pending is not None:
                res_done[pending].synchronize()
                yield res_host[pending].tolist()
            pending = cur
            i += 1
        res_done[pending].synchronize()
        yield res_host[pending].tolist()

    @torch.no_grad()
    def step(self, x_local: torch.Tensor, slot: int = 0):
        out, per_image, scalars = self._graphed_local(x_local, slot) if self.graph else self._local(x_local)
        if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(self.group) == 1:
            return out, scalars_to_terms(scalars, per_image)
        per_image = gather_per_image(per_image, self.group)
        return out, rd_terms_on_device(per_image, x_local.shape[2] * x_local.shape[3], self.lambda_rd)


# ---- data-parallel training step (BASELINE configs[3]; reference Trainer.py:79-86, single process there) -------------------

def grad_buckets(params, bucket_bytes: int = 32 << 20):
    """Parameters grouped, in REVERSE registration order (the order backward produces their gradients), into buckets of about
    `bucket_bytes` of fp32 gradient: a handful of NCCL launches for the 7.3 M parameters instead of one per tensor.  The default
    (32 MB) puts this model's 29 MB of gradients in ONE bucket: the whole backward is one autograd node / one graph replay, so
    there is nothing to overlap a second bucket with, and one all-reduce costs one launch latency instead of four."""
    buckets, cur, size = [], [], 0
    for p in reversed(list(params)):
        if not p.requires_grad:
            continue
        cur.append(p)
        size += p.numel() * 4
        if size >= bucket_bytes:
            buckets.append(cur)
            cur, size = [], 0
    if cur:
        buckets.append(cur)
    return buckets


def allreduce_gradients(buckets, group=None, flats=None, average: bool = True):
    """Average .grad over the ranks: each bucket is flattened into one buffer, summed with one all-reduce (NCCL over NVLink on
    the GPUs; gloo in the CPU tests), divided by the world size and scattered back.  The reference's loss is a mean over the batch
    (RateDistortionLoss.py:19-27), so with equal shards the average of the per-rank gradients is the full-batch gradient.
    average=False leaves the SUM in .grad (training.Adam then applies 1 / world inside its update kernel: grad_scale).
    Returns the async work handles' count (all are waited before returning)."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return 0
    world = dist.get_world_size(group)
    works = []
    for bi, bucket in enumerate(buckets):
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in bucket]
        n = sum(g.numel() for g in grads)
        flat = None if flats is None else flats[bi]
        if flat is None or flat.numel() != n or flat.device != grads[0].device:
            flat = torch.empty(n, dtype=torch.float32, device=grads[0].device)
            if flats is not None:
                flats[bi] = flat
        torch.cat([g.reshape(-1).float() for g in grads], out=flat)
        works.append((dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=True), flat, bucket))
    for work, flat, bucket in works:
        work.wait()
        if average:
            flat.div_(world)
        off = 0
        for p in bucket:
            n = p.numel()
            # .grad becomes a VIEW of the averaged bucket (no copy back; with `flats` given the buffer persists until the next call,
            # which is after the optimizer has consumed it)
            p.grad = flat[off:off + n].view_as(p) if flats is not None else flat[off:off + n].view_as(p).clone()
            off += n
    return len(works)


class ShardedTrainer:
    """One training step per call on this rank's shard: model(x) -> rd_loss -> backward -> gradient all-reduce -> Adam.

    Mirrors the body of Trainer.train (Trainer.py:79-86) with the optimizer of Main.ipynb:133; every rank holds the full
    model and must start from identical weights.  Noise is drawn per rank from the rank's own generator state (seed the
    ranks differently) or injected through `noise`.

    graph=True captures forward + loss + backward (+ the Adam launch when there is a single rank) in a CUDA graph per input
    shape and replays it: the ~380 kernel launches of a step, their tensor-map encodes and the Python around them are paid
    once.  The noise comes from torch's graph-safe Philox state (a fresh draw every replay).  The returned dict then holds
    device tensors only ('loss', 'scalars' = the 8 rd scalars of nic_rd_finalize); read them when needed.  Steps with injected
    noise run eagerly.

    distortion="ms-ssim" trains for MS-SSIM (RateDistortionLoss.ms_ssim_rd_loss: loss = bpp + lambda * (1 - MS-SSIM), no 255^2);
    'scalars' then has a 9th entry, the batch MS-SSIM.  The all-reduce is the same: with equal shards the average of the per-rank
    gradients of a batch-mean loss is the global gradient.  Not built for ScalableImageCoding (vision_rd_loss is its loss)."""

    def __init__(self, model, lambda_rd: float, lr: float = 1e-4, group=None, bucket_bytes: int = 32 << 20, optimizer=None,
                 graph: bool = False, distortion: str = "mse"):
        from .training import DISTORTIONS, Adam
        self._scalable = type(model).__name__ == "ScalableImageCoding"
        if distortion not in DISTORTIONS:
            raise ValueError(f"distortion must be one of {DISTORTIONS}, got {distortion!r}")
        if self._scalable and distortion != "mse":
            raise ValueError("ScalableImageCoding trains with vision_rd_loss (MSE); distortion='ms-ssim' is not built for it")
        self.model, self.lambda_rd, self.group, self.graph, self.distortion = model, lambda_rd, group, graph, distortion
        self.optimizer = optimizer if optimizer is not None else Adam(model.parameters(), lr=lr)
        self.buckets = grad_buckets(model.parameters(), bucket_bytes)
        self._flats = [None] * len(self.buckets)
        self._graphs = {}
        self.step_count = 0

    def _distributed(self) -> bool:
        return dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1

    def _allreduce(self):
        """Gradient all-reduce; with training.Adam the division by the world size happens inside the update kernel."""
        fold = hasattr(self.optimizer, "grad_scale") and self._distributed()
        if fold:
            self.optimizer.grad_scale = 1.0 / dist.get_world_size(self.group)
        allreduce_gradients(self.buckets, self.group, self._flats, average=not fold)

    def _forward_backward(self, x_local, noise=None, partial_hook=None):
        """forward + loss + backward on the calling thread and stream (training.step_gradients: the same kernels loss.backward()
        runs, without the autograd engine, whose device thread cannot take part in a stream capture)."""
        self.optimizer.zero_grad()
        if self._scalable:                                   # two-head model, vision_rd_loss (training_scalable.py)
            from .training_scalable import step_gradients as scalable_step
            loss, terms = scalable_step(self.model, x_local, self.lambda_rd, noise=noise)
            return loss, None, torch.stack([terms[k] for k in ("bpp_y1", "bpp_y2", "bpp_z", "mse", "psnr", "loss")])
        from .training import step_gradients
        return step_gradients(self.model, x_local, self.lambda_rd, noise=noise, partial_hook=partial_hook, distortion=self.distortion)

    # ---- gradient all-reduce INSIDE the captured step, overlapped with g_a's backward -------------------------------------------
    def _comm_setup(self, device):
        """Two flat fp32 buckets: 'early' = every parameter except g_a's (their gradients are final before g_a's backward starts),
        'late' = g_a's.  The gradients are copied into the buckets inside the graph, the buckets are summed over the ranks by NCCL
        launches captured in the same graph (the early one on a side stream, beside g_a's backward), and .grad becomes views of
        the buckets; training.Adam divides by the world size inside its update kernel."""
        if getattr(self, "_comm", None) is not None:
            return self._comm
        enc = {id(p) for p in self.model.encoder.parameters()}
        early = [p for p in self.model.parameters() if p.requires_grad and id(p) not in enc]
        late = [p for p in self.model.parameters() if p.requires_grad and id(p) in enc]
        mk = lambda ps: torch.zeros(sum(p.numel() for p in ps), dtype=torch.float32, device=device)      # noqa: E731
        self._comm = {"early": early, "late": late, "flat_early": mk(early), "flat_late": mk(late),
                      "stream": torch.cuda.Stream(device=device)}
        return self._comm

    @staticmethod
    def _views(params, flat):
        out, off = {}, 0
        for p in params:
            out[id(p)] = flat[off:off + p.numel()].view_as(p)
            off += p.numel()
        return out

    def _reduce_bucket(self, params, flat, grads):
        """grads of `params` -> flat -> all-reduce(SUM) on the current stream; returns {id: view of flat}."""
        views = self._views(params, flat)
        srcs = [grads[id(p)] if id(p) in grads else None for p in params]
        dsts = [views[id(p)] for p in params]
        for d, g in zip(dsts, srcs):
            if g is None:
                d.zero_()
        torch._foreach_copy_([d for d, g in zip(dsts, srcs) if g is not None], [g.reshape(d.shape) for d, g in zip(dsts, srcs) if g is not None])
        # the sources were produced on other streams than the one that copies them: hold them until the capture ends, so that the
        # allocator cannot hand their memory to a later tensor of the same graph
        self._comm.setdefault("keep", []).extend(g for g in srcs if g is not None)
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        return views

    def _graphed(self, x_local):
        key = (tuple(x_local.shape), x_local.device)
        ent = self._graphs.get(key)
        dist_on = self._distributed()
        has_launch = hasattr(self.optimizer, "launch")
        # data parallel: the all-reduce (and with it Adam) joins the graph unless NIC_GRAPH_ALLREDUCE=0
        comm_in_graph = dist_on and has_launch and not self._scalable and hasattr(self.optimizer, "grad_scale") \
            and os.environ.get("NIC_GRAPH_ALLREDUCE", "1") != "0"
        fuse_adam = has_launch and (not dist_on or comm_in_graph)
        if ent is None:
            static_x = torch.empty_like(x_local)
            static_x.copy_(x_local)
            side = torch.cuda.Stream(device=x_local.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                     # warm-up: allocations, attribute setting, the device status word
                self._forward_backward(static_x)
                if comm_in_graph:                              # ... and the NCCL communicator
                    c = self._comm_setup(x_local.device)
                    dist.all_reduce(c["flat_early"], group=self.group); dist.all_reduce(c["flat_late"], group=self.group)
            torch.cuda.current_stream().wait_stream(side)
            if fuse_adam:
                self.optimizer.prepare(x_local.device)
            if comm_in_graph:
                self.optimizer.grad_scale = 1.0 / dist.get_world_size(self.group)
            # every derived cache (packed conv weights, adjoint packs, GDN effective parameters, the factorized table, the masked
            # conv's zeroing) is keyed on the parameters' version counters: bump them so that the capture RECORDS the kernels that
            # rebuild those caches - a replay must re-derive them from the weights the previous replay's Adam launch wrote
            for p in self.model.parameters():
                torch.autograd.graph.increment_version(p)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                hook = None
                if comm_in_graph:
                    c = self._comm_setup(x_local.device)
                    cur = torch.cuda.current_stream()

                    def hook(grads, streams, c=c):
                        # every gradient outside g_a is enqueued: sum them over the ranks on the side stream while g_a's backward runs
                        for st in streams:
                            c["stream"].wait_stream(st)
                        with torch.cuda.stream(c["stream"]):
                            grads.update(self._reduce_bucket(c["early"], c["flat_early"], grads))
                res = self._forward_backward(static_x, partial_hook=hook)
                if comm_in_graph:
                    late = self._reduce_bucket(c["late"], c["flat_late"], {id(p): p.grad for p in c["late"] if p.grad is not None})
                    for p in c["late"]:
                        p.grad = late[id(p)]
                    cur.wait_stream(c["stream"])              # join: the early bucket is reduced
                if fuse_adam:
                    self.optimizer.launch()                  # counter increment + update: the step count lives on the device
            # the gradients the capture produced: every replay rewrites THESE tensors, so .grad must point at them again after
            # a replay (the all-reduce below re-points .grad at views of its averaged buckets)
            ent = (g, static_x, res, [p.grad for p in self.model.parameters()])
            self._graphs[key] = ent
            if comm_in_graph:
                self._comm["keep"] = []
        g, static_x, res, static_grads = ent
        if static_x.data_ptr() != x_local.data_ptr():
            static_x.copy_(x_local, non_blocking=True)
        if fuse_adam and hasattr(self.optimizer, "sync_lr"):
            self.optimizer.sync_lr()                          # a scheduler's new lr reaches the captured update through device memory
        g.replay()
        for p, sg in zip(self.model.parameters(), static_grads):
            p.grad = sg
        if fuse_adam:
            self.optimizer.t += 1
            for p in self.model.parameters():                 # updated inside the replay: packed-weight caches key on _version
                torch.autograd.graph.increment_version(p)
        return res, fuse_adam, comm_in_graph

    def step(self, x_local: torch.Tensor, noise=None) -> dict:
        if (self.graph and noise is None) or self._scalable:
            reduced = False
            if self.graph and noise is None:
                (loss, per_image, scalars), adam_done, reduced = self._graphed(x_local)
            else:
                (loss, per_image, scalars), adam_done = self._forward_backward(x_local, noise), False
            if not reduced:
                self._allreduce()
            if not adam_done:
                self.optimizer.step()
            self.step_count += 1
            # scalars: the 8 rd scalars of nic_rd_finalize (+ the batch MS-SSIM with distortion='ms-ssim'); ScalableImageCoding: (bpp_y1, bpp_y2, bpp_z, mse, psnr, loss)
            return {"loss": loss, "scalars": scalars, "mse_per_image": None if per_image is None else per_image[2]}
        from .RateDistortionLoss import ms_ssim_rd_loss, rd_loss
        if self.distortion == "ms-ssim":
            from .RateDistortionLoss import check_ms_ssim_shape
            check_ms_ssim_shape(tuple(x_local.shape))
        self.optimizer.zero_grad()
        out = self.model(x_local, training=True, noise=noise, lean=True)
        rd = (ms_ssim_rd_loss if self.distortion == "ms-ssim" else rd_loss)(out, x_local, self.lambda_rd)
        rd["loss"].backward()
        self._allreduce()
        self.optimizer.step()
        self.step_count += 1
        return rd
