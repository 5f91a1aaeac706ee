"""Pipeline trace of conv_tc_kernel for one layer (GPU box):  python tools/trace_layer.py k2|d2|d3|k3|ep3|k2c|d2c|gs3 [bf16|bf16x3]
(k2c / d2c: the conv alone with a bias epilogue and f32 NHWC output, as the bf16x3 arm runs it before gdn_x3_kernel;
gs3: g_s layer 3's conv as the bf16x3 arm runs it before its IGDN - bias epilogue, bf16-pair output, CTA-pair form)
Ends with a per-phase summary over every CTA that issues MMAs: mainloop (first A slot ready -> last MMA issued) against
epilogue (accumulator ready -> last store issued) per tile, in SM clocks."""
import ctypes as C, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch, torch.nn as nn
from neural_image_compression_b200 import engine, _lib
from neural_image_compression_b200._lib import EPI_BIAS, EPI_GDN, EPI_IGDN, EPI_LRELU, LAYOUT_NCHW, LAYOUT_NHWC
from neural_image_compression_b200.gdn import GDN

which = sys.argv[1] if len(sys.argv) > 1 else "k2"
prec = sys.argv[2] if len(sys.argv) > 2 else "bf16"
B = 16
dev = torch.device("cuda:0")
cfg = {
    "k2": (nn.Conv2d(128, 128, 5, 2, 2), EPI_GDN, (256, 384), {}),
    "k3": (nn.Conv2d(128, 128, 5, 2, 2), EPI_GDN, (128, 192), {}),
    "d2": (nn.ConvTranspose2d(128, 128, 5, 2, 2, output_padding=1), EPI_IGDN, (128, 192), {}),
    "d3": (nn.ConvTranspose2d(128, 3, 5, 2, 2, output_padding=1), EPI_BIAS, (256, 384), dict(out_layout=LAYOUT_NCHW, out_dtype=torch.float32)),
    "ep3": (nn.Conv2d(640, 1152, 1), EPI_BIAS, (32, 48), dict(out_layout=LAYOUT_NCHW, out_dtype=torch.float32)),
    "ep1": (nn.Conv2d(512, 640, 1), EPI_LRELU, (32, 48), {}),
    "ep2": (nn.Conv2d(640, 640, 1), EPI_LRELU, (32, 48), {}),
    "hs3": (nn.Conv2d(192, 256, 3, 1, 1), EPI_BIAS, (32, 48), {}),
    "hs2": (nn.ConvTranspose2d(128, 192, 5, 2, 2, output_padding=1), EPI_LRELU, (16, 24), {}),
    "ha1": (nn.Conv2d(128, 128, 3, 1, 1), EPI_LRELU, (32, 48), {}),
    "ha2": (nn.Conv2d(128, 128, 5, 2, 2), EPI_LRELU, (32, 48), {}),
    "ctx": (nn.Conv2d(128, 256, 5, 1, 2), EPI_BIAS, (32, 48), {}),
    "l1": (nn.Conv2d(3, 128, 5, 2, 2), EPI_GDN, (512, 768), dict(in_layout=LAYOUT_NCHW)),
    "k2c": (nn.Conv2d(128, 128, 5, 2, 2), EPI_BIAS, (256, 384), dict(out_dtype=torch.float32)),
    "k2p": (nn.Conv2d(128, 128, 5, 2, 2), EPI_BIAS, (256, 384), {}),      # pair (bf16x3) or bf16 output: the swapped orientation
    "d2p": (nn.ConvTranspose2d(128, 128, 5, 2, 2, output_padding=1), EPI_BIAS, (128, 192), {}),
    "d2c": (nn.ConvTranspose2d(128, 128, 5, 2, 2, output_padding=1), EPI_BIAS, (128, 192), dict(out_dtype=torch.float32)),
    "gs3": (nn.ConvTranspose2d(128, 128, 5, 2, 2, output_padding=1), EPI_BIAS, (128, 192), {}),
}[which]
conv, epi, (h, w), kw = cfg
conv = conv.to(dev)
g = GDN(128, inverse=(epi == EPI_IGDN)).to(dev) if epi in (EPI_GDN, EPI_IGDN) else None
op = engine.ConvOp(conv, epi, gdn=g)
x = torch.randn(B, h, w, conv.in_channels, device=dev)
x = engine.to_pair(x) if prec == "bf16x3" else x.to(torch.bfloat16)
if which == "l1":
    x = torch.rand(B, 3, h, w, device=dev)
    names_l1 = ["P:start", "P:patch_ready", "P:fetched_next", "P:a_empty", "P:built", "M:acc_empty", "M:a_full", "E:acc_full",
                "e:start", "e:sqdone", "e:synced", "e:gdn", "e:computed", "e:synced2", "E:done"]
lib = _lib.load()
lib.nic_debug_set_trace.argtypes = [C.c_void_p]; lib.nic_debug_set_trace.restype = None
for _ in range(3):
    op.run(x, B, h, w, prec, **kw)
torch.cuda.synchronize()
buf = torch.zeros(148 * 32 * 16, dtype=torch.int64, device=dev)
lib.nic_debug_set_trace(buf.data_ptr())
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); op.run(x, B, h, w, prec, **kw); e1.record()
torch.cuda.synchronize()
lib.nic_debug_set_trace(None)
t = buf.cpu().reshape(148, 32, 16)
print(f"{which}: {e0.elapsed_time(e1)*1000:.1f} us")
names = names_l1 if which == "l1" else ["mma:acc_empty", "mma:first_a", "mma:issued", "epi:acc_full", "epi:done", "A:first", "A:last", "-",
         "e0:start", "e0:sqdone", "e0:synced", "e0:gdn", "e0:computed", "e0:synced2"]
for cta in (0, 77):
    base = int(t[cta, 0][t[cta, 0] > 0].min())
    print(f"CTA {cta} (clk relative to its first stamp)")
    for i in range(10):
        row = t[cta, i]
        if int(row[0]) == 0:
            break
        print("  tile %2d: " % i + "  ".join(f"{n}={int(row[j]) - base:6d}" for j, n in enumerate(names) if n != "-" and int(row[j]) != 0))
    live = [i for i in range(16) if int(t[cta, i][0]) and int(t[cta, i][15])]
    if len(live) > 2:
        a, b = live[1], live[-1]
        dclk, dns = int(t[cta, b][0]) - int(t[cta, a][0]), int(t[cta, b][15]) - int(t[cta, a][15])
        print(f"  SM clock during the kernel: {dclk / dns * 1000:.0f} MHz ({dclk} clk in {dns} ns, tiles {a}..{b})")
if which != "l1":
    # slot 7: the tile's phase (stamped by the MMA issuer); tile 0 of each CTA is left out (it starts on an idle pipeline)
    import collections
    acc = collections.defaultdict(lambda: [0, 0, 0])
    for cta in range(148):
        for i in range(1, 16):
            row = t[cta, i]
            if int(row[1]) and int(row[2]) and int(row[8]) and int(row[4]):
                a = acc[int(row[7])]
                a[0] += 1; a[1] += int(row[2]) - int(row[1]); a[2] += int(row[4]) - int(row[8])
    for ph in sorted(acc):
        n, ml, ep = acc[ph]
        print(f"phase {ph}: {n:4d} tiles  mainloop {ml / n:8.0f} clk  epilogue {ep / n:8.0f} clk per tile")
