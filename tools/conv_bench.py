"""Timing of the channels-last tensor-core convolution (dba_conv_nhwc) at the update operator's layer shapes, 48x64, CUDA events.
Prints TFLOP/s per shape."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import droid_slam_b200

be = droid_slam_b200.install()
DEV = "cuda:0"
E = int(os.environ.get("CB_E", 256))
ht, wd = 48, 64
SHAPES = {"zr": (128, 320, 3, 256), "q": (128, 320, 3, 128), "stem": (128, 0, 3, 384), "c3x3": (128, 0, 3, 128), "heads": (256, 0, 3, 32), "c1x1": (256, 0, 1, 128)}
which = os.environ.get("CB_SHAPES", "zr,q,stem,c3x3,heads,c1x1").split(",")
g = torch.Generator(device=DEV).manual_seed(0)
for name in which:
    c0, c1, ks, n = SHAPES[name]
    x0 = torch.randn(E, ht, wd, c0, device=DEV, generator=g).half()
    x1 = torch.randn(E, ht, wd, c1, device=DEV, generator=g).half() if c1 else None
    w = (torch.randn(ks * ks, n, c0 + c1, device=DEV, generator=g) * 0.03).half()
    b = torch.zeros(n, device=DEV)
    for _ in range(2):
        out = be.conv_nhwc(x0, x1, w, b, ks, True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        out = be.conv_nhwc(x0, x1, w, b, ks, True)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    fl = 2.0 * E * ht * wd * n * (c0 + c1) * ks * ks
    print("%-6s E=%d: %8.3f ms  %7.1f TFLOP/s" % (name, E, ms, fl / ms / 1e9), flush=True)
