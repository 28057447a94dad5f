"""CUDA-event timing of 200 back-to-back damped SPD solves and their error against fp64 LAPACK.
usage: python tools/chol_timing.py [n]   (n <= 448 runs the resident-tile kernel, larger n the barrier kernel)"""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
n = int(sys.argv[1]) if len(sys.argv) > 1 else 426
import torch  # noqa: E402
from droid_slam_b200 import c_api  # noqa: E402

L = c_api.load()
g = torch.Generator().manual_seed(0)
A = torch.randn(n, n + 8, generator=g, dtype=torch.float64)
Hc = A @ A.t() + 1e-3 * torch.eye(n, dtype=torch.float64)
bc = torch.randn(n, generator=g, dtype=torch.float64)
H, b = Hc.cuda(), bc.cuda()
ws = torch.empty(L.dba_solve_workspace_bytes(n), dtype=torch.uint8, device="cuda")
x = torch.zeros(n, device="cuda")
fail = torch.zeros(1, dtype=torch.int32, device="cuda")


def solve():
    L.dba_solve_spd(ctypes.c_void_p(H.data_ptr()), ctypes.c_void_p(b.data_ptr()), n, ctypes.c_float(1e-4), ctypes.c_float(0.1), ctypes.c_void_p(x.data_ptr()),
                    ctypes.c_void_p(fail.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws.numel(), None)


for it in range(20):
    solve()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for it in range(200):
    solve()
e1.record()
torch.cuda.synchronize()
Hd = Hc.clone()
Hd.diagonal().add_(0.1 + 1e-4 * Hc.diagonal())
ref = torch.linalg.solve(Hd, bc)
err = float((x.cpu().double() - ref).abs().max() / ref.abs().max())
print("n=%d  %s kernel: %.1f us per solve (200 back-to-back), fail=%d, max rel err vs fp64 LAPACK %.2e"
      % (n, "barrier" if n > 448 else "resident", 1e3 * e0.elapsed_time(e1) / 200, int(fail), err))
