"""Runs the Cholesky trailing update (gpk_syrk_lower_dev, n=4096, k=4096) a few times -- target of `ncu --set full`."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gp_algos_b200 import _lib
ts = torch.cuda.Stream(); torch.cuda.set_stream(ts)
h = _lib.Handle(0, ts.cuda_stream)
n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
k = int(sys.argv[2]) if len(sys.argv) > 2 else n
P = torch.randn(k, n, dtype=torch.float64, device="cuda")
Cm = torch.zeros(n, n, dtype=torch.float64, device="cuda")
for _ in range(3):
    h.check(h.lib.gpk_syrk_lower_dev(h.h, P.data_ptr(), n, Cm.data_ptr(), n, n, k))
torch.cuda.synchronize()
e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(3):
    h.check(h.lib.gpk_syrk_lower_dev(h.h, P.data_ptr(), n, Cm.data_ptr(), n, n, k))
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 3
print(f"syrk n={n} k={k}: {ms:.3f} ms  {n*n*k/ms*1e-9:.2f} TFLOP/s")
