"""Phase timeline of the FAST pipeline k_flow_pipe (CTA 0, pipeline steps 264..279) from a -DGLABC_FLOW_TRACE build:
   python -c "import sys; sys.path.insert(0,'gl-abc-mcmc_b200'); import build; build.build(variant='trace', extra_flags=['-DGLABC_FLOW_TRACE'])"
   GLABC_LIB=$PWD/gl-abc-mcmc_b200/csrc/libglabc.trace.so python profiles/micro/k4_trace.py [fast|precise]
`precise` times the PRECISE pipeline only: it records no timeline."""
import ctypes
import sys
import time

import numpy as np
import torch

sys.path.insert(0, '/root/repo')
import glabc_b200  # noqa: E402,F401
from glabc_b200 import _abi  # noqa: E402
from glabc_b200.flows import RealNVP  # noqa: E402

torch.manual_seed(0)
f = RealNVP(device="cuda")
with torch.no_grad():
    f.w3.copy_(0.05 * torch.randn_like(f.w3))
eng = f.train_init()
eps = torch.randn(1 << 21, 2, device="cuda")
mode = sys.argv[1] if len(sys.argv) > 1 else "fast"
for _ in range(3):
    f.fused_sample_from(eps, eng, precision=mode)
torch.cuda.synchronize()
best = 0.0
for rep in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        f.fused_sample_from(eps, eng, precision=mode)
    e1.record()
    torch.cuda.synchronize()
    best = max(best, 20 * eps.shape[0] / (e0.elapsed_time(e1) * 1e-3))
print("samples/s", best)
lib = ctypes.CDLL(_abi.LIB_PATH)
if hasattr(lib, "glabc_debug_pipe_trace") and mode == "fast":
    buf = np.zeros((6, 64, 6), dtype=np.int64)
    rc = lib.glabc_debug_pipe_trace(buf.ctypes.data_as(ctypes.c_void_p))
    assert rc == 0, rc
    base = buf[buf > 0].min()
    np.set_printoptions(linewidth=250)
    names = ["M1 (two threads, alternate steps): top, a1_full, acc_empty, MMA1 issued", "U warp 0: top, out_full, update done",
             "Y warp 8: top, waits done, L1 done", "Y warp 12: top, waits done, L1 done",
             "M2: top, act_full, MMA2 issued", "E warp 4: top, acc_full, done"]
    for r in range(6):
        print(names[r])
        for st in range(8, 24):
            row = buf[r, st]
            print(st, [int(x - base) if x > 0 else -1 for x in row])
