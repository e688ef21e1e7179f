"""Per-tile event clocks of CTA 0 of edge_wide_tc (CGS_DEBUG_TRACE): where a band's time goes."""
import ctypes as C
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "collaborative-gan-sampling_b200"))
import numpy as np
import torch
from cgs import lib as L, nets as N, synthetic as S

lib = L.load()
lib.cgs_debug_set_flags(L.DEBUG_TRACE | int(os.environ.get("EXTRA", "0")))
dev = torch.device("cuda", 0)
arch = N.get_arch("dcgan64_l1")
spec = N.NetSpec(arch, S.init_weights(arch, gain=2.5), dev)
layer = arch["d"][0]
desc = spec.d.layer_desc(0)
B = 1024
x = torch.randn(B, 64, 64, 4, device=dev)
y = torch.empty(B, 32, 32, 64, device=dev)
ws = torch.empty(int(lib.cgs_layer_workspace_bytes(C.byref(desc), B)), dtype=torch.uint8, device=dev)
for _ in range(3):
    L.check(lib.cgs_layer_forward(C.byref(desc), 0, B, L.ptr(x), L.ptr(y), L.ptr(ws), ws.numel(), L.stream_ptr()))
torch.cuda.synchronize()
buf = np.zeros((8, 64), np.int64)
lib.cgs_debug_trace_tc.argtypes = [C.c_void_p]
print("entries", lib.cgs_debug_trace_tc(buf.ctypes.data))
names = ["tma: stage free", "mma: tmem free", "mma: patch landed", "mma: committed", "epi: start wait", "epi: acc ready", "epi: tile done"]
t0 = buf[0, 0]
for t in range(0, 22):
    print("tile %2d " % t + "  ".join("%s %7d" % (names[r].split(":")[1].strip()[:10], buf[r, t] - t0) for r in range(7)))
