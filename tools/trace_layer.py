"""Run one layer pass with the CTA-0 pipeline trace on (CGS_DEBUG_TRACE) and print per-role event timelines.

The trace code is compiled out of the product build: rebuild first with
    CGS_NVCC_EXTRA=-DCGS_TRACE python collaborative-gan-sampling_b200/build.py -f
(and rebuild without it afterwards).
"""
import argparse
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "collaborative-gan-sampling_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from cgs import lib as L, nets as N, synthetic as S  # noqa: E402

os.environ["CGS_DEBUG"] = str(int(os.environ.get("CGS_DEBUG", "0")) | L.DEBUG_TRACE)   # read when libcgs loads

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="mnist")
ap.add_argument("--layer", default="d_conv2")
ap.add_argument("--bwd", action="store_true")
ap.add_argument("--batch", type=int, default=1024)
a = ap.parse_args()
dev = torch.device("cuda", 0)
lib = L.load()
arch = N.get_arch(a.workload)
spec = N.NetSpec(arch, S.init_weights(arch, gain=2.5), dev)
chain = [(l, spec.gtail.layer_desc(i)) for i, l in enumerate(arch["gtail"])] + \
        [(l, spec.d.layer_desc(i)) for i, l in enumerate(arch["d"][:-1])]
layer, desc = [c for c in chain if c[0]["name"] == a.layer][0]
B = a.batch
cin, cout = layer["cin"], layer["cout"]
if layer["type"] == "fc":
    xs, ys = (B, cin), (B, N.cstride(cout))
elif layer["type"] == "conv":
    xs = (B, layer["hin"], layer["win"], N.cstride(cin)); ys = (B, (layer["hin"] + 1) // 2, (layer["win"] + 1) // 2, N.cstride(cout))
else:
    xs = (B, layer["hin"], layer["win"], N.cstride(cin)); ys = (B, layer["hin"] * 2, layer["win"] * 2, N.cstride(cout))
x = torch.randn(xs, device=dev); y = torch.empty(ys, device=dev); dy = torch.randn(ys, device=dev); dx = torch.empty(xs, device=dev)
buf = np.zeros(32768, np.uint64)
ws = torch.empty(int(lib.cgs_layer_workspace_bytes(C.byref(desc), B)), dtype=torch.uint8, device=dev)
for rep in range(2):
    if a.bwd:
        L.check(lib.cgs_layer_backward(C.byref(desc), 0, B, L.ptr(dy), L.ptr(dx), L.ptr(x), 1, L.ptr(ws), ws.numel(), L.stream_ptr()))
    else:
        L.check(lib.cgs_layer_forward(C.byref(desc), 0, B, L.ptr(x), L.ptr(y), L.ptr(ws), ws.numel(), L.stream_ptr()))
    n = lib.cgs_debug_trace(buf.ctypes.data, 32768)
ev = [(int(v >> 60), int((v >> 56) & 0xf), int((v >> 32) & 0xffffff), int(v & 0xffffffff)) for v in buf[:n].tolist() if v]
t0 = min(e[3] for e in ev)
names = {(0, 0): "P.wait_empty", (0, 1): "P.issued", (1, 0): "T.wait_empty", (2, 0): "M.wait_full", (2, 1): "M.commit",
         (2, 2): "M.tmem_empty", (3, 0): "E.tmem_full", (3, 1): "E.released", (3, 2): "E.done",
         (5, 0): "M5.loop_top", (5, 1): "M5.waited", (5, 3): "M5.mma_issued", (5, 2): "M5.loop_end",
         (4, 0): "C.ld_done", (4, 1): "C.math_done", (4, 2): "C.stored", (4, 3): "C.synced"}
print("events", len(ev))
chunk = {}
for e in ev:
    if e[0] == 4:
        chunk.setdefault(e[2], {})[e[1]] = (e[3] - t0) & 0xffffffff
print("per chunk (idx = tile_count*8 + chunk): ld_done math_done stored synced")
for k in sorted(chunk)[:24]:
    print("   %4d  %s" % (k, "  ".join("%7d" % chunk[k].get(i, -1) for i in range(4))))
for key in sorted(names):
    rows = sorted([(e[2], (e[3] - t0) & 0xffffffff) for e in ev if (e[0], e[1]) == key])
    ts = [t for _, t in rows]
    d = np.diff(ts) if len(ts) > 1 else []
    print("%-14s n=%4d first=%7d last=%8d  mean dt=%7.1f  first 40 t: %s" % (names[key], len(ts), ts[0] if ts else -1, ts[-1] if ts else -1,
          float(np.mean(d)) if len(d) else 0.0, ts[:40]))
# steady-state table: per ring stage the time the weight-TMA thread saw the slot empty, the MMA thread saw it full and
# committed it (cycles since the first event; dM = commit -> next commit)
by = {}
for e in ev:
    if e[0] in (1, 2):
        by.setdefault(e[2], {})[(e[0], e[1])] = (e[3] - t0) & 0xffffffff
lo = int(os.environ.get("TRACE_FROM", "144"))
print("stage  T.got_empty  M.got_full  M.commit   full-empty  commit-full  commit-prev_commit")
prev = None
for k in range(lo, lo + 80):
    r = by.get(k)
    if not r:
        continue
    te, mf, mc = r.get((1, 0), -1), r.get((2, 0), -1), r.get((2, 1), -1)
    print("%5d  %10d  %10d  %9d  %9d  %9d  %9s" % (k, te, mf, mc, mf - te, mc - mf, (mc - prev) if prev is not None else "-"))
    prev = mc
tiles = {}
for e in ev:
    if e[0] == 3:
        tiles.setdefault(e[2], {})[e[1]] = (e[3] - t0) & 0xffffffff
print("tile  E.tmem_full  E.released  E.done")
for k in sorted(tiles)[:16]:
    print("%4d  %s" % (k, "  ".join("%9d" % tiles[k].get(i, -1) for i in range(3))))
