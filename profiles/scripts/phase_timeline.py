"""Phase timeline of the fused YOLO decode+NMS kernel (block 0) using the -DDET_DEBUG_PHASES build."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PKG = os.path.join(ROOT, "object-detection-pytorch-rust_b200")
sys.path.insert(0, PKG)
import importlib.util
spec = importlib.util.spec_from_file_location("b", os.path.join(PKG, "build.py"))
b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
dbg = b.build(debug_phases=True)
import det_b200._native as N
N._LIB_PATH = dbg
import torch
import det_b200 as det

yh = det.YoloGridHead(7, 2, 20, (448, 448))
heads = torch.randn(4, 256, 7, 7, 30, generator=torch.Generator().manual_seed(1)).cuda()
out = None
for i in range(4):
    out = yh.detect(heads[i], 0.25, 0.5, max_det=300, out=out)
torch.cuda.synchronize()
buf = (ctypes.c_longlong * 32)()
assert N.lib().det_debug_read_phases(buf) == 0
names = {0: "start", 1: "A staged+decoded", 2: "B scores/stats/tier", 5: "E pair filter", 8: "R resolve (class 0)",
         3: "all classes done", 4: "counting-sort merge", 15: "output"}
order = [0, 1, 2, 5, 8, 3, 4, 15]
prev = buf[0]
for i in order:
    if buf[i]:
        print(f"{names[i]:>26s}: +{buf[i] - prev:7d} cycles  (t={buf[i] - buf[0]})")
        prev = buf[i]
