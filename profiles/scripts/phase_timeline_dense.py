"""Phase timeline (block 0) of dense_detect_nms_kernel using the -DDET_DEBUG_PHASES build."""
import ctypes, os, sys
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
C = 80
strides = [8, 16, 32]
wh = [[[10, 13], [16, 30], [33, 23]], [[30, 61], [62, 45], [59, 119]], [[116, 90], [156, 198], [373, 326]]]
dh = det.DenseAnchorHead(strides, wh, C)
n = 32
g = torch.Generator(device="cuda").manual_seed(3)
hs = [torch.randn(n, 3 * (5 + C), 640 // s, 640 // s, device="cuda", generator=g) for s in strides]
for h in hs:
    h.view(n, 3, 5 + C, h.shape[2], h.shape[3])[:, :, 4] -= 4.0
names = {0: "start", 1: "keys+stats", 2: "counting sort", 3: "gather+file", 6: "suppressors (own category)", 4: "pairs across categories", 5: "rounds", 14: "output"}
order = [0, 1, 2, 3, 6, 4, 5, 14]
for thr, cap in ((0.1, 2048), (0.25, 1024)):
    for _ in range(3):
        r = dh.detect_thresholded(hs, thr, 0.5, max_det=300, cand_cap=cap, check=False)
    torch.cuda.synchronize()
    cnts = (torch.cat([x.flatten(1) for x in dh.decode(hs)[1:2]], 1) > thr).sum(1).cpu()
    r = dh.detect_thresholded(hs, thr, 0.5, max_det=300, cand_cap=cap, check=False)
    torch.cuda.synchronize()
    buf = (ctypes.c_longlong * 32)()
    assert N.lib().det_debug_read_phases_dense(buf) == 0
    print(f"thr {thr} cap {cap}: kept {float(r['count'].float().mean())}")
    prev = buf[0]
    for i in order:
        if buf[i]:
            print(f"{names[i]:>22s}: +{buf[i] - prev:8d} cycles  (t={buf[i] - buf[0]})")
            prev = buf[i]
    blk = (ctypes.c_longlong * (64 * 16))()
    assert N.lib().det_debug_read_phase_blocks_dense(blk) == 0
    tot = [(blk[b * 16 + 14] - blk[b * 16 + 0], b) for b in range(n)]
    print("boxes reaching below -1 per image:", [blk[b * 16 + 7] for b in range(n)])
    print("per-image CTA cycles:", sorted(t for t, _ in tot))
    _, worst = max(tot)
    print(f"slowest CTA {worst}: candidates {int(cnts[worst])}")
    prev = blk[worst * 16]
    for i in order:
        v = blk[worst * 16 + i]
        if v:
            print(f"{names[i]:>22s}: +{v - prev:8d} cycles")
            prev = v
