"""det_dense_detect (decode + threshold + per-class NMS + top 300) at the bench's settings, graph-replayed: ms per batch and
the fraction of the HBM copy peak."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "object-detection-pytorch-rust_b200"))
import torch
import det_b200 as det
from bench import time_graph, load_peaks
dev = torch.device("cuda", 0)
C80, R = 80, 25200
strides = [8, 16, 32]
wh = [[[10, 13], [16, 30], [33, 23]], [[30, 61], [62, 45], [59, 119]], [[116, 90], [156, 198], [373, 326]]]
dh = det.DenseAnchorHead(strides, wh, C80)
peak = load_peaks()[0]
for n in [int(a) for a in sys.argv[1:]] or [32, 256]:
    g = torch.Generator(device=dev).manual_seed(3)
    pool = 2 if n > 64 else 4
    heads = []
    for _ in range(pool):
        hs = [torch.randn(n, 3 * (5 + C80), 640 // s, 640 // s, device=dev, generator=g) for s in strides]
        for h in hs:
            h.view(n, 3, 5 + C80, h.shape[2], h.shape[3])[:, :, 4] -= 4.0
        heads.append(hs)
    for thr, cap in ((0.1, 2048), (0.25, 1024)):
        ws = (torch.empty((det._native.fn("det_dense_detect_workspace_bytes")(n, cap),), dtype=torch.uint8, device=dev)
              if os.environ.get("DET_PLAIN_WS") == "1" else det.DenseDetectWorkspace(n, cap, dev))
        r = dh.detect_thresholded(heads[0], thr, 0.5, max_det=300, cand_cap=cap, gate=False, check=True, workspace=ws)
        fns = [(lambda hs=hs_: dh.detect_thresholded(hs, thr, 0.5, max_det=300, cand_cap=cap, gate=False, check=False, out=r,
                                                     workspace=ws)) for hs_ in heads]
        ms = time_graph(fns, 10)
        k = float(r["count"].float().mean())
        by = n * (4 * R * (5 + C80) + (36 * k + 4))
        print(f"N={n} thr={thr}: {ms * 1e3:.1f} us per batch, kept {k:.1f}/image, {by / ms / 1e6:.0f} GB/s = {by / ms / 1e6 / peak:.3f} of the copy peak")
    del heads
    torch.cuda.empty_cache()
