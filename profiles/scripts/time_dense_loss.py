"""det_rpn_loss (dense gradients) at N=1024, R=50127: ms per call (CUDA events)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "object-detection-pytorch-rust_b200"))
import torch
import det_b200 as det
from bench import synth_gt, time_region
dev = torch.device("cuda")
strides = (4, 8, 16, 32, 64)
rpn = det.RegionProposalNetwork(list(strides))
hw = [(448 // s, 448 // s) for s in strides]
anchors = torch.cat(rpn.anchor_generator.grid_anchors(hw, dev), 0)
grid = rpn.anchor_generator.grid_layout(hw)
nb = 1024
gtb, _, off, tot = synth_gt(nb, 3, dev)
R = anchors.shape[0]
matched, labels, stats = rpn.anchor_matcher.match_packed(gtb, off, nb, anchors, grid=grid, with_stats=True)
det.subsample_labels_(labels, 256, 0.5, 1, stats=stats)
asg = det.Assignment(labels, matched, gtb, off)
logits = torch.randn(nb, R, device=dev); deltas = torch.randn(nb, R, 4, device=dev) * 0.5
gl, gd = torch.empty_like(logits), torch.empty_like(deltas)
ms = time_region(lambda: rpn._run_loss(anchors, logits, deltas, asg, nb, None, gl, gd), 20)
by = nb * 21 * R + nb * 256 * 4 + nb * 128 * 40
print(f"{ms*1e3:.1f} us  {by/ms/1e6:.0f} GB/s  frac {by/ms/1e6/6537.6:.3f}")
