#!/usr/bin/env python
"""Second-stage (Fast R-CNN box predictor) training losses: det_b200.FastRCNNOutputs.losses_batched
(det_fast_rcnn_loss_typed: one kernel) against a torch-CUDA restatement of detectron2's FastRCNNOutputLayers.losses
(_log_classification_stats, F.cross_entropy, box_reg_loss with smooth-L1) plus autograd's backward, on the same inputs.

    python profiles/scripts/time_fast_rcnn_loss.py [--out FILE] [--rounds 7] [--quick]

Sizes: N = 16 and 2 images x 512 sampled rows (ROI_HEADS.BATCH_SIZE_PER_IMAGE), K = 80 classes, class-specific deltas,
25 % foreground rows, smooth-L1 with beta 0; fp32 rows and bf16 rows (an autocast box head; the torch restatement
computes on .float() as autocast does for cross_entropy).  Each size and dtype is timed forward only (ours: one launch,
sums only; torch: the forward with the autograd graph recorded) and forward + backward (ours: the fused launch,
with_grads=True; torch: forward + backward()).

Timing: CUDA events, warmed up, median over `rounds` rounds that alternate ours and torch.  Ours is captured in a CUDA
graph that runs the call on R distinct copies of the inputs, R * input bytes > 2 * L2, so every call reads its rows
from HBM: ms per call = replay time / R.  Ours is also timed eager (back-to-back Python calls, host overhead included).
The torch restatement synchronises the host (nonzero) and is timed around back-to-back calls on the same R copies.
Kernel time: torch.profiler over separate graph replays (kernel durations / calls), set against the algorithmic bytes
M * (e(K+1) + 8) + fg * (4e + 32) read and, with gradients, M * e(5K+1) written (e = element bytes).
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "object-detection-pytorch-rust_b200"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

L2 = 126 * 1024 * 1024
K, P = 80, 512
FG = 0.25
WEIGHTS = (10.0, 10.0, 5.0, 5.0)
CLAMP = math.log(1000.0 / 16)


def make_inputs(n, seed, dev, dtype):
    g = torch.Generator().manual_seed(seed)
    M = n * P
    logits = torch.randn(M, K + 1, generator=g) * 2.0
    deltas = torch.randn(M, 4 * K, generator=g) * 0.5
    xy = torch.rand(M, 2, generator=g) * torch.tensor([1100.0, 700.0])
    wh = 16.0 + torch.rand(M, 2, generator=g) * torch.tensor([300.0, 200.0])
    props = torch.cat([xy, xy + wh], 1)
    fg = torch.rand(M, generator=g) < FG
    classes = torch.where(fg, torch.randint(0, K, (M,), generator=g), torch.full((M,), K))
    gtb = torch.where(fg[:, None], props + (torch.rand(M, 4, generator=g) - 0.5) * 20, props)
    return [logits.to(dev, dtype), deltas.to(dev, dtype), props.to(dev), classes.to(dev), gtb.to(dev)]


def torch_losses(logits, deltas, props, gt_classes, gt_boxes):
    """detectron2 v0.6 FastRCNNOutputLayers.losses (softmax CE, smooth-L1 beta 0, class-specific) in torch"""
    logits, deltas = logits.float(), deltas.float()
    pred = logits.argmax(dim=1)
    fg_inds = (gt_classes >= 0) & (gt_classes < K)
    num_fg = fg_inds.nonzero().numel()
    fg_gt, fg_pred = gt_classes[fg_inds], pred[fg_inds]
    stats = (num_fg, (fg_pred == K).nonzero().numel(), (pred == gt_classes).nonzero().numel(),
             (fg_pred == fg_gt).nonzero().numel())
    loss_cls = F.cross_entropy(logits, gt_classes, reduction="mean")
    fg = torch.nonzero((gt_classes >= 0) & (gt_classes < K), as_tuple=True)[0]
    d = deltas.view(-1, K, 4)[fg, gt_classes[fg]]
    src, tgt = props[fg], gt_boxes[fg]
    sw, sh = src[:, 2] - src[:, 0], src[:, 3] - src[:, 1]
    scx, scy = src[:, 0] + 0.5 * sw, src[:, 1] + 0.5 * sh
    tw, th = tgt[:, 2] - tgt[:, 0], tgt[:, 3] - tgt[:, 1]
    tcx, tcy = tgt[:, 0] + 0.5 * tw, tgt[:, 1] + 0.5 * th
    wx, wy, ww, wh = WEIGHTS
    t = torch.stack((wx * (tcx - scx) / sw, wy * (tcy - scy) / sh, ww * torch.log(tw / sw), wh * torch.log(th / sh)), 1)
    loss_box = torch.abs(d - t).sum() / max(gt_classes.numel(), 1.0)
    return loss_cls, loss_box, stats


def config(det, n, dtype, rounds, quick):
    dev = torch.device("cuda", 0)
    M = n * P
    e = torch.tensor([], dtype=dtype).element_size()
    in_bytes = M * (e * (K + 1) + e * 4 * K + 16 + 8 + 16)
    R = 2 if quick else max(2, math.ceil(2 * L2 / in_bytes) + 1)
    sets = [make_inputs(n, 100 + r, dev, dtype) for r in range(R)]
    fr = det.FastRCNNOutputs(K, det.Box2BoxTransform(WEIGHTS, CLAMP))
    n_fg = int(((sets[0][3] >= 0) & (sets[0][3] < K)).sum())
    read_bytes = M * (e * (K + 1) + 8) + n_fg * (4 * e + 32)
    write_bytes = M * e * (5 * K + 1)
    med = lambda v: sorted(v)[len(v) // 2]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"images": n, "rows": M, "classes": K, "dtype": str(dtype).replace("torch.", ""), "fg_rows": n_fg,
           "input_sets_per_replay": R, "input_bytes_per_call": in_bytes}
    for mode in ("forward", "forward_backward"):
        grads = mode == "forward_backward"
        outs = [None] * R

        def call_all():
            for r, s in enumerate(sets):
                outs[r] = fr.losses_batched(*s, with_grads=grads)

        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            call_all()
        torch.cuda.current_stream().wait_stream(st)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=st):
            call_all()
        for _ in range(3):
            graph.replay()
        call_all()
        torch.cuda.synchronize()

        def torch_all():
            for lg, dl, pr, gc, gb in sets:
                lg = lg.detach().requires_grad_(True)
                dl = dl.detach().requires_grad_(True)
                lc, lb, _ = torch_losses(lg, dl, pr, gc, gb)
                if grads:
                    (lc + lb).backward()

        torch_all()
        torch.cuda.synchronize()
        reps = 2 if quick else 10
        ours_graph, ours_eager, ref = [], [], []
        for _ in range(rounds):
            e0.record()
            for _ in range(reps):
                graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ours_graph.append(e0.elapsed_time(e1) / (reps * R))
            e0.record()
            call_all()
            e1.record()
            torch.cuda.synchronize()
            ours_eager.append(e0.elapsed_time(e1) / R)
            e0.record()
            torch_all()
            e1.record()
            torch.cuda.synchronize()
            ref.append(e0.elapsed_time(e1) / R)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize()
        tot, calls = 0.0, 0
        for ev in prof.events():
            if ev.device_type.name == "CUDA" and "fast_rcnn_loss_kernel" in ev.name:
                tot += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                calls += 1
        kern_us = tot / calls if calls else None
        algo = read_bytes + (write_bytes if grads else 0)
        # agreement with the torch restatement on the first input set
        lc, lb, stats = torch_losses(*sets[0])
        o = outs[0]["sums"]
        agree = {"loss_cls_rel_diff": abs(float(o[0]) - float(lc)) / abs(float(lc)),
                 "loss_box_reg_rel_diff": abs(float(o[1]) - float(lb)) / max(abs(float(lb)), 1e-30),
                 "counts_equal": [int(o[2]), int(o[5]), int(o[3]), int(o[4])] == list(stats)}
        res[mode] = {"ours_graph_us_per_call": 1000 * med(ours_graph), "ours_graph_us_rounds": [1000 * v for v in ours_graph],
                     "ours_eager_us_per_call": 1000 * med(ours_eager),
                     "torch_us_per_call": 1000 * med(ref), "torch_us_rounds": [1000 * v for v in ref],
                     "speedup_graph_vs_torch": med(ref) / med(ours_graph),
                     "speedup_eager_vs_torch": med(ref) / med(ours_eager),
                     "kernel_us": kern_us, "kernel_launches_profiled": calls, "algorithmic_bytes": algo,
                     "algorithmic_tb_per_s": (algo / (kern_us * 1e-6) / 1e12) if kern_us else None,
                     "agreement_with_torch": agree}
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    import det_b200 as det
    props = torch.cuda.get_device_properties(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        power = f"unavailable ({e})"
    res = {"gpu": props.name, "sms": props.multi_processor_count, "power_limit_and_max_sm_clock": power,
           "l2_bytes_assumed": L2, "timing": __doc__.split("Timing: ")[1].strip()}
    print(json.dumps({k: res[k] for k in ("gpu", "sms", "power_limit_and_max_sm_clock")}), flush=True)
    sizes = (2,) if args.quick else (16, 2)
    res["configs"] = {f"n{n}_{str(dt).replace('torch.', '')}": config(det, n, dt, 2 if args.quick else args.rounds,
                                                                       args.quick)
                      for n in sizes for dt in (torch.float32, torch.bfloat16)}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
