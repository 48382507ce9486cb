#!/usr/bin/env python
"""Second-stage (Fast R-CNN box predictor) inference: det_b200.FastRCNNOutputs.inference_batched (det_roi_detect_typed:
the select kernel + the NMS kernel) against a torch-CUDA restatement of detectron2's fast_rcnn_inference loop on the
same inputs.

    python profiles/scripts/time_roi_detect.py [--out FILE] [--rounds 5] [--quick]

Sizes: COCO-like, N = 8 and 64 images x P = 1000 proposals, K = 80 classes, class-specific deltas, score_thresh 0.05,
IoU 0.5, top-100.  Logits: randn, background column + 4 + U(-0.5, 1) per image, so that a few hundred to two thousand
(proposal, class) pairs per image pass the threshold (the count is reported).

Timing: CUDA events.  Ours is captured in a CUDA graph (owned workspace: exactly two launches per call) that runs the
call on R distinct copies of the inputs, R * bytes > 2 * L2, so every call reads its rows from HBM; ms per call =
replay time / R, median of `rounds`.  The select kernel's own time comes from torch.profiler over separate replays
(kernel durations / calls) and is set against its algorithmic bytes M * (4(K+1) + 16K + 16) read plus the candidates
it writes (28 bytes each).  The torch loop synchronises per image (nonzero), so it is timed around back-to-back calls on
the same R copies.
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
import torchvision  # noqa: E402

L2 = 126 * 1024 * 1024
K, P = 80, 1000
WEIGHTS = (10.0, 10.0, 5.0, 5.0)
CLAMP = math.log(1000.0 / 16)


def make_inputs(n, seed, dev):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(n * P, K + 1, generator=g)
    logits.view(n, P, K + 1)[:, :, K] += 4.0 + (torch.rand(n, 1, generator=g) * 1.5 - 0.5)
    deltas = torch.randn(n * P, 4 * K, generator=g) * 0.5
    h, w = 800, 1216
    xy = torch.rand(n * P, 2, generator=g) * torch.tensor([w * 0.9, h * 0.9])
    wh = 16.0 + torch.rand(n * P, 2, generator=g) * torch.tensor([w * 0.3, h * 0.3])
    props = torch.cat([xy, xy + wh], 1)
    off = torch.arange(n + 1, dtype=torch.int32) * P
    sizes = torch.tensor([[h, w]] * n, dtype=torch.int32)
    return [t.to(dev) for t in (logits, deltas, props, off, sizes)]


def torch_loop(logits, deltas, props, sizes_host, thr, iou, topk):
    """detectron2's FastRCNNOutputLayers.predict_probs / predict_boxes + fast_rcnn_inference, in torch on the GPU"""
    n = len(sizes_host)
    probs = F.softmax(logits, dim=-1)
    d = deltas.view(-1, K, 4)
    wx, wy, ww, wh = WEIGHTS
    w = (props[:, 2] - props[:, 0])[:, None]
    h = (props[:, 3] - props[:, 1])[:, None]
    cx, cy = props[:, 0:1] + 0.5 * w, props[:, 1:2] + 0.5 * h
    dw = torch.clamp(d[..., 2] / ww, max=CLAMP)
    dh = torch.clamp(d[..., 3] / wh, max=CLAMP)
    pcx, pcy = d[..., 0] / wx * w + cx, d[..., 1] / wy * h + cy
    pw, ph = torch.exp(dw) * w, torch.exp(dh) * h
    boxes = torch.stack((pcx - 0.5 * pw, pcy - 0.5 * ph, pcx + 0.5 * pw, pcy + 0.5 * ph), dim=-1)
    out = []
    for i in range(n):
        s, b = probs[i * P:(i + 1) * P], boxes[i * P:(i + 1) * P]
        valid = torch.isfinite(b).flatten(1).all(1) & torch.isfinite(s).all(1)
        s, b = s[valid][:, :-1], b[valid]
        hh, ww_ = sizes_host[i]
        b = torch.stack((b[..., 0].clamp(0, ww_), b[..., 1].clamp(0, hh), b[..., 2].clamp(0, ww_),
                         b[..., 3].clamp(0, hh)), -1)
        mask = s > thr
        idx = mask.nonzero()
        bb, ss = b[mask], s[mask]
        keep = torchvision.ops.batched_nms(bb, ss, idx[:, 1], iou)[:topk]
        out.append((idx[keep, 0] * K + idx[keep, 1], ss[keep]))
    return out


def config(det, n, rounds, quick):
    dev = torch.device("cuda", 0)
    row_bytes = 4 * (K + 1) + 16 * K + 16
    in_bytes = n * P * (row_bytes + 4) + 8 * n
    R = max(2, math.ceil(2 * L2 / in_bytes) + 1)
    if quick:
        R = 2
    sets = [make_inputs(n, 100 + r, dev) for r in range(R)]
    fr = det.FastRCNNOutputs(K, det.Box2BoxTransform(WEIGHTS, CLAMP), 0.05, 0.5, 100, cand_cap=4096)
    ws = det.DenseDetectWorkspace(n, 4096, dev)
    outs = [None] * R

    def call_all():
        for r, (lg, dl, pr, off, sz) in enumerate(sets):
            outs[r] = fr.inference_batched(lg, dl, pr, off, sz, out=outs[r], workspace=ws, check=False)

    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        call_all()
    torch.cuda.current_stream().wait_stream(st)
    torch.cuda.synchronize()
    assert all(int(o["overflow"].item()) == 0 for o in outs)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call_all()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3 if quick else 20
    ours = []
    for _ in range(rounds):
        e0.record()
        for _ in range(reps):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
        ours.append(e0.elapsed_time(e1) / (reps * R))
    # kernel durations from the profiler, in a run of their own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            graph.replay()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = "select" if "roi_detect_kernel" in ev.name else ("nms" if "dense_detect_nms_kernel" in ev.name else None)
        if name:
            t = kern.setdefault(name, [0.0, 0])
            t[0] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            t[1] += 1
    kern_us = {k: v[0] / v[1] for k, v in kern.items() if v[1]}
    # candidates written by the select kernel: the number that passed
    n_cand = []
    for lg, dl, pr, off, sz in sets[:1]:
        p = F.softmax(lg, -1)[:, :K]
        n_cand = (p > 0.05).view(n, P * K).sum(1).tolist()
    algo_bytes = n * P * row_bytes + 28 * sum(n_cand)
    sel_us = kern_us.get("select")
    # the torch loop on the same inputs
    sizes_host = [(800, 1216)] * n
    torch_loop(*sets[0][:3], sizes_host, 0.05, 0.5, 100)
    torch.cuda.synchronize()
    loop = []
    for _ in range(rounds):
        e0.record()
        for lg, dl, pr, off, sz in sets:
            torch_loop(lg, dl, pr, sizes_host, 0.05, 0.5, 100)
        e1.record()
        torch.cuda.synchronize()
        loop.append(e0.elapsed_time(e1) / R)
    # agreement with the loop (its softmax sums in another order, so a score at the threshold or a tie may differ)
    ref = torch_loop(*sets[0][:3], sizes_host, 0.05, 0.5, 100)
    o = outs[0]
    same = sum(int(torch.equal(o["idx"][i, :int(o["count"][i])], ref[i][0])) for i in range(n))
    med = lambda v: sorted(v)[len(v) // 2]
    res = {"images": n, "proposals_per_image": P, "classes": K, "input_sets_per_replay": R,
           "input_bytes_per_call": in_bytes, "candidates_per_image": {"min": min(n_cand), "max": max(n_cand),
                                                                       "mean": sum(n_cand) / n},
           "ours_ms_per_call": med(ours), "ours_ms_rounds": ours, "ours_us_per_image": 1000 * med(ours) / n,
           "kernel_us": kern_us, "select_algorithmic_bytes": algo_bytes,
           "select_tb_per_s": (algo_bytes / (sel_us * 1e-6) / 1e12) if sel_us else None,
           "torch_loop_ms_per_call": med(loop), "torch_loop_ms_rounds": loop,
           "speedup_vs_torch_loop": med(loop) / med(ours), "images_with_identical_idx_vs_torch_loop": same}
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
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
    res["configs"] = {f"n{n}": config(det, n, 2 if args.quick else args.rounds, args.quick)
                      for n in ((2,) if args.quick else (8, 64))}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
