#!/usr/bin/env python
"""Batched ROI-head proposal sampling: det_b200.ROIHeads.sample_proposals_batched (det_roi_sample_proposals: two
launches) against the existing per-image label_and_sample_proposals loop and a torch-CUDA restatement of detectron2's
per-image loop (cat gt -> pairwise_iou -> Matcher -> class labels -> subsample_labels with torch.randperm -> gather),
on the same inputs.

    python profiles/scripts/time_roi_sample.py [--out FILE] [--rounds 7] [--quick]

Sizes: N in {2, 16} images x P in {1000, 2000} proposals per image (detectron2's FPN / C4 training counts), G ~ U[1, 60]
gt boxes per image (seeded), S = 512 samples per image, positive fraction 0.25, K = 80 classes, Matcher([0.5], [0, 1])
without low-quality matches, gt appended.

Timing: CUDA events, warmed up, median over `rounds` rounds that alternate the arms.  Ours graph-replayed: a CUDA graph
of R back-to-back calls that also advances the device seed, ms per call = replay time / R.  Ours eager: R back-to-back
Python calls (host overhead included).  The two per-image loops synchronise the host and are timed around R calls.
The whole working set (< 1 MB) stays in L2, as it does in a training step.  Kernel time: torch.profiler over separate
graph replays (kernel durations / calls).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "object-detection-pytorch-rust_b200"))

import torch  # noqa: E402

K, S, FRAC = 80, 512, 0.25
R = 20


def make_inputs(n, P, seed):
    g = torch.Generator().manual_seed(seed)
    images = []
    for _ in range(n):
        G = int(torch.randint(1, 61, (1,), generator=g))
        xy = torch.rand(G, 2, generator=g) * 900
        gt = torch.cat([xy, xy + 16 + torch.rand(G, 2, generator=g) * 250], 1)
        xy = torch.rand(P, 2, generator=g) * 900
        props = torch.cat([xy, xy + 8 + torch.rand(P, 2, generator=g) * 300], 1)
        k = min(P // 4, 8 * G)  # an RPN's proposals crowd around the objects
        props[:k] = gt.repeat(8, 1)[:k] + (torch.rand(k, 4, generator=g) - 0.5) * 40
        images.append((props, gt, torch.randint(0, K, (G,), generator=g)))
    return images


def pairwise_iou(a, b):
    area1 = (a[:, 2] - a[:, 0]) * (a[:, 3] - a[:, 1])
    area2 = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    wh = (torch.min(a[:, None, 2:], b[None, :, 2:]) - torch.max(a[:, None, :2], b[None, :, :2])).clamp(min=0)
    inter = wh.prod(dim=2)
    return torch.where(inter > 0, inter / (area1[:, None] + area2 - inter), torch.zeros(1, dtype=inter.dtype,
                                                                                         device=inter.device))


def detectron2_loop(props_list, gt_list, cls_list):
    """detectron2 v0.6 ROIHeads.label_and_sample_proposals restated on torch CUDA tensors (boxes and the gathered
    fields only)."""
    out = []
    for props, gt, gcls in zip(props_list, gt_list, cls_list):
        cand = torch.cat([props, gt])
        q = pairwise_iou(gt, cand)
        vals, idx = q.max(dim=0)
        labels = (vals >= 0.5).to(torch.int8)
        cls = gcls[idx]
        cls[labels == 0] = K
        pos = torch.nonzero((cls != -1) & (cls != K), as_tuple=True)[0]
        neg = torch.nonzero(cls == K, as_tuple=True)[0]
        num_pos = min(pos.numel(), int(S * FRAC))
        num_neg = min(neg.numel(), S - num_pos)
        p1 = torch.randperm(pos.numel(), device=cand.device)[:num_pos]
        p2 = torch.randperm(neg.numel(), device=cand.device)[:num_neg]
        sampled = torch.cat([pos[p1], neg[p2]])
        out.append((cand[sampled], cls[sampled], gt[idx[sampled]]))
    return out


def med(v):
    v = sorted(v)
    return v[len(v) // 2]


def config(det, n, P, rounds, seed):
    dev = torch.device("cuda")
    images = make_inputs(n, P, seed)
    heads = det.ROIHeads(K, S, FRAC, det.Matcher([0.5], [0, 1], allow_low_quality_matches=False), True)
    pb = torch.stack([p for p, _, _ in images]).to(dev)
    counts = torch.full((n,), P, dtype=torch.int32, device=dev)
    table, off = det.Matcher.pack_gt([gt.to(dev) for _, gt, _ in images], dev)
    classes = torch.cat([c for _, _, c in images]).to(dev)
    seed_t = torch.tensor([seed], dtype=torch.int64, device=dev)
    props_l = [p.to(dev) for p, _, _ in images]
    gt_l = [gt.to(dev) for _, gt, _ in images]
    cls_l = [c.to(dev) for _, _, c in images]
    proposals, targets = [], []
    for p, gt, c in zip(props_l, gt_l, cls_l):
        pi = det.Instances((1200, 1200))
        pi.proposal_boxes = det.Boxes(p)
        pi.objectness_logits = torch.zeros(P, device=dev)
        t = det.Instances((1200, 1200))
        t.gt_boxes = det.Boxes(gt)
        t.gt_classes = c
        proposals.append(pi)
        targets.append(t)
    args = (pb, counts, table, off, classes, seed_t)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ws = heads.sample_workspace(n, P, table.shape[0], dev)
        out = heads.sample_proposals_batched(*args, workspace=ws)
    torch.cuda.current_stream().wait_stream(st)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=st):
        for _ in range(R):
            heads.sample_proposals_batched(*args, out=out, workspace=ws)
            seed_t.add_(1)
    for _ in range(3):
        graph.replay()
        heads.sample_proposals_batched(*args)
        heads.label_and_sample_proposals(proposals, targets)
        detectron2_loop(props_l, gt_l, cls_l)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    arms = {
        "ours_graph": graph.replay,
        "ours_eager": lambda: [heads.sample_proposals_batched(*args) for _ in range(R)],
        "existing_loop": lambda: [heads.label_and_sample_proposals(proposals, targets) for _ in range(R)],
        "detectron2_torch_loop": lambda: [detectron2_loop(props_l, gt_l, cls_l) for _ in range(R)],
    }
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(1000.0 * e0.elapsed_time(e1) / R)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "roi_sample" in ev.name:
            name = "label" if "label" in ev.name else "select"
            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            s, c = kern.get(name, (0.0, 0))
            kern[name] = (s + t, c + 1)
    gts = [gt.shape[0] for _, gt, _ in images]
    res = {"n": n, "P": P, "G_per_image": gts, "pairs": sum((P + g) * g for g in gts),
           "mean_count": float(out["count"].float().mean()), "mean_num_fg": float(out["num_fg"].float().mean())}
    for k, v in times.items():
        res[k + "_us_per_call"] = med(v)
        res[k + "_us_rounds"] = v
    for k, (s, c) in kern.items():
        res[f"kernel_{k}_us"] = s / c
    res["speedup_graph_vs_existing_loop"] = med(times["existing_loop"]) / med(times["ours_graph"])
    res["speedup_graph_vs_detectron2_loop"] = med(times["detectron2_torch_loop"]) / med(times["ours_graph"])
    print(json.dumps({k: v for k, v in res.items() if not k.endswith("rounds")}), flush=True)
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
           "timing": __doc__.split("Timing: ")[1].strip()}
    print(json.dumps({k: res[k] for k in ("gpu", "sms", "power_limit_and_max_sm_clock")}), flush=True)
    sizes = [(2, 1000)] if args.quick else [(n, P) for n in (2, 16) for P in (1000, 2000)]
    res["configs"] = {f"n{n}_p{P}": config(det, n, P, 2 if args.quick else args.rounds, 100 + n + P)
                      for n, P in sizes}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
