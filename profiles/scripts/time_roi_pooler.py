#!/usr/bin/env python
"""ROIPooler: the ROIPool type against the reference's per-level loop, and bf16 feature pyramids read natively against
the route a 16-bit pyramid took before the pooling kernels read bf16 / fp16.

    python profiles/scripts/time_roi_pooler.py [--out FILE] [--rounds 3] [--quick]

Sizes: the reference config (FPN-18: 64 channels, 448x448, strides 4..32) and a detectron2-sized batch (256 channels,
800x1344, strides 4..32), 16 images x 512 boxes each, 7x7 output.  Timing: CUDA events around `iters` back-to-back calls
(the reference loop synchronises on nonzero(), so it cannot be graph-captured; every arm is timed the same way), arms
alternated in rounds, median.  The features are not re-written between calls: the FPN-18 pyramid (68 MB in fp32) stays
in the 126 MB L2, as it does in real use right after the FPN wrote it; the detectron2-sized one (1.46 GB in fp32) does
not.

  ROIPool, fp32, forward and forward+backward: ours (det_roi_levels + one det_roi_pool_levels launch) against the
  reference's loop over levels (nonzero -> torchvision CUDA roi_pool -> index_put_), as prof_roi.py does for ROIAlign.
  ROIAlignV2 and ROIPool on a bf16 pyramid, forward and forward+backward, three arms:
    (a) fp32 features;  (b) bf16 features through the previous route (f.float(), the fp32 call, .to(bf16));
    (c) bf16 features read natively.  (c) is checked bit-identical to (b) in forward.
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
import torchvision  # noqa: E402

L2 = 126 * 1024 * 1024
STRIDES = [4, 8, 16, 32]


def timed(fn, iters):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def arms(fns, iters, rounds):
    """median ms per call of each arm over `rounds` alternated rounds"""
    ms = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            ms[k].append(timed(f, iters))
    return {k: sorted(v)[len(v) // 2] for k, v in ms.items()}, ms


def boxes_for(n_img, per_img, hw, g):
    h, w = hw
    out = []
    for _ in range(n_img):
        sz = torch.exp(torch.rand(per_img, generator=g) * math.log(400.0 / 8.0)) * 8.0   # 8 .. 400 px: every level
        ar = torch.exp((torch.rand(per_img, generator=g) - 0.5) * 1.6)
        bw, bh = sz * torch.sqrt(ar), sz / torch.sqrt(ar)
        cx, cy = torch.rand(per_img, generator=g) * w, torch.rand(per_img, generator=g) * h
        out.append(torch.stack((cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2), 1))
    return out


def reference_loop(feats, scales, bl, pool):
    """reference ROIPooler.forward (roi_poolers.py:269-331) over torchvision's CUDA kernels"""
    rois = torch.cat([torch.cat((torch.full_like(b[:, :1], i), b), 1) for i, b in enumerate(bl)], 0)
    allb = torch.cat(bl, 0)
    area = (allb[:, 2] - allb[:, 0]) * (allb[:, 3] - allb[:, 1])
    lv = torch.clamp(torch.floor(4 + torch.log2(torch.sqrt(area) / 224 + 1e-8)), min=2, max=5).to(torch.int64) - 2
    out = torch.zeros((rois.shape[0], feats[0].shape[1], 7, 7), device=rois.device, dtype=feats[0].dtype)
    for l, (f, s) in enumerate(zip(feats, scales)):
        inds = torch.nonzero(lv == l, as_tuple=True)[0]
        r = rois[inds]
        out = out.index_put((inds,), torchvision.ops.roi_pool(f, r, (7, 7), s) if pool
                            else torchvision.ops.roi_align(f, r, (7, 7), s, 0, True))
    return out


def fwd_bwd(run, feats, gout):
    """one forward and the gradients w.r.t. every feature map (no accumulation into .grad)"""
    out = run(feats)
    return torch.autograd.grad(out, feats, gout)


def config(det, name, n_img, C, hw, per_img, iters, rounds):
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(1)
    scales = [1.0 / s for s in STRIDES]
    f16 = [torch.randn(n_img, C, hw[0] // s, hw[1] // s, generator=g).to(dev).to(torch.bfloat16) for s in STRIDES]
    f32 = [f.float() for f in f16]           # the same values: (a) reads exactly what (b) and (c) compute on
    bl = [b.to(dev) for b in boxes_for(n_img, per_img, hw, g)]
    boxes = [det.Boxes(b) for b in bl]
    m = n_img * per_img
    elems = sum(f.numel() for f in f32)
    res = {"images": n_img, "boxes_per_image": per_img, "channels": C, "image_hw": list(hw), "output": [7, 7],
           "pyramid_elements": elems, "pyramid_bytes_fp32": 4 * elems, "pyramid_bytes_bf16": 2 * elems,
           "fp32_pyramid_fits_l2": 4 * elems <= L2, "output_bytes_fp32": m * C * 49 * 4, "cases": {}}
    print(json.dumps({name: {k: v for k, v in res.items() if k != "cases"}}), flush=True)
    for ptype in ("ROIPool", "ROIAlignV2"):
        pooler = det.ROIPooler(scales, 0, 7, ptype)
        ours = lambda fs: pooler(fs, boxes)
        prev = lambda fs: pooler([f.float() for f in fs], boxes).to(torch.bfloat16)  # the route before native reads
        # (c) == (b) bitwise, forward
        c_out, b_out = ours(f16), prev(f16)
        ident = torch.equal(c_out.view(torch.int16), b_out.view(torch.int16))
        gout16 = torch.randn(c_out.shape, device=dev, generator=torch.Generator(device=dev).manual_seed(2)).bfloat16()
        gout32 = gout16.float()
        r16 = [f.clone().requires_grad_(True) for f in f16]
        r32 = [f.clone().requires_grad_(True) for f in f32]
        case = {}
        if ptype == "ROIPool":   # ours vs the reference loop on torchvision CUDA, fp32
            ref_out = reference_loop(f32, scales, bl, True)
            a_out = ours(f32)
            exact = torch.equal(ref_out, a_out)
            ms, samples = arms({"ours": lambda: ours(f32), "reference_loop": lambda: reference_loop(f32, scales, bl, True)},
                               iters, rounds)
            case["fp32_vs_reference_forward"] = {"ms": ms, "ms_rounds": samples, "speedup": ms["reference_loop"] / ms["ours"],
                                                 "outputs_equal": exact}
            print(json.dumps({f"{name}/{ptype}/fp32_vs_reference_forward": ms}), flush=True)
            ms, samples = arms({"ours": lambda: fwd_bwd(ours, r32, gout32),
                                "reference_loop": lambda: fwd_bwd(lambda fs: reference_loop(fs, scales, bl, True), r32,
                                                                  gout32)}, iters, rounds)
            case["fp32_vs_reference_forward_backward"] = {"ms": ms, "ms_rounds": samples,
                                                          "speedup": ms["reference_loop"] / ms["ours"]}
            print(json.dumps({f"{name}/{ptype}/fp32_vs_reference_forward_backward": ms}), flush=True)
        ms, samples = arms({"a": lambda: ours(f32), "b": lambda: prev(f16), "c": lambda: ours(f16)}, iters, rounds)
        case["bf16_forward"] = {"ms": ms, "ms_rounds": samples, "speedup_c_over_b": ms["b"] / ms["c"],
                                "c_over_a": ms["c"] / ms["a"], "c_equals_b_bitwise": ident}
        print(json.dumps({f"{name}/{ptype}/bf16_forward": ms, "c_equals_b_bitwise": ident}), flush=True)
        ms, samples = arms({"a": lambda: fwd_bwd(ours, r32, gout32), "b": lambda: fwd_bwd(prev, r16, gout16),
                            "c": lambda: fwd_bwd(ours, r16, gout16)}, iters, rounds)
        case["bf16_forward_backward"] = {"ms": ms, "ms_rounds": samples, "speedup_c_over_b": ms["b"] / ms["c"],
                                         "c_over_a": ms["c"] / ms["a"]}
        print(json.dumps({f"{name}/{ptype}/bf16_forward_backward": ms}), flush=True)
        res["cases"][ptype] = case
        del r16, r32
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
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
           "l2_bytes_assumed": L2,
           "timing": f"CUDA events around back-to-back calls, median of {args.rounds} alternated rounds; "
                     "features not re-written between calls",
           "arms": {"a": "fp32 features", "b": "bf16 features, f.float() then the fp32 call, then .to(bf16)",
                    "c": "bf16 features read natively"}}
    print(json.dumps({k: res[k] for k in ("gpu", "sms", "power_limit_and_max_sm_clock")}), flush=True)
    sizes = [("fpn18_448", 16, 64, (448, 448), 512, 20), ("detectron2_800x1344", 16, 256, (800, 1344), 512, 10)]
    if args.quick:
        sizes = [("fpn18_448", 2, 64, (448, 448), 64, 3)]
    res["configs"] = {name: config(det, name, n, C, hw, per, 3 if args.quick else it, args.rounds)
                      for name, n, C, hw, per, it in sizes}
    res["all_c_equal_b_bitwise"] = all(c["bf16_forward"]["c_equals_b_bitwise"] for cfg in res["configs"].values()
                                       for c in cfg["cases"].values())
    print(json.dumps({"all_c_equal_b_bitwise": res["all_c_equal_b_bitwise"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")
    assert res["all_c_equal_b_bitwise"], "bf16 native forward differs from the f.float() route"


if __name__ == "__main__":
    main()
