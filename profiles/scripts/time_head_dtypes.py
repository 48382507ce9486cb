#!/usr/bin/env python
"""16-bit detection heads: native reads against the fp32 path and against the route a 16-bit head took before the
decode kernels read bf16 / fp16 (an explicit .float() copy, then the fp32 call).

    python profiles/scripts/time_head_dtypes.py [--dtype bf16|fp16] [--out FILE] [--quick]

Three arms per configuration, alternated (a b c a b c ...), each timed from one CUDA graph (bench.time_graph) over a
pool of input sets larger than the 126 MB L2:
  (a) fp32 head;  (b) 16-bit head, .float() then the fp32 call;  (c) 16-bit head read natively.
Arm (c) computes bit-identical results to (b) (tests/test_gpu_head_dtypes.py); the script checks that once per
configuration as well.  Algorithmic bytes use the element size `e` of the head the kernel reads (4 for (a), 2 for (c));
the peak is bench.load_peaks()'s.  The host pipeline arm times YoloHostPipeline end to end (pinned host batch -> H2D ->
kernel -> D2H, 8 slots on 8 streams) with the host-side fill of the pinned input inside the timed loop.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "object-detection-pytorch-rust_b200"))

import torch  # noqa: E402

import bench  # noqa: E402

L2 = 126 * 1024 * 1024
STRIDES = [8, 16, 32]
WH = [[[10, 13], [16, 30], [33, 23]], [[30, 61], [62, 45], [59, 119]], [[116, 90], [156, 198], [373, 326]]]


def pool_size(set_bytes, minimum=2):
    return max(minimum, -(-2 * L2 // set_bytes))  # at least twice the L2 per pool


def three_arms(fa, fb, fc, iters, rounds):
    """median ms per step of each arm over `rounds` alternated rounds"""
    ms = {"a": [], "b": [], "c": []}
    for _ in range(rounds):
        for k, f in (("a", fa), ("b", fb), ("c", fc)):
            ms[k].append(bench.time_graph(f, iters))
    return {k: sorted(v)[len(v) // 2] for k, v in ms.items()}, ms


def same(x, y):
    if isinstance(x, dict):
        return all(same(x[k], y[k]) for k in x if torch.is_tensor(x[k]))
    if isinstance(x, (tuple, list)):
        return all(same(a, b) for a, b in zip(x, y))
    if x.dtype == torch.float32:
        return torch.equal(x.view(torch.int32), y.view(torch.int32))
    return torch.equal(x, y)


def detect_same(r16, r32):
    if not torch.equal(r16["count"], r32["count"]):
        return False
    for i, k in enumerate(r16["count"].tolist()):
        k = max(k, 0)
        if not all(same(r16[key][i, :k], r32[key][i, :k]) for key in ("idx", "boxes", "scores", "classes")):
            return False
    return True


def entry(ms, bytes_a, bytes_c, peak, formula, samples, identical):
    e = {"ms": ms, "ms_rounds": samples, "c_faster_than_b": ms["c"] < ms["b"], "speedup_c_over_b": ms["b"] / ms["c"],
         "c_over_a": ms["c"] / ms["a"], "c_equals_b_bitwise": identical}
    if bytes_a is not None:
        e["roofline"] = {"formula": formula, "bytes_a": bytes_a, "bytes_c": bytes_c,
                         "frac_a": bytes_a / ms["a"] / 1e6 / peak, "frac_c": bytes_c / ms["c"] / 1e6 / peak}
    return e


def dense(det, dev, dt, peak, quick, rounds, out):
    C = 80
    dh = det.DenseAnchorHead(STRIDES, WH, C)
    R = 25200
    for n in ((8,) if quick else (32, 256)):
        g = torch.Generator(device=dev).manual_seed(3)
        set16 = n * R * (5 + C) * 2
        pool = pool_size(set16)
        h32, h16 = [], []
        for _ in range(pool):
            hs = [torch.randn(n, 3 * (5 + C), 640 // s, 640 // s, device=dev, generator=g) for s in STRIDES]
            for h in hs:
                h.view(n, 3, 5 + C, h.shape[2], h.shape[3])[:, :, 4] -= 4.0  # objectness bias (SURVEY Cfg4)
            h16.append([h.to(dt) for h in hs])
            h32.append([h.float() for h in h16[-1]])  # the same values: arm (a) reads exactly what (b) and (c) compute on
        iters = 3 if quick else (10 if n > 64 else 40)
        ob = (torch.empty((n, R, 4), device=dev), torch.empty((n, R), device=dev),
              torch.empty((n, R), dtype=torch.int64, device=dev))
        ms, samples = three_arms([lambda hs=hs: dh.decode(hs, out=ob) for hs in h32],
                                 [lambda hs=hs: dh.decode([h.float() for h in hs], out=ob) for hs in h16],
                                 [lambda hs=hs: dh.decode(hs, out=ob) for hs in h16], iters, rounds)
        ident = same(dh.decode(h16[0]), dh.decode([h.float() for h in h16[0]]))
        out[f"dense_decode_n{n}"] = entry(ms, n * (4 * R * (5 + C) + 28 * R), n * (2 * R * (5 + C) + 28 * R), peak,
                                          "N * (e*R*(5+C) read + 28*R written), R=25200, C=80", samples, ident)
        print(json.dumps({f"dense_decode_n{n}": out[f"dense_decode_n{n}"]["ms"]}), flush=True)
        del ob
        for thr in (0.1, 0.25):
            for gate in (False, True):
                cap, max_det = 2048, 300
                ws = {k: det.DenseDetectWorkspace(n, cap, dev) for k in "abc"}
                res = {k: dh.detect_thresholded(h16[0] if k == "c" else h32[0], thr, 0.5, max_det=max_det, cand_cap=cap,
                                                gate=gate, check=True, workspace=ws[k]) for k in "abc"}
                run = lambda k, hs: dh.detect_thresholded(hs, thr, 0.5, max_det=max_det, cand_cap=cap, gate=gate,
                                                          check=False, out=res[k], workspace=ws[k])
                ms, samples = three_arms([lambda hs=hs: run("a", hs) for hs in h32],
                                         [lambda hs=hs: run("b", [h.float() for h in hs]) for hs in h16],
                                         [lambda hs=hs: run("c", hs) for hs in h16], iters, rounds)
                r16 = dh.detect_thresholded(h16[0], thr, 0.5, max_det=max_det, cand_cap=cap, gate=gate, check=True)
                r32 = dh.detect_thresholded(h32[0], thr, 0.5, max_det=max_det, cand_cap=cap, gate=gate, check=True)
                k_mean = float(r32["count"].float().mean())
                key = f"dense_detect_n{n}_thr{thr}_{'gate' if gate else 'nogate'}"
                e = entry(ms, None if gate else n * (4 * R * (5 + C) + 36 * k_mean + 4),
                          None if gate else n * (2 * R * (5 + C) + 36 * k_mean + 4), peak,
                          "N * (e*R*(5+C) read + (36*K + 4) written), K = kept per image (gate off: whole head streamed)",
                          samples, detect_same(r16, r32))
                e["kept_per_image"] = k_mean
                if n >= 256 and thr == 0.1 and not gate:  # how tie-prone the 16-bit candidate lists are
                    sc = dh.decode(h16[0])[1]
                    ties = 0
                    for i in range(n):
                        s = sc[i][sc[i] > thr]
                        ties += int(s.numel() - s.unique().numel())
                    e["equal_candidate_scores_per_image"] = ties / n
                out[key] = e
                print(json.dumps({key: e["ms"]}), flush=True)
        del h32, h16
        torch.cuda.empty_cache()


def rpn(det, dev, dt, peak, quick, rounds, out):
    strides = [4, 8, 16, 32, 64]
    r = det.RegionProposalNetwork(strides, [[32], [64], [128], [256], [512]], [[0.5, 1.0, 2.0]]).eval()
    img, R = 448, 50127
    for n in ((8,) if quick else (64, 256)):
        g = torch.Generator(device=dev).manual_seed(5)
        pool = pool_size(n * R * 5 * 2)
        s16, s32 = [], []
        for _ in range(pool):
            obj = [torch.randn(n, 3, img // s, img // s, device=dev, generator=g).to(dt) for s in strides]
            dlt = [(torch.randn(n, 12, img // s, img // s, device=dev, generator=g) * 0.3).to(dt) for s in strides]
            s16.append((obj, dlt))
            s32.append(([o.float() for o in obj], [d.float() for d in dlt]))
        up = lambda p: ([o.float() for o in p[0]], [d.float() for d in p[1]])
        iters = 3 if quick else 20
        ms, samples = three_arms([lambda p=p: r.decode_heads(*p) for p in s32],
                                 [lambda p=p: r.decode_heads(*up(p)) for p in s16],
                                 [lambda p=p: r.decode_heads(*p) for p in s16], iters, rounds)
        ident = same(r.decode_heads(*s16[0])[:2], r.decode_heads(*up(s16[0]))[:2])
        out[f"rpn_decode_heads_n{n}"] = entry(ms, n * R * (4 * 5 + 20), n * R * (2 * 5 + 20), peak,
                                              "N * R * (e*5 read (objectness + 4 deltas) + 20 written), R=50127",
                                              samples, ident)
        print(json.dumps({f"rpn_decode_heads_n{n}": ms}), flush=True)
        sizes = torch.tensor([[img, img]] * n, dtype=torch.int32, device=dev)
        ms, samples = three_arms([lambda p=p: r.proposals_from_heads(*p, sizes) for p in s32],
                                 [lambda p=p: r.proposals_from_heads(*up(p), sizes) for p in s16],
                                 [lambda p=p: r.proposals_from_heads(*p, sizes) for p in s16], iters, rounds)
        ident = same(r.proposals_from_heads(*s16[0], sizes), r.proposals_from_heads(*up(s16[0]), sizes))
        out[f"rpn_proposals_from_heads_n{n}"] = entry(ms, None, None, peak, None, samples, ident)
        print(json.dumps({f"rpn_proposals_from_heads_n{n}": ms}), flush=True)
        del s16, s32
        torch.cuda.empty_cache()


def yolo(det, dev, dt, peak, quick, rounds, out):
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    n = 32 if quick else 256
    set16 = n * 7 * 7 * 30 * 2
    pool = pool_size(set16)
    g = torch.Generator(device=dev).manual_seed(7)
    h16 = [torch.randn(n, 7, 7, 30, device=dev, generator=g).to(dt) for _ in range(pool)]
    h32 = [h.float() for h in h16]
    res = {k: yh.detect(h32[0], 0.25, 0.5, max_det=300) for k in "abc"}
    run = lambda k, h: yh.detect(h, 0.25, 0.5, max_det=300, out=res[k])
    ms, samples = three_arms([lambda h=h: run("a", h) for h in h32], [lambda h=h: run("b", h.float()) for h in h16],
                             [lambda h=h: run("c", h) for h in h16], 3 if quick else 20, rounds)
    ident = same(yh.detect(h16[0], 0.25, 0.5, max_det=300), yh.detect(h16[0].float(), 0.25, 0.5, max_det=300))
    out[f"yolo_detect_n{n}"] = entry(ms, None, None, peak, None, samples, ident)
    out[f"yolo_detect_n{n}"]["pool_sets"] = pool
    print(json.dumps({f"yolo_detect_n{n}": ms}), flush=True)


def host_pipeline(det, dev, dt, quick, rounds, out):
    yh = det.YoloGridHead(7, 2, 20, (448, 448))
    batch, depth = (32, 4) if quick else (256, 8)
    g = torch.Generator().manual_seed(11)
    host16 = [torch.randn(batch, 7, 7, 30, generator=g).to(dt) for _ in range(16)]
    host32 = [h.float() for h in host16]
    pipes = {"a": det.YoloHostPipeline(yh, batch, 0.25, 0.5, 300, depth=depth, index_dtype=torch.int32),
             "b": det.YoloHostPipeline(yh, batch, 0.25, 0.5, 300, depth=depth, index_dtype=torch.int32),
             "c": det.YoloHostPipeline(yh, batch, 0.25, 0.5, 300, depth=depth, index_dtype=torch.int32, input_dtype=dt)}
    src = {"a": host32, "b": host16, "c": host16}  # (b) converts the 16-bit host batch into the fp32 pinned input

    def run(k, steps):
        p = pipes[k]
        for i in range(steps):
            s = i % depth
            if i >= depth:
                p.wait(s)
            p.input(s).copy_(src[k][i % len(src[k])])
            p.launch(s)
        for s in range(depth):
            p.wait(s)

    steps = 64 if quick else 2000
    samples = {"a": [], "b": [], "c": []}
    for k in "abc":
        run(k, 2 * depth)  # warm-up
    for _ in range(rounds):
        for k in "abc":
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(k, steps)
            samples[k].append((time.perf_counter() - t0) * 1e3 / steps)
    ms = {k: sorted(v)[len(v) // 2] for k, v in samples.items()}
    ident = True
    for k in "bc":
        got = pipes[k].run(host16[0])
        want = yh.detect(host16[0].cuda().float(), 0.25, 0.5, max_det=300, index_dtype=torch.int32)
        cnt = got["count"]
        ident = ident and torch.equal(cnt, want["count"].cpu()) and all(
            same(got[key][i, :c], want[key][i, :c].cpu()) for i, c in enumerate(cnt.tolist()) for key in ("flat", "boxes", "scores"))
    e = entry(ms, None, None, 0, None, samples, ident)
    e.update({"batch": batch, "depth": depth, "steps": steps, "h2d_bytes": {k: p.h2d_bytes for k, p in pipes.items()},
              "d2h_bytes": pipes["a"].d2h_bytes, "images_per_s": {k: batch / v * 1e3 for k, v in ms.items()}})
    out[f"yolo_host_pipeline_b{batch}_depth{depth}"] = e
    print(json.dumps({"host_pipeline": ms}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    import det_b200 as det
    dev = torch.device("cuda", 0)
    dt = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    peak, peak_src = bench.load_peaks()
    props = torch.cuda.get_device_properties(dev)
    power = None
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        power = f"unavailable ({e})"
    res = {"gpu": props.name, "sms": props.multi_processor_count, "power_limit_and_max_sm_clock": power,
           "dtype": args.dtype, "peak_gbs": peak, "peak_source": peak_src,
           "arms": {"a": "fp32 head", "b": f"{args.dtype} head, .float() then the fp32 call (the route before native reads)",
                    "c": f"{args.dtype} head read natively"},
           "timing": "bench.time_graph: ms per step from one CUDA graph over a pool of input sets > 126 MB L2, median of "
                     f"{args.rounds} alternated rounds; host pipeline: wall clock over its steps, synchronised"}
    print(json.dumps({k: res[k] for k in ("gpu", "power_limit_and_max_sm_clock", "peak_gbs", "peak_source")}), flush=True)
    res["configs"] = {}
    dense(det, dev, dt, peak, args.quick, args.rounds, res["configs"])
    rpn(det, dev, dt, peak, args.quick, args.rounds, res["configs"])
    yolo(det, dev, dt, peak, args.quick, args.rounds, res["configs"])
    host_pipeline(det, dev, dt, args.quick, args.rounds, res["configs"])
    res["all_c_faster_than_b"] = all(e["c_faster_than_b"] for e in res["configs"].values())
    res["all_c_equal_b_bitwise"] = all(e["c_equals_b_bitwise"] for e in res["configs"].values())
    print(json.dumps({"all_c_faster_than_b": res["all_c_faster_than_b"], "all_c_equal_b_bitwise": res["all_c_equal_b_bitwise"]}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:  # one line per configuration
            cfg = res.pop("configs")
            head = [f" {json.dumps(k)}: {json.dumps(v)}," for k, v in res.items()]
            body = [f"  {json.dumps(k)}: {json.dumps(v)}" for k, v in cfg.items()]
            f.write("{\n" + "\n".join(head) + '\n "configs": {\n' + ",\n".join(body) + "\n }\n}\n")


if __name__ == "__main__":
    main()
