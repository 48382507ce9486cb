"""Device time of the fused YOLO decode+NMS launch (det_yolo_decode_nms, 7x7x30 head, 256 images, max_det 300) on three
input regimes, for one or more source trees, each tree timed in a subprocess of its own and the trees alternated:

  bench      bench.py's inputs: seeded randn logits, score > 0.25, IoU 0.5 (about 845 candidates per image)
  overlap    tests/test_gpu_yolo.py test_yolo_fast_path_heavy_overlap: priors 300/380, w/h logits x 0.05, score > 0.2,
             IoU 0.3 (long suppression chains inside every class)
  low_score  bench inputs with score > 0.02: about 1 900 candidates per image, the per-category branch

    python profiles/scripts/time_yolo_regimes.py [--rounds 3] [TREE ...]     (default TREE: this repository)

A pool of 8 input batches (12 MB, L2-resident after the first pass) is replayed from one CUDA graph of 200 launches;
the time is CUDA events around 20 replays.  Prints one JSON line per (round, tree) and a summary (median us per launch)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def inputs(name, torch):
    g = torch.Generator().manual_seed(1)
    heads = torch.randn(8, 256, 7, 7, 30, generator=g)
    priors, score, iou = None, 0.25, 0.5
    if name == "overlap":
        heads[..., 2:4] *= 0.05
        heads[..., 7:9] *= 0.05
        priors, score, iou = [[300, 300], [380, 380]], 0.2, 0.3
    elif name == "low_score":
        score = 0.02
    return heads, priors, score, iou


def worker(tree):
    sys.path.insert(0, os.path.join(tree, "object-detection-pytorch-rust_b200"))
    import torch
    import det_b200 as det
    det._native.lib()
    out = {"tree": tree, "device": torch.cuda.get_device_name(0)}
    for name in ("bench", "overlap", "low_score"):
        heads, priors, score, iou = inputs(name, torch)
        yh = det.YoloGridHead(7, 2, 20, (448, 448), priors=priors)
        heads = heads.cuda()
        res = yh.detect(heads[0], score, iou, max_det=300)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            yh.detect(heads[1], score, iou, max_det=300, out=res)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            for i in range(200):
                yh.detect(heads[i % 8], score, iou, max_det=300, out=res)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        out[name] = {"us_per_launch": e0.elapsed_time(e1) * 1e3 / 4000,
                     "kept_per_image": float(res["count"].float().mean())}
    print(json.dumps(out))


def main():
    args = sys.argv[1:]
    if args[:1] == ["--worker"]:
        worker(args[1])
        return
    rounds = 3
    if args[:1] == ["--rounds"]:
        rounds, args = int(args[1]), args[2:]
    trees = [os.path.abspath(t) for t in args] or [ROOT]
    rows = []
    for r in range(rounds):
        for t in trees:
            line = subprocess.check_output([sys.executable, os.path.abspath(__file__), "--worker", t], text=True)
            row = json.loads(line.strip().splitlines()[-1])
            row["round"] = r
            rows.append(row)
            print(json.dumps(row), flush=True)
    summary = {}
    for t in trees:
        mine = [x for x in rows if x["tree"] == t]
        summary[t] = {k: sorted(x[k]["us_per_launch"] for x in mine)[len(mine) // 2] for k in ("bench", "overlap", "low_score")}
    print(json.dumps({"median_us_per_launch": summary}))


if __name__ == "__main__":
    main()
