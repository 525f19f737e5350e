#!/usr/bin/env python
"""Throughput of PoseEngine.infer_images on a photo-like mix of frame sizes: frames bucketed by raw shape (the default)
versus ragged runs (ragged=True), on the same frames, with identical person rows asserted between the two.

  python tools/bench_ragged.py [--frames 512] [--reps 3] [--out FILE.json] [--parent-tree DIR --ab-reps 3]

Frames: seeded uniform-noise uint8 BGR frames; sizes drawn half from five common photo sizes (480x640, 640x480, 427x640,
612x612, 375x500) and half uniformly from [240, 720]^2.  Weights: seeded He-normal (as bench.py).  Every shape is warmed up
by one untimed pass of each path; the timed passes alternate the two paths.  The canvas fill fraction (useful pixels /
computed pixels of the ragged runs) is computed from the shapes.  With --parent-tree (a built checkout of another
revision) the unchanged uniform benchmark, `bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline` (batch 32 @368x368),
first runs alternately in that tree and in this one, so that the two builds are compared within the same run-to-run
spread.  Prints one JSON object (also written to --out)."""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import _b200_alias  # noqa: E402

PHOTO_SIZES = [(480, 640), (640, 480), (427, 640), (612, 612), (375, 500)]


def frame_sizes(n, seed):
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        if rs.rand() < 0.5:
            out.append(PHOTO_SIZES[rs.randint(len(PHOTO_SIZES))])
        else:
            out.append((int(rs.randint(240, 721)), int(rs.randint(240, 721))))
    return out


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [s.strip() for s in q.split(",")[:2]]
    except Exception as e:     # the figure is then reported without it, and says so
        info["power_limit"] = "unknown (%s)" % type(e).__name__
    return info


BENCH_ARGS = ["--gpus", "1", "--steps", "20", "--warmup", "5", "--no-cpu-baseline"]


def bench_py(tree):
    """frames/s of bench.py run from `tree` (its own package and library)."""
    r = subprocess.run([sys.executable, "bench.py"] + BENCH_ARGS, cwd=tree, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise SystemExit("bench.py in %s failed (rc %d): %s" % (tree, r.returncode, r.stderr[-2000:]))
    return float(json.loads(lines[-1])["value"])


def bench_ab(parent_tree, reps):
    runs = {"parent": [], "this": []}
    for _ in range(reps):
        runs["parent"].append(bench_py(os.path.abspath(parent_tree)))
        runs["this"].append(bench_py(ROOT))
    med = {k: statistics.median(v) for k, v in runs.items()}
    return {"command": "python bench.py " + " ".join(BENCH_ARGS), "parent_tree": parent_tree,
            "frames_per_s_each_run": runs, "median": med, "this_over_parent": round(med["this"] / med["parent"], 4),
            "spread_parent": round((max(runs["parent"]) - min(runs["parent"])) / med["parent"], 4),
            "spread_this": round((max(runs["this"]) - min(runs["this"])) / med["this"], 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--batch-cap", type=int, default=32)
    ap.add_argument("--mode", default="bf16", choices=["bf16", "bf16x3", "fp32"])
    ap.add_argument("--dest-size", type=int, default=368)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    ap.add_argument("--parent-tree", default="", help="built tree of the revision to compare bench.py against")
    ap.add_argument("--ab-reps", type=int, default=3)
    args = ap.parse_args()

    _b200_alias.load_package()
    import torch
    engine = importlib.import_module(_b200_alias.PKG + ".engine")
    nat = importlib.import_module(_b200_alias.PKG + "._native")
    syn = importlib.import_module(_b200_alias.PKG + ".synthetic")
    if not torch.cuda.is_available():
        raise SystemExit("bench_ragged.py measures the B200: no CUDA device here")
    ab = bench_ab(args.parent_tree, args.ab_reps) if args.parent_tree else None     # before this process holds the GPU

    sizes = frame_sizes(args.frames, args.seed)
    rs = np.random.RandomState(args.seed + 1)
    frames = [rs.randint(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
    # noise frames up to 368 x 1104 (46 x 138 maps): about 1 300 peaks per part, hence the largest peak capacity
    pe = engine.PoseEngine(syn.he_state_arrays(1234), 0, mode=args.mode, batch_cap=args.batch_cap, peak_cap=2048,
                           human_cap=2048)

    # shapes: buckets of the default path, runs of the ragged one, canvas fill
    pads = [nat.crop_geometry(h, w, args.dest_size, 8)[2] for h, w in sizes]
    buckets = {}
    for i, s in enumerate(sizes):
        buckets.setdefault(s, []).append(i)
    n_bucket_runs = sum((len(v) + args.batch_cap - 1) // args.batch_cap for v in buckets.values())
    runs = engine.ragged_groups(pads, args.batch_cap)
    useful = sum(ph * pw for ph, pw in pads)
    computed = sum(len(part) * ch * cw for part, (ch, cw) in runs)

    # warm-up of every shape of both paths; identical person rows
    a = pe.infer_images_arrays(frames, args.dest_size)
    b = pe.infer_images_arrays(frames, args.dest_size, ragged=True)
    for i, (x, y) in enumerate(zip(a, b)):
        if not np.array_equal(x, y):
            raise SystemExit("frame %d: ragged person rows differ from the bucketed path" % i)
    persons = int(sum(len(x) for x in a))

    times = {"bucketed": [], "ragged": []}
    for _ in range(args.reps):
        for name, ragged in (("bucketed", False), ("ragged", True)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = pe.infer_images_arrays(frames, args.dest_size, ragged=ragged)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
            if any(not np.array_equal(x, y) for x, y in zip(res, a)):
                raise SystemExit("%s pass: person rows changed between passes" % name)
    fps = {k: [round(args.frames / t, 1) for t in v] for k, v in times.items()}
    med = {k: statistics.median(v) for k, v in fps.items()}
    out = {
        "metric": "frames/s of PoseEngine.infer_images_arrays over %d mixed-size frames (host frames -> person rows)"
                  % args.frames,
        "gpu": gpu_info(),
        "mode": args.mode, "batch_cap": args.batch_cap, "dest_size": args.dest_size, "seed": args.seed,
        "frames_per_s": {"bucketed": med["bucketed"], "ragged": med["ragged"],
                         "speedup": round(med["ragged"] / med["bucketed"], 3)},
        "frames_per_s_each_rep": fps,
        "identical_person_rows": True, "persons": persons,
        "distinct_raw_shapes": len(buckets), "bucketed_runs": n_bucket_runs,
        "bucketed_mean_batch": round(args.frames / n_bucket_runs, 2),
        "ragged_runs": len(runs), "ragged_mean_batch": round(args.frames / len(runs), 2),
        "canvas_fill": round(useful / computed, 4),
        "useful_megapixels": round(useful / 1e6, 3), "computed_megapixels": round(computed / 1e6, 3),
        "bench_py_ab": ab if ab is not None else "not run (no --parent-tree)",
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
