"""Detection on decoded images of any size, end to end: the routes from a list of uint8 (h, w, 3) images to boxes, on the
default model in bf16 at batch 64, one JSON line on stdout.

The images are a seeded mix of COCO-like sizes, so the letterbox does real resizing on every image.  Routes:
  today          per-image preprocess_image (numpy in, float32 608 x 608 out), np.stack, detect (host float32 batch)
  images_sync    detect_images on numpy lists, one synchronous call per batch
  images_submit  submit_images / collect with two batches in flight, from pageable and from page-locked lists
  device         detect_images on lists of CUDA uint8 tensors against detect on the same images already letterboxed into a
                 float32 CUDA batch, alternated round by round in the same process; plus the "patchify" category time per
                 step of both (CUDA events around the patch kernel, in a separate profiled pass)
Every timing is warmed up and ends in a device synchronise.  The device-resident sources (64 images of 0.4-1.2 MB of uint8)
fit the 126 MB L2, as a batch the caller has just decoded and copied there would.

    python scripts/bench_images.py [--steps 20] [--warmup 3] [--rounds 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from collections import deque

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [(640, 480), (480, 640), (427, 640), (640, 427), (500, 375), (612, 612), (640, 640), (333, 500)]   # (height, width)


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power}
    except Exception as e:         # the measurement is still valid; say what is missing
        return {"name": None, "power_limit": None, "error": str(e)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5, help="alternated rounds of the device-resident comparison")
    ap.add_argument("--today-steps", type=int, default=3, help="steps of the per-image preprocess route (slow)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    import vision_transformer_detector_b200 as vd
    if not torch.cuda.is_available():
        raise SystemExit("bench_images.py needs a CUDA device")
    B, K, W = args.batch, args.steps, args.warmup
    rng = np.random.default_rng(args.seed)
    sizes = [SIZES[i] for i in rng.integers(0, len(SIZES), 2 * B)]
    batches = [[rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for h, w in sizes[i * B:(i + 1) * B]] for i in range(2)]
    m = vd.create_vision_transformer_detector(seed=0, compute_mode="bf16")
    target = m.config.input_shape[:2]

    def timed(fn, steps, warmup=W) -> float:
        """seconds per call"""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) / steps

    step = [0]

    def next_batch():
        step[0] += 1
        return batches[step[0] % 2]

    res = {"metric": "images_per_s", "batch": B, "mode": "bf16", "config": "default", "sizes": [list(s) for s in SIZES],
           "steps": K, "warmup": W}
    # 1. today's route
    today = timed(lambda: m.detect(np.stack([vd.preprocess_image(im, target) for im in next_batch()])), args.today_steps, 1)
    res["today_preprocess_stack_detect"] = B / today
    # 2. one synchronous detect_images per batch
    res["detect_images_numpy_sync"] = B / timed(lambda: m.detect_images(next_batch()), K)
    # 3. two submissions in flight

    def pipelined(lists, steps):
        def run(n):
            q = deque()
            for i in range(n):
                if len(q) == 2:
                    m.collect(q.popleft())
                q.append(m.submit_images(lists[i % 2]))
            while q:
                m.collect(q.popleft())
        run(2 * W)
        torch.cuda.synchronize()
        t = time.perf_counter()
        run(steps)
        torch.cuda.synchronize()
        return B * steps / (time.perf_counter() - t)

    res["submit_images_pageable"] = pipelined(batches, K)
    pinned = [[torch.from_numpy(im).pin_memory().numpy() for im in b] for b in batches]
    res["submit_images_pinned"] = pipelined(pinned, K)
    # 4. device resident: CUDA uint8 lists against detect on the same images letterboxed into a float32 batch
    dev_lists = [[torch.from_numpy(im).cuda() for im in b] for b in batches]
    dev_f32 = [torch.stack([vd.preprocess_image(t, target) for t in b]) for b in dev_lists]
    # the two routes compute the same records
    a, b = m.detect_images(dev_lists[0]), m.detect(dev_f32[0])
    res["device_records_identical"] = bool(all(torch.equal(getattr(a, f), getattr(b, f))
                                                for f in ("logits", "decoded", "class_id", "class_conf", "keep", "corners")))

    def alternate(fn, inputs):
        def call():
            fn(inputs[step[0] % 2])
            next_batch()
        return call

    rounds = {"detect_images_cuda_list": [], "detect_letterboxed_f32": []}
    for _ in range(args.rounds):
        rounds["detect_images_cuda_list"].append(B / timed(alternate(m.detect_images, dev_lists), K))
        rounds["detect_letterboxed_f32"].append(B / timed(alternate(m.detect, dev_f32), K))
    for k, v in rounds.items():
        res[k] = statistics.median(v)
        res[k + "_rounds"] = v
    res["pipelined_pinned_over_device_detect"] = res["submit_images_pinned"] / res["detect_letterboxed_f32"]
    # 5. patch-stage device time per step of both sides of 4 (profiled pass of its own)
    m.profile_enable(["patchify"])
    for name, fn in (("detect_images_cuda_list", lambda: m.detect_images(dev_lists[0])),
                     ("detect_letterboxed_f32", lambda: m.detect(dev_f32[0]))):
        for _ in range(W):
            fn()
        torch.cuda.synchronize()
        m.profile_read(reset=True)
        timed(fn, K, 0)
        ms, n = m.profile_read(reset=True).get("patchify", (0.0, 0))
        res[f"patchify_ms_per_step_{name}"] = ms / K
        res[f"patchify_launches_per_step_{name}"] = n / K
    m.profile_enable(None)
    res["card"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    m.close()


if __name__ == "__main__":
    main()
