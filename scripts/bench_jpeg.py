"""Detection on JPEG files, end to end: the routes from a list of JPEG files to boxes, on the default model in bf16 at batch
64, one JSON line on stdout.

The files are 64-per-batch seeded, photo-like synthetic images in bench_images.py's mix of COCO sizes, encoded by PIL at
quality 75-95, mostly 4:2:0 with some 4:4:4 and greyscale.  The decode time follows the compressed size, and synthetic
content compresses differently from photographs, so the mean bytes per file is reported with the results.  Routes:
  pil_*_submit_images   PIL decode (Image.open + convert("RGB") + np.asarray) with one thread, a thread pool and a process
                        pool over all host cores, each followed by submit_images with two batches in flight
  detect_jpeg_sync      detect_jpeg, one synchronous call per batch
  submit_jpeg_*         submit_jpeg / collect with two batches in flight, from pageable bytes and from page-locked arrays
  device_detect_images  detect_images on the same images already decoded into CUDA uint8 tensors: the upper bound
  decode_stage_*        decode_jpeg of one batch: CUDA events around the call (its H2D copy of the files included), and the
                        device time of the jpeg_* kernels alone from torch.profiler, in ms per batch
  repair                subsequences of the parallel Huffman decode per batch, and how many of them and how many symbols
                        the sync passes and the repair re-decoded
Every timing is warmed up and ends in a device synchronise.

    python scripts/bench_jpeg.py [--steps 20] [--warmup 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import io
import json
import os
import sys
import time
from collections import deque
from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_images import SIZES, card  # noqa: E402


def photo(h, w, rng):
    """Smooth colour fields, a few edges and sensor-like noise."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    f = rng.uniform(0.005, 0.05, (3, 2))
    img = np.stack([128 + 80 * np.sin(xx * f[c, 0] + c) * np.cos(yy * f[c, 1] + 2 * c) for c in range(3)], -1)
    for _ in range(6):
        y0, x0 = rng.integers(0, h), rng.integers(0, w)
        img[y0:y0 + h // 4, x0:x0 + w // 4] += rng.uniform(-60, 60, 3).astype(np.float32)
    return np.clip(img + rng.normal(0, 6, img.shape), 0, 255).astype(np.uint8)


def encode(img, rng) -> bytes:
    from PIL import Image
    b = io.BytesIO()
    kind = rng.choice(["420"] * 6 + ["444", "grey"])
    q = int(rng.integers(75, 96))
    if kind == "grey":
        Image.fromarray(img).convert("L").save(b, "JPEG", quality=q)
    else:
        Image.fromarray(img).save(b, "JPEG", quality=q, subsampling=0 if kind == "444" else 2)
    return b.getvalue()


def pil_decode(data: bytes) -> np.ndarray:
    from PIL import Image
    with Image.open(io.BytesIO(data)) as im:
        return np.asarray(im.convert("RGB"))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pil-steps", type=int, default=4, help="steps of the PIL routes (slow)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    import vision_transformer_detector_b200 as vd
    from vision_transformer_detector_b200 import _capi
    from vision_transformer_detector_b200 import vision_transformer_utilities as vu
    if not torch.cuda.is_available():
        raise SystemExit("bench_jpeg.py needs a CUDA device")
    B, K, W = args.batch, args.steps, args.warmup
    rng = np.random.default_rng(args.seed)
    sizes = [SIZES[i] for i in rng.integers(0, len(SIZES), 2 * B)]
    files = [encode(photo(h, w, rng), rng) for h, w in sizes]
    batches = [files[:B], files[B:]]
    m = vd.create_vision_transformer_detector(seed=0, compute_mode="bf16")

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

    def pipelined(submit, lists, steps):
        """images/s of `submit(list) -> ticket` with two tickets in flight"""
        def run(n):
            q = deque()
            for i in range(n):
                if len(q) == 2:
                    m.collect(q.popleft())
                q.append(submit(lists[i % 2]))
            while q:
                m.collect(q.popleft())
        run(2 * W)
        torch.cuda.synchronize()
        t = time.perf_counter()
        run(steps)
        torch.cuda.synchronize()
        return B * steps / (time.perf_counter() - t)

    res = {"metric": "images_per_s", "batch": B, "mode": "bf16", "config": "default", "sizes": [list(s) for s in SIZES],
           "steps": K, "warmup": W, "mean_bytes_per_file": float(np.mean([len(f) for f in files])),
           "corpus": "synthetic photo-like images, PIL-encoded at q75-95, 6/8 4:2:0, 1/8 4:4:4, 1/8 greyscale"}
    # the decoded images of both batches: the GPU decode gives PIL's pixels, and the records agree
    decoded = [[pil_decode(f) for f in b] for b in batches]
    gpu = vu.decode_jpeg(batches[0])
    res["decode_equals_pil"] = bool(all(np.array_equal(g.cpu().numpy(), d) for g, d in zip(gpu, decoded[0])))
    a, b = m.detect_jpeg(batches[0]), m.detect_images(decoded[0])
    res["records_identical"] = bool(all(np.array_equal(getattr(a, f), getattr(b, f)) for f in
                                        ("logits", "decoded", "class_id", "class_conf", "keep", "corners", "boxes_original")))
    # 1. PIL decode on the host, then submit_images, two batches in flight
    cores = os.cpu_count() or 1
    res["host_cores"] = cores
    with ThreadPoolExecutor(cores) as tp, ProcessPoolExecutor(cores) as pp:
        for name, dec in (("pil_1thread", lambda fs: [pil_decode(f) for f in fs]),
                          ("pil_threads", lambda fs: list(tp.map(pil_decode, fs))),
                          ("pil_processes", lambda fs: list(pp.map(pil_decode, fs, chunksize=max(1, len(fs) // cores))))):
            res[f"{name}_submit_images"] = pipelined(lambda fs: m.submit_images(dec(fs)), batches, args.pil_steps)
    # 2. detect_jpeg, one synchronous call per batch
    res["detect_jpeg_sync"] = B / timed(lambda: m.detect_jpeg(next_batch()), K)
    # 3. submit_jpeg, two batches in flight
    res["submit_jpeg_pageable"] = pipelined(m.submit_jpeg, batches, K)
    pinned = [[torch.frombuffer(bytearray(f), dtype=torch.uint8).pin_memory().numpy() for f in b] for b in batches]
    res["submit_jpeg_pinned"] = pipelined(m.submit_jpeg, pinned, K)
    # 4. device-resident detect_images on the same decoded images
    dev_lists = [[torch.from_numpy(im).cuda() for im in b] for b in decoded]
    def device_step():
        m.detect_images(dev_lists[step[0] % 2])
        next_batch()
    res["device_detect_images"] = B / timed(device_step, K)
    res["submit_jpeg_pinned_over_device"] = res["submit_jpeg_pinned"] / res["device_detect_images"]
    res["submit_jpeg_pageable_over_device"] = res["submit_jpeg_pageable"] / res["device_detect_images"]
    # 5. the decode stage alone
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(W):
        vu.decode_jpeg(batches[0])
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(K):
        vu.decode_jpeg(batches[0])
    ev[1].record()
    torch.cuda.synchronize()
    res["decode_stage_ms_per_batch_events_with_h2d"] = ev[0].elapsed_time(ev[1]) / K
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(K):
            vu.decode_jpeg(batches[0])
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        if "jpeg_" in e.key and "kernel" in e.key:
            t = getattr(e, "device_time_total", None)
            t = e.cuda_time_total if t is None else t
            kernels[e.key.split("jpeg_")[1].split("(")[0]] = t / 1e3 / K
    res["decode_stage_kernel_ms_per_batch"] = kernels
    res["decode_stage_kernel_ms_per_batch_total"] = sum(kernels.values())
    stats = np.zeros(3, np.int64)
    _capi.check(_capi.load().vitdet_jpeg_stats(vu._decoder(torch.cuda.current_device()), C.c_void_p(stats.ctypes.data)))
    res["repair"] = {"subsequences": int(stats[0]), "redecoded_subsequences": int(stats[1]), "redecoded_symbols": int(stats[2])}
    res["card"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    m.close()


if __name__ == "__main__":
    main()
