"""Detection on camera-size JPEG files: the decode at full size against the decode at the scale PIL's draft() picks for the
letterbox (detect_jpeg / submit_jpeg(ratio="auto")), on the default model in bf16 at batch 64, one JSON line on stdout.

The files are seeded, photo-like synthetic images of about 12 MP (4032 x 3024 and 3024 x 4032, 4000 x 3000, 4608 x 2592),
encoded by PIL at quality 85-95, 6/8 of them 4:2:0, 1/8 4:2:2 and 1/8 greyscale.  Synthetic content compresses differently
from photographs, so the mean bytes per file is reported with the results.  Routes:
  submit_jpeg_ratio1 / _auto     submit_jpeg / collect with two batches in flight, pageable bytes, at ratio 1 and "auto"
  pil_draft_threads_submit_images  a 16-thread PIL pool decoding with draft("RGB", letterbox size), then submit_images
                                 with two batches in flight
  decode_stage_kernel_ms_*       device time of the jpeg_* kernels of decode_jpeg on one batch, by kernel, from
                                 torch.profiler, in ms per batch, at ratio 1 and at the auto ratios
  decode_buffer_bytes_*          the device bytes of one batch's decode: coefficients, component planes and RGB images
                                 (what jpeg_plan sizes; the compact bit streams and subsequence states do not depend on
                                 the ratio and are left out)
Every timing is warmed up and ends in a device synchronise.

    python scripts/bench_jpeg_large.py [--steps 6] [--warmup 2] [--out FILE]
"""
from __future__ import annotations

import argparse
import io
import json
import os
import sys
import time
from collections import deque
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from bench_images import card  # noqa: E402
from bench_jpeg import photo  # noqa: E402

SIZES = [(3024, 4032), (4032, 3024), (3000, 4000), (2592, 4608)]        # (height, width), about 12 MP


def make_files(B: int, bases, rng) -> list:
    """B files from the base images, each flipped, sampled and quantised on its own."""
    from PIL import Image
    out = []
    for i in range(B):
        img = bases[i % len(bases)]
        if rng.random() < 0.5:
            img = img[:, ::-1]
        if rng.random() < 0.5:
            img = img[::-1]
        kind = rng.choice(["420"] * 6 + ["422", "grey"])
        q = int(rng.integers(85, 96))
        b = io.BytesIO()
        if kind == "grey":
            Image.fromarray(np.ascontiguousarray(img)).convert("L").save(b, "JPEG", quality=q)
        else:
            Image.fromarray(np.ascontiguousarray(img)).save(b, "JPEG", quality=q, subsampling=2 if kind == "420" else 1)
        out.append(b.getvalue())
    return out


def decode_buffer_bytes(files, ratios) -> int:
    """Coefficient, plane and RGB bytes of one batch's decode, as jpeg_plan sizes them."""
    import jpeg_oracle as jo
    import jpeg_scaled_oracle as js
    a256 = lambda v: (v + 255) // 256 * 256                                  # noqa: E731
    total = 0
    for d, r in zip(files, ratios):
        j = jo.parse(d)
        g = js.scaled_geometry(j, r)
        nmcu = j["mcux"] * j["mcuy"]
        mcu_coefs, full = 0, False
        for c, _, _ in j["blocks"]:
            dc_only = g["comps"][c]["size"] == 1
            if not dc_only:
                mcu_coefs = (mcu_coefs + 7) // 8 * 8
            mcu_coefs += 1 if dc_only else 64
            full |= not dc_only
        if full:
            mcu_coefs = (mcu_coefs + 7) // 8 * 8
        total += 2 * ((nmcu * mcu_coefs + 7) // 8 * 8)
        total += sum(a256(nmcu * j["hs"][c] * j["vs"][c] * g["comps"][c]["size"] ** 2) for c in range(j["ncomp"]))
        total += a256(g["height"] * g["width"] * 3)
    return total


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    from PIL import Image
    import vision_transformer_detector_b200 as vd
    from vision_transformer_detector_b200 import vision_transformer_utilities as vu
    if not torch.cuda.is_available():
        raise SystemExit("bench_jpeg_large.py needs a CUDA device")
    B, K, W = args.batch, args.steps, args.warmup
    rng = np.random.default_rng(args.seed)
    bases = [photo(*SIZES[i % len(SIZES)], rng) for i in range(8)]
    batches = [make_files(B, bases, rng), make_files(B, bases, rng)]
    m = vd.create_vision_transformer_detector(seed=0, compute_mode="bf16")
    th, tw = m.config.input_shape[:2]

    def size(d):
        with Image.open(io.BytesIO(d)) as im:
            return im.height, im.width

    auto = [[vu.jpeg_auto_ratio(*size(d)) for d in b] for b in batches]

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

    def pil_draft(d):
        im = Image.open(io.BytesIO(d))
        rh, rw, _, _ = vu.resize_with_pad_geometry(im.height, im.width, th, tw)
        im.draft("RGB", (rw, rh))
        return np.asarray(im.convert("RGB"))

    res = {"metric": "images_per_s", "batch": B, "mode": "bf16", "config": "default", "sizes": [list(s) for s in SIZES],
           "steps": K, "warmup": W, "mean_bytes_per_file": float(np.mean([len(f) for b in batches for f in b])),
           "auto_ratios": {str(r): sum(a.count(r) for a in auto) for r in (1, 2, 4, 8)},
           "corpus": "synthetic photo-like images of about 12 MP, PIL-encoded at q85-95, 6/8 4:2:0, 1/8 4:2:2, 1/8 greyscale"}
    # the auto decode is PIL's draft decode, and detect_jpeg(ratio="auto") is detect_images on it
    draft = [pil_draft(d) for d in batches[0]]
    gpu = vu.decode_jpeg(batches[0], ratio=auto[0])
    res["auto_decode_equals_pil_draft"] = bool(all(np.array_equal(g.cpu().numpy(), d) for g, d in zip(gpu, draft)))
    a, b = m.detect_jpeg(batches[0], ratio="auto"), m.detect_images(draft)
    res["auto_records_identical"] = bool(all(np.array_equal(getattr(a, f), getattr(b, f)) for f in
                                             ("logits", "decoded", "class_id", "class_conf", "keep", "corners")))
    del gpu
    # 1. submit_jpeg with two batches in flight, at ratio 1 and at auto
    res["submit_jpeg_ratio1"] = pipelined(lambda fs: m.submit_jpeg(fs), batches, K)
    res["submit_jpeg_auto"] = pipelined(lambda fs: m.submit_jpeg(fs, ratio="auto"), batches, K)
    res["auto_over_ratio1"] = res["submit_jpeg_auto"] / res["submit_jpeg_ratio1"]
    # 2. a thread pool decoding with PIL's draft for the letterbox size, then submit_images
    with ThreadPoolExecutor(args.threads) as tp:
        res[f"pil_draft_{args.threads}threads_submit_images"] = pipelined(lambda fs: m.submit_images(list(tp.map(pil_draft, fs))),
                                                                         batches, K)
    # 3. the decode kernels by stage, and the decode buffers, at ratio 1 and auto
    from torch.profiler import ProfilerActivity, profile
    for name, ratio in (("ratio1", [1] * B), ("auto", auto[0])):
        for _ in range(W):
            vu.decode_jpeg(batches[0], ratio=ratio)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(K):
                vu.decode_jpeg(batches[0], ratio=ratio)
            torch.cuda.synchronize()
        kernels = {}
        for e in prof.key_averages():
            if "jpeg_" in e.key and "kernel" in e.key:
                t = getattr(e, "device_time_total", None)
                t = e.cuda_time_total if t is None else t
                kernels[e.key.split("jpeg_")[1].split("(")[0]] = t / 1e3 / K
        res[f"decode_stage_kernel_ms_per_batch_{name}"] = kernels
        res[f"decode_stage_kernel_ms_per_batch_{name}_total"] = sum(kernels.values())
        res[f"decode_buffer_bytes_{name}"] = decode_buffer_bytes(batches[0], ratio)
    res["card"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    m.close()


if __name__ == "__main__":
    main()
