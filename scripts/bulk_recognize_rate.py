"""Bulk recognition of pre-cropped word images: Recognizer.recognize_batch against the ways there were before it.

    python scripts/bulk_recognize_rate.py [--crops 4096] [--loop-crops 512] [--rounds 2] [--out profiles/bulk_recognize_rate.json]

``--crops`` seeded word-like crops (a random word rendered with cv2.putText, dark on light, resized to a seeded size:
heights 12..120, widths 20..900, some exactly 31 x 200), read by a default 31 x 200 Recognizer (seeded synthetic
weights) in four ways:

* ``loop``: ``[rec.recognize(c) for c in crops]`` on the first ``--loop-crops`` crops (one crop per call);
* ``host_fit``: tools.fit + cv2.cvtColor on the host, then ``recognize_crops`` on the stacked crops, 1024 at a time;
* ``batch_host``: ``recognize_batch`` of the host arrays (pinned staging, one upload per chunk);
* ``batch_device``: ``recognize_batch`` of the crops already on the GPU as CUDA tensors.

Each is warmed up once, then timed with a host clock in ``--rounds`` rounds that alternate the four (every call ends
with the strings on the host, i.e. after a device synchronise).  The script also records the host-to-device bytes of
each way, computed from the shapes; the time of ``fit_crops_kernel`` (CUDA events around ``--reps`` launches over one
1024-crop chunk of device sources) with the bytes it reads and writes, next to ``b2o_crnn_forward`` over the same
chunk; and the GPU's name and power limit, read in the same process.  All four ways must return the same strings.
"""
import argparse
import json
import os
import string
import sys
import time

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from crnn_geometry_rate import gpu_identity  # noqa: E402
from keras_ocr_b200 import tools, weights as W  # noqa: E402
from keras_ocr_b200.recognition import Recognizer  # noqa: E402

CHUNK = 1024


def word_crops(seed, n, exact_fraction=0.05):
    rng = np.random.default_rng(seed)
    alphabet = string.digits + string.ascii_lowercase
    crops = []
    for _ in range(n):
        word = "".join(rng.choice(list(alphabet), int(rng.integers(3, 11))))
        (tw, th), base = cv2.getTextSize(word, cv2.FONT_HERSHEY_SIMPLEX, 1.0, 2)
        canvas = np.full((th + base + 8, tw + 8, 3), int(rng.integers(180, 256)), np.uint8)
        colour = tuple(int(c) for c in rng.integers(0, 90, 3))
        cv2.putText(canvas, word, (4, th + 4), cv2.FONT_HERSHEY_SIMPLEX, 1.0, colour, 2, cv2.LINE_AA)
        if rng.random() < exact_fraction:
            h, w = 31, 200
        else:
            h = int(np.exp(rng.uniform(np.log(12), np.log(121))))
            w = int(np.clip(h * canvas.shape[1] / canvas.shape[0] * rng.uniform(0.5, 2.0), 20, 900))
        crops.append(np.ascontiguousarray(cv2.resize(canvas, (w, h), interpolation=cv2.INTER_AREA)))
    return crops


def fit_kind(crop, height=31, width=200):
    plan = tools.fit_plan(crop.shape, width, height)
    if plan is None:
        return "exact"
    return "downscaled" if plan[0] < crop.shape[0] or plan[1] < crop.shape[1] else "upscaled"


def run_loop(rec, crops):
    return [rec.recognize(c) for c in crops]


def run_host_fit(rec, crops):
    out = []
    for s in range(0, len(crops), CHUNK):
        fitted = [cv2.cvtColor(tools.fit(c, rec.width, rec.height, cval=0), cv2.COLOR_RGB2GRAY) for c in crops[s:s + CHUNK]]
        out += rec.recognize_crops(np.stack(fitted))
    return out


def h2d_bytes(rec, crops):
    """Host-to-device bytes of each way, from the shapes."""
    n, crop = len(crops), rec.height * rec.width
    chunks = [crops[s:s + CHUNK] for s in range(0, len(crops), CHUNK)]
    table = sum((len(c) * 24 + 15) // 16 * 16 for c in chunks)
    return {"loop": n * crop, "host_fit": n * crop, "batch_host": table + sum(c.size for c in crops),
            "batch_device": table, "batch_device_sources_uploaded_beforehand": sum(c.size for c in crops)}


def fit_kernel_time(rec, device_crops, reps):
    """fit_crops_kernel alone over one chunk of device sources (pointer table built once), and the CRNN over it."""
    srcs = device_crops[:CHUNK]
    b = len(srcs)
    table = np.zeros(b * 24, np.uint8)
    table[: b * 8].view(np.uint64)[:] = [t.data_ptr() for t in srcs]
    dims = np.array([rec._fit_dims(t.shape) for t in srcs], np.int32)
    table[b * 8:].view(np.int32)[:] = dims.reshape(-1)
    table_dev = torch.from_numpy(table).to(rec.device)
    ptrs, dims_dev = table_dev.data_ptr(), table_dev.data_ptr() + b * 8
    crnn_in, _ = rec._fit_table(ptrs, dims_dev, b, False)
    rec.predict_device(crnn_in)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        rec._fit_table(ptrs, dims_dev, b, False)
    stop.record()
    stop.synchronize()
    fit_ms = start.elapsed_time(stop) / reps
    start.record()
    for _ in range(3):
        rec.predict_device(crnn_in)
    stop.record()
    stop.synchronize()
    crnn_ms = start.elapsed_time(stop) / 3
    src_bytes = int(sum(t.numel() for t in srcs))
    written = b * rec.height * rec.width * 2
    read = src_bytes + b * 24
    return {"crops": b, "reps": reps, "fit_ms": fit_ms, "fit_us_per_crop": fit_ms * 1e3 / b,
            "bytes_read_sources_and_table": read, "bytes_written_crnn_in": written,
            "gb_per_s": (read + written) / (fit_ms / 1e3) / 1e9,
            "note_bytes": "sources counted once in full; a downscale reads only the rows and columns it samples",
            "crnn_forward_ms": crnn_ms, "fit_share_of_fit_plus_crnn": fit_ms / (fit_ms + crnn_ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--crops", type=int, default=4096)
    ap.add_argument("--loop-crops", type=int, default=512)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bulk_recognize_rate.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bulk_recognize_rate.py measures on the GPU"
    result = {"gpu": gpu_identity(), "crops": args.crops, "loop_crops": args.loop_crops, "chunk": CHUNK}
    crops = word_crops(7, args.crops)
    hs, ws = np.array([c.shape[0] for c in crops]), np.array([c.shape[1] for c in crops])
    result["crop_sizes"] = {"height_min": int(hs.min()), "height_max": int(hs.max()), "width_min": int(ws.min()),
                            "width_max": int(ws.max()), "exact_31x200": int(((hs == 31) & (ws == 200)).sum()),
                            **{k: sum(fit_kind(c) == k for c in crops) for k in ("upscaled", "downscaled")}}
    rec = Recognizer(weights=W.synthetic_crnn_weights(seed=2))
    device = [torch.from_numpy(c).to(rec.device) for c in crops]
    torch.cuda.synchronize()
    ways = {"loop": lambda: run_loop(rec, crops[: args.loop_crops]),
            "host_fit": lambda: run_host_fit(rec, crops),
            "batch_host": lambda: rec.recognize_batch(crops),
            "batch_device": lambda: rec.recognize_batch(device)}
    texts = {name: fn() for name, fn in ways.items()}              # warm-up: modules, workspace, pinned buffers
    assert texts["host_fit"] == texts["batch_host"] == texts["batch_device"]
    assert texts["loop"] == texts["batch_host"][: args.loop_crops]
    seconds = {name: [] for name in ways}
    for _ in range(args.rounds):                                     # the four ways alternate within every round
        for name, fn in ways.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            seconds[name].append(time.perf_counter() - t0)
    result["ways"] = {}
    for name in ways:
        n = args.loop_crops if name == "loop" else args.crops
        result["ways"][name] = {"crops": n, "seconds": seconds[name], "crops_per_s": n / min(seconds[name])}
    base = result["ways"]["loop"]["crops_per_s"]
    for w in result["ways"].values():
        w["rate_vs_loop"] = w["crops_per_s"] / base
    result["h2d_bytes"] = h2d_bytes(rec, crops)
    result["fit_crops_kernel"] = fit_kernel_time(rec, device, args.reps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    for name, w in result["ways"].items():
        print(f"{name:13s} {w['crops_per_s']:10.0f} crops/s ({w['rate_vs_loop']:.1f}x loop), "
              f"runs {['%.3f' % s for s in w['seconds']]} s, H2D {result['h2d_bytes'][name] / 1e6:.1f} MB")
    k = result["fit_crops_kernel"]
    print(f"fit_crops_kernel: {k['fit_ms']:.3f} ms / {k['crops']} crops ({k['fit_us_per_crop']:.2f} us/crop, "
          f"{k['gb_per_s']:.0f} GB/s); CRNN {k['crnn_forward_ms']:.2f} ms; fit share {k['fit_share_of_fit_plus_crnn']:.1%}")
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
