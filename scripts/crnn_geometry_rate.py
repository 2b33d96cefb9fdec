"""Recognizer throughput at several crop geometries (build_params height / width / rnn_steps_to_discard).

    python scripts/crnn_geometry_rate.py [--crops 1024] [--reps 5] [--rounds 2] [--out profiles/crnn_geometry_rate.json]

For each geometry -- the default 31 x 200 and the three of tests/golden/crnn_geometry.npz (A: 31 x 400; B: 35 x 250, 3
steps discarded; C: 48 x 128, none discarded, no spatial transformer, RGB) -- a Recognizer with seeded synthetic weights
reads ``--crops`` seeded noise crops (CRNN input prepared once, so only ``b2o_crnn_forward`` is timed):

* crops/s from CUDA events around ``--reps`` forward passes after two warm-up passes, in ``--rounds`` rounds that
  alternate the geometries (the spread between rounds is the run-to-run noise);
* the tensor-core conv kernel's time and algorithmic FLOPs over one pass (``b2o_profile_enable`` / ``b2o_profile_read``)
  and the whole CRNN's algorithmic FLOPs per crop, computed below from the layer shapes (13.444 GFLOP at 31 x 200,
  SURVEY.md C.2);
* per-kernel device times of one pass from ``torch.profiler`` (a separate, traced pass);
* the GPU's name and power limit, read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from keras_ocr_b200 import weights as W  # noqa: E402
from keras_ocr_b200.recognition import Recognizer  # noqa: E402

# tag: (height, width, rnn_steps_to_discard, stn, color)
GEOMETRIES = {"default": (31, 200, 2, True, False), "A": (31, 400, 2, True, False),
              "B": (35, 250, 3, True, False), "C": (48, 128, 0, False, True)}


def crnn_flop_per_crop(height, width, stn=True, color=False, classes=37):
    """Algorithmic FLOPs (2 x MAC) of one crop through build_model (recognition.py:214-329), from the layer shapes."""
    w0, h0, w1, h1, t, hf = width, height, width // 2, height // 2, width // 4, height // 4
    mac = w0 * h0 * 9 * (3 if color else 1) * 64                    # conv_1
    mac += w0 * h0 * 9 * 64 * 128 + w0 * h0 * 9 * 128 * 256           # conv_2, conv_3 (-> pool)
    mac += w1 * h1 * 9 * 256 * 256 + w1 * h1 * 9 * 256 * 512          # conv_4, conv_5 (-> pool)
    mac += 2 * t * hf * 9 * 512 * 512                                 # conv_6, conv_7
    if stn:                                                           # localisation net + bilinear sampler
        mac += t * hf * 25 * 512 * 16 + t * hf * 25 * 16 * 32 + t * hf * 32 * 64 + 64 * 6 + t * hf * 512 * 4
    mac += t * hf * 512 * 128                                         # fc_9
    mac += 4 * t * 2 * 128 * 512                                      # 4 LSTMs: input + recurrent products
    mac += t * 256 * classes                                          # fc_12
    return 2 * mac


def gpu_identity():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        name, limit, clock = (x.strip() for x in r.stdout.strip().split(","))
        out.update({"smi_name": name, "power_limit_w": float(limit), "max_sm_clock_mhz": float(clock)})
    except Exception as e:                                            # noqa: BLE001 - reported, not hidden
        out["power_limit_w"] = None
        out["smi_error"] = repr(e)
    return out


def setup(tag, n_crops):
    h, w, d, stn, color = GEOMETRIES[tag]
    rec = Recognizer(weights=W.synthetic_crnn_weights(seed=2, stn=stn, color=color, height=h, width=w),
                     build_params={"height": h, "width": w, "rnn_steps_to_discard": d, "stn": stn, "color": color})
    tail = (3,) if color else ()
    crops = torch.from_numpy(np.random.default_rng(1).integers(0, 256, (n_crops, h, w) + tail, dtype=np.uint8)).to(rec.device)
    x = torch.empty((n_crops, w, h) + tail, dtype=torch.float16, device=rec.device)
    rec.ctx.crops_to_input(crops.data_ptr(), n_crops, x.data_ptr(), torch.cuda.current_stream().cuda_stream, color=color)
    for _ in range(2):                                                # warm-up: modules, workspace, launch attributes
        rec.predict_device(x)
    torch.cuda.synchronize()
    return rec, x


def time_passes(rec, x, reps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        rec.predict_device(x)
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / reps


def tc_profile(rec, x):
    rec.ctx.profile_enable(1)
    rec.predict_device(x)
    torch.cuda.synchronize()
    ms, flop, launches = rec.ctx.profile_read()
    rec.ctx.profile_enable(0)
    return {"tc_ms": ms, "tc_flop": flop, "tc_launches": launches, "tc_tflops": flop / ms / 1e9 if ms > 0 else None}


def kernel_times(rec, x, top=12):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rec.predict_device(x)
        torch.cuda.synchronize()
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            rows.append({"kernel": ev.key[:120], "calls": ev.count, "ms": t / 1e3})
    rows.sort(key=lambda r: -r["ms"])
    return rows[:top]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--crops", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "crnn_geometry_rate.json"))
    args = ap.parse_args()
    assert round(crnn_flop_per_crop(31, 200) / 1e9, 3) == 13.444, crnn_flop_per_crop(31, 200)   # SURVEY.md C.2
    assert torch.cuda.is_available(), "crnn_geometry_rate.py measures on the GPU"
    result = {"gpu": gpu_identity(), "crops": args.crops, "reps": args.reps, "geometries": {}}
    state = {tag: setup(tag, args.crops) for tag in GEOMETRIES}
    rounds = {tag: [] for tag in GEOMETRIES}
    for _ in range(args.rounds):                                      # geometries alternate within every round
        for tag, (rec, x) in state.items():
            rounds[tag].append(time_passes(rec, x, args.reps))
    for tag, (rec, x) in state.items():
        h, w, d, stn, color = GEOMETRIES[tag]
        flop = crnn_flop_per_crop(h, w, stn, color)
        ms = min(rounds[tag])
        result["geometries"][tag] = {
            "height": h, "width": w, "rnn_steps_to_discard": d, "stn": stn, "color": color,
            "time_steps": w // 4, "label_steps": w // 4 - d, "gflop_per_crop": flop / 1e9,
            "ms_per_pass": rounds[tag], "crops_per_s": args.crops / (ms / 1e3),
            "crnn_tflops_algorithmic": flop * args.crops / (ms / 1e3) / 1e12,
            **tc_profile(rec, x),
        }
    for tag, (rec, x) in state.items():                               # traced passes last: the profiler slows the host
        result["geometries"][tag]["kernels"] = kernel_times(rec, x)
    base = result["geometries"]["default"]["crops_per_s"]
    for tag, g in result["geometries"].items():
        g["rate_vs_default"] = g["crops_per_s"] / base
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    for tag, g in result["geometries"].items():
        print(f"{tag:8s} {g['height']}x{g['width']}: {g['crops_per_s']:9.0f} crops/s ({g['rate_vs_default']:.2f}x default), "
              f"{g['gflop_per_crop']:.3f} GFLOP/crop, tensor-core conv {g['tc_tflops']:.0f} TFLOP/s, "
              f"passes {['%.2f' % t for t in g['ms_per_pass']]} ms")
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
