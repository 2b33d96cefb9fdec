"""bench.py -- images/sec of end-to-end ``Pipeline.recognize`` (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W                # this repository (B200 kernels)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR   # also write the last timed step's results

One step = one ``recognize`` pass over a batch of 32 synthetic pages (768x768 RGB, 32 rendered
words each, ``Pipeline(scale=2)`` -> 32x1536x1536 detector input, BASELINE.json configs[3]); with
N GPUs every rank owns its own 32 pages (configs[4]: 256 pages over 8 GPUs, weak scaling) and the
per-image (count, boxes, labels) records -- written on the device -- are gathered to rank 0 over NCCL
once per step (``distributed.recognize_sharded``) and decoded there.

Timed region: K steps bracketed by barrier + cuda synchronize, CUDA events, max over ranks.
``value``  : sources resident in HBM when the step starts (resize/pad ... CTC decode + result D2H).
``e2e``    : the same through the public API with HOST numpy images: pinned H2D copy of the step's
             inputs and D2H of the results inside the timed region.
``roofline``: the dominant kernel (tcgen05 conv) -- algorithmic FLOPs of its launches in one step
             / their CUDA-event time, against the measured bf16 peak (MEASURED_PEAKS.json).
``cpu_baseline``: the oracle port of the reference path on the host cores, bounded sample.

``--dump-outputs DIR`` writes what the last timed step of ``value`` returned (``dump_outputs``).  Pages and weights are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

PAGES_PER_RANK = 32
PAGE_H = PAGE_W = 768
WORDS_PER_PAGE = 32
SCALE = 2
METRIC = "images/sec end-to-end Pipeline.recognize"
UNIT = "images/s"


def workload_config(n_gpus):
    return {
        "workload": "e2e_recognize_b32_768x768_scale2_to_1536x1536" if n_gpus == 1
        else f"e2e_recognize_b{PAGES_PER_RANK * n_gpus}_1536x1536_sharded_{n_gpus}gpu",
        "pages_per_gpu": PAGES_PER_RANK, "global_batch": PAGES_PER_RANK * n_gpus,
        "source": f"{PAGE_H}x{PAGE_W}x3 uint8, {WORDS_PER_PAGE} cv2.putText words/page",
        "detector_input": "1536x1536", "scale": SCALE, "parallelism": f"dp{n_gpus}",
        "weights": "no pretrained files offline: CRAFT seeded synthetic with textlike routing; CRNN = the reference architecture "
                   "trained on rendered Hershey-font words (oracle/train_crnn_full.py) -- the words found are the rendered words",
        "l2": "per-step activations (>40 GB) exceed the 126 MB L2; no explicit flush needed",
    }


def make_pages(rank, with_layout=False):
    from oracle import synth
    if not with_layout:
        images, _ = synth.text_images(seed=1000 + rank, n=PAGES_PER_RANK, h=PAGE_H, w=PAGE_W, n_words=WORDS_PER_PAGE)
        return images
    rng = np.random.default_rng(1000 + rank)                     # the same stream as text_images
    laid = [synth.text_image(rng, PAGE_H, PAGE_W, WORDS_PER_PAGE, return_layout=True) for _ in range(PAGES_PER_RANK)]
    return np.stack([p[0] for p in laid]), [p[1] for p in laid], [p[2] for p in laid]


def words_read(result, words, rects):
    """(rendered words found with the right text, rendered words): a (text, box) counts when the box centre lies in
    exactly one rendered word's glyph rectangle and the text equals that word.  Outside the timed region: a
    full-size sanity check of WHAT the benchmarked step produced, not only how fast."""
    hit = 0
    for group, page_words, page_rects in zip(result, words, rects):
        found = set()
        for text, box in group:
            c = np.asarray(box).mean(0)
            inside = [k for k, (x0, y0, x1, y1) in enumerate(page_rects) if x0 <= c[0] <= x1 and y0 <= c[1] <= y1]
            if len(inside) == 1 and page_words[inside[0]] == text:
                found.add(inside[0])
        hit += len(found)
    return hit, sum(len(w) for w in words)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(result, out_dir):
    """Writes a ``recognize`` result (per image, a list of (text, box)) as float32 arrays, images and words in order:

    ``counts.npy`` (n_images,)          words found in each image
    ``boxes.npy``  (n_words, 4, 2)      word quads in source-image pixels
    ``texts.npy``  (n_words, max_len)   Unicode code points of each word's text, zero-padded
    """
    texts = [text for group in result for text, _ in group]
    codes = np.zeros((len(texts), max((len(t) for t in texts), default=0)), np.float32)
    for i, text in enumerate(texts):
        codes[i, :len(text)] = [ord(c) for c in text]
    arrays = {
        "counts": np.array([len(group) for group in result], np.float32),
        "boxes": np.array([box for group in result for _, box in group], np.float32).reshape(-1, 4, 2),
        "texts": codes,
    }
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"outputs of one step take {total} bytes, more than the {DUMP_LIMIT_BYTES} a dump may hold")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1400.0))), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.device_index = device_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.device_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_sample(threads=None, n_images=1, rank=0):
    """Oracle port of the reference path on the host cores; returns (images/s, description, cores)."""
    import torch
    from keras_ocr_b200 import weights as W
    from oracle.pipeline import OraclePipeline

    if threads:
        torch.set_num_threads(threads)
    cores = torch.get_num_threads()
    pages = make_pages(rank)[:n_images]
    pipe = OraclePipeline(W.synthetic_craft_weights(3, textlike=True), W.synthetic_crnn_weights(2, decisive=True), scale=SCALE)
    t0 = time.perf_counter()
    out = pipe.recognize(pages)
    dt = time.perf_counter() - t0
    words = sum(len(g) for g in out)
    desc = (f"{n_images} page(s) {PAGE_H}x{PAGE_W} -> 1536x1536 of the same workload, {words} words found, "
            f"stages s: " + ", ".join(f"{k}={v:.2f}" for k, v in pipe.timings.items()))
    return n_images / dt, desc, cores


def host_threads():
    """Physical cores of the box.  torchrun exports OMP_NUM_THREADS=1 to every rank, which would leave the CPU arm on a
    single thread; the arm runs on rank 0 alone, so it sets torch's intra-op thread count explicitly.  (All logical
    threads -- 2 per core -- made the CRAFT forward 10x slower on these hosts: 59 s vs 6 s per page.)"""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except ImportError:
        n = None
    n = int(n or max(1, (os.cpu_count() or 2) // 2))
    try:
        n = min(n, len(os.sched_getaffinity(0)))        # a container may see fewer CPUs than the box has cores
    except AttributeError:
        pass
    return max(n, 1)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0                                        # rank 0 alone runs the CPU arm
    threads = host_threads()
    for _ in range(1 if args.warmup > 0 else 0):        # one warm-up pass pages everything in (each pass is ~6 s)
        cpu_sample(threads, 1)
    t0 = time.perf_counter()
    desc, used = "", 0
    for _ in range(args.steps):
        _, desc, used = cpu_sample(threads, 1)
    dt = time.perf_counter() - t0
    value = args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port",
                         "sample": "each step = 1 page of the workload's batch (bounded sample), rank 0 only; oracle port "
                                   "(torch-CPU fp32 CRAFT+CRNN, OpenCV getBoxes/warpBox) -- the reference needs TensorFlow, "
                                   "which is not installable offline; " + desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback (use --impl reference)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    from keras_ocr_b200 import distributed as D, weights as W
    from keras_ocr_b200.detection import Detector
    from keras_ocr_b200.pipeline import Pipeline
    from keras_ocr_b200.recognition import Recognizer

    det = Detector(weights=W.synthetic_craft_weights(3, textlike=True), device=local_rank)
    rec = Recognizer(weights=W.synthetic_crnn_weights(2, decisive=True), device=local_rank)
    pipe = Pipeline(detector=det, recognizer=rec, scale=SCALE, max_size=2048)
    pages, page_words, page_rects = make_pages(rank, with_layout=True)
    pages_dev = torch.from_numpy(pages).to(device)
    # the e2e leg's inputs live in PINNED host memory (the contract's "from pinned host memory"); the numpy
    # view below is what the user-facing call receives, and Pipeline uploads an already-pinned array as is
    pages_pinned = torch.from_numpy(pages).pin_memory()
    pages = pages_pinned.numpy()
    max_boxes = 128
    stats = {"words": 0}

    def step(inputs):
        if world == 1:
            result = pipe.recognize(inputs)
        else:
            # every rank runs its own 32 pages; the (count, boxes, labels) records are written on the device
            # (b2o_pack_records), gathered to rank 0 in ONE NCCL gather and decoded there -- the other ranks
            # never bring a result to the host
            result = D.recognize_sharded(pipe, inputs, max_boxes=max_boxes, presharded=True)
        if result is not None:
            stats["words"] = sum(len(g) for g in result)
            stats["last"] = result
        return result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: the K steps run as a stream, rank 0 decoding step k-1's gathered words while every GPU already works on step k
    # (distributed.ShardedStream); all K results are produced inside the timed region (the last one by flush()).  Measured on
    # 2 GPUs (profiles/r2d_bench_2gpu_*.json): 972.9 img/s against 969.2 with the per-step gather + decode
    # (B2O_BENCH_STREAM=0 selects that).
    stream = D.ShardedStream(pipe, max_boxes=max_boxes) if world > 1 and os.environ.get("B2O_BENCH_STREAM", "1") != "0" else None

    def timed(inputs, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if stream is not None:
            for _ in range(steps):
                stream.submit(inputs)
            result = stream.flush()
            if result is not None:
                stats["words"] = sum(len(g) for g in result)
                stats["last"] = result
        else:
            for _ in range(steps):
                step(inputs)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            every = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(every, ms)
            stats["per_rank_ms"] = [round(float(t.item()) / steps, 3) for t in every]   # names the limiter: rank 0 (decode) or a slow clock
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    for _ in range(max(args.warmup, 3)):
        step(pages_dev)
    step(pages)                                          # warm the host-input path too (pinned staging)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = det.ctx.launch_count() + rec.ctx.launch_count()
    D.stats["decode_ms"], D.stats["decodes"] = 0.0, 0
    stats["last"] = None
    ms_dev = timed(pages_dev, args.steps)
    last_result = stats["last"]                          # what the last timed step returned (rank 0)
    per_rank_dev = stats.get("per_rank_ms")
    decode_ms = D.stats["decode_ms"] / max(D.stats["decodes"], 1)
    launches = det.ctx.launch_count() + rec.ctx.launch_count() - launches0
    ms_e2e = timed(pages, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    h2d, d2h = pipe.last_stats.get("h2d_bytes", 0), pipe.last_stats.get("d2h_bytes", 0)
    if world > 1:                                        # rank 0 also reads the gathered record blocks
        d2h += world * PAGES_PER_RANK * det.ctx.record_floats(max_boxes) * 4

    # roofline leg: one extra step with per-launch CUDA events around the tensor-core conv kernel
    det.ctx.profile_enable(1); rec.ctx.profile_enable(1)
    step(pages_dev)
    torch.cuda.synchronize()
    ms_d, fl_d, n_d = det.ctx.profile_read()
    ms_r, fl_r, n_r = rec.ctx.profile_read()
    det.ctx.profile_enable(0); rec.ctx.profile_enable(0)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record(); step(pages_dev); a1.record(); torch.cuda.synchronize()
    step_ms_plain = a0.elapsed_time(a1)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    # what the benchmarked step produced, checked at full size on rank 0's pages (outside the timed region)
    hit, rendered = words_read(pipe.recognize(pages_dev), page_words, page_rects)
    total_pages = PAGES_PER_RANK * world
    value = total_pages * args.steps / (ms_dev / 1e3)
    e2e_value = total_pages * args.steps / (ms_e2e / 1e3)
    peak, peak_src = measured_peaks()
    tc_ms, tc_flop, tc_n = ms_d + ms_r, fl_d + fl_r, n_d + n_r
    achieved = tc_flop / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get("conv_tc_dram_bytes_per_launch")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16", "data": "synthetic",
        "config": dict(workload_config(world), **({"host_decode": "pipelined one step deep (ShardedStream)"} if stream else {})),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "conv_tc_kernel (tcgen05 implicit-GEMM conv/dense)",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "peak_source": peak_src, "launches_per_step": int(tc_n),
                     "flop_per_step": tc_flop, "kernel_ms_per_step": tc_ms,
                     "kernel_share_of_step": tc_ms / step_ms_plain if step_ms_plain > 0 else None,
                     "traffic": traffic},
        "words_per_step": stats["words"],
        "words_read_correctly": {"rank0_pages": PAGES_PER_RANK, "rendered": rendered, "read": hit},
    }
    if hit < 0.9 * rendered:                                # reported, never fatal: the line above is the measurement
        sys.stderr.write(f"bench.py: only {hit} of {rendered} rendered words were read correctly\n")
    if world > 1:
        line["per_rank_ms_per_step"] = per_rank_dev
        line["rank0_decode_ms_per_step"] = round(decode_ms, 3)
    if world == 1:
        v, desc, cores = cpu_sample(host_threads(), 1)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": "oracle port of the reference path (TensorFlow not installable offline): " + desc}
    if args.dump_outputs:
        dump_outputs(last_result, args.dump_outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results to DIR/<name>.npy (b200 only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    sys.exit(run_reference(args) if args.impl == "reference" else run_b200(args))


if __name__ == "__main__":
    main()
