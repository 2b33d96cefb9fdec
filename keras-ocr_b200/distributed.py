"""Multi-GPU ``Pipeline.recognize``: one process per GPU, images sharded by batch, ONE gather.

The reference is single-process (SURVEY.md 2.3); images are fully independent in
``Pipeline.recognize`` (reference pipeline.py:28-75), so the path shards with no data-path
collective.  Each rank runs the whole pipeline on its contiguous slice and the per-image result
records -- ``count`` (int32), ``boxes`` (M,4,2) float32, ``labels`` (M,steps) int8 -- are gathered to
rank 0 with a single ``torch.distributed.gather`` over NCCL/NVLink (``gloo`` in the CPU tests).  ``steps`` is the
recognizer's label row length (``Recognizer.steps``: 48 for the default 31 x 200 crops).
"""
import numpy as np
import torch
import torch.distributed as dist

STEPS = 48                                             # label row length of the default recognizer


def label_slots(steps):
    """float32 slots per word of a record's label area: ``steps`` int8 labels, 4 per slot (b2o_record_floats_steps)."""
    return (int(steps) + 3) // 4


def _steps_of(pipeline):
    return int(getattr(pipeline.recognizer, "steps", STEPS))


def shard_bounds(n_items, world_size, rank):
    """Contiguous shard [lo, hi) of ``n_items`` for ``rank`` (first ``n_items % world`` ranks get one more)."""
    base, extra = divmod(n_items, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def pack_records(counts, boxes, labels, per_rank, max_boxes, steps=STEPS):
    """Fixed-size record block for one rank: float32 tensor (per_rank, 1 + max_boxes*8 + max_boxes*ceil(steps/4)).

    labels (int8, ``steps`` per word) are bit-packed 4 per float32 slot so that a single dtype travels; the words'
    labels lie back to back and the bytes after the last one are -1 (the layout of b2o_pack_records_steps).
    counts (n,), boxes (n,M,4,2) float32, labels (sum(counts),steps) int -> one contiguous CPU tensor.
    """
    n = len(counts)
    slots = label_slots(steps)
    rec = np.zeros((per_rank, 1 + max_boxes * 8 + max_boxes * slots), dtype=np.float32)
    lab_area = np.full((per_rank, max_boxes * slots * 4), -1, dtype=np.int8)
    lab8 = lab_area[:, :max_boxes * steps].reshape(per_rank, max_boxes, steps)
    start = 0
    for i in range(n):
        c = min(int(counts[i]), max_boxes)
        rec[i, 0] = int(counts[i])                     # what the image HAS; unpack_blocks refuses counts > max_boxes
        rec[i, 1:1 + c * 8] = np.asarray(boxes[i][:c], dtype=np.float32).reshape(-1)
        if c:
            lab8[i, :c] = np.asarray(labels[start:start + c], dtype=np.int8)
        start += int(counts[i])
    rec[:, 1 + max_boxes * 8:] = lab_area.view(np.float32)
    rec[n:, 0] = -1                                    # padding rows of a short last shard
    return torch.from_numpy(rec)


def unpack_records(rec, max_boxes, steps=STEPS):
    """Inverse of pack_records for one rank's block -> list of (count, boxes (c,4,2), labels (c,steps))."""
    counts, boxes, labels = unpack_blocks([rec], max_boxes, steps=steps)
    ends = np.cumsum(counts)
    return [(int(c), boxes[e - c:e], labels[e - c:e].astype(np.int32)) for c, e in zip(counts, ends)]


class RecordOverflow(ValueError):
    """An image has more words than a fixed-size record holds (``max_boxes``)."""


def unpack_blocks(blocks, max_boxes, strict=True, steps=STEPS):
    """All gathered blocks at once (rank order = global image order): returns (counts (n_images,), boxes (total,4,2)
    float32, labels (total,steps) int8) with the words of image i at [sum(counts[:i]), +counts[i]).  Only the used
    prefix of every record is touched (two concatenations of per-image views), not the 75 % padding.

    A record's count field is the number of words its image HAS; a record holds ``max_boxes`` of them.  The
    single-GPU ``Pipeline.recognize`` grows its box table on demand (as the reference returns every box), so a
    count above ``max_boxes`` raises ``RecordOverflow`` rather than dropping words (``strict=False``: keep the
    first ``max_boxes``, for callers that asked for a cap)."""
    box_parts, lab_parts, counts = [], [], []
    lab0 = (1 + max_boxes * 8) * 4                     # byte offset of the label area inside a record
    for r, block in enumerate(blocks):
        rec = np.ascontiguousarray(np.asarray(block.cpu() if isinstance(block, torch.Tensor) else block))
        rec8 = rec.view(np.int8)
        for i, c in enumerate(rec[:, 0].astype(np.int64).tolist()):
            if c < 0:                                  # padding row of a short shard
                continue
            if c > max_boxes:
                if strict:
                    raise RecordOverflow(f"image {i} of rank {r} has {c} words but the gathered records hold "
                                         f"max_boxes={max_boxes}: pass a larger max_boxes (or max_boxes='auto')")
                c = max_boxes
            counts.append(c)
            if c:
                box_parts.append(rec[i, 1:1 + c * 8])
                lab_parts.append(rec8[i, lab0:lab0 + c * steps])
    boxes = np.concatenate(box_parts).reshape(-1, 4, 2) if box_parts else np.zeros((0, 4, 2), np.float32)
    labels = np.concatenate(lab_parts).reshape(-1, steps) if lab_parts else np.zeros((0, steps), np.int8)
    return np.asarray(counts, dtype=np.int64), boxes, labels


def gather_records(local, world_size, rank, device=None):
    """The single collective: gather every rank's record block to rank 0.  Returns the list of blocks
    on rank 0, None elsewhere."""
    if world_size == 1:
        return [local]
    t = local.to(device) if device is not None else local
    blocks = [torch.empty_like(t) for _ in range(world_size)] if rank == 0 else None
    dist.gather(t, gather_list=blocks, dst=0)
    return blocks


def _host_records(pipeline, local, per_rank, max_boxes, steps=STEPS):
    """Record block of a duck-typed pipeline: pack the (word, box) lists its ``recognize`` returned on the host."""
    alphabet = pipeline.recognizer.alphabet
    counts = [len(g) for g in local]
    boxes = [np.array([b for _, b in g], dtype=np.float32).reshape(-1, 4, 2) for g in local]
    labels = np.full((sum(counts), steps), -1, dtype=np.int8)
    k = 0
    for g in local:
        for text, _ in g:
            labels[k, :len(text)] = [alphabet.index(ch) for ch in text]
            k += 1
    return pack_records(counts, boxes, labels, per_rank, max_boxes, steps)


def recognize_sharded(pipeline, images, max_boxes=128, presharded=False, steps=None):
    """Run ``pipeline.recognize`` on this rank's shard of ``images`` and gather to rank 0.

    ``images`` is the global batch (every rank passes the same list and takes its contiguous slice) or, with
    ``presharded=True``, this rank's own slice (equal length on every rank).  A pipeline that offers
    ``recognize_records`` (this package's ``Pipeline`` with its own Detector / Recognizer) never brings its
    results to the host: the record block is written by ``b2o_pack_records`` on the device, gathered over
    NCCL/NVLink, and copied to the host once, on rank 0.  Any other pipeline goes through ``recognize`` and
    ``pack_records``.

    ``steps``: label row length of the records (default: ``pipeline.recognizer.steps``, 48 for the default recognizer).

    Returns, on rank 0, the same list-of-lists as ``Pipeline.recognize`` for ALL images (global
    order); ``None`` on the other ranks.  Boxes are in source-image pixels.
    """
    steps = _steps_of(pipeline) if steps is None else int(steps)
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    if presharded:
        mine, per_rank = images, len(images)
    else:
        lo, hi = shard_bounds(len(images), world, rank)
        mine, per_rank = images[lo:hi], shard_bounds(len(images), world, 0)[1]
    alphabet = pipeline.recognizer.alphabet
    assert len(alphabet) + 1 <= 127, "record labels travel as int8: alphabets up to 126 characters"
    if per_rank == 0:
        return [] if rank == 0 else None
    native = getattr(pipeline, "recognize_records", None) is not None and getattr(pipeline, "_native", lambda: True)()
    if native:
        if getattr(pipeline, "records_counts", None) is not None:
            state = pipeline.records_begin(mine, rows=per_rank, rec_boxes=16 if max_boxes == "auto" else max_boxes)
            if max_boxes == "auto":
                max_boxes = agree_max_boxes(pipeline.records_counts(state), _collective_device(pipeline))
            local = pipeline.records_end(state, rec_boxes=max_boxes)
        else:                                           # a pipeline that only offers the one-call form
            assert max_boxes != "auto", "max_boxes='auto' needs records_begin / records_counts / records_end"
            local = pipeline.recognize_records(mine, rows=per_rank, rec_boxes=max_boxes)
        device = None                                   # already where the backend wants it
    else:
        result = pipeline.recognize(mine) if len(mine) else []
        if max_boxes == "auto":
            max_boxes = agree_max_boxes([len(g) for g in result], _collective_device(pipeline))
        local = _host_records(pipeline, result, per_rank, max_boxes, steps)
        device = _collective_device(pipeline)
    blocks = gather_records(local, world, rank, device)
    if rank != 0:
        return None
    return _decode_blocks(blocks, max_boxes, alphabet, steps)


def _collective_device(pipeline):
    """Where tensors must live for the process group's collectives: the GPU under NCCL, the host under gloo."""
    return pipeline.detector.device if dist.is_initialized() and dist.get_backend() == "nccl" else None


def agree_max_boxes(counts, device=None, floor=16):
    """``max_boxes='auto'``: every rank contributes its largest per-image word count; ONE all-reduce (MAX) of a
    single int gives the record size all ranks use for this batch (next power of two, at least ``floor``), so a dense
    page costs nothing on sparse batches and nothing is ever dropped.  Costs one extra tiny collective + sync per
    batch, which is why a fixed ``max_boxes`` (overflow = ``RecordOverflow`` on rank 0) stays the default."""
    local = int(max(counts)) if len(counts) else 0
    if dist.is_initialized() and dist.get_world_size() > 1:
        t = torch.tensor([local], dtype=torch.int32, device=device if device is not None else "cpu")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        local = int(t.item())
    size = floor
    while size < local:
        size *= 2
    return size


stats = {"decode_ms": 0.0, "decodes": 0}      # rank 0's serial host work (bench.py reports it per step)


def _decode_blocks(blocks, max_boxes, alphabet, steps=STEPS):
    import time

    from . import recognition

    t0 = time.perf_counter()
    try:
        return _decode_blocks_impl(blocks, max_boxes, alphabet, recognition, steps)
    finally:
        stats["decode_ms"] += (time.perf_counter() - t0) * 1e3
        stats["decodes"] += 1


def _decode_blocks_impl(blocks, max_boxes, alphabet, recognition, steps):
    counts, boxes, labels = unpack_blocks(blocks, max_boxes, steps=steps)
    texts = recognition.labels_to_text(labels, alphabet)
    quads, out, start = list(boxes), [], 0             # one (4,2) view per word, made once
    for c in counts.tolist():
        out.append(list(zip(texts[start:start + c], quads[start:start + c])))
        start += c
    return out


class ShardedStream:
    """``recognize_sharded`` for a STREAM of batches, software-pipelined one batch deep: while every rank's GPU works
    on batch k, rank 0 decodes the gathered words of batch k-1 (the only serial host work of the multi-GPU path:
    ~3 ms for 8 x 1028 words).  Every rank passes its own, equally long, slice of each batch.

        stream = ShardedStream(pipeline)
        for batch in batches:
            done = stream.submit(batch)      # rank 0: results of the PREVIOUS batch (None for the first); other ranks: None
        last = stream.flush()                # rank 0: results of the last batch

    With this package's ``Pipeline`` the records stay on the device until the gather and reach the host through ONE
    asynchronous copy into pinned memory; any other pipeline (``recognize`` only) is served too, without the overlap.
    ``max_boxes``: words a record holds (an image with more raises ``RecordOverflow`` on rank 0 when its batch is
    decoded) or ``"auto"`` (sized per batch by ``agree_max_boxes``).  ``steps``: label row length of the records
    (default: ``pipeline.recognizer.steps``, 48 for the default recognizer)."""

    def __init__(self, pipeline, max_boxes=128, steps=None):
        self.pipeline, self.max_boxes = pipeline, max_boxes
        self.steps = _steps_of(pipeline) if steps is None else int(steps)
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.alphabet = pipeline.recognizer.alphabet
        assert len(self.alphabet) + 1 <= 127, "record labels travel as int8: alphabets up to 126 characters"
        self._native = (getattr(pipeline, "records_begin", None) is not None
                        and getattr(pipeline, "_native", lambda: True)())
        self._pending = None                             # (host blocks, event or None) of the batch in flight
        self._side = None                                # communication stream (CUDA tensors only)
        self._keep = None

    def _take_pending(self):
        if self._pending is None or self.rank != 0:
            self._pending = None
            return None
        host, event, max_boxes = self._pending
        self._pending = None
        if event is not None:
            event.synchronize()
        return _decode_blocks(list(host), max_boxes, self.alphabet, self.steps)

    def submit(self, images):
        rows = len(images)
        if rows == 0:
            return self._take_pending()
        max_boxes = self.max_boxes
        if self._native:
            state = self.pipeline.records_begin(images, rows=rows, rec_boxes=16 if max_boxes == "auto" else max_boxes)   # GPU busy from here on
            previous = self._take_pending()              # ... while the host decodes the batch before
            if max_boxes == "auto":
                max_boxes = agree_max_boxes(self.pipeline.records_counts(state), _collective_device(self.pipeline))
            local = self.pipeline.records_end(state, rec_boxes=max_boxes)
            device = None
        else:
            previous = self._take_pending()
            result = self.pipeline.recognize(images)
            if max_boxes == "auto":
                max_boxes = agree_max_boxes([len(g) for g in result], _collective_device(self.pipeline))
            local = _host_records(self.pipeline, result, rows, max_boxes, self.steps)
            device = _collective_device(self.pipeline)
        if local.is_cuda or device is not None:
            self._gather_on_side_stream(local.to(device) if device is not None else local, max_boxes)
            return previous
        blocks = gather_records(local, self.world, self.rank, None)      # host tensors (gloo): plain blocking gather
        if self.rank == 0:
            self._pending = (torch.stack(list(blocks)), None, max_boxes)
        return previous

    def _gather_on_side_stream(self, local, max_boxes):
        """The gather and rank 0's copy to the host run on a SIDE stream that waits for this batch's records; the compute
        stream is never made to wait for another rank (with the collective on the compute stream, rank 0's next batch queued
        behind a gather that completes only when the slowest rank has sent: measured on 8 GPUs, rank 0 66.0 ms per step against
        62.4-65.0 for the others, profiles/r2scale8_bench_8gpu.json)."""
        main = torch.cuda.current_stream(local.device)
        if self._side is None:
            self._side = torch.cuda.Stream(device=local.device)
        ready = torch.cuda.Event()
        ready.record(main)
        with torch.cuda.stream(self._side):
            self._side.wait_event(ready)
            local.record_stream(self._side)
            blocks = gather_records(local, self.world, self.rank, None)
            if self.rank == 0:
                stacked = torch.stack(list(blocks))
                host = torch.empty(stacked.shape, dtype=stacked.dtype, pin_memory=True)
                host.copy_(stacked, non_blocking=True)   # one asynchronous copy into pinned memory; waited for at decode time
                event = torch.cuda.Event()
                event.record(self._side)
                self._pending = (host, event, max_boxes)
                self._keep = (stacked, blocks)           # alive until the copy has run
            else:
                self._keep = local                       # alive until the send has run (next submit replaces it)

    def flush(self):
        return self._take_pending()
