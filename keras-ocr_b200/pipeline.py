"""Pipeline: drop-in for ``keras_ocr.pipeline.Pipeline`` (reference pipeline.py:7-75)."""
import numpy as np
import torch

from . import detection, recognition, tools


class Pipeline:
    """A wrapper for a combination of detector and recognizer.

    Args:
        detector: The detector to use (default: ``detection.Detector()``)
        recognizer: The recognizer to use (default: ``recognition.Recognizer()``)
        scale: The scale factor to apply to input images
        max_size: The maximum single-side dimension of images for inference.

    Any object with ``detect`` / ``recognize_from_boxes`` can be injected, as in the reference
    (pipeline.py:18-26, 62-65); with this package's own Detector and Recognizer the whole call
    stays on the GPU between the host->device copy of the images and the device->host copy of
    (counts, boxes, labels).
    """

    def __init__(self, detector=None, recognizer=None, scale=2, max_size=2048, inflight=1, gpu_decode=False):
        if detector is None:
            detector = detection.Detector()
        if recognizer is None:
            recognizer = recognition.Recognizer()
        self.scale = scale
        self.detector = detector
        self.recognizer = recognizer
        self.max_size = max_size
        # inflight > 1: batches of >= inflight * min_chunk images are processed as `inflight` sub-batches,
        # software-pipelined on one stream: while the host waits for the box counts of one sub-batch (the path's
        # one data-dependent synchronisation) or decodes its labels, the GPU already runs the next one.  Results
        # are identical to the unsplit batch (images are independent; the padding is that of the whole batch).
        # Measured on the 32-page bench: ~2 % faster device-resident, but the half-size recurrent / box kernels
        # lose what the overlap gains and the end-to-end number does not move, hence the default of 1.
        self.inflight = inflight
        # gpu_decode: JPEG files / buffers in ``images`` are decoded by nvJPEG into device memory (tools.read_device)
        # instead of cv2 on the host (reference tools.py:19-38); pixels may differ from libjpeg's by a few levels, which is
        # why it is opt-in for a drop-in.
        self.gpu_decode = gpu_decode
        self.min_chunk = 4
        self.last_stats = {}
        self._h2d_stream = None

    def _native(self):
        return isinstance(self.detector, detection.Detector) and isinstance(self.recognizer, recognition.Recognizer)

    def _upload(self, array):
        """Host uint8 array -> CUDA tensor through pinned memory on a side stream, so the copy overlaps kernels
        already queued on the compute stream; the compute stream waits for the copy's event."""
        det = self.detector
        if self._h2d_stream is None:
            self._h2d_stream = torch.cuda.Stream(device=det.device)
        main = torch.cuda.current_stream(det.device)
        pinned = torch.from_numpy(np.ascontiguousarray(array))
        if not pinned.is_pinned():                       # callers that already hold pinned pages skip the staging copy
            pinned = pinned.pin_memory()
        if self.inflight <= 1:                           # nothing queued to overlap with: plain stream-ordered copy
            return pinned.to(det.device, non_blocking=True)
        with torch.cuda.stream(self._h2d_stream):
            t = pinned.to(det.device, non_blocking=True)
            done = torch.cuda.Event()
            done.record(self._h2d_stream)
        t.record_stream(main)
        main.wait_event(done)
        return t

    def _plans(self, images):
        """(scale, height, width) after tools.resize_image for every image (one rule for a 4-D batch)."""
        if isinstance(images, (np.ndarray, torch.Tensor)) and images.ndim == 4:
            return [tools.resize_plan(tuple(images.shape[1:]), self.scale, self.max_size)] * len(images)
        return [tools.resize_plan(tuple(image.shape), self.scale, self.max_size) for image in images]

    def prepare_device(self, images, pad_to=None, want_gray=False):
        """resize_image + pad (pipeline.py:44-57) on the GPU.  Returns ((N,H,W,3) u8 CUDA tensor, scales), plus
        the gray batch (N,H,W) u8 (recognition.py:510) or None when ``want_gray``: equally sized sources (a 4-D
        array / tensor) are resized in ONE launch that also writes the gray image the recognizer needs.
        ``pad_to``: (height, width) of the padded batch when ``images`` is part of a larger batch."""
        det = self.detector
        plans = self._plans(images)
        scales = [p[0] for p in plans]
        hp, wp = pad_to if pad_to is not None else (max(p[1] for p in plans), max(p[2] for p in plans))
        n = len(images)
        stream = torch.cuda.current_stream(det.device).cuda_stream
        batch = torch.empty((n, hp, wp, 3), dtype=torch.uint8, device=det.device)
        same = isinstance(images, np.ndarray) and images.ndim == 4
        h2d, gray = 0, None
        if isinstance(images, torch.Tensor):
            # sources already resident in HBM (bench.py's device-resident leg): no copy
            assert images.is_cuda and images.dtype == torch.uint8 and images.dim() == 4
            src_all, same = images.contiguous(), True
        elif same:
            assert images.shape[3] == 3 and images.dtype == np.uint8, "images must be HxWx3 uint8"
            src_all = self._upload(images)
            h2d = src_all.numel()
        if same:
            _, hr, wr = plans[0]
            gray = torch.empty((n, hp, wp), dtype=torch.uint8, device=det.device)
            det.ctx.resize_pad_batch(src_all.data_ptr(), n, src_all.shape[1], src_all.shape[2], hr, wr, batch.data_ptr(),
                                     hp, wp, gray.data_ptr(), stream)
        else:
            for i, image in enumerate(images):
                if isinstance(image, torch.Tensor):                # decoded on the device (gpu_decode) or supplied resident
                    assert image.is_cuda and image.dim() == 3 and image.shape[2] == 3 and image.dtype == torch.uint8
                    src = image.contiguous()
                else:
                    assert image.ndim == 3 and image.shape[2] == 3 and image.dtype == np.uint8, "images must be HxWx3 uint8"
                    src = self._upload(image)
                    h2d += src.numel()
                _, hr, wr = plans[i]
                det.ctx.resize_pad(src.data_ptr(), image.shape[0], image.shape[1], hr, wr, batch.data_ptr(), i, hp, wp, stream)
        self.last_stats["h2d_bytes"] = self.last_stats.get("h2d_bytes", 0) + int(h2d)
        return (batch, scales, gray) if want_gray else (batch, scales)

    # ---------------------------------------------------------------- the three stages of one sub-batch
    def _stage_detect(self, images, pad_to, thresholds):
        batch, scales, gray = self.prepare_device(images, pad_to, want_gray=True)
        scores = self.detector.predict_device(batch)
        return {"batch": batch, "scales": scales, "gray": gray,
                "boxes_state": self.detector.boxes_enqueue(scores, **thresholds)}

    def _stage_recognize(self, st):
        det, rec = self.detector, self.recognizer
        bst = st.pop("boxes_state")
        boxes, counts = det.boxes_finish(bst)
        labels = rec.recognize_from_boxes_device(st["batch"], boxes, counts, gray=st["gray"], flat=bst["flat"],
                                                 image_index=bst["image_index"])
        st["counts"] = counts
        st["boxes_host"] = torch.empty(boxes.shape, dtype=boxes.dtype, pin_memory=True)
        st["boxes_host"].copy_(boxes, non_blocking=True)
        if labels is not None:
            st["labels_host"] = torch.empty(labels.shape, dtype=labels.dtype, pin_memory=True)
            st["labels_host"].copy_(labels, non_blocking=True)
        st["keep"] = (boxes, labels)                     # alive until the copies have run
        st["done"] = torch.cuda.Event()
        st["done"].record(torch.cuda.current_stream(det.device))

    def _stage_finish(self, st):
        st["done"].synchronize()
        boxes_host, counts = st["boxes_host"].numpy(), st["counts"]
        d2h = boxes_host.nbytes + counts.nbytes
        if "labels_host" in st:
            labels_host = st["labels_host"].numpy()
            d2h += labels_host.nbytes
            texts = recognition.labels_to_text(labels_host, self.recognizer.alphabet)
        else:
            texts = []
        self.last_stats["d2h_bytes"] += int(d2h)
        out, start = [], 0
        for i, (c, scale) in enumerate(zip(counts, st["scales"])):
            c = int(c)
            group = boxes_host[i, :c].copy()
            if scale != 1:
                group = tools.adjust_boxes(boxes=group, boxes_format="boxes", scale=1 / scale)
            out.append(list(zip(texts[start:start + c], group)))
            start += c
        return out

    def recognize(self, images, detection_kwargs=None, recognition_kwargs=None):
        """Run the pipeline on one or multiple images (reference pipeline.py:28-75).

        Returns a list (one entry per image) of lists of (text, box) tuples, boxes (4,2) float32 in
        the coordinates of the *input* image.
        """
        if not isinstance(images, (np.ndarray, torch.Tensor)):
            if self.gpu_decode and self._native():
                images = [tools.read_device(image, self.detector.ctx, self.detector.device) for image in images]
            else:
                images = [tools.read(image) for image in images]
        if detection_kwargs is None:
            detection_kwargs = {}
        if recognition_kwargs is None:
            recognition_kwargs = {}
        if not self._native():
            return self._recognize_generic(images, detection_kwargs, recognition_kwargs)
        thresholds = {k: detection_kwargs[k] for k in ("detection_threshold", "text_threshold", "link_threshold",
                                                        "size_threshold") if k in detection_kwargs}
        n = len(images)
        self.last_stats = {"h2d_bytes": 0, "d2h_bytes": 0}
        if n == 0:
            return []
        plans = self._plans(images)
        pad_to = (max(p[1] for p in plans), max(p[2] for p in plans))      # of the WHOLE batch (pipeline.py:48-57)
        k = max(1, min(int(self.inflight), n // self.min_chunk))
        bounds = [n * i // k for i in range(k + 1)]
        states, out = [], []
        for step in range(k + 2):                        # detect(i) | recognize(i-1) | finish(i-2)
            if step < k:
                states.append(self._stage_detect(images[bounds[step]:bounds[step + 1]], pad_to, thresholds))
            if 1 <= step <= k:
                self._stage_recognize(states[step - 1])
            if step >= 2:
                out.extend(self._stage_finish(states[step - 2]))
                states[step - 2] = None
        return out

    def recognize_records(self, images, rows=None, rec_boxes=128, detection_kwargs=None):
        """``recognize`` without the trip to the host: returns the results as a CUDA float32 tensor of fixed-size
        per-image records, ``(rows, b2o_record_floats_steps(rec_boxes, steps))`` = [count | rec_boxes x (4,2) boxes in
        source pixels | rec_boxes x steps int8 labels], steps = ``recognizer.steps`` (48 for the default recognizer;
        ``distributed.unpack_blocks(..., steps=steps)`` decodes it; rows beyond ``len(images)`` carry count -1).  This is the payload of the multi-GPU gather (SURVEY.md 8(e)): only the per-image box
        counts ever reach the host on this rank."""
        return self.records_end(self.records_begin(images, rows, rec_boxes, detection_kwargs))

    def records_begin(self, images, rows=None, rec_boxes=128, detection_kwargs=None):
        """First half of ``recognize_records``: queues resize/pad, CRAFT and getBoxes and returns at once (no
        synchronisation), so the caller can use the host while the GPU works (``distributed.ShardedStream`` decodes the
        previous batch's words here).  Pass the returned state to ``records_end``."""
        assert self._native(), "recognize_records needs this package's Detector and Recognizer"
        assert len(self.recognizer.alphabet) + 1 <= 127, "record labels travel as int8: alphabets up to 126 characters"
        if not isinstance(images, (np.ndarray, torch.Tensor)):
            if self.gpu_decode:
                images = [tools.read_device(image, self.detector.ctx, self.detector.device) for image in images]
            else:
                images = [tools.read(image) for image in images]
        thresholds = {k: v for k, v in (detection_kwargs or {}).items()
                      if k in ("detection_threshold", "text_threshold", "link_threshold", "size_threshold")}
        n = len(images)
        rows = n if rows is None else int(rows)
        assert rows >= n and rows > 0
        self.last_stats = {"h2d_bytes": 0, "d2h_bytes": 0}
        state = {"n": n, "rows": rows, "rec_boxes": rec_boxes}
        if n:
            plans = self._plans(images)
            state["st"] = self._stage_detect(images, (max(p[1] for p in plans), max(p[2] for p in plans)), thresholds)
        return state

    def records_counts(self, state):
        """Waits for the box counts of ``records_begin`` (the path's one synchronisation) and returns them (host
        ndarray, one per image) -- what a caller needs to size ``rec_boxes`` before ``records_end``."""
        if state["n"] == 0:
            return np.zeros((0,), np.int32)
        if "counts" not in state:
            st = state["st"]
            bst = st["boxes_state"]
            state["boxes"], state["counts"] = self.detector.boxes_finish(bst)
        return state["counts"]

    def records_end(self, state, rec_boxes=None):
        """Second half of ``recognize_records``: waits for the box counts (the path's one synchronisation), queues
        warp + CRNN + ``b2o_pack_records`` and returns the CUDA record tensor.  A record holds ``rec_boxes`` words;
        its count field carries what the image has, so the reader (``distributed.unpack_blocks``) notices an image
        that does not fit instead of losing words."""
        det, rec = self.detector, self.recognizer
        n, rows = state["n"], state["rows"]
        rec_boxes = state["rec_boxes"] if rec_boxes is None else int(rec_boxes)
        records = torch.empty((rows, det.ctx.record_floats(rec_boxes, rec.steps)), dtype=torch.float32, device=det.device)
        if n == 0:
            records.zero_()
            records[:, 0] = -1
            return records
        counts = self.records_counts(state)
        st = state["st"]
        bst = st.pop("boxes_state")
        boxes = state["boxes"]
        labels = rec.recognize_from_boxes_device(st["batch"], boxes, counts, gray=st["gray"], flat=bst["flat"],
                                                 image_index=bst["image_index"])
        inv = torch.tensor([1.0 / s for s in st["scales"]], dtype=torch.float32).to(det.device, non_blocking=True)
        det.ctx.pack_records(boxes.data_ptr(), bst["counts"].data_ptr(), labels.data_ptr() if labels is not None else None,
                             inv.data_ptr(), n, boxes.shape[1], rows, rec_boxes, records.data_ptr(),
                             torch.cuda.current_stream(det.device).cuda_stream, steps=rec.steps)
        self.last_stats["d2h_bytes"] = int(counts.nbytes)
        return records

    def _recognize_generic(self, images, detection_kwargs, recognition_kwargs):
        """Reference flow for injected (duck-typed) detectors / recognizers: host arrays between stages."""
        import cv2

        resized = []
        for image in images:
            scale, hr, wr = tools.resize_plan(image.shape, self.scale, self.max_size)
            resized.append((cv2.resize(image, dsize=(wr, hr)), scale))
        max_height, max_width = np.array([im.shape[:2] for im, _ in resized]).max(axis=0)
        scales = [s for _, s in resized]
        padded = []
        for im, _ in resized:
            canvas = np.zeros((max_height, max_width, 3), dtype=im.dtype) + 255
            canvas[: im.shape[0], : im.shape[1]] = im
            padded.append(canvas)
        batch = np.array(padded)
        box_groups = self.detector.detect(images=batch, **detection_kwargs)
        prediction_groups = self.recognizer.recognize_from_boxes(images=batch, box_groups=box_groups, **recognition_kwargs)
        box_groups = [tools.adjust_boxes(boxes=boxes, boxes_format="boxes", scale=1 / scale) if scale != 1 else boxes
                      for boxes, scale in zip(box_groups, scales)]
        return [list(zip(predictions, boxes)) for predictions, boxes in zip(prediction_groups, box_groups)]
