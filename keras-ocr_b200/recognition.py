"""Recognizer: drop-in for ``keras_ocr.recognition.Recognizer`` (reference recognition.py:353-537)."""
import string
import typing

import numpy as np
import torch

from . import _lib, tools, weights as weights_mod

DEFAULT_ALPHABET = string.digits + string.ascii_lowercase      # reference recognition.py:25
TARGET_HEIGHT, TARGET_WIDTH, STEPS = 31, 200, 48                # DEFAULT_BUILD_PARAMS, recognition.py:13-23 (the defaults;
                                                                # a Recognizer's own are its height / width / steps)
DEFAULT_BUILD_PARAMS = {"height": 31, "width": 200, "color": False, "filters": (64, 128, 256, 256, 512, 512, 512),
                        "rnn_units": (128, 128), "dropout": 0.25, "rnn_steps_to_discard": 2, "pool_size": 2}


def labels_to_text(rows, alphabet=DEFAULT_ALPHABET):
    """reference recognition.py:527-534: drop blank / -1, map indices to characters.

    Vectorised: the kept labels of all rows are gathered into ONE byte string with a newline after every row, decoded
    once and split (no per-character and no per-row Python work besides the split); alphabets that are not ASCII or
    contain a newline, and tables with out-of-range indices, take the reference's element-wise filter."""
    blank = len(alphabet)
    rows = np.asarray(rows)
    if rows.ndim == 2 and rows.size and alphabet.isascii() and "\n" not in alphabet:
        keep = (rows != blank) & (rows != -1)
        flat = rows[keep]
        if flat.size == 0 or (int(flat.min()) >= 0 and int(flat.max()) < blank):
            out = np.full(flat.size + rows.shape[0], 10, dtype=np.uint8)          # 10 = "\n"
            ends = np.cumsum(keep.sum(1) + 1) - 1
            chars = np.ones(out.size, dtype=bool)
            chars[ends] = False
            out[chars] = np.frombuffer(alphabet.encode("ascii"), dtype=np.uint8)[flat]
            return out.tobytes().decode("ascii").split("\n")[:-1]
    return ["".join(alphabet[idx] for idx in row if idx not in (blank, -1)) for row in rows]


class Recognizer:
    """A text recognizer using the CRNN architecture, running as sm_100a CUDA kernels.

    Args:
        alphabet: the characters the model recognises (default ``0-9a-z``; up to 1023 characters).  The
            checkpoint's ``fc_12`` must have ``len(alphabet) + 1`` classes; if it does not, the reference's
            "backbone weights only" behaviour applies (recognition.py:399-411): the top layer is
            re-initialised (Glorot uniform, zero bias) and has to be trained before it is useful.
        weights: ``None`` builds an untrained model for ``alphabet`` (as the reference does); ``"kurapan"`` looks for ``crnn_kurapan.npz`` (exported) or the reference's ``crnn_kurapan.h5``
            (read with h5py where installed) in the cache dir; otherwise a ``.npz`` / ``.h5`` path or a dict
            keyed like ``weights.py``.
        build_params: ``None`` / the defaults (reference recognition.py:13-23), optionally with ``"stn": False`` (the
            recognizer without the spatial transformer, recognition.py:243), ``"color": True`` (RGB crops into a
            3-channel ``conv_1``, recognition.py:214), another crop size ``"height"`` / ``"width"`` and another
            ``"rnn_steps_to_discard"`` (recognition.py:214, 328); ``"dropout"`` is accepted and has no effect at
            inference.  Crops are ``height x width``; the model reads ``T = width // 4`` time steps and returns label
            rows of ``T - rnn_steps_to_discard`` (the instance's ``steps``; 48 by default).  Supported: height 16..64,
            width 32..800, ``0 <= rnn_steps_to_discard < width // 4`` -- ValueError otherwise.  Other ``filters``,
            ``rnn_units`` or ``pool_size`` raise NotImplementedError.
    """

    def __init__(self, alphabet=None, weights="kurapan", build_params=None, device=None):
        assert alphabet or weights, "At least one of alphabet or weights must be provided."
        # build_params (recognition.py:13-23, 365-368): the CUDA recognizer implements the default layer stack; of the
        # build options ``stn`` (with / without the spatial transformer, recognition.py:243), ``color`` (RGB instead of
        # gray crops, recognition.py:214), the crop size and the discarded steps (214, 328) may differ, and ``dropout``
        # is an inference no-op (321)
        params = dict(DEFAULT_BUILD_PARAMS, **(build_params or {}))
        self.stn = bool(params.pop("stn", True))
        self.color = bool(params.pop("color"))                    # RGB crops, no gray conversion (recognition.py:214, 508-510)
        self.height, self.width = params.pop("height"), params.pop("width")
        self.rnn_steps_to_discard = params.pop("rnn_steps_to_discard")
        params.pop("dropout")
        changed = sorted(k for k in params if params[k] != DEFAULT_BUILD_PARAMS.get(k))
        if changed:
            raise NotImplementedError(f"build_params other than the defaults are not supported by the CUDA recognizer: {changed}")
        self._check_geometry()
        self.steps = self.width // 4 - self.rnn_steps_to_discard  # label row length (CTC input_length)
        if not torch.cuda.is_available():
            raise _lib.B2OError("keras-ocr_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.alphabet = alphabet or DEFAULT_ALPHABET              # recognition.py:369-375
        if len(self.alphabet) + 1 > _lib.MAX_CLASSES:
            raise ValueError(f"alphabet too long: at most {_lib.MAX_CLASSES - 1} characters")
        self.blank_label_idx = len(self.alphabet)
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        if isinstance(weights, dict):
            tensors = weights
        elif weights is None:
            # reference recognition.py:382-383: no weights -> the freshly built (untrained) model for this alphabet
            tensors = weights_mod.synthetic_crnn_weights(seed=0, alphabet=self.alphabet, stn=self.stn, color=self.color,
                                                         height=self.height, width=self.width)
        elif isinstance(weights, str) and weights.endswith(".npz"):
            tensors = weights_mod.load_npz(weights)
        elif isinstance(weights, str) and weights.endswith(".h5"):
            tensors = weights_mod.load_keras_h5(weights)
        elif weights == "kurapan":                                # recognition.py:27-44: cache file, sha256-verified
            import os
            cache = tools.get_default_cache_dir()
            if os.path.isfile(os.path.join(cache, "crnn_kurapan.npz")):
                tensors = weights_mod.load_npz(os.path.join(cache, "crnn_kurapan.npz"))
            else:
                tensors = weights_mod.load_keras_h5(tools.find_cached(
                    "crnn_kurapan.h5", sha256="a7d8086ac8f5c3d6a0a828f7d6fbabcaf815415dd125c32533013f85603be46d"))
        else:
            raise NotImplementedError(f"Cannot load weights from {weights}")
        has_stn = "stn.conv_a.kernel" in tensors
        if has_stn and not self.stn:                              # stn=False with a checkpoint that has one: drop it
            tensors = {k: v for k, v in tensors.items() if not k.startswith("stn.")}
        elif self.stn and not has_stn:
            raise ValueError("the checkpoint has no spatial-transformer tensors: pass build_params={'stn': False}")
        self._check_checkpoint_geometry(tensors)
        in_ch = int(np.shape(tensors["conv_1.kernel"])[2]) if "conv_1.kernel" in tensors else 1
        if in_ch != (3 if self.color else 1):
            raise ValueError(f"conv_1.kernel takes {in_ch} input channel(s): pass build_params={{'color': {in_ch == 3}}}")
        n_classes = len(self.alphabet) + 1
        top = tensors.get("fc_12.kernel")
        if top is None or tuple(np.shape(top)) != (256, n_classes):
            print("Provided alphabet does not match pretrained alphabet. Using backbone weights only.")
            tensors = dict(tensors)
            limit = float(np.sqrt(6.0 / (256 + n_classes)))           # keras Dense default: glorot_uniform, zeros
            tensors["fc_12.kernel"] = np.random.default_rng(0).uniform(-limit, limit, (256, n_classes)).astype(np.float32)
            tensors["fc_12.bias"] = np.zeros(n_classes, np.float32)
        self.ctx = _lib.Context(self.device_index)
        self.ctx.set_crnn_geometry(self.height, self.width, self.rnn_steps_to_discard)
        self.ctx.load_crnn(tensors)
        self._keep_workspace = False     # tests set keep_workspace to read intermediate taps
        self._last_ws = None
        self._ws = None                  # reusable CRNN workspace (grown on demand)

    def _check_geometry(self):
        """The crop size and discarded steps the kernels support (include/b2ocr.h, b2o_set_crnn_geometry)."""
        (h_lo, h_hi), (w_lo, w_hi) = _lib.CRNN_HEIGHTS, _lib.CRNN_WIDTHS
        for key, value in (("height", self.height), ("width", self.width), ("rnn_steps_to_discard", self.rnn_steps_to_discard)):
            if isinstance(value, bool) or not isinstance(value, (int, np.integer)):
                raise ValueError(f"build_params[{key!r}] must be an integer, got {value!r}")
        self.height, self.width, self.rnn_steps_to_discard = int(self.height), int(self.width), int(self.rnn_steps_to_discard)
        if not h_lo <= self.height <= h_hi or not w_lo <= self.width <= w_hi:
            raise ValueError(f"crops of {self.height} x {self.width} are not supported: height {h_lo}..{h_hi}, width {w_lo}..{w_hi}")
        if not 0 <= self.rnn_steps_to_discard < self.width // 4:
            raise ValueError(f"rnn_steps_to_discard={self.rnn_steps_to_discard} must be in 0..{self.width // 4 - 1}: "
                             f"crops {self.width} wide give {self.width // 4} time steps")

    def _check_checkpoint_geometry(self, tensors):
        """fc_9 reads height // 4 * 512 features per step and stn.dense_a the flattened (width // 4, height // 4, 32)
        localisation map (recognition.py:275, 282): a checkpoint built for another crop size does not fit."""
        feat_h, t = self.height // 4, self.width // 4
        fc9 = tensors.get("fc_9.kernel")
        if fc9 is not None and int(np.shape(fc9)[0]) != feat_h * 512:
            rows = int(np.shape(fc9)[0])
            hint = (f"pass build_params with a 'height' in {4 * (rows // 512)}..{4 * (rows // 512) + 3}" if rows % 512 == 0
                    else "no crop height fits it")
            raise ValueError(f"fc_9.kernel has {rows} rows but crops {self.height} high need {feat_h * 512}: {hint}")
        dense = tensors.get("stn.dense_a.kernel") if self.stn else None
        if dense is not None and int(np.shape(dense)[0]) != t * feat_h * 32:
            rows = int(np.shape(dense)[0])
            hint = (f"pass build_params with a 'width' in {4 * (rows // (feat_h * 32))}..{4 * (rows // (feat_h * 32)) + 3}"
                    if rows % (feat_h * 32) == 0 else "no crop width fits it")
            raise ValueError(f"stn.dense_a.kernel has {rows} rows but {self.height} x {self.width} crops need "
                             f"{t * feat_h * 32}: {hint}")

    @property
    def keep_workspace(self):
        return self._keep_workspace

    @keep_workspace.setter
    def keep_workspace(self, on):
        """Debug: keep the last forward pass's workspace for ``tap`` and make the CRNN write its fp32 logits
        (off on the product path: the fused Dense + CTC kernel then stores labels only)."""
        self._keep_workspace = bool(on)
        self.ctx.set_debug_taps(self._keep_workspace)

    # ------------------------------------------------------------------ device-resident API
    def gray_device(self, images_t):
        n, h, w, _ = images_t.shape
        gray = torch.empty((n, h, w), dtype=torch.uint8, device=self.device)
        self.ctx.rgb_to_gray(images_t.data_ptr(), n, h, w, gray.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        return gray

    def warp_device(self, gray, boxes_flat, image_index, want_crops=False):
        """tools.warpBox for every box.  ``gray``: (N,H,W) u8 -- or the RGB batch (N,H,W,3) for a color recognizer.
        Returns (crnn_in (B,width,height[,3]) fp16, crops (B,height,width[,3]) u8 or None); 200 x 31 by default."""
        n, h, w = gray.shape[:3]
        color = gray.dim() == 4
        assert color == self.color, "a color recognizer warps the RGB batch, a gray one the gray batch"
        tail = (3,) if color else ()
        b = boxes_flat.shape[0]
        crnn_in = torch.empty((b, self.width, self.height) + tail, dtype=torch.float16, device=self.device)
        crops = torch.empty((b, self.height, self.width) + tail, dtype=torch.uint8, device=self.device) if want_crops else None
        self.ctx.warp_boxes(gray.data_ptr(), n, h, w, boxes_flat.data_ptr(), image_index.data_ptr(), b,
                            crops.data_ptr() if want_crops else None, crnn_in.data_ptr(),
                            torch.cuda.current_stream(self.device).cuda_stream, color=color)
        return crnn_in, crops

    def _fit_dims(self, shape):
        """(sh, sw, rh, rw) of one (H,W,3) crop for b2o_fit_crops; raises what tools.fit raises for it."""
        if len(shape) != 3 or shape[2] != 3:
            raise ValueError(f"crops must be (H, W, 3) uint8 RGB, got shape {tuple(shape)}")
        h, w = int(shape[0]), int(shape[1])
        return (h, w) + (tools.fit_plan(shape, self.width, self.height) or (h, w))

    def _fit_table(self, srcs_dev, dims_dev, b, want_crops):
        """b2o_fit_crops on the current stream: crop pointers and dims already on the device."""
        tail = (3,) if self.color else ()
        crnn_in = torch.empty((b, self.width, self.height) + tail, dtype=torch.float16, device=self.device)
        crops = torch.empty((b, self.height, self.width, 3), dtype=torch.uint8, device=self.device) if want_crops else None
        self.ctx.fit_crops(srcs_dev, dims_dev, b, crops.data_ptr() if want_crops else None, crnn_in.data_ptr(),
                           torch.cuda.current_stream(self.device).cuda_stream)
        return crnn_in, crops

    def fit_device(self, sources, want_crops=False):
        """tools.fit(cval=0) + the gray conversion of ``recognize`` for crops already on the GPU, in one launch.
        ``sources``: a list of (H,W,3) uint8 CUDA tensors of any sizes, read in place.  Returns (crnn_in
        (B,width,height[,3]) fp16, crops (B,height,width,3) u8 -- what tools.fit returns -- or None)."""
        for s in sources:
            if not (isinstance(s, torch.Tensor) and s.is_cuda and s.dtype == torch.uint8 and s.device == self.device):
                raise ValueError(f"fit_device takes uint8 CUDA tensors on {self.device}")
        sources = [s.contiguous() for s in sources]
        b = len(sources)
        table = np.zeros(b * 8 + b * 16, dtype=np.uint8)
        table[: b * 8].view(np.uint64)[:] = [s.data_ptr() for s in sources]
        table[b * 8:].view(np.int32)[:] = np.array([self._fit_dims(s.shape) for s in sources], np.int32).reshape(-1)
        if b == 0:
            return self._fit_table(None, None, 0, want_crops)
        table_dev = torch.from_numpy(table).to(self.device)
        return self._fit_table(table_dev.data_ptr(), table_dev.data_ptr() + b * 8, b, want_crops)

    def predict_device(self, crnn_in):
        """CRNN + greedy CTC.  crnn_in: (B,width,height) fp16 -> labels (B,steps) int32 (-1 padded); (B,200,31) -> (B,48)
        by default."""
        b = crnn_in.shape[0]
        labels = torch.empty((b, self.steps), dtype=torch.int32, device=self.device)
        nbytes = self.ctx.crnn_workspace_bytes(b)
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        ws = self._ws
        self.ctx.crnn_forward(crnn_in.data_ptr(), b, labels.data_ptr(), ws.data_ptr(), nbytes,
                              torch.cuda.current_stream(self.device).cuda_stream)
        self._last_ws = (ws, b) if self.keep_workspace else None
        return labels

    def tap(self, name, shape, dtype):
        """Debug: copy an intermediate of the last predict_device call (needs keep_workspace=True)."""
        ws, b = self._last_ws
        out = torch.empty(shape, dtype=dtype, device=self.device)
        self.ctx.crnn_tap(name, ws.data_ptr(), b, out.data_ptr(), out.numel() * out.element_size(),
                          torch.cuda.current_stream(self.device).cuda_stream)
        return out

    def recognize_crops(self, crops):
        """crops: (B,height,width) uint8 -- (B,height,width,3) for a color recognizer -- i.e. what tools.warpBox returns at
        the model's crop size (31 x 200 by default) -> list[str]."""
        t = crops if isinstance(crops, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(crops))
        t = t.to(self.device).contiguous()
        b = t.shape[0]
        if b == 0:
            return []
        tail = (3,) if self.color else ()
        assert t.shape[1:] == (self.height, self.width) + tail, f"crops must be (B,{self.height},{self.width}{',3' if tail else ''})"
        crnn_in = torch.empty((b, self.width, self.height) + tail, dtype=torch.float16, device=self.device)
        self.ctx.crops_to_input(t.data_ptr(), b, crnn_in.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream,
                                color=self.color)
        return labels_to_text(self.predict_device(crnn_in).cpu().numpy(), self.alphabet)

    def recognize(self, image):
        """Recognize text from a single pre-cropped image (reference recognition.py:467-489): fit to the model's
        width x height (200 x 31 by default) with zero fill (host, as upstream), gray conversion, then the CUDA CRNN."""
        import cv2

        image = tools.read_and_fit(filepath_or_array=image, width=self.width, height=self.height, cval=0)
        if not self.color and image.ndim == 3 and image.shape[-1] == 3:      # recognition.py:481-483
            image = cv2.cvtColor(image, code=cv2.COLOR_RGB2GRAY)
        return self.recognize_crops(np.ascontiguousarray(image.reshape((1, self.height, self.width) + ((3,) if self.color else ()))))[0]

    def recognize_batch(self, images, chunk=1024) -> typing.List[str]:
        """``[self.recognize(image) for image in images]`` for many pre-cropped images of any sizes, with the fit and
        the gray conversion on the GPU (``b2o_fit_crops``) and the CRNN run over ``chunk`` crops at a time.

        ``images``: a list of (H,W,3) uint8 RGB arrays, image paths (read with tools.read like ``recognize``) or
        (H,W,3) uint8 CUDA tensors (read in place, no copy), or one (N,H,W,3) uint8 array of equally sized crops.
        Host crops of a chunk are packed into a pinned staging buffer and sent with one host-to-device copy on a
        side stream; two buffers alternate, so chunk k+1 is read, packed and copied while chunk k runs, and the
        labels of chunk k are decoded once chunk k+1 is queued.  ``chunk`` bounds the CRNN workspace (about 9.5 MB
        per crop at 31 x 200).  A crop tools.fit cannot fit raises what ``recognize`` raises (ZeroDivisionError,
        cv2.error) before its chunk is queued; crops given as arrays or tensors are all checked before any work."""
        if isinstance(images, np.ndarray) and images.ndim != 4:
            raise ValueError("an array of crops must be (N, H, W, 3) uint8")
        if isinstance(chunk, bool) or not isinstance(chunk, (int, np.integer)) or chunk < 1:
            raise ValueError(f"chunk must be a positive integer, got {chunk!r}")
        n = len(images)
        if n == 0:
            return []
        if isinstance(images, np.ndarray):
            self._check_host_crop(images[0])
            dims = [self._fit_dims(images.shape[1:])] * n
        else:
            images = list(images)
            dims = [None if isinstance(im, str) else self._fit_dims(self._check_device_crop(im).shape) for im in images]
        stream = torch.cuda.current_stream(self.device)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self.device)
            self._staging = [{"host": None, "dev": None, "labels": None, "copied": None, "fitted": None} for _ in range(2)]
        out, pending = [], None
        for k, start in enumerate(range(0, n, chunk)):
            slot = self._staging[k % 2]
            b = min(chunk, n - start)
            crops = [self._check_device_crop(tools.read(c) if isinstance(c, str) else c) for c in images[start:start + b]]
            cdims = [d if d is not None else self._fit_dims(c.shape) for c, d in zip(crops, dims[start:start + b])]
            head = b * 24
            offsets, nbytes = [], (head + 15) // 16 * 16
            for c in crops:
                offsets.append(None if isinstance(c, torch.Tensor) and c.is_cuda else nbytes)
                if offsets[-1] is not None:
                    nbytes += c.shape[0] * c.shape[1] * 3
            if slot["copied"] is not None:
                slot["copied"].synchronize()                  # chunk k-2's copy out of this host buffer is done
            if slot["host"] is None or slot["host"].numel() < nbytes:
                size = max(nbytes, nbytes * 5 // 4)
                slot["host"] = torch.empty(size, dtype=torch.uint8, pin_memory=True)
                with torch.cuda.stream(stream):
                    slot["dev"] = torch.empty(size, dtype=torch.uint8, device=self.device)
                slot["dev"].record_stream(self._copy_stream)
                self._copy_stream.wait_stream(stream)         # the new block may still be in use by queued kernels
            host = slot["host"].numpy()
            base = slot["dev"].data_ptr()
            ptrs = host[: b * 8].view(np.uint64)
            for i, (c, off) in enumerate(zip(crops, offsets)):
                if off is None:
                    c = c.contiguous()
                    crops[i] = c                              # keep a contiguous copy alive until the launch
                    ptrs[i] = c.data_ptr()
                else:
                    host[off:off + c.size].reshape(c.shape)[...] = c
                    ptrs[i] = base + off
            host[b * 8:head].view(np.int32)[:] = np.asarray(cdims, np.int32).reshape(-1)
            with torch.cuda.stream(self._copy_stream):
                if slot["fitted"] is not None:
                    self._copy_stream.wait_event(slot["fitted"])   # chunk k-2 has read this device buffer
                slot["dev"][:nbytes].copy_(slot["host"][:nbytes], non_blocking=True)
                slot["copied"] = torch.cuda.Event()
                slot["copied"].record(self._copy_stream)
            stream.wait_event(slot["copied"])
            with torch.cuda.stream(stream):
                crnn_in, _ = self._fit_table(base, base + b * 8, b, False)
                slot["fitted"] = torch.cuda.Event()
                slot["fitted"].record(stream)
                labels = self.predict_device(crnn_in)
                if slot["labels"] is None or slot["labels"].shape[0] < b:
                    slot["labels"] = torch.empty((max(b, chunk), self.steps), dtype=torch.int32, pin_memory=True)
                host_labels = slot["labels"][:b]
                host_labels.copy_(labels, non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(stream)
            if pending is not None:
                out.extend(self._decode(*pending))
            pending = (ready, host_labels)
        out.extend(self._decode(*pending))
        return out

    def _decode(self, ready, host_labels):
        ready.synchronize()
        return labels_to_text(host_labels.numpy(), self.alphabet)

    @staticmethod
    def _check_host_crop(image):
        """A crop recognize_batch accepts: a (H,W,3) uint8 ndarray or tensor; CPU tensors come back as arrays."""
        if isinstance(image, torch.Tensor):
            ok = image.dtype == torch.uint8
            image = image if image.is_cuda else image.numpy()
        else:
            ok = isinstance(image, np.ndarray) and image.dtype == np.uint8
        if not ok or image.ndim != 3 or image.shape[2] != 3:
            raise ValueError("recognize_batch takes (H, W, 3) uint8 RGB crops, paths or CUDA tensors")
        return image

    def _check_device_crop(self, image):
        if isinstance(image, torch.Tensor) and image.is_cuda and image.device != self.device:
            raise ValueError(f"CUDA crops must be on {self.device}, got {image.device}")
        return self._check_host_crop(image)

    def recognize_from_boxes_device(self, images_t, boxes, counts, gray=None, flat=None, image_index=None):
        """images_t (N,H,W,3) u8 CUDA; boxes (N,M,4,2) f32 CUDA; counts host ndarray -> labels (B,steps) i32 CUDA.

        Optional device-side by-products of the earlier stages, so that nothing but the kernel launches is
        left to do once the host knows the counts: ``gray`` (N,H,W) u8 from ``b2o_resize_pad_batch``;
        ``flat`` (>=B,4,2) / ``image_index`` (>=B,) from ``b2o_compact_boxes``."""
        counts = np.asarray(counts)
        m = boxes.shape[1]
        total = int(np.minimum(counts, m).sum())
        if total == 0:
            return None
        if self.color:
            gray = images_t                                       # color recognizer: crops come straight from the RGB batch
        elif gray is None:
            gray = self.gray_device(images_t)
        if flat is None or image_index is None:
            n = len(counts)
            flat = torch.empty((n * m, 4, 2), dtype=torch.float32, device=self.device)
            image_index = torch.empty((n * m,), dtype=torch.int32, device=self.device)
            counts_dev = torch.from_numpy(counts.astype(np.int32)).to(self.device)
            self.ctx.compact_boxes(boxes.data_ptr(), counts_dev.data_ptr(), n, m, flat.data_ptr(),
                                   image_index.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        crnn_in, _ = self.warp_device(gray, flat[:total], image_index[:total])
        return self.predict_device(crnn_in)

    # ------------------------------------------------------------------ reference API
    def recognize_from_boxes(self, images, box_groups, **kwargs) -> typing.List[typing.List[str]]:
        """Same contract as reference recognition.py:491-537."""
        assert len(box_groups) == len(images), "You must provide the same number of box groups as images."
        from .detection import _as_device_images

        images_t = _as_device_images(images, self.device)
        counts = np.array([len(b) for b in box_groups], dtype=np.int64)
        if counts.sum() == 0:
            return [[]] * len(images)
        flat = np.concatenate([np.asarray(b, dtype=np.float32).reshape(-1, 4, 2) for b in box_groups if len(b)])
        # caller-supplied quads: tools.warpBox first replaces each by its minimum rotated rectangle and divides by its
        # truncated width / height (tools.py:88-95; ZeroDivisionError for a degenerate box).  Rectangles -- everything
        # a Detector returns -- pass through bit for bit.
        flat = tools.rectify_boxes(flat)
        flat_t = torch.from_numpy(np.ascontiguousarray(flat)).to(self.device)
        idx = torch.from_numpy(np.repeat(np.arange(len(counts), dtype=np.int32), counts)).to(self.device)
        crnn_in, _ = self.warp_device(images_t if self.color else self.gray_device(images_t), flat_t, idx)
        predictions = labels_to_text(self.predict_device(crnn_in).cpu().numpy(), self.alphabet)
        ends = np.cumsum(counts)
        return [predictions[int(e - c):int(e)] for c, e in zip(counts, ends)]
