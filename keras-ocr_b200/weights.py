"""Weight dictionaries for the CRAFT detector and the CRNN recognizer.

The product consumes weights in the reference's own naming so that the real
checkpoints drop in unchanged:

* CRAFT  -- the PyTorch state-dict keys of ``craft_mlt_25k.pth`` after the ``module.``
  prefix is stripped (reference keras_ocr/detection.py:428-468 maps exactly these names
  onto the Keras layers): ``<conv>.weight`` (O,I,kh,kw), ``<conv>.bias``,
  ``<bn>.{weight,bias,running_mean,running_var}``.
* CRNN   -- Keras layer names of ``build_model`` (reference recognition.py:214-329) with
  Keras layouts: ``conv_N.kernel`` (kh,kw,I,O), ``bn_N.{gamma,beta,moving_mean,moving_variance}``,
  ``lstm_N.{kernel,recurrent_kernel,bias}``, ``fc_N.{kernel,bias}``; the auto-named
  localisation net is exposed as ``stn.conv_a / stn.conv_b / stn.dense_a / stn.dense_b``.

No pretrained files exist offline, so ``synthetic_*`` build seeded weights with realistic
statistics (He-scaled kernels, batch-norm statistics moved away from (0,1) so that folding
mistakes show up in the parity tests).
"""
import numpy as np

# name, cin, cout, kernel, dilation, batch-norm name (or None), relu after
CRAFT_CONVS = [
    ("basenet.slice1.0", 3, 64, 3, 1, "basenet.slice1.1", True),
    ("basenet.slice1.3", 64, 64, 3, 1, "basenet.slice1.4", True),
    ("basenet.slice1.7", 64, 128, 3, 1, "basenet.slice1.8", True),
    ("basenet.slice1.10", 128, 128, 3, 1, "basenet.slice1.11", True),
    ("basenet.slice2.14", 128, 256, 3, 1, "basenet.slice2.15", True),
    ("basenet.slice2.17", 256, 256, 3, 1, "basenet.slice2.18", True),
    ("basenet.slice3.20", 256, 256, 3, 1, "basenet.slice3.21", True),
    ("basenet.slice3.24", 256, 512, 3, 1, "basenet.slice3.25", True),
    ("basenet.slice3.27", 512, 512, 3, 1, "basenet.slice3.28", True),
    ("basenet.slice4.30", 512, 512, 3, 1, "basenet.slice4.31", True),
    ("basenet.slice4.34", 512, 512, 3, 1, "basenet.slice4.35", True),
    ("basenet.slice4.37", 512, 512, 3, 1, "basenet.slice4.38", False),
    ("basenet.slice5.1", 512, 1024, 3, 6, None, False),
    ("basenet.slice5.2", 1024, 1024, 1, 1, None, False),
    ("upconv1.conv.0", 1536, 512, 1, 1, "upconv1.conv.1", True),
    ("upconv1.conv.3", 512, 256, 3, 1, "upconv1.conv.4", True),
    ("upconv2.conv.0", 768, 256, 1, 1, "upconv2.conv.1", True),
    ("upconv2.conv.3", 256, 128, 3, 1, "upconv2.conv.4", True),
    ("upconv3.conv.0", 384, 128, 1, 1, "upconv3.conv.1", True),
    ("upconv3.conv.3", 128, 64, 3, 1, "upconv3.conv.4", True),
    ("upconv4.conv.0", 192, 64, 1, 1, "upconv4.conv.1", True),
    ("upconv4.conv.3", 64, 32, 3, 1, "upconv4.conv.4", True),
    ("conv_cls.0", 32, 32, 3, 1, None, True),
    ("conv_cls.2", 32, 32, 3, 1, None, True),
    ("conv_cls.4", 32, 16, 3, 1, None, True),
    ("conv_cls.6", 16, 16, 1, 1, None, True),
    ("conv_cls.8", 16, 2, 1, 1, None, False),
]

CRAFT_MAC_PER_PIXEL = 355720          # SURVEY.md 8(a): MAC per detector-input pixel
CRAFT_FLOP_PER_PIXEL = 2 * CRAFT_MAC_PER_PIXEL
CRNN_FLOP_PER_CROP = 13.444e9         # SURVEY.md 8(d)

# name, cin, cout, kernel, batch-norm after the ReLU (or None)
CRNN_CONVS = [
    ("conv_1", 1, 64, 3, None),
    ("conv_2", 64, 128, 3, None),
    ("conv_3", 128, 256, 3, "bn_3"),
    ("conv_4", 256, 256, 3, None),
    ("conv_5", 256, 512, 3, "bn_5"),
    ("conv_6", 512, 512, 3, None),
    ("conv_7", 512, 512, 3, "bn_7"),
]
CRNN_LSTMS = ["lstm_10", "lstm_10_back", "lstm_11", "lstm_11_back"]
ALPHABET = "0123456789abcdefghijklmnopqrstuvwxyz"     # reference recognition.py:25


def _he(rng, shape, fan_in, gain=2.0):
    return (rng.standard_normal(shape) * np.sqrt(gain / fan_in)).astype(np.float32)


# "textlike" routing: channel 0 carries a fine "ink" signal (strokes), channel 1 a coarse one (whole
# words) through the layers listed here; see synthetic_craft_weights(textlike=True).
_FINE = ["basenet.slice1.3", "basenet.slice1.7", "basenet.slice1.10"]
_COARSE = ["basenet.slice2.14", "basenet.slice2.17", "basenet.slice3.20", "basenet.slice3.24", "basenet.slice3.27"]
TEXTLIKE_HEAD = {"text_gain": 0.5, "text_bias": 0.0, "link_gain": 2.0, "link_bias": 0.0}   # calibrated on cv2.putText pages


def _route(w, name, bn, out_ch, in_ch, mode, gain=1.0, bias=0.0):
    """Make output channel ``out_ch`` of conv ``name`` depend only on input channel ``in_ch``:
    mode "blur" = 3x3 box filter, "id" = centre tap (or the single tap of a 1x1)."""
    k = w[name + ".weight"]
    k[out_ch] = 0.0
    if mode == "blur":
        k[out_ch, in_ch] = gain / (k.shape[2] * k.shape[3])
    else:
        k[out_ch, in_ch, k.shape[2] // 2, k.shape[3] // 2] = gain
    w[name + ".bias"][out_ch] = bias
    if bn is not None:
        w[bn + ".weight"][out_ch] = 1.0
        w[bn + ".bias"][out_ch] = 0.0
        w[bn + ".running_mean"][out_ch] = 0.0
        w[bn + ".running_var"][out_ch] = 1.0


def synthetic_craft_weights(seed=0, textlike=False):
    """Seeded CRAFT weights keyed like the reference's ``.pth`` (prefix stripped).

    ``textlike=True`` overwrites two channels per layer so that, on dark-text-on-light pages, the
    network output is a usable (text, link) pair: text = blurred ink at half resolution, link = a
    coarse blob per word routed through the H/8 tap and the decoder.  Every other channel keeps
    its random weights (the arithmetic cost is unchanged); the point is that ``getBoxes`` and the
    recognizer see realistic word boxes although no pretrained checkpoint exists offline.
    """
    rng = np.random.default_rng(seed)
    w = {}
    for name, cin, cout, k, _dil, bn, relu in CRAFT_CONVS:
        gain = 2.0 if relu else 1.0
        w[name + ".weight"] = _he(rng, (cout, cin, k, k), cin * k * k, gain)
        w[name + ".bias"] = (rng.standard_normal(cout) * 0.05).astype(np.float32)
        if bn is not None:
            w[bn + ".weight"] = rng.uniform(0.8, 1.2, cout).astype(np.float32)
            w[bn + ".bias"] = (rng.standard_normal(cout) * 0.1).astype(np.float32)
            w[bn + ".running_mean"] = (rng.standard_normal(cout) * 0.1).astype(np.float32)
            w[bn + ".running_var"] = rng.uniform(0.8, 1.25, cout).astype(np.float32)
    if textlike:
        bn_of = {name: bn for name, _ci, _co, _k, _d, bn, _r in CRAFT_CONVS}
        # ink = relu(1 - mean(normalised RGB)): 0 on white, ~2.3 on dark strokes
        k = w["basenet.slice1.0.weight"]
        k[0] = 0.0
        k[0, :, 1, 1] = -1.0 / 3.0
        w["basenet.slice1.0.bias"][0] = 1.0
        for key, val in ((".weight", 1.0), (".bias", 0.0), (".running_mean", 0.0), (".running_var", 1.0)):
            w["basenet.slice1.1" + key][0] = val
        for name in _FINE + _COARSE:
            _route(w, name, bn_of[name], 0, 0, "blur")
        _route(w, "upconv2.conv.0", "upconv2.conv.1", 1, 256, "id")       # concat [y1(256), s3(512)] -> s3 ch0
        _route(w, "upconv2.conv.3", "upconv2.conv.4", 1, 1, "blur")
        _route(w, "upconv3.conv.0", "upconv3.conv.1", 1, 1, "id")         # concat [y2(128), s2(256)] -> y2 ch1
        _route(w, "upconv3.conv.3", "upconv3.conv.4", 1, 1, "blur")
        _route(w, "upconv4.conv.0", "upconv4.conv.1", 0, 64, "id")        # concat [y3(64), s1(128)] -> s1 ch0
        _route(w, "upconv4.conv.0", "upconv4.conv.1", 1, 1, "id")         #                          -> y3 ch1
        _route(w, "upconv4.conv.3", "upconv4.conv.4", 0, 0, "id")
        _route(w, "upconv4.conv.3", "upconv4.conv.4", 1, 1, "blur")
        for name in ("conv_cls.0", "conv_cls.2", "conv_cls.4", "conv_cls.6"):
            _route(w, name, None, 0, 0, "id")
            _route(w, name, None, 1, 1, "id")
        h = TEXTLIKE_HEAD
        _route(w, "conv_cls.8", None, 0, 0, "id", h["text_gain"], h["text_bias"])
        _route(w, "conv_cls.8", None, 1, 1, "id", h["link_gain"], h["link_bias"])
    return w


HERSHEY = "crnn_hershey.npz"                # keras-ocr_b200/data/: the reference CRNN trained on rendered words (see below)


def synthetic_crnn_weights(seed=1, alphabet=ALPHABET, decisive=False, stn=True, color=False, height=31, width=200):
    """Seeded CRNN weights keyed by Keras layer name (Keras layouts); the top layer has len(alphabet)+1 classes.

    ``color=True``: ``conv_1`` takes 3 input channels (``build_model(color=True)``, recognition.py:214).
    ``stn=False``: no spatial-transformer tensors (the ``build_model(stn=False)`` variant, recognition.py:196, 243).
    ``height`` / ``width``: the crop size of ``build_model(height, width)``; it sets the input widths of ``fc_9``
    (``height // 4 * 512``) and ``stn.dense_a`` (``width // 4 * height // 4 * 32``).  The defaults give 31 x 200.
    ``decisive=True`` (default alphabet, gray, with STN; ``seed`` is ignored): every tensor comes from
    ``data/crnn_hershey.npz`` -- the reference architecture TRAINED with CTC loss on words rendered in cv2's Hershey font
    and cut out as the oracle pipeline cuts them (``oracle/train_crnn_full.py``; 3.5 minutes on one B200; no pretrained file
    involved).  It reads the synthetic pages (99.7 % of unseen synthetic crops, 100 % of the crops of pages it never saw), its
    per-step argmax is decided by a wide margin and its strings do not change when a box moves by a pixel, so decoded
    strings can be compared for identity (BASELINE.json north_star) instead of up to the near-ties random weights leave."""
    if decisive:
        import os
        assert alphabet == ALPHABET and stn and not color and (height, width) == (31, 200), \
            "the trained recognizer is the default architecture / alphabet"
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", HERSHEY)
        with np.load(path) as data:
            return {k: data[k].astype(np.float32) for k in data.files}
    rng = np.random.default_rng(seed)
    steps, feat_h = width // 4, height // 4          # both 2x2 max pools floor (recognition.py:227, 235)
    w = {}
    for name, cin, cout, k, bn in CRNN_CONVS:
        w[name + ".kernel"] = _he(rng, (k, k, cin, cout), cin * k * k)
        w[name + ".bias"] = (rng.standard_normal(cout) * 0.05).astype(np.float32)
        if bn is not None:
            w[bn + ".gamma"] = rng.uniform(0.8, 1.2, cout).astype(np.float32)
            w[bn + ".beta"] = (rng.standard_normal(cout) * 0.1).astype(np.float32)
            w[bn + ".moving_mean"] = (rng.uniform(0.2, 0.6, cout)).astype(np.float32)
            w[bn + ".moving_variance"] = rng.uniform(0.5, 1.2, cout).astype(np.float32)
    w["stn.conv_a.kernel"] = _he(rng, (5, 5, 512, 16), 512 * 25)
    w["stn.conv_a.bias"] = (rng.standard_normal(16) * 0.05).astype(np.float32)
    w["stn.conv_b.kernel"] = _he(rng, (5, 5, 16, 32), 16 * 25)
    w["stn.conv_b.bias"] = (rng.standard_normal(32) * 0.05).astype(np.float32)
    w["stn.dense_a.kernel"] = _he(rng, (steps * feat_h * 32, 64), steps * feat_h * 32)
    w["stn.dense_a.bias"] = (rng.standard_normal(64) * 0.05).astype(np.float32)
    # a trained STN sits near the identity transform [[1,0,0],[0,1,0]] with small deviations
    w["stn.dense_b.kernel"] = (rng.standard_normal((64, 6)) * 0.01).astype(np.float32)
    w["stn.dense_b.bias"] = (np.array([1, 0, 0, 0, 1, 0]) + rng.standard_normal(6) * 0.02).astype(np.float32)
    w["fc_9.kernel"] = _he(rng, (feat_h * 512, 128), feat_h * 512)
    w["fc_9.bias"] = (rng.standard_normal(128) * 0.05).astype(np.float32)
    for name in CRNN_LSTMS:
        w[name + ".kernel"] = _he(rng, (128, 512), 128, 1.0)
        w[name + ".recurrent_kernel"] = _he(rng, (128, 512), 128, 1.0)
        b = (rng.standard_normal(512) * 0.05).astype(np.float32)
        b[128:256] += 1.0                                   # unit_forget_bias
        w[name + ".bias"] = b
    w["fc_12.kernel"] = _he(rng, (256, len(alphabet) + 1), 256, 8.0)
    w["fc_12.bias"] = (rng.standard_normal(len(alphabet) + 1) * 0.1).astype(np.float32)
    if color:                                       # build_model(color=True): conv_1 over RGB crops (own stream: the rest is unchanged)
        w["conv_1.kernel"] = _he(np.random.default_rng(seed + 7919), (3, 3, 3, 64), 27)
    if not stn:                                     # build_model(stn=False): the same model without the localisation net
        w = {k: v for k, v in w.items() if not k.startswith("stn.")}
    return w


def load_craft_pth(path):
    """Read the reference's ``craft_mlt_25k.pth`` (sha256 in detection.py:647-652)."""
    import torch

    state = torch.load(path, map_location="cpu")
    out = {}
    for key, value in state.items():
        if key.endswith("num_batches_tracked"):
            continue
        name = key[len("module."):] if key.startswith("module.") else key
        out[name] = value.detach().cpu().numpy().astype(np.float32)
    return out


def load_npz(path):
    """Weights exported to a flat ``.npz`` with the key names documented above."""
    with np.load(path) as data:
        return {k: data[k].astype(np.float32) for k in data.files}


# --------------------------------------------------------------------------------------- Keras HDF5
_CRNN_NAMED = ({f"conv_{i}" for i in range(1, 8)} | {"bn_3", "bn_5", "bn_7", "fc_9", "fc_12"} | set(CRNN_LSTMS))
_KINDS = ("kernel", "recurrent_kernel", "bias", "gamma", "beta", "moving_mean", "moving_variance")
_STN_BY_SHAPE = {(5, 5, 512, 16): "stn.conv_a.kernel", (5, 5, 16, 32): "stn.conv_b.kernel",
                 (11200, 64): "stn.dense_a.kernel", (64, 6): "stn.dense_b.kernel",
                 (16,): "stn.conv_a.bias", (32,): "stn.conv_b.bias", (64,): "stn.dense_a.bias", (6,): "stn.dense_b.bias"}


def map_keras_datasets(flat):
    """Keras (TF2 ``save_weights`` HDF5) dataset paths -> the keys of this module.

    ``flat`` maps a dataset path such as ``conv_3/conv_3/kernel:0`` or ``lstm_10/lstm_10/lstm_cell/bias:0`` to its
    array.  Named layers of ``build_model`` (reference recognition.py:214-329) map by name; the nested localisation
    model of the spatial transformer is auto-named by Keras (``model_N/conv2d_M/...``, recognition.py:263-277), so its
    eight tensors are told apart by their shapes, which are all distinct (``dense_a``'s kernel by its 64 columns: its
    row count depends on the crop size)."""
    out = {}
    for path, arr in flat.items():
        parts = [q for q in path.split("/") if q]
        kind = parts[-1].split(":")[0]
        if kind not in _KINDS:
            continue
        arr = np.asarray(arr, dtype=np.float32)
        if parts[0] in _CRNN_NAMED:
            key = f"{parts[0]}.{kind}"
        else:
            key = _STN_BY_SHAPE.get(tuple(arr.shape))
            if key is None and kind == "kernel" and arr.ndim == 2 and arr.shape[1] == 64:
                key = "stn.dense_a.kernel"          # Flatten of the (T, Hf, 32) map: rows follow the crop size (build_model height / width)
            if key is None or not key.endswith(kind):
                raise ValueError(f"unrecognised tensor {path} with shape {arr.shape} in Keras weight file")
        if key in out:
            raise ValueError(f"two tensors map to {key} (second: {path})")
        out[key] = arr
    return out


def load_keras_h5(path):
    """Read the reference's ``crnn_kurapan.h5`` / ``crnn_kurapan_notop.h5`` (recognition.py:27-44; loaded there by
    ``model.load_weights``, 386-392) with this package's own HDF5 reader (``hdf5.py``; no h5py needed).  Both Keras
    layouts are accepted: ``save_weights`` (layer groups at the root) and ``model.save`` (under ``model_weights``)."""
    from . import hdf5

    flat = hdf5.read_datasets(path)
    if any(k.startswith("model_weights/") for k in flat):
        flat = {k[len("model_weights/"):]: v for k, v in flat.items() if k.startswith("model_weights/")}
    return map_keras_datasets(flat)
