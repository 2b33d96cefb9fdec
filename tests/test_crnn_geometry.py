"""CPU: recognizers built with another crop size (build_params height / width / rnn_steps_to_discard, reference
recognition.py:13-23, 214, 328) -- the oracle against the reference-source fixture, the synthetic weights' shapes, the
record layout of other label lengths and the argument checks of Recognizer that run before the device check."""
import os

import numpy as np
import pytest
import torch

from keras_ocr_b200 import distributed as D, weights as W
from keras_ocr_b200.recognition import Recognizer

GEOMETRIES = ("A", "B", "C")


def _geometry(g, tag):
    h, w, d, stn, color = (int(v) for v in g[f"{tag}_geometry"])
    return h, w, d, bool(stn), bool(color)


@pytest.mark.parametrize("tag", GEOMETRIES)
def test_crnn_oracle_matches_reference_source_at_other_geometries(golden_dir, tag):
    """tests/golden/crnn_geometry.npz: the reference's own build_model / CTCDecoder source on oracle/keras_shim.py at
    A (31 x 200 -> 31 x 400), B (35 x 250, 3 steps discarded) and C (48 x 128, none discarded, no STN, RGB)."""
    from oracle import crnn
    from tests.geometry_oracle import crnn_logits
    g = np.load(os.path.join(golden_dir, "crnn_geometry.npz"))
    h, w, d, stn, color = _geometry(g, tag)
    crops = g[f"{tag}_crops"]
    assert crops.shape[1:3] == (h, w) and (crops.ndim == 4) == color
    wts = W.synthetic_crnn_weights(seed=int(g[f"{tag}_seed"]), stn=stn, color=color, height=h, width=w)
    probs, _ = crnn_logits(wts, crops.astype(np.float32) / 255, d)
    assert probs.shape == (len(crops), w // 4 - d, 37)
    assert float(np.abs(probs.numpy() - g[f"{tag}_probs"]).max()) <= 1e-4
    assert np.array_equal(crnn.ctc_greedy(probs), g[f"{tag}_labels"])
    assert float(g[f"{tag}_margin_fraction"]) >= 0.5


def test_synthetic_crnn_weight_shapes_follow_the_crop_size():
    default = W.synthetic_crnn_weights(seed=5)
    explicit = W.synthetic_crnn_weights(seed=5, height=31, width=200)
    assert set(default) == set(explicit) and all(np.array_equal(default[k], explicit[k]) for k in default)
    assert default["fc_9.kernel"].shape == (3584, 128) and default["stn.dense_a.kernel"].shape == (11200, 64)
    for h, w in [(31, 400), (35, 250), (48, 128), (16, 32), (64, 800), (17, 33)]:
        wts = W.synthetic_crnn_weights(seed=5, height=h, width=w)
        assert wts["fc_9.kernel"].shape == (h // 4 * 512, 128)
        assert wts["stn.dense_a.kernel"].shape == (w // 4 * (h // 4) * 32, 64)
        assert all(wts[k].shape == default[k].shape for k in default if k not in ("fc_9.kernel", "stn.dense_a.kernel"))
    assert "stn.dense_a.kernel" not in W.synthetic_crnn_weights(seed=5, stn=False, height=48, width=128)


@pytest.mark.parametrize("steps", [98, 59, 48, 1])
def test_records_round_trip_with_other_label_lengths(steps):
    rng = np.random.default_rng(steps)
    counts = np.array([3, 0, 5, 2])
    boxes = [rng.uniform(0, 500, (c, 4, 2)).astype(np.float32) for c in counts]
    labels = rng.integers(-1, 37, (int(counts.sum()), steps)).astype(np.int8)
    rec = D.pack_records(counts, boxes, labels, 6, 8, steps=steps)
    assert rec.shape == (6, 1 + 8 * 8 + 8 * ((steps + 3) // 4))
    lab_area = rec.numpy()[:, 1 + 8 * 8:].view(np.int8)
    assert (lab_area[:, 8 * steps:] == -1).all()                        # tail bytes of the last slot
    got = D.unpack_records(rec, 8, steps=steps)
    assert [c for c, _, _ in got] == counts.tolist()
    ends = np.cumsum(counts)
    for (c, b, lab), box, e in zip(got, boxes, ends):
        assert np.array_equal(b, box) and np.array_equal(lab, labels[e - c:e].astype(np.int32))
    counts2, boxes2, labels2 = D.unpack_blocks([rec, rec], 8, steps=steps)
    assert labels2.shape == (2 * int(counts.sum()), steps) and np.array_equal(labels2[:len(labels)], labels)
    if steps == 48:                                                     # the default layout is unchanged
        assert np.array_equal(rec.numpy().view(np.uint32), D.pack_records(counts, boxes, labels, 6, 8).numpy().view(np.uint32))


def test_recognizer_geometry_arguments_are_checked_before_the_device():
    w = W.synthetic_crnn_weights(0)
    for bad in [{"height": 15}, {"height": 65}, {"width": 31}, {"width": 801}, {"rnn_steps_to_discard": -1},
                {"width": 128, "rnn_steps_to_discard": 32}, {"height": 31.5}, {"width": "200"}]:
        with pytest.raises(ValueError):
            Recognizer(weights=w, build_params=bad)
    for other in [{"filters": (32, 128, 256, 256, 512, 512, 512)}, {"rnn_units": (64, 64)}, {"pool_size": 3}]:
        with pytest.raises(NotImplementedError):
            Recognizer(weights=w, build_params=other)
    if torch.cuda.is_available():
        return
    from keras_ocr_b200 import _lib
    # supported geometries (odd sizes included) and any dropout get as far as the device check
    for good in [{"height": 16, "width": 32}, {"height": 64, "width": 800}, {"height": 35, "width": 250, "rnn_steps_to_discard": 3},
                 {"height": 17, "width": 33, "rnn_steps_to_discard": 7}, {"dropout": 0.0}, {"dropout": 0.9}]:
        with pytest.raises(_lib.B2OError):
            Recognizer(weights=w, build_params=good)


def test_keras_checkpoint_of_another_crop_size_reads_back(tmp_path):
    """A Keras ``save_weights`` file of a 35 x 250 recognizer: the auto-named localisation net's dense_a kernel is found
    by its 64 columns whatever its row count (15872 = 62 x 8 x 32 here)."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from h5_writer import write
    w = W.synthetic_crnn_weights(seed=4, height=35, width=250)
    stn = {"stn.conv_a": ("model_1", "conv2d_8"), "stn.conv_b": ("model_1", "conv2d_9"),
           "stn.dense_a": ("model_1", "dense_3"), "stn.dense_b": ("model_1", "dense_4")}
    tree = {}
    for key, arr in w.items():
        layer, kind = key.rsplit(".", 1)
        parts = [*stn[layer], f"{kind}:0"] if layer in stn else (
            [layer, layer, "lstm_cell_7", f"{kind}:0"] if layer.startswith("lstm") else [layer, layer, f"{kind}:0"])
        node = tree
        for part in parts[:-1]:
            node = node.setdefault(part, {})
        node[parts[-1]] = arr
    path = str(tmp_path / "crnn_35x250.h5")
    write(path, tree)
    back = W.load_keras_h5(path)
    assert set(back) == set(w) and all(np.array_equal(back[k], w[k]) for k in w)
    assert back["stn.dense_a.kernel"].shape == (15872, 64)
