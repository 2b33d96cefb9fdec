"""GPU: recognizers built with another crop size (build_params height / width / rnn_steps_to_discard, reference
recognition.py:13-23, 214, 328), at the three geometries of tests/golden/crnn_geometry.npz -- A: 31 x 400 (98-long label
rows); B: 35 x 250 with 3 steps discarded (odd sizes on both axes, 59-long rows); C: 48 x 128, none discarded, no
spatial transformer, RGB crops (fc_9 over 12 feature rows) -- against the reference's own source and the fp32 oracle."""
import os
import sys

import numpy as np
import pytest
import torch

from keras_ocr_b200 import distributed as D, weights as W

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from h5_writer import write  # noqa: E402

pytestmark = pytest.mark.gpu

GEOMETRIES = ("A", "B", "C")
MARGIN = 0.3              # the fixture's top-2 logit margin: twice the logit bound below, so fp16 cannot flip such a step


def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.fixture(scope="module")
def golden(golden_dir):
    return dict(np.load(os.path.join(golden_dir, "crnn_geometry.npz")))


class Case:
    """One geometry: its fixture arrays, weights and a Recognizer built for it (workspace kept for the taps)."""

    def __init__(self, g, tag):
        from keras_ocr_b200.recognition import Recognizer
        self.tag = tag
        self.h, self.w, self.d, stn, color = (int(v) for v in g[f"{tag}_geometry"])
        self.stn, self.color = bool(stn), bool(color)
        self.t, self.hf, self.keep = self.w // 4, self.h // 4, self.w // 4 - self.d
        self.g = {k[len(tag) + 1:]: v for k, v in g.items() if k.startswith(tag + "_")}
        self.params = {"height": self.h, "width": self.w, "rnn_steps_to_discard": self.d, "stn": self.stn, "color": self.color}
        self.weights = W.synthetic_crnn_weights(seed=int(self.g["seed"]), stn=self.stn, color=self.color, height=self.h, width=self.w)
        self.rec = Recognizer(weights=self.weights, build_params=self.params)
        self.rec.keep_workspace = True

    def crnn_input(self, crops):
        rec = self.rec
        t = torch.from_numpy(np.ascontiguousarray(crops)).to(rec.device)
        x = torch.empty((t.shape[0], self.w, self.h) + ((3,) if self.color else ()), dtype=torch.float16, device=rec.device)
        rec.ctx.crops_to_input(t.data_ptr(), t.shape[0], x.data_ptr(), _stream(), color=self.color)
        return x


@pytest.fixture(scope="module")
def cases(cuda_device, golden):
    return {tag: Case(golden, tag) for tag in GEOMETRIES}


@pytest.mark.parametrize("tag", GEOMETRIES)
def test_warp_boxes_at_other_crop_sizes(cases, cuda_device, tag):
    """b2o_warp_boxes[_color] at the recognizer's crop size vs the reference's tools.warpBox(target_height, target_width)."""
    c = cases[tag]
    image, quads, ref = c.g["image"], c.g["quads"], c.g["warp_crops"]
    img = torch.from_numpy(image[None]).to(cuda_device).contiguous()
    idx = torch.zeros(len(quads), dtype=torch.int32, device=cuda_device)
    crnn_in, crops = c.rec.warp_device(img, torch.from_numpy(quads).to(cuda_device), idx, want_crops=True)
    crops = crops.cpu().numpy()
    assert crops.shape == ref.shape == (len(quads), c.h, c.w) + ((3,) if c.color else ())
    diff = np.abs(crops.astype(np.int16) - ref.astype(np.int16))
    assert diff.max() <= 1 and (diff > 0).mean() <= 1e-3, (int(diff.max()), float((diff > 0).mean()))
    assert torch.equal(crnn_in, c.crnn_input(crops))               # both routes to the CRNN input agree bit for bit


@pytest.mark.parametrize("tag", GEOMETRIES)
def test_crnn_at_other_crop_sizes_vs_oracle_and_reference(cases, tag):
    """Taps vs the fp32 oracle (the tolerances of test_crnn_vs_oracle), labels = the exact greedy collapse of the device's
    own logits, softmax vs the reference-source fixture, and the reference's argmax at every step it decides by a margin."""
    from oracle import crnn
    from tests.geometry_oracle import crnn_logits
    c = cases[tag]
    crops = c.g["crops"]
    b = len(crops)
    labels = c.rec.predict_device(c.crnn_input(crops)).cpu().numpy()
    assert labels.shape == (b, c.keep)
    _, inter = crnn_logits(c.weights, crops.astype(np.float32) / 255, c.d)

    def rel(a, ref):
        return float((a - ref).abs().max() / max(ref.abs().max(), 1e-6))

    tap = c.rec.tap
    feat = tap("features", (b, c.t, c.hf, 512), torch.float16).float().cpu()
    assert rel(feat, inter["features"].permute(0, 2, 3, 1)) <= 2e-2
    if c.stn:
        assert float((tap("theta", (b, 6), torch.float32).cpu() - inter["theta"]).abs().max()) <= 2e-2
        assert rel(tap("warped", (b, c.t, c.hf, 512), torch.float16).float().cpu(), inter["warped"]) <= 5e-2
    assert rel(tap("fc_9", (b, c.t, 128), torch.float16).float().cpu(), inter["fc_9"]) <= 5e-2
    assert float((tap("l2", (b, c.t, 256), torch.float16).float().cpu() - inter["l2"]).abs().max()) <= 5e-2
    logits = tap("logits", (b, c.keep, 37), torch.float32).cpu()
    assert float((logits - inter["logits"]).abs().max()) <= 0.15
    probs = torch.softmax(logits, -1)
    assert np.array_equal(labels, crnn.ctc_greedy(probs))            # integer work: exact
    ref_probs = c.g["probs"]
    assert float(np.abs(probs.numpy() - ref_probs).max()) <= 5e-2
    logp = np.log(ref_probs.astype(np.float64))
    top2 = np.sort(logp, -1)[..., -2:]
    decided = (top2[..., 1] - top2[..., 0]) >= MARGIN
    assert decided.mean() >= 0.5 and np.isclose(decided.mean(), float(c.g["margin_fraction"]))
    assert np.array_equal(logits.numpy().argmax(-1)[decided], ref_probs.argmax(-1)[decided])


@pytest.mark.parametrize("tag", GEOMETRIES)
def test_crop_labels_do_not_depend_on_the_batch_at_other_crop_sizes(cases, tag):
    c = cases[tag]
    rng = np.random.default_rng(3)
    crops = np.concatenate([c.g["crops"], rng.integers(0, 256, (37 - len(c.g["crops"]),) + c.g["crops"].shape[1:], dtype=np.uint8)])
    batch = c.rec.predict_device(c.crnn_input(crops)).cpu().numpy()
    for i in (0, 5, 36):
        alone = c.rec.predict_device(c.crnn_input(crops[i:i + 1])).cpu().numpy()
        assert np.array_equal(alone[0], batch[i])


@pytest.mark.parametrize("tag", GEOMETRIES)
def test_public_api_at_other_crop_sizes(cases, cuda_device, tag):
    """recognize_crops / recognize / recognize_from_boxes return labels_to_text of the device labels."""
    from keras_ocr_b200 import tools
    from keras_ocr_b200.recognition import labels_to_text
    c = cases[tag]
    crops = c.g["crops"]
    texts = labels_to_text(c.rec.predict_device(c.crnn_input(crops)).cpu().numpy())
    assert c.rec.recognize_crops(crops) == texts
    rgb = crops[0] if c.color else np.repeat(crops[0][..., None], 3, axis=2)     # RGB -> gray is exact on equal channels
    assert c.rec.recognize(rgb) == texts[0]
    small = np.ascontiguousarray(rgb[: c.h // 2 + 3, : c.w // 3 + 5])              # fit() letterboxes to the model's size
    fitted = tools.fit(small, c.w, c.h, cval=0)
    assert c.rec.recognize(small) == c.rec.recognize_crops((fitted if c.color else fitted[..., 0])[None])[0]
    image, quads = c.g["image"], c.g["quads"]
    rgb_image = image if c.color else np.repeat(image[..., None], 3, axis=2)
    img = torch.from_numpy(image[None]).to(cuda_device).contiguous()
    idx = torch.zeros(len(quads), dtype=torch.int32, device=cuda_device)
    crnn_in, _ = c.rec.warp_device(img, torch.from_numpy(quads).to(cuda_device), idx)
    want = labels_to_text(c.rec.predict_device(crnn_in).cpu().numpy())
    assert c.rec.recognize_from_boxes([rgb_image], [quads]) == [want]


def _keras_h5_tree(w):
    stn = {"stn.conv_a": ("model_1", "conv2d_8"), "stn.conv_b": ("model_1", "conv2d_9"),
           "stn.dense_a": ("model_1", "dense_3"), "stn.dense_b": ("model_1", "dense_4")}
    tree = {}
    for key, arr in w.items():
        layer, kind = key.rsplit(".", 1)
        if layer in stn:
            parts = [*stn[layer], f"{kind}:0"]
        elif layer.startswith("lstm"):
            parts = [layer, layer, "lstm_cell_7", f"{kind}:0"]
        else:
            parts = [layer, layer, f"{kind}:0"]
        node = tree
        for part in parts[:-1]:
            node = node.setdefault(part, {})
        node[parts[-1]] = arr
    return tree


def test_keras_checkpoint_of_another_crop_size(cases, tmp_path):
    """A Keras .h5 checkpoint of geometry B loads with its build_params and reads like the weight dict; with the default
    build_params its fc_9 / stn.dense_a do not fit and the error names the build_params that would."""
    from keras_ocr_b200.recognition import Recognizer
    c = cases["B"]
    path = str(tmp_path / "crnn_35x250.h5")
    write(path, _keras_h5_tree(c.weights))
    rec = Recognizer(weights=path, build_params=c.params)
    crops = c.g["crops"]
    assert rec.recognize_crops(crops) == c.rec.recognize_crops(crops)
    with pytest.raises(ValueError, match="height"):
        Recognizer(weights=path)
    with pytest.raises(ValueError, match="width"):
        Recognizer(weights=path, build_params={"height": 35})


def test_default_build_params_spelled_out_are_the_default(cuda_device):
    from keras_ocr_b200.recognition import DEFAULT_BUILD_PARAMS, Recognizer
    w = W.synthetic_crnn_weights(seed=2)
    crops = np.random.default_rng(8).integers(0, 256, (9, 31, 200), dtype=np.uint8)
    a = Recognizer(weights=w)
    b = Recognizer(weights=w, build_params=dict(DEFAULT_BUILD_PARAMS, stn=True))
    assert (a.height, a.width, a.steps) == (b.height, b.width, b.steps) == (31, 200, 48)
    x = torch.from_numpy(crops).to(a.device)
    outs = []
    for r in (a, b):
        inp = torch.empty((9, 200, 31), dtype=torch.float16, device=r.device)
        r.ctx.crops_to_input(x.data_ptr(), 9, inp.data_ptr(), _stream())
        outs.append(r.predict_device(inp).cpu().numpy())
    assert np.array_equal(outs[0], outs[1])


def test_pipeline_with_a_wider_recognizer(cases, cuda_device):
    """Pipeline with recognizer A (31 x 400, 98-long rows): the detector half is unchanged; recognize ==
    recognize_records decoded by distributed.unpack_blocks == the sharded gather == detect + recognize_from_boxes."""
    from keras_ocr_b200 import recognition
    from keras_ocr_b200.detection import Detector
    from keras_ocr_b200.pipeline import Pipeline
    from keras_ocr_b200.recognition import Recognizer
    from oracle import synth
    c = cases["A"]
    assert c.rec.steps == 98
    det = Detector(weights=W.synthetic_craft_weights(3, textlike=True))
    pages, _ = synth.text_images(seed=21, n=2, h=192, w=384, n_words=4)
    pipe = Pipeline(detector=det, recognizer=c.rec, scale=2)
    got = pipe.recognize(pages)
    default = Pipeline(detector=det, recognizer=Recognizer(weights=W.synthetic_crnn_weights(2)), scale=2).recognize(pages)
    assert [len(g) for g in got] == [len(g) for g in default] and sum(len(g) for g in got) >= 6
    assert all(np.array_equal(a, b) for ga, gb in zip(got, default) for (_, a), (_, b) in zip(ga, gb))
    rec = pipe.recognize_records(pages, rows=3, rec_boxes=16)
    assert rec.shape == (3, 1 + 16 * 8 + 16 * 25)
    counts, boxes, labels = D.unpack_blocks([rec], 16, steps=98)
    assert labels.shape[1] == 98 and counts.tolist() == [len(g) for g in got]
    assert recognition.labels_to_text(labels) == [t for g in got for t, _ in g]
    assert np.array_equal(boxes, np.concatenate([np.stack([b for _, b in g]) for g in got if g]))
    for result in (D.recognize_sharded(pipe, pages, max_boxes=16), D.recognize_sharded(pipe, pages, max_boxes="auto")):
        assert [[t for t, _ in g] for g in result] == [[t for t, _ in g] for g in got]
    stream = D.ShardedStream(pipe, max_boxes=16)
    assert stream.submit(pages) is None
    assert [[t for t, _ in g] for g in stream.flush()] == [[t for t, _ in g] for g in got]
    # the reference flow: Detector.detect on the padded batch, then recognize_from_boxes
    batch = pipe.prepare_device(pages)[0].cpu().numpy()
    groups = det.detect(batch)
    texts = c.rec.recognize_from_boxes(batch, groups)
    assert texts == [[t for t, _ in g] for g in got]


@pytest.mark.parametrize("steps", [98, 59])
def test_pack_records_steps_matches_host_bookkeeping(cuda_device, steps):
    """b2o_pack_records_steps == distributed.pack_records(..., steps) bit for bit, as the 48-step test checks b2o_pack_records."""
    from keras_ocr_b200 import _lib
    ctx = _lib.Context(0)
    rng = np.random.default_rng(steps)
    n, m, rows, rec_boxes = 5, 8, 7, 6
    counts = np.array([3, 0, 8, 11, 1], np.int32)
    held = np.minimum(counts, m)
    boxes = rng.uniform(0, 3000, (n, m, 4, 2)).astype(np.float32)
    labels = rng.integers(-1, 37, (int(held.sum()), steps)).astype(np.int32)
    inv = np.array([0.5, 1.0, 1 / 1.6, 0.5, 1 / 3], np.float32)
    b_t, c_t = torch.from_numpy(boxes).to(cuda_device), torch.from_numpy(counts).to(cuda_device)
    labels_t, inv_t = torch.from_numpy(labels).to(cuda_device), torch.from_numpy(inv).to(cuda_device)
    rec = torch.zeros((rows, ctx.record_floats(rec_boxes, steps)), dtype=torch.float32, device=cuda_device)
    assert rec.shape[1] == 1 + rec_boxes * 8 + rec_boxes * ((steps + 3) // 4)
    ctx.pack_records(b_t.data_ptr(), c_t.data_ptr(), labels_t.data_ptr(), inv_t.data_ptr(), n, m, rows, rec_boxes,
                     rec.data_ptr(), _stream(), steps=steps)
    scaled = [boxes[i, :held[i]] * inv[i] for i in range(n)]
    expect = D.pack_records(held, scaled, labels.astype(np.int8), rows, rec_boxes, steps=steps)
    assert np.array_equal(rec.cpu().numpy().view(np.uint32), expect.numpy().view(np.uint32))
    ctx.close()
