"""GPU: Recognizer.recognize_batch / fit_device (b2o_fit_crops, fit_crops_kernel) -- the single-crop API of reference
recognition.py:467-489 over many crops at once.  The fitted u8 crops equal tools.fit(cval=0) byte for byte and the CRNN
input equals b2o_crops_to_input of what ``recognize`` feeds it, at the default geometry and at 35 x 250 gray and
48 x 128 colour; the strings equal the ``recognize`` loop for every input form and chunk size."""
import os
import sys

import cv2
import numpy as np
import pytest
import torch

from keras_ocr_b200 import tools, weights as W

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from fitmodel import sweep_sizes  # noqa: E402

pytestmark = pytest.mark.gpu

# (height, width, rnn_steps_to_discard, stn, color): the default, and geometries B and C of crnn_geometry.npz
GEOMETRIES = {"default": (31, 200, 2, True, False), "35x250": (35, 250, 3, True, False), "48x128": (48, 128, 0, False, True)}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _recognizer(tag, seed=0):
    from keras_ocr_b200.recognition import Recognizer
    h, w, d, stn, color = GEOMETRIES[tag]
    weights = W.synthetic_crnn_weights(seed=seed, stn=stn, color=color, height=h, width=w)
    return Recognizer(weights=weights, build_params={"height": h, "width": w, "rnn_steps_to_discard": d, "stn": stn,
                                                     "color": color})


@pytest.fixture(scope="module")
def recognizers(cuda_device):
    return {tag: _recognizer(tag) for tag in GEOMETRIES}


@pytest.fixture(scope="module")
def decisive(cuda_device):
    from keras_ocr_b200.recognition import Recognizer
    return Recognizer(weights=W.synthetic_crnn_weights(decisive=True))


def _crops_to_input(rec, fitted):
    """What ``recognize`` feeds the CRNN: cvtColor(tools.fit(...)) (the RGB fit for colour) through b2o_crops_to_input."""
    crops = fitted if rec.color else np.stack([cv2.cvtColor(f, cv2.COLOR_RGB2GRAY) for f in fitted])
    t = torch.from_numpy(np.ascontiguousarray(crops)).to(rec.device)
    x = torch.empty((len(crops), rec.width, rec.height) + ((3,) if rec.color else ()), dtype=torch.float16, device=rec.device)
    rec.ctx.crops_to_input(t.data_ptr(), len(crops), x.data_ptr(), _stream(), color=rec.color)
    return x


@pytest.mark.parametrize("tag", list(GEOMETRIES))
def test_fit_device_matches_tools_fit_byte_for_byte(recognizers, golden_dir, tag):
    rec = recognizers[tag]
    rng = np.random.default_rng(17)
    sizes = sweep_sizes(11, 560, rec.height, rec.width)
    images = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
    g = np.load(os.path.join(golden_dir, "inputs.npz"))
    goldens = ("wide", "tall", "exact")
    images += [g[f"fit_{k}_src"] for k in goldens]
    srcs = [torch.from_numpy(im).to(rec.device) for im in images]
    crnn_in, crops = rec.fit_device(srcs, want_crops=True)
    crops = crops.cpu().numpy()
    want = np.stack([tools.fit(im, rec.width, rec.height, cval=0) for im in images])
    bad = [sizes[i] if i < len(sizes) else goldens[i - len(sizes)] for i in range(len(images)) if not np.array_equal(crops[i], want[i])]
    assert not bad, bad[:10]
    if tag == "default":                                     # the reference's own tools.fit outputs (cval 0, letterbox)
        for i, k in enumerate(goldens):
            assert tuple(g[f"fit_{k}_params"]) == (0, 0)
            assert np.array_equal(crops[len(sizes) + i], g[f"fit_{k}_dst"])
    assert torch.equal(crnn_in, _crops_to_input(rec, want))
    alone, none = rec.fit_device(srcs[:1])                   # crops are optional and independent of the batch
    assert none is None and torch.equal(alone, crnn_in[:1])


def test_fit_crops_from_one_staging_buffer_and_argument_checks(recognizers):
    """The pointer table may point into one packed buffer (what recognize_batch uploads); bad arguments are refused."""
    from keras_ocr_b200 import _lib
    rec = recognizers["default"]
    rng = np.random.default_rng(4)
    images = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in [(20, 90), (31, 200), (80, 60), (1, 40), (7, 1)]]
    packed = torch.from_numpy(np.concatenate([im.reshape(-1) for im in images])).to(rec.device)
    offsets = np.cumsum([0] + [im.size for im in images])[:-1]
    ptrs = torch.from_numpy(np.array([packed.data_ptr() + int(o) for o in offsets], np.uint64).view(np.int64)).to(rec.device)
    dims = torch.tensor([rec._fit_dims(im.shape) for im in images], dtype=torch.int32, device=rec.device)
    crnn_in, crops = rec._fit_table(ptrs.data_ptr(), dims.data_ptr(), len(images), True)
    want = np.stack([tools.fit(im, 200, 31, cval=0) for im in images])
    assert np.array_equal(crops.cpu().numpy(), want)
    assert torch.equal(crnn_in, _crops_to_input(rec, want))
    rec.ctx.fit_crops(None, None, 0, None, None, _stream())                 # b == 0: nothing to do
    for args in ((None, dims.data_ptr(), 5), (ptrs.data_ptr(), None, 5), (ptrs.data_ptr(), dims.data_ptr(), -1)):
        with pytest.raises(_lib.B2OError, match="b2o_fit_crops"):
            rec.ctx.fit_crops(*args, None, crnn_in.data_ptr(), _stream())
    with pytest.raises(_lib.B2OError):
        rec.ctx.fit_crops(ptrs.data_ptr(), dims.data_ptr(), 5, None, None, _stream())


def _word_crops(seed, n_pages=12):
    """Word crops cut from rendered pages with random margins, rescaled by 0.4x..3x, plus blurred-noise crops."""
    from oracle import synth
    rng = np.random.default_rng(seed)
    crops, words = [], []
    for _ in range(n_pages):
        page, ws, rects = synth.text_image(rng, 256, 384, 6, return_layout=True)
        for word, (x0, y0, x1, y1) in zip(ws, rects):
            m = int(rng.integers(0, 10))
            x0, y0 = max(x0 - m, 0), max(y0 - int(rng.integers(0, 8)), 0)
            x1, y1 = min(x1 + int(rng.integers(0, 10)), page.shape[1]), min(y1 + int(rng.integers(0, 8)), page.shape[0])
            crop = page[y0:y1, x0:x1]
            s = float(np.exp(rng.uniform(np.log(0.4), np.log(3.0))))
            size = (max(int(crop.shape[1] * s), 1), max(int(crop.shape[0] * s), 1))
            crops.append(np.ascontiguousarray(cv2.resize(crop, size)))
            words.append(word)
    for _ in range(12):
        h, w = int(rng.integers(5, 90)), int(rng.integers(5, 500))
        crops.append(np.repeat(synth.noise_gray(rng, h, w)[..., None], 3, axis=2))
        words.append(None)
    crops.append(np.ascontiguousarray(crops[0][:31, :200]) if crops[0].shape[0] >= 31 and crops[0].shape[1] >= 200
                 else cv2.resize(crops[0], (200, 31)))                  # an exact-size crop: no resize
    words.append(words[0])
    return crops, words


def test_recognize_batch_equals_the_recognize_loop(decisive, tmp_path):
    rec = decisive
    crops, words = _word_crops(31)
    loop = [rec.recognize(c) for c in crops]
    read = np.mean([t == w for t, w in zip(loop, words) if w is not None])
    print(f"\n{len(crops)} crops, {read:.1%} of the word crops read as the rendered word")
    for chunk in (1, 7, 1024):
        assert rec.recognize_batch(crops, chunk=chunk) == loop, chunk
    paths = []
    for i, c in enumerate(crops):
        paths.append(str(tmp_path / f"crop_{i}.png"))
        cv2.imwrite(paths[-1], cv2.cvtColor(c, cv2.COLOR_RGB2BGR))
    assert rec.recognize_batch(paths, chunk=7) == [rec.recognize(p) for p in paths] == loop
    cuda = [torch.from_numpy(c).to(rec.device) for c in crops]
    assert rec.recognize_batch(cuda, chunk=7) == loop
    mixed = [paths[i] if i % 3 == 0 else cuda[i] if i % 3 == 1 else crops[i] for i in range(len(crops))]
    assert rec.recognize_batch(mixed, chunk=5) == loop
    same = np.stack([cv2.resize(c, (150, 24)) for c in crops])
    assert rec.recognize_batch(same, chunk=7) == [rec.recognize(c) for c in same]


def test_recognize_batch_edge_cases(decisive):
    rec = decisive
    assert rec.recognize_batch([]) == [] and rec.recognize_batch(np.zeros((0, 10, 10, 3), np.uint8)) == []
    rng = np.random.default_rng(2)
    good = [rng.integers(0, 256, (20, 60, 3), dtype=np.uint8) for _ in range(3)]
    for bad, exc in (((0, 10, 3), ZeroDivisionError), ((10, 0, 3), ZeroDivisionError), ((1, 1000, 3), cv2.error),
                     ((1000, 1, 3), cv2.error)):
        img = np.zeros(bad, np.uint8)
        with pytest.raises(exc):
            rec.recognize(img)
        with pytest.raises(exc):
            rec.recognize_batch(good + [img])
        with pytest.raises(exc):
            rec.recognize_batch(good * 3 + [img], chunk=4)
        with pytest.raises(exc):
            rec.fit_device([torch.from_numpy(img).to(rec.device)])
    with pytest.raises(ValueError):
        rec.recognize_batch([np.zeros((20, 60), np.uint8)])
    with pytest.raises(ValueError):
        rec.recognize_batch(good, chunk=0)
    assert rec.recognize_batch(good, chunk=2) == [rec.recognize(g) for g in good]     # still works afterwards


@pytest.mark.parametrize("tag", ["A", "B", "C"])
def test_recognize_batch_at_other_crop_sizes(cuda_device, golden_dir, tag):
    """A recognizer of each crnn_geometry.npz case gives its recognize loop's strings; its crops and pages are cut
    into ragged word-sized pieces."""
    from keras_ocr_b200.recognition import Recognizer
    g = dict(np.load(os.path.join(golden_dir, "crnn_geometry.npz")))
    h, w, d, stn, color = (int(v) for v in g[f"{tag}_geometry"])
    rec = Recognizer(weights=W.synthetic_crnn_weights(seed=int(g[f"{tag}_seed"]), stn=bool(stn), color=bool(color),
                                                      height=h, width=w),
                     build_params={"height": h, "width": w, "rnn_steps_to_discard": d, "stn": bool(stn), "color": bool(color)})
    rgb = lambda a: a if a.ndim == 3 else np.repeat(a[..., None], 3, axis=2)      # noqa: E731
    rng = np.random.default_rng(6)
    image = rgb(g[f"{tag}_image"])
    crops = [rgb(c) for c in g[f"{tag}_crops"]]
    for _ in range(40):
        ch, cw = int(rng.integers(8, 120)), int(rng.integers(10, 600))
        y, x = int(rng.integers(0, max(image.shape[0] - ch, 1))), int(rng.integers(0, max(image.shape[1] - cw, 1)))
        crops.append(np.ascontiguousarray(image[y:y + ch, x:x + cw]))
    loop = [rec.recognize(c) for c in crops]
    assert rec.recognize_batch(crops, chunk=16) == loop
    assert rec.recognize_batch([torch.from_numpy(c).to(rec.device) for c in crops]) == loop
