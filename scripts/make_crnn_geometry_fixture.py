"""Write tests/golden/crnn_geometry.npz: recognizers built with other crop sizes, pinned to the reference's own source.

    python scripts/make_crnn_geometry_fixture.py [--out tests/golden/crnn_geometry.npz]

Runs only where the reference checkout is (``KERAS_OCR_REFERENCE``, as ``oracle/validate_against_reference.py``, whose
AST-lifting helpers it uses).  Like that script's ``check_crnn``, it executes the reference's ``build_model`` /
``CTCDecoder`` on ``oracle/keras_shim.py`` and its ``tools.warpBox``, at each of CRNN_GEOMETRIES, asserts that the fp32
oracle (``tests/geometry_oracle.py``) equals them, and stores inputs and reference outputs only.
"""
import argparse
import ast
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from keras_ocr_b200 import weights as W  # noqa: E402
from oracle import crnn as o_crnn, imageops as o_img, keras_shim as shim, synth  # noqa: E402
from oracle.validate_against_reference import GOLDEN, REF, lift, reference_tools  # noqa: E402
from tests.geometry_oracle import crnn_logits  # noqa: E402

# Each breaks a different assumption of the default 31 x 200 -- A: 98-long label rows; B: odd sizes on both axes
# (250 -> 125 -> 62, 35 -> 17 -> 8) and rows that are not a multiple of 4 long; C: no transformer, RGB crops, fc_9 over
# 12 feature rows.
CRNN_GEOMETRIES = {
    "A": {"height": 31, "width": 400, "rnn_steps_to_discard": 2, "stn": True, "color": False},
    "B": {"height": 35, "width": 250, "rnn_steps_to_discard": 3, "stn": True, "color": False},
    "C": {"height": 48, "width": 128, "rnn_steps_to_discard": 0, "stn": False, "color": True},
}
MARGIN = 0.3            # top-2 logit gap at which fp16 cannot flip a step's argmax (twice the GPU tests' logit bound)


def make(tools, out):
    """Crops are warpBox's own output on a blurred-noise image (RGB for the color model) plus noise crops.  Weights:
    ``synthetic_crnn_weights`` at the first seed for which at least half of all kept steps have a top-2 logit margin
    >= MARGIN (stored as ``<tag>_margin_fraction``), so that a GPU run can be held to the reference's argmax there."""
    path = os.path.join(REF, "keras_ocr", "recognition.py")
    with open(path) as f:
        tree = ast.parse(f.read())
    defaults = next(ast.literal_eval(n.value) for n in tree.body if isinstance(n, ast.Assign)
                    and getattr(n.targets[0], "id", "") == "DEFAULT_BUILD_PARAMS")
    scope = lift(path, ["_repeat", "_meshgrid", "_transform", "CTCDecoder", "build_model"],
                 {"tf": shim.tf, "keras": shim.keras, "np": np})
    alphabet = "0123456789abcdefghijklmnopqrstuvwxyz"
    for tag, geo in CRNN_GEOMETRIES.items():
        h, w, d, stn, color = geo["height"], geo["width"], geo["rnn_steps_to_discard"], geo["stn"], geo["color"]
        rng = np.random.default_rng(41)
        gray = synth.noise_gray(rng, 240, 480)
        image = np.stack([gray, synth.noise_gray(rng, 240, 480), synth.noise_gray(rng, 240, 480)], -1) if color else gray
        quads = synth.random_quads(rng, 10, 240, 480)
        warped = np.stack([tools.warpBox(image=image, box=q, target_height=h, target_width=w) for q in quads])
        if not color:
            for q, crop in zip(quads[:3], warped):
                assert np.array_equal(crop, o_img.warp_box(gray, q, target_height=h, target_width=w))
        noise = rng.integers(0, 256, (3,) + warped.shape[1:], dtype=np.uint8)
        crops = np.concatenate([warped, noise]).astype(np.uint8)
        x = crops.astype("float32") / 255                                    # recognition.py:524-526
        if not color:
            x = x[..., np.newaxis]
        params = dict(defaults, height=h, width=w, rnn_steps_to_discard=d, color=color, stn=stn)
        for seed in range(100, 140):
            shim.reset()
            backbone, model, _, prediction_model = scope["build_model"](alphabet=alphabet, **params)
            wts = W.synthetic_crnn_weights(seed=seed, stn=stn, color=color, height=h, width=w)
            used = shim.load_weights(wts)
            assert used == set(wts), sorted(set(wts) - used)
            probs_ref = model.predict(x).numpy()
            logp = np.log(probs_ref.astype(np.float64))                      # logits up to a per-step constant
            top2 = np.sort(logp, -1)[..., -2:]
            fraction = float(((top2[..., 1] - top2[..., 0]) >= MARGIN).mean())
            if fraction >= 0.5:
                break
        assert fraction >= 0.5, (tag, fraction)
        labels_ref = prediction_model.predict(x).numpy()
        probs, taps = crnn_logits(wts, x, d)
        labels = o_crnn.ctc_greedy(probs)
        t, keep = w // 4, w // 4 - d
        assert probs_ref.shape == (len(crops), keep, 37) and labels_ref.shape == (len(crops), keep), (probs_ref.shape, labels_ref.shape)
        assert taps["features"].shape == (len(crops), 512, t, h // 4)
        e_p = float(np.abs(probs.numpy() - probs_ref).max())
        print(f"  {tag} {h}x{w} discard {d} stn={stn} color={color}: weights seed {seed}, {fraction:.2f} of the steps "
              f"decided by >= {MARGIN}; softmax max|ref-oracle| = {e_p:.2e}, labels equal: {np.array_equal(labels, labels_ref)}")
        assert e_p < 1e-4, e_p
        assert np.array_equal(labels, labels_ref)
        out[f"{tag}_geometry"] = np.array([h, w, d, int(stn), int(color)], np.int64)
        out[f"{tag}_seed"] = np.array(seed)
        out[f"{tag}_margin_fraction"] = np.array(fraction)
        out[f"{tag}_image"] = image
        out[f"{tag}_quads"] = quads
        out[f"{tag}_warp_crops"] = warped
        out[f"{tag}_crops"] = crops
        out[f"{tag}_probs"] = probs_ref.astype(np.float32)
        out[f"{tag}_labels"] = labels_ref.astype(np.int64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(GOLDEN, "crnn_geometry.npz"))
    args = ap.parse_args()
    assert os.path.isdir(REF), f"reference not found at {REF}"
    out = {}
    make(reference_tools(), out)
    np.savez_compressed(args.out, **out)
    print(f"wrote {args.out} ({os.path.getsize(args.out) / 1e3:.0f} kB); oracle == reference at every geometry")


if __name__ == "__main__":
    main()
