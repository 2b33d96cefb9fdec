"""The reference's one real known-answer test (reference tests/test_pipeline.py:6-20, BASELINE.json configs[0]):
``Pipeline()`` with the pretrained ``craft_mlt_25k.pth`` + ``crnn_kurapan.h5`` on ``tests/test_image.jpg`` -> exactly one
prediction, ``"eventdock"``; a blank image -> no prediction.

Neither weight file exists offline (no network, SURVEY.md 8(c)), so the test SKIPS unless they are present in the
keras-ocr cache directory (``~/.keras-ocr`` or ``$KERAS_OCR_CACHE_DIR``, reference tools.py:495-498) with the reference's
sha256 digests (detection.py:647-658, recognition.py:27-44).  The reference's test image is stored as
``tests/golden/test_image.jpg``.  Everything between the files and the assertion is the product path:
``weights.load_craft_pth`` (torch.load), ``hdf5.read_datasets`` (own HDF5 reader), the CUDA pipeline."""
import os

import numpy as np
import pytest

from keras_ocr_b200 import tools

pytestmark = pytest.mark.gpu

CRAFT = ("craft_mlt_25k.pth", "4a5efbfb48b4081100544e75e1e2b57f8de3d84f213004b14b85fd4b3748db17")
CRNN = ("crnn_kurapan.h5", "a7d8086ac8f5c3d6a0a828f7d6fbabcaf815415dd125c32533013f85603be46d")


def test_pipeline_known_answer_eventdock(cuda_device, golden_dir):
    cache = tools.get_default_cache_dir()
    missing = [name for name, _ in (CRAFT, CRNN) if not os.path.isfile(os.path.join(cache, name))]
    if missing:
        pytest.skip(f"pretrained weights not in {cache}: {', '.join(missing)} (no network to download them)")
    image_path = os.path.join(golden_dir, "test_image.jpg")
    for name, digest in (CRAFT, CRNN):
        assert tools.sha256sum(os.path.join(cache, name)) == digest, f"{name}: sha256 mismatch"

    from keras_ocr_b200.pipeline import Pipeline
    pipeline = Pipeline()                                    # defaults = the pretrained pair, like the reference

    # We shouldn't find any text in a blank image.
    assert len(pipeline.recognize(images=[np.zeros((256, 256, 3), dtype="uint8")])[0]) == 0

    image = tools.read(image_path)
    predictions = pipeline.recognize(images=[image])[0]      # a list of (text, box) tuples
    assert len(predictions) == 1
    assert predictions[0][0] == "eventdock"
    assert predictions[0][1].shape == (4, 2) and predictions[0][1].dtype == np.float32
