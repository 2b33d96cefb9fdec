"""Crop-size sweep and NumPy model of ``fit_crops_kernel`` (keras-ocr_b200/csrc/image.cu): tools.fit_plan picks the
cv2.resize size, cvmodels.resize_model resamples, the rest of the crop is 0 (``Recognizer.recognize`` fits with
cval=0).  tests/test_fit_batch.py pins the model to tools.fit / cv2 on the CPU; the GPU tests pin the kernel to both."""
import numpy as np

from cvmodels import resize_model
from keras_ocr_b200 import tools

GEOMETRIES = ((31, 200), (35, 250), (48, 128))      # (height, width): the default and two of crnn_geometry.npz


def sweep_sizes(seed, n, height, width, max_h=400, max_w=1200):
    """n seeded (h, w) crop sizes in 1..max_h x 1..max_w: log-uniform (up- and downscales, extreme aspect ratios),
    plus exact-size crops, crops equal to the target on one axis, 2x / 1/2x and 1-pixel rows and columns.  Sizes whose
    resized side would be 0 (tools.fit raises cv2.error) are left out."""
    rng = np.random.default_rng(seed)
    special = [(height, width), (height, width), (height, 1 + width // 2), (height, 3 * width), (height // 2, width),
               (4 * height, width), (2 * height, 2 * width), (height // 2 + 1, width // 2), (1, 1), (1, 7), (9, 1),
               (1, width // 10), (height, 1), (max_h, max_w), (max_h, 1 + width // 8), (1 + height // 30, max_w)]
    sizes = [s for s in special if not resize_is_empty(s, height, width)]
    while len(sizes) < n:
        h = int(np.exp(rng.uniform(0, np.log(max_h + 1))))
        w = int(np.exp(rng.uniform(0, np.log(max_w + 1))))
        r = rng.random()
        if r < 0.06:
            h = height
        elif r < 0.12:
            w = width
        size = (min(max(h, 1), max_h), min(max(w, 1), max_w))
        if not resize_is_empty(size, height, width):
            sizes.append(size)
    return sizes


def resize_is_empty(size, height, width):
    h, w = size
    sx, sy = width / w, height / h
    if sx == 1 and sy == 1:
        return False
    return int(sx * h) == 0 if sx <= sy else int(sy * w) == 0


def gray_model(rgb):
    """cv2.cvtColor(RGB2GRAY) on uint8 (gray_of in image.cu)."""
    r, g, b = (rgb[..., c].astype(np.int32) for c in range(3))
    return ((9798 * r + 19235 * g + 3735 * b + 16384) >> 15).astype(np.uint8)


def fit_model(img, height, width):
    """The fitted RGB crop fit_crops_kernel writes: tools.fit(img, width, height, cval=0)."""
    plan = tools.fit_plan(img.shape, width, height)
    if plan is None:
        return img.copy()
    rh, rw = plan
    out = np.zeros((height, width, 3), np.uint8)
    out[:rh, :rw] = resize_model(img, rw, rh)[:height, :width]
    return out


def crnn_input_model(fitted, color):
    """(height, width[, 3]) u8 fitted crop -> the (width, height[, 3]) fp16 CRNN input of b2o_crops_to_input."""
    crop = fitted if color else gray_model(fitted)
    x = np.flip(crop, 0).swapaxes(0, 1)
    return (x.astype(np.float32) / np.float32(255)).astype(np.float16)
