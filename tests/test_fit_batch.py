"""CPU: the host plan and the arithmetic of batched crop fitting (Recognizer.recognize_batch, b2o_fit_crops).
tools.fit_plan gives the sizes tools.fit resizes to, and the model of fit_crops_kernel (fit_plan + the cv2.resize model
of tests/cvmodels.py + zero fill) reproduces tools.fit(cval=0) -- i.e. cv2 itself -- bit for bit, downscales included,
over a sweep of crop sizes at three crop geometries."""
import os
import sys

import cv2
import numpy as np
import pytest

from keras_ocr_b200 import tools

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from fitmodel import GEOMETRIES, fit_model, gray_model, resize_is_empty, sweep_sizes  # noqa: E402

N_SIZES = 2000


def _image(rng, h, w):
    return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


@pytest.mark.parametrize("height,width", GEOMETRIES)
def test_fit_plan_gives_the_sizes_fit_resizes_to(height, width):
    """fit_plan == the extent of the resized image inside tools.fit's letterbox: fitting an all-255 image with cval=0
    leaves exactly the resized rows and columns non-zero; None exactly when fit returns the image itself."""
    sizes = sweep_sizes(1, N_SIZES, height, width)
    assert len(sizes) == N_SIZES
    kinds = set()
    for h, w in sizes:
        img = np.full((h, w, 3), 255, np.uint8)
        out = tools.fit(img, width, height, cval=0)
        plan = tools.fit_plan(img.shape, width, height)
        if plan is None:
            assert out is img and (h, w) == (height, width)
            kinds.add("exact")
            continue
        rh, rw = plan
        assert 1 <= rh <= height and 1 <= rw <= width and (rh == height or rw == width), (h, w, plan)
        rows, cols = np.nonzero(out[..., 0])
        assert (rows.max() + 1, cols.max() + 1) == (rh, rw), (h, w, plan)
        assert out[:rh, :rw].min() == 255
        kinds.add("up" if rh * rw > h * w else "down")
        if (rh, rw) == (h, w):
            kinds.add("one axis equal, no resize")
    assert kinds == {"exact", "up", "down", "one axis equal, no resize"}


@pytest.mark.parametrize("height,width", GEOMETRIES)
def test_fit_crops_model_matches_fit_bit_for_bit(height, width):
    """fit_crops_kernel's model == tools.fit(img, width, height, cval=0) (cv2.resize INTER_LINEAR), and its gray plane ==
    cv2.cvtColor of it, for every size of the sweep."""
    rng = np.random.default_rng(height * 1000 + width)
    sizes = sweep_sizes(2, N_SIZES, height, width)
    down = 0
    for h, w in sizes:
        img = _image(rng, h, w)
        want = tools.fit(img, width, height, cval=0)
        got = fit_model(img, height, width)
        assert np.array_equal(got, want), (h, w, int((got != want).sum()))
        assert np.array_equal(gray_model(got), cv2.cvtColor(want, cv2.COLOR_RGB2GRAY)), (h, w)
        down += h > height or w > width
    assert down >= len(sizes) // 3


def test_fit_plan_downscale_corner_cases():
    """Large one-axis downscales, exact 2x / 1/2x and 1 x 1 up to a full crop height match cv2.resize."""
    rng = np.random.default_rng(5)
    for h, w in [(31, 3000), (992, 200), (62, 400), (16, 100), (1, 1), (1, 200), (31, 1), (400, 13)]:
        img = _image(rng, h, w)
        assert np.array_equal(fit_model(img, 31, 200), tools.fit(img, 200, 31, cval=0)), (h, w)


@pytest.mark.parametrize("shape", [(0, 10, 3), (10, 0, 3), (0, 0, 3)])
def test_fit_plan_raises_zero_division_for_empty_crops(shape):
    img = np.zeros(shape, np.uint8)
    with pytest.raises(ZeroDivisionError):
        tools.fit(img, 200, 31, cval=0)
    with pytest.raises(ZeroDivisionError):
        tools.fit_plan(shape, 200, 31)


@pytest.mark.parametrize("shape,height,width", [((1, 1000, 3), 31, 200), ((1000, 1, 3), 31, 200), ((1, 300, 3), 48, 128)])
def test_fit_plan_raises_cv2_error_when_a_resized_side_is_empty(shape, height, width):
    assert resize_is_empty(shape[:2], height, width)
    with pytest.raises(cv2.error):
        tools.fit(np.zeros(shape, np.uint8), width, height, cval=0)
    with pytest.raises(cv2.error):
        tools.fit_plan(shape, width, height)


def test_fit_return_scale_and_crop_mode_unchanged():
    """fit's scale (min of the two ratios for letterbox, max for crop) and the crop mode still follow the reference."""
    img = np.zeros((40, 300, 3), np.uint8)
    _, scale = tools.fit(img, 200, 31, cval=0, return_scale=True)
    assert scale == 200 / 300
    out, scale = tools.fit(img, 200, 31, mode="crop", return_scale=True)
    assert scale == 31 / 40 and out.shape == (31, 200, 3)
    assert tools.fit_plan(img.shape, 200, 31, mode="crop") == (31, int(31 / 40 * 300))
    assert tools.fit(np.zeros((31, 200, 3), np.uint8), 200, 31, return_scale=True)[1] == 1
