"""Host-side helpers of the hot path (reference keras_ocr/tools.py, hot subset only)."""
import hashlib
import io
import os
import typing

import numpy as np


def read(filepath_or_buffer: typing.Union[str, io.BytesIO, np.ndarray]):
    """tools.read (reference tools.py:19-38): ndarrays pass through; files / buffers are decoded to
    RGB on the host (image decode stays host-side, SURVEY.md 8(a) row 2).  URLs need a network and
    are not supported offline."""
    if isinstance(filepath_or_buffer, np.ndarray):
        return filepath_or_buffer
    import cv2

    if hasattr(filepath_or_buffer, "read"):
        data = np.asarray(bytearray(filepath_or_buffer.read()), dtype=np.uint8)
        image = cv2.imdecode(data, cv2.IMREAD_UNCHANGED)
    elif isinstance(filepath_or_buffer, str):
        assert os.path.isfile(filepath_or_buffer), "Could not find image at path: " + filepath_or_buffer
        image = cv2.imread(filepath_or_buffer)
    else:
        raise TypeError(f"cannot read image from {type(filepath_or_buffer)!r}")
    return cv2.cvtColor(image, cv2.COLOR_BGR2RGB)


def read_device(filepath_or_buffer, ctx, device):
    """``read`` with the decode on the GPU where possible (SURVEY.md 8(f)2): a JPEG file / buffer is handed to nvJPEG
    through ``b2o_decode_jpeg`` and comes back as an (H, W, 3) uint8 RGB CUDA tensor -- only the compressed bytes cross
    PCIe.  Everything else (arrays, PNG, JPEG flavours nvJPEG refuses, a box without nvJPEG) goes through ``read`` and is
    returned as the host array the caller uploads as before."""
    import torch

    if isinstance(filepath_or_buffer, (np.ndarray, torch.Tensor)):
        return filepath_or_buffer
    if isinstance(filepath_or_buffer, str):
        assert os.path.isfile(filepath_or_buffer), "Could not find image at path: " + filepath_or_buffer
        with open(filepath_or_buffer, "rb") as f:
            data = f.read()
    elif hasattr(filepath_or_buffer, "read"):
        data = filepath_or_buffer.read()
    else:
        raise TypeError(f"cannot read image from {type(filepath_or_buffer)!r}")
    if data[:2] == b"\xff\xd8":                                  # JPEG start-of-image marker
        info = ctx.jpeg_info(data)
        if info is not None and info[2] in (1, 3):
            h, w, _ = info
            out = torch.empty((h, w, 3), dtype=torch.uint8, device=device)
            if ctx.decode_jpeg(data, out.data_ptr(), h, w, torch.cuda.current_stream(device).cuda_stream):
                return out
    return read(io.BytesIO(data))


def resize_plan(shape, max_scale, max_size):
    """The scale and output size tools.resize_image (reference tools.py:378-398) would pick.

    Returns (scale, out_h, out_w).  ``max(shape)`` includes the channel axis, as upstream."""
    longest = max(shape)
    scale = max_size / longest if longest * max_scale > max_size else max_scale
    return scale, int(shape[0] * scale), int(shape[1] * scale)


def adjust_boxes(boxes, scale=1, boxes_format="boxes"):
    """tools.adjust_boxes (reference tools.py:232-260)."""
    if scale == 1:
        return boxes
    if boxes_format == "boxes":
        return np.array(boxes) * scale
    if boxes_format == "lines":
        return [[(np.array(box) * scale, character) for box, character in line] for line in boxes]
    if boxes_format == "predictions":
        return [(word, np.array(box) * scale) for word, box in boxes]
    raise NotImplementedError(f"Unsupported boxes format: {boxes_format}")


def fit_plan(shape, width, height, mode="letterbox"):
    """The cv2.resize size tools.fit (reference tools.py:402-452) picks for an image of ``shape``: None when it returns
    the image unchanged (it already is ``height`` x ``width``), else ``(new_h, new_w)``.  Python floats as upstream:
    ``sx = width / w``, ``sy = height / h``, letterbox scales by the width when ``sx <= sy`` (crop when ``sx >= sy``),
    the other side is truncated with ``int()``.  Raises what ``fit`` raises: ZeroDivisionError for an image without
    rows or columns, cv2.error when a resized side would be 0 (e.g. 1 x 1000 into 31 x 200).  ``fit`` and the batched
    GPU fit (``Recognizer.recognize_batch``, ``b2o_fit_crops``) both follow this plan."""
    h, w = int(shape[0]), int(shape[1])
    sx, sy = width / w, height / h
    if sx == 1 and sy == 1:
        return None
    if mode not in ("letterbox", "crop"):
        raise NotImplementedError(f"Unsupported mode: {mode}")
    use_width = (sx <= sy) if mode == "letterbox" else (sx >= sy)
    new_h, new_w = (int(sx * h), width) if use_width else (height, int(sy * w))
    if new_h <= 0 or new_w <= 0:
        import cv2

        raise cv2.error(f"tools.fit: {h} x {w} resized to {new_h} x {new_w}; cv2.resize needs a non-empty size")
    return new_h, new_w


def fit(image, width, height, cval=255, mode="letterbox", return_scale=False):
    """tools.fit (reference tools.py:402-452): scale the image to fit ``width`` x ``height`` keeping
    its aspect ratio, then letterbox (pad bottom/right with ``cval``) or crop.  Host-side like the
    reference; the size comes from ``fit_plan``.  ``Recognizer.recognize`` uses it for one crop; bulk
    recognition (``Recognizer.recognize_batch``) runs the same plan on the GPU with ``b2o_fit_crops``."""
    import cv2

    plan = fit_plan(image.shape, width, height, mode)
    if plan is None:
        return (image, 1) if return_scale else image
    sx, sy = width / image.shape[1], height / image.shape[0]
    scale = min(sx, sy) if mode == "letterbox" else max(sx, sy)
    new_h, new_w = plan
    resized = cv2.resize(image, dsize=(new_w, new_h))
    if mode == "letterbox":
        fitted = np.zeros((height, width, 3), dtype="uint8") + cval
        fitted[: resized.shape[0], : resized.shape[1]] = resized[:height, :width]
    else:
        fitted = resized[:height, :width]
    return (fitted, scale) if return_scale else fitted


def read_and_fit(filepath_or_array, width, height, cval=255, mode="letterbox"):
    """tools.read_and_fit (reference tools.py:455-481)."""
    image = read(filepath_or_array) if isinstance(filepath_or_array, str) else filepath_or_array
    return fit(image=image, width=width, height=height, cval=cval, mode=mode)


def sha256sum(filename):
    """tools.sha256sum (reference tools.py:484-492)."""
    h = hashlib.sha256()
    with open(filename, "rb") as f:
        for chunk in iter(lambda: f.read(128 * 1024), b""):
            h.update(chunk)
    return h.hexdigest()


def get_default_cache_dir():
    """tools.get_default_cache_dir (reference tools.py:495-498)."""
    return os.environ.get("KERAS_OCR_CACHE_DIR", os.path.expanduser(os.path.join("~", ".keras-ocr")))


def find_cached(filename, sha256=None, cache_dir=None):
    """Offline half of tools.download_and_verify (reference tools.py:501-530): locate and verify a
    weight file that is already in the cache; there is no network here to download it."""
    path = os.path.join(cache_dir or get_default_cache_dir(), filename)
    assert os.path.isfile(path), (
        f"{path} not found and no network is available to download it; pass weights=<dict|path> instead")
    assert sha256 is None or sha256 == sha256sum(path), "Error occurred verifying sha256."
    return path


# ----------------------------------------------------------------------------------- box geometry (host)
def _convex_hull(points):
    """Counter-clockwise convex hull (Andrew's monotone chain) of (n,2) float64 points, collinear points dropped."""
    pts = sorted(set(map(tuple, np.asarray(points, dtype=np.float64).tolist())))
    if len(pts) <= 2:
        return np.array(pts, dtype=np.float64).reshape(-1, 2)

    def cross(o, a, b):
        return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])

    lower, upper = [], []
    for p in pts:
        while len(lower) >= 2 and cross(lower[-2], lower[-1], p) <= 0:
            lower.pop()
        lower.append(p)
    for p in reversed(pts):
        while len(upper) >= 2 and cross(upper[-2], upper[-1], p) <= 0:
            upper.pop()
        upper.append(p)
    return np.array(lower[:-1] + upper[:-1], dtype=np.float64)


def minimum_rotated_rectangle(points):
    """shapely ``MultiPoint(points).minimum_rotated_rectangle`` as the reference uses it (tools.py:544-547), restated:
    for every edge of the convex hull, the axis-parallel bounding rectangle in that edge's frame; the one of least
    area, transformed back.  Returns (4,2) float64, or None when the hull has no area (shapely then returns a point
    or a line, ``.exterior`` raises AttributeError and the reference falls back to the raw points, tools.py:548-550).
    shapely is not installable offline, so this follows its published algorithm (PARITY UNPINNED beyond that)."""
    hull = _convex_hull(points)
    if len(hull) < 3:
        return None
    best, best_area = None, None
    for i in range(len(hull)):
        dx, dy = hull[(i + 1) % len(hull)] - hull[i]
        length = float(np.hypot(dx, dy))
        ux, uy = dx / length, dy / length
        vx, vy = -uy, ux
        a, b = hull @ np.array([ux, uy]), hull @ np.array([vx, vy])          # coordinates in the edge's frame
        area = (a.max() - a.min()) * (b.max() - b.min())
        # Ties are common (two edges whose rectangles are spanned by the same triangle of the quad have equal areas in
        # exact arithmetic): an edge only wins if it is smaller by more than rounding, i.e. the FIRST edge in hull order
        # (counter-clockwise from the lexicographically smallest vertex) wins a tie.
        if best_area is None or area < best_area * (1.0 - 1e-9):
            corners = np.array([[a.min(), b.min()], [a.max(), b.min()], [a.max(), b.max()], [a.min(), b.max()]])
            best = corners @ np.array([[ux, uy], [vx, vy]])                  # back to image coordinates
            best_area = area
    return best


def get_rotated_box(points):
    """tools.get_rotated_box (reference tools.py:533-581): minimum rotated rectangle of the points, corners ordered
    top-left, top-right, bottom-right, bottom-left (the imutils rule), float32, plus the rotation angle."""
    points = np.asarray(points)
    pts = minimum_rotated_rectangle(points)
    if pts is None:
        pts = points
    x_sorted = pts[np.argsort(pts[:, 0]), :]
    left, right = x_sorted[:2, :], x_sorted[2:, :]
    tl, bl = left[np.argsort(left[:, 1]), :]
    d = np.sqrt(((right - tl[np.newaxis]) ** 2).sum(1))
    br, tr = right[np.argsort(d)[::-1], :]
    out = np.array([tl, tr, br, bl], dtype="float32")
    with np.errstate(divide="ignore", invalid="ignore"):
        rotation = np.arctan((tl[0] - bl[0]) / (tl[1] - bl[1]))
    return out, rotation


def get_rotated_width_height(box):
    """tools.get_rotated_width_height (reference tools.py:41-57): truncated mean lengths of opposite sides."""
    box = np.asarray(box, dtype=np.float64)

    def dist(a, b):
        return float(np.sqrt(((box[a] - box[b]) ** 2).sum()))

    return int((dist(0, 1) + dist(2, 3)) / 2), int((dist(0, 3) + dist(1, 2)) / 2)


def rectify_boxes(boxes, tolerance=1e-3):
    """What ``tools.warpBox`` does to a caller-supplied quad before it builds the homography (reference
    tools.py:88-95): replace it by its minimum rotated rectangle and measure that rectangle.  A quad that already IS
    a rectangle (every corner within ``tolerance`` px of the rectified one -- everything ``getBoxes`` emits) is kept
    bit for bit, so boxes that come from the detector are not perturbed by the fp64 round trip.  Raises
    ZeroDivisionError for a box whose width or height truncates to 0, as the reference does (tools.py:95).
    boxes: (n,4,2) -> (n,4,2) float32."""
    boxes = np.asarray(boxes, dtype=np.float32).reshape(-1, 4, 2)
    out = boxes.copy()
    for k, quad in enumerate(boxes):
        rect, _ = get_rotated_box(quad)
        w, h = get_rotated_width_height(rect)
        if w == 0 or h == 0:
            raise ZeroDivisionError("division by zero")          # scale = min(target_width / w, target_height / h)
        nearest = np.abs(rect[:, None, :] - quad[None, :, :]).max(-1).min(-1)      # each rectified corner vs the quad's
        if nearest.max() > tolerance:
            out[k] = rect
    return out


# ----------------------------------------------------------------------------------- drawing (host, cv2)
def _plain_boxes(boxes, boxes_format):
    """The (4,2) corner arrays inside any of the three box containers the reference passes around."""
    if boxes_format == "lines":
        return [quad for line in boxes for quad, _character in line]
    if boxes_format == "predictions":
        return [quad for _word, quad in boxes]
    return list(boxes)


def drawBoxes(image, boxes, color=(255, 0, 0), thickness=5, boxes_format="boxes"):
    """tools.drawBoxes (reference tools.py:189-229): the outlines of ``boxes`` on a copy of ``image``.  ``boxes_format``:
    "boxes" = (N,4,2) array as from ``Detector.detect``; "lines" = lists of (box, character); "predictions" = (word, box)
    tuples as from ``Pipeline.recognize``.  An empty container returns the image itself, as upstream."""
    import cv2

    if len(boxes) == 0:
        return image
    canvas = image.copy()
    for quad in _plain_boxes(boxes, boxes_format):
        cv2.polylines(canvas, np.asarray(quad)[np.newaxis].astype("int32"), True, color, thickness)
    return canvas


def drawAnnotations(image, predictions, ax=None):
    """tools.drawAnnotations (reference tools.py:150-186): the boxes on the image plus every recognised word in the
    margin -- words whose box starts in the left half on the left, the others on the right, each column top to bottom
    in the order of the boxes' upper edges, joined to its box by a red arrow.  Needs matplotlib, like upstream."""
    import matplotlib.pyplot as plt

    if ax is None:
        ax = plt.subplots()[1]
    ax.imshow(drawBoxes(image, predictions, boxes_format="predictions"))
    ax.set_xticks([])
    ax.set_yticks([])
    height, width = image.shape[:2]
    columns = {"left": [], "right": []}
    for word, quad in sorted(predictions, key=lambda item: item[1][:, 1].min()):
        columns["left" if quad[:, 0].min() < width / 2 else "right"].append((word, quad))
    for side, entries in columns.items():
        for rank, (word, quad) in enumerate(entries):
            anchor = (quad[0][0] / width, 1 - quad[0][1] / height)              # axes fraction, y upwards
            label_at = (-0.05 if side == "left" else 1.05, 1 - rank / len(entries))
            ax.annotate(text=word, xy=anchor, xytext=label_at, xycoords="axes fraction", color="r", fontsize=14,
                        arrowprops={"arrowstyle": "->", "color": "r"},
                        horizontalalignment="right" if side == "left" else "left")
    return ax
