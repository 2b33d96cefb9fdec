"""CPU: the dependency-free HDF5 reader (keras_ocr_b200/hdf5.py) that loads the reference's Keras weight files
(crnn_kurapan.h5, reference recognition.py:27-44, 386-392) without h5py."""
import sys
import os

import numpy as np
import pytest

from keras_ocr_b200 import hdf5, weights as W

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from h5_writer import write  # noqa: E402


def test_round_trip_groups_contiguous_and_chunked(tmp_path):
    rng = np.random.default_rng(0)
    big = rng.standard_normal((70, 33)).astype(np.float32)            # chunked 32 x 16 with ragged edge chunks
    tree = {
        "a": {"a": {"kernel:0": rng.standard_normal((3, 3, 4, 8)).astype(np.float32), "bias:0": np.arange(8, dtype=np.float32)}},
        "many": {f"d{i:02d}": np.full((i + 1,), i, np.float64) for i in range(21)},     # three symbol-table nodes
        "ints": np.arange(-5, 7, dtype=np.int32).reshape(3, 4),
        "big": big,
        "scalar": np.float32(2.5).reshape(()),
    }
    for userblock in (0, 512):
        path = str(tmp_path / f"t{userblock}.h5")
        write(path, tree, chunked={id(big): (32, 16)}, userblock=userblock)
        got = hdf5.read_datasets(path)
        flat = {"a/a/kernel:0": tree["a"]["a"]["kernel:0"], "a/a/bias:0": tree["a"]["a"]["bias:0"], "ints": tree["ints"],
                "big": big, "scalar": tree["scalar"], **{f"many/{k}": v for k, v in tree["many"].items()}}
        assert set(got) == set(flat)
        for k, v in flat.items():
            assert got[k].dtype == v.dtype and got[k].shape == v.shape and np.array_equal(got[k], v), k
    with pytest.raises(hdf5.Hdf5Error):
        hdf5.read_datasets(b"not an hdf5 file at all" * 100)


def test_reads_a_file_written_by_the_hdf5_c_library(golden_dir):
    """A real HDF5 file: scipy's MATLAB v7.3 test fixture, stored in tests/golden (HDF5 1.8 C library, 512-byte user
    block, object-header continuation blocks).  Its twin in MATLAB's own v7 format, read by scipy, holds the same
    variable."""
    import scipy.io
    got = hdf5.read_datasets(os.path.join(golden_dir, "testhdf5_7.4_GLNX86.mat"))
    assert list(got) == ["testdouble"] and got["testdouble"].dtype == np.float64
    twin = scipy.io.loadmat(os.path.join(golden_dir, "testdouble_7.4_GLNX86.mat"))["testdouble"]
    assert np.array_equal(got["testdouble"].ravel(), twin.ravel())


def test_keras_checkpoint_round_trip_through_hdf5(tmp_path):
    """A full CRNN checkpoint laid out as Keras ``save_weights`` does (``<layer>/<layer>/<kind>:0``, the spatial
    transformer's localisation net under auto-generated names, LSTM weights one group deeper), written to disk and read
    back through ``weights.load_keras_h5`` -- no h5py involved."""
    w = W.synthetic_crnn_weights(4)
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
    for wrapped in (False, True):                                       # model.save() nests everything under model_weights
        path = str(tmp_path / f"crnn_{wrapped}.h5")
        write(path, {"model_weights": tree} if wrapped else tree)
        back = W.load_keras_h5(path)
        assert set(back) == set(w)
        assert all(np.array_equal(back[k], w[k]) for k in w)
