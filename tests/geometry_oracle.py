"""The fp32 oracle of a recognizer built with another crop size (build_params height / width / rnn_steps_to_discard).

``oracle.crnn.crnn_logits`` is shape-generic up to the LSTM outputs (the time axis is width // 4 long, the feature height
height // 4) but drops the default 2 steps; this applies fc_12 to its full-length ``l2`` and drops ``rnn_steps_to_discard``
instead (the ``x[:, d:]`` Lambda of the reference, recognition.py:328).  Used by the crop-geometry tests and by
``scripts/make_crnn_geometry_fixture.py``."""
import numpy as np
import torch

from oracle import crnn


def crnn_logits(weights, crops, rnn_steps_to_discard):
    """crops (B,h,w[,C]) float32 in [0,1] -> (softmax (B,w//4-d,K), intermediates with "logits" (B,w//4-d,K))."""
    with torch.no_grad():
        _, inter = crnn.crnn_logits(weights, crops, return_intermediates=True)
        k = torch.as_tensor(np.asarray(weights["fc_12.kernel"]), dtype=torch.float32)
        b = torch.as_tensor(np.asarray(weights["fc_12.bias"]), dtype=torch.float32)
        logits = inter["l2"] @ k + b
    d = int(rnn_steps_to_discard)
    return torch.softmax(logits, -1)[:, d:], dict(inter, logits=logits[:, d:])
