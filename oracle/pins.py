"""TEST INFRASTRUCTURE ONLY -- digests of the values that the oracle-vs-reference tests compare with the reference.

``tests/golden/reference_pins.json`` maps a test id to one short digest per item of the values the test compares
(per person, per round, ...), so that without the reference tree the oracle is still checked against what the reference
returned, and a mismatch names the item that diverged.
"""
import hashlib
import json

import numpy as np
import torch


def digest(values):
    """SHA-256 over nested lists / tuples of arrays, tensors and JSON-able values: dtype, shape and bytes of every array."""
    h = hashlib.sha256()

    def feed(v):
        if isinstance(v, (list, tuple)):
            h.update(b"[%d;" % len(v))
            for x in v:
                feed(x)
        elif isinstance(v, torch.Tensor):
            feed(v.detach().cpu().numpy())
        elif isinstance(v, (np.ndarray, np.generic)):
            a = np.ascontiguousarray(v)
            h.update(("%s%s;" % (a.dtype.str, a.shape)).encode() + a.tobytes())
        else:
            h.update(json.dumps(v, sort_keys=True, default=lambda x: x.tolist()).encode() + b";")
    feed(values)
    return h.hexdigest()


def item_digests(values):
    """One 64-bit digest (hex) per item of a list / tuple, or a single one for anything else."""
    items = values if isinstance(values, (list, tuple)) else [values]
    return [digest(v)[:16] for v in items]


def mismatch(recorded, got):
    """None if the two digest lists agree, else a short description of where they differ."""
    if recorded == got:
        return None
    if len(recorded) != len(got):
        return "%d items recorded, %d computed" % (len(recorded), len(got))
    bad = [i for i, (a, b) in enumerate(zip(recorded, got)) if a != b]
    return "items %s of %d differ" % (bad[:20], len(got))
