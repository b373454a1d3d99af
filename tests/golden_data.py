"""The committed reference outputs, tests/golden/<case>.npz, as make_golden.py writes them and the tests read them.

A file holds one float32 array per output.  To keep every fixture under 1 MB, an output of more than MAX_ELEMS elements
is stored as a fixed sample: `<key>` holds its values at MAX_ELEMS positions drawn once from a seeded generator, in
flattened order, and `<key>_mask` marks those positions (np.packbits of a boolean array of the output's size)."""
import numpy as np
import torch

MAX_ELEMS = 200_000


def shrink(arrays, seed):
    """The arrays to store for one case: small outputs whole, larger ones as a sample plus its mask."""
    out = {}
    for key, a in arrays.items():
        if a.size <= MAX_ELEMS:
            out[key] = a
            continue
        mask = np.zeros(a.size, dtype=bool)
        mask[np.random.default_rng(seed).choice(a.size, MAX_ELEMS, replace=False)] = True
        out[key] = a.reshape(-1)[mask]
        out[key + "_mask"] = np.packbits(mask)
    return out


def stored(gold, key, a):
    """`a` (a numpy array or tensor of the output's full shape) at the positions `gold` holds for `key`, flattened in the
    same order, or `a` itself when `key` is stored whole."""
    if key + "_mask" not in gold.files:
        return a
    mask = np.unpackbits(gold[key + "_mask"], count=int(np.prod(a.shape))).astype(bool).reshape(tuple(a.shape))
    return a[mask] if isinstance(a, np.ndarray) else a[torch.from_numpy(mask)]
