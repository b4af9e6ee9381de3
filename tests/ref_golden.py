"""Golden outputs of the reference's compiled code (tests/golden/ref/<name>.npz), shared by the tests that pin the oracle
and the Python mirror to the reference. tests/golden/make_ref_golden.py records them by running those tests with
LIMAP_REF_RECORD=1, where oracle/_ref has been built; everywhere else the tests read them."""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")
RECORD = os.environ.get("LIMAP_REF_RECORD") == "1"


def _narrow(a):
    """Integers are stored in the narrowest type that holds them (the tests compare values, not types)."""
    if a.dtype.kind == "i" and a.size:  # signed only: uint8 byte streams stay bytes
        for t in (np.int8, np.int16, np.int32):
            if np.iinfo(t).min <= a.min() and a.max() <= np.iinfo(t).max:
                return a.astype(t)
    return a


def reference(name, compute):
    """The compiled reference's outputs for one test: tests/golden/ref/<name>.npz, recomputed by `compute` (which calls
    oracle/_ref) and stored again when LIMAP_REF_RECORD=1. The arrays of one test are stored as one byte stream
    (`data`) and one line per array in `index` ("name dtype shape"): a file holds dozens of small arrays, and one
    compressed stream keeps it a fraction of the size of one .npy entry each."""
    path = os.path.join(GOLD, name + ".npz")
    if RECORD:
        os.makedirs(GOLD, exist_ok=True)
        arrays = {k: np.array(_narrow(np.asarray(v)), order="C") for k, v in compute().items()}
        index = [f"{k} {a.dtype.str} {','.join(map(str, a.shape))}" for k, a in arrays.items()]
        data = b"".join(a.tobytes() for a in arrays.values())
        np.savez_compressed(path, index=np.array(index), data=np.frombuffer(data, np.uint8))
    with np.load(path) as z:
        index, data = z["index"], z["data"].tobytes()
    out, pos = {}, 0
    for line in index:
        k, dt, shape = str(line).split(" ")
        shape = tuple(int(n) for n in shape.split(",") if n)
        a = np.frombuffer(data, np.dtype(dt), count=int(np.prod(shape, dtype=np.int64)), offset=pos).reshape(shape)
        out[k] = a.copy()
        pos += a.nbytes
    return out
