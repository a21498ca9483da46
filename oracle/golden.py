"""Golden-vector files (tests/golden/*.npz) whose largest arrays are stored as a sample.

Golden files stay under 1 MB.  Where a case's whole arrays would not fit, ``sample`` keeps a fixed,
seeded sample of the elements of the arrays it is given:

    <key>          the sampled values, 1-D, in flat-index order
    <key>_index    their flat indices into the whole array (sorted)
    <key>_shape    the whole array's shape
    <key>_rms      the whole array's rms, so a tolerance relative to it is the one of the whole array

``Golden`` reads both kinds of file; ``pick`` takes the same elements out of a whole computed array.
"""
import numpy as np


def sample(arrays, keys, fraction, seed=0):
    """``arrays`` with each array named in ``keys`` replaced by a seeded sample of ``fraction`` of its elements."""
    out = dict(arrays)
    rng = np.random.default_rng(seed)
    for k in keys:
        a = np.asarray(arrays[k])
        idx = np.sort(rng.choice(a.size, int(round(a.size * fraction)), replace=False)).astype(np.int32)
        out[k] = a.reshape(-1)[idx]
        out[k + "_index"] = idx
        out[k + "_shape"] = np.array(a.shape, dtype=np.int64)
        out[k + "_rms"] = np.array(np.sqrt(np.mean(np.square(a, dtype=np.float64))))
    return out


class Golden:
    """One golden .npz; ``g[key]`` is the stored array (the sample, for a sampled key)."""

    def __init__(self, path):
        self.d = np.load(path)

    def __getitem__(self, key):
        return self.d[key]

    def sampled(self, key):
        return key + "_index" in self.d.files

    def shape(self, key):
        return tuple(int(s) for s in self.d[key + "_shape"]) if self.sampled(key) else self.d[key].shape

    def rms(self, key):
        if self.sampled(key):
            return float(self.d[key + "_rms"])
        return float(np.sqrt(np.mean(np.square(self.d[key], dtype=np.float64))))

    def pick(self, key, a):
        """The elements of ``a`` (the whole array of ``key``, or one that broadcasts to it) the file stores for ``key``."""
        a = np.asarray(a)
        if not self.sampled(key):
            return a
        return np.broadcast_to(a, self.shape(key)).reshape(-1)[self.d[key + "_index"]]
