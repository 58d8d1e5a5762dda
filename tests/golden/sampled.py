"""Fixed samples of large reference outputs, so the golden fixtures stay small.

At the test sizes the reference's outputs are tens of megabytes of float data that does not compress.  A fixture keeps
masks and small arrays whole; for a large array it keeps the values at a fixed set of positions (every channel of each
position) together with the array's shape and channel axis.  The positions are a Weyl sequence over the flattened
non-channel axes: evenly spread and derived from the shape alone, with no random generator, so they are the same with
any numpy.  A test compares its own full output at the same positions (Golden.pick).
"""
import math

import numpy as np

_PHI = 0.6180339887498949


def positions(n_total: int, n: int) -> np.ndarray:
    """`n` distinct flat indices spread evenly over [0, n_total), ascending (all of them when n >= n_total)."""
    if n >= n_total:
        return np.arange(n_total)
    step = max(1, int(n_total * _PHI))
    while math.gcd(step, n_total) != 1:
        step += 1
    return np.sort((np.arange(n, dtype=np.int64) * step) % n_total)


def _numpy(a) -> np.ndarray:
    return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)


def take(a, axis: int, n: int) -> np.ndarray:
    """[n, C]: the channel vectors (C = a.shape[axis]) of `a` at `n` fixed positions."""
    a = np.moveaxis(_numpy(a), axis, -1)
    rows = a.reshape(-1, a.shape[-1])
    return rows[positions(rows.shape[0], n)]


def shrink(arrays: dict, spec: dict) -> dict:
    """Fixture contents: arrays named in `spec` ({name: (channel axis, positions)}) are sampled, the rest stay whole."""
    out = {}
    for k, a in arrays.items():
        a = _numpy(a)
        if k in spec:
            axis, n = spec[k]
            axis %= a.ndim
            out[k] = take(a, axis, n)
            out[k + "__shape"] = np.array(a.shape, dtype=np.int64)
            out[k + "__axis"] = np.array(axis, dtype=np.int64)
        else:
            out[k] = a
    return out


class Golden:
    """Read side of a fixture written by shrink(): g[k] is what was stored (the samples, for a sampled array)."""

    def __init__(self, path: str):
        with np.load(path) as z:
            self._z = {k: z[k] for k in z.files}

    def __getitem__(self, k: str) -> np.ndarray:
        return self._z[k]

    def shape(self, k: str) -> tuple:
        return tuple(int(v) for v in self._z[k + "__shape"]) if k + "__shape" in self._z else self._z[k].shape

    def pick(self, k: str, a) -> np.ndarray:
        """The values of `a` -- a full output of the shape stored for sampled array `k`, or a per-position array (the
        same shape without the channel axis, such as a mask) -- at k's positions: [n, C] or [n].  For an array stored
        whole, `a` itself after checking its shape."""
        a = _numpy(a)
        if k + "__shape" not in self._z:
            assert a.shape == self._z[k].shape, (k, a.shape, self._z[k].shape)
            return a
        shape, axis, n = self.shape(k), int(self._z[k + "__axis"]), self._z[k].shape[0]
        if a.shape == shape[:axis] + shape[axis + 1:]:
            return take(np.expand_dims(a, axis), axis, n)[:, 0]
        assert a.shape == shape, (k, a.shape, shape)
        return take(a, axis, n)
