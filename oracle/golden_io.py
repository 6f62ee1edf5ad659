"""Fixture files under tests/golden/ stay below 1 MB each: save() cuts an array that would not fit along one axis over
<name>.npz, <name>.part1.npz, ..., and load() joins it back, so a test sees exactly the array the generator computed."""
from __future__ import annotations

import numpy as np

MAX_SPLIT_BYTES = 900_000            # raw bytes of the cut array per file (float heatmaps barely compress)


def save(path: str, arrays: dict, split_key: str | None = None, axis: int = 1) -> None:
    """np.savez_compressed(path, **arrays); arrays[split_key], if larger than MAX_SPLIT_BYTES, is cut along `axis` into
    as many equal parts as keep each below it, the first stored in `path` and part i in <path without .npz>.part<i>.npz."""
    arrays = dict(arrays)
    if split_key is not None and arrays[split_key].nbytes > MAX_SPLIT_BYTES:
        parts = np.array_split(arrays[split_key], -(-arrays[split_key].nbytes // MAX_SPLIT_BYTES), axis=axis)
        arrays.update({split_key: parts[0], "split_key": np.array(split_key), "split": np.array([axis, len(parts)], np.int64)})
        for i, p in enumerate(parts[1:], 1):
            np.savez_compressed(f"{path[:-4]}.part{i}.npz", **{split_key: p})
    np.savez_compressed(path, **arrays)


def load(path: str) -> dict:
    """The arrays save() was given."""
    g = dict(np.load(path))
    if "split_key" in g:
        key = str(g.pop("split_key"))
        axis, n = (int(v) for v in g.pop("split"))
        g[key] = np.concatenate([g[key]] + [np.load(f"{path[:-4]}.part{i}.npz")[key] for i in range(1, n)], axis=axis)
    return g
