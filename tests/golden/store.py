"""Storage format of the golden ``.npz`` files: an array of at most ``SAMPLE`` elements is stored whole; a larger one keeps
the ``SAMPLE`` elements at ``sample_index`` of its flattened form, with its shape under ``<name>.shape``.  This keeps each
file well under 1 MB while every test still compares whole-output shapes and a spread of elements."""

from __future__ import annotations

import math

import numpy as np
import torch

SAMPLE = 8192


def sample_index(numel: int, k: int = SAMPLE) -> np.ndarray:
    """``k`` distinct flat indices in ``[0, numel)``: a multiplicative stride coprime with ``numel``, so every row and column
    residue is reached.  Pure integer arithmetic, so the selection never changes with a library version."""
    if numel <= k:
        return np.arange(numel)
    p = int(numel * 0.6180339887)
    while math.gcd(p, numel) != 1:
        p += 1
    return (np.arange(k, dtype=np.int64) * p) % numel


def pack(arrays: dict) -> dict:
    """What ``np.savez_compressed`` writes for ``arrays`` (name -> full output)."""
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.size > SAMPLE:
            out[name] = a.reshape(-1)[sample_index(a.size)]
            out[name + ".shape"] = np.array(a.shape, dtype=np.int64)
        else:
            out[name] = a
    return out


class Golden:
    """A golden file; ``pair(name, got)`` checks ``got``'s shape and returns (the stored elements of ``got``, the golden ones)."""

    def __init__(self, path: str) -> None:
        self.z = np.load(path)

    def __getitem__(self, name: str) -> np.ndarray:
        assert name + ".shape" not in self.z.files, f"{name} is stored as a sample: compare through pair()"
        return self.z[name]

    def pair(self, name: str, got: torch.Tensor):
        ref = torch.from_numpy(self.z[name])
        shape = tuple(int(s) for s in self.z[name + ".shape"]) if name + ".shape" in self.z.files else tuple(ref.shape)
        assert tuple(got.shape) == shape, (name, tuple(got.shape), shape)
        got = got.detach().cpu()
        if name + ".shape" in self.z.files:
            got = got.reshape(-1)[torch.from_numpy(sample_index(got.numel()))]
        return got, ref
