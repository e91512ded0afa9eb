"""Shared by the CPU and GPU test files: deterministic inputs (identical to tests/golden/make_golden.py)."""
import ast
import hashlib

import numpy as np


def gen_input(seed, shape, dt):
    rng = np.random.Generator(np.random.PCG64(seed))
    if dt == "u8":
        return rng.integers(0, 256, size=shape, dtype=np.uint8)
    if dt == "i64":
        return rng.integers(-2**40, 2**40, size=shape, dtype=np.int64)
    if dt == "bool":
        return rng.integers(0, 2, size=shape).astype(np.bool_)
    return rng.standard_normal(size=shape).astype(np.float32)


def batcher_trials(golden):
    return [ast.literal_eval(str(t)) for t in golden["trials"]]


def batcher_random_seed(trial, mode, item):
    """Input seed of item `item` of random Batcher trial `trial` (tests/golden/batcher_random_golden.npz)."""
    return 100000 + 200 * trial + 100 * (mode == "cat") + item


def digest(a):
    """64 bits of the SHA-256 of an array's dtype, shape and bytes: stands in for outputs too large to store verbatim."""
    h = hashlib.sha256(f"{a.dtype.str}{tuple(a.shape)}".encode() + np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest()[:8], dtype="<u8")[0]


def tree_masks(n):
    """All arrival-order bitmasks that matter for an n-peer tree (nodes with two children)."""
    nodes = [p for p in range(1, n) if 2 * p + 1 < n]
    masks = []
    for bits in range(1 << len(nodes)):
        m = 0
        for k, p in enumerate(nodes):
            if (bits >> k) & 1:
                m |= 1 << p
        masks.append(m)
    return masks
