"""Golden fixtures stay under 1 MB a file.  An output too large for that is stored as a fixed sample of its elements
(`<key>_sample`, with the full shape in `<key>_shape`); a smaller one is stored whole under `<key>`.  The generators
write through `pack`, the tests read through `pair`, so both agree on which elements were kept.

TEST INFRASTRUCTURE.  Never imported by `latte_b200/`."""
import math

import numpy as np
import torch

SAMPLE = 1 << 17        # elements kept of a sampled output (512 KB of float32)
_STRIDE = 1_000_003     # prime: i * _STRIDE mod n visits distinct elements spread over the whole array


def sample_index(n: int, k: int) -> np.ndarray:
    """`k` distinct flat indices into `n` elements, sorted.  Integer arithmetic only, so it is the same everywhere."""
    assert 0 < k <= n and math.gcd(_STRIDE, n) == 1, (n, k)
    return np.sort(np.arange(k, dtype=np.int64) * _STRIDE % n)


def pack(key: str, a: np.ndarray, k: int = SAMPLE) -> dict:
    """`{key: a}` when `a` has at most `k` elements, else its `k` elements at `sample_index` and its shape."""
    if a.size <= k:
        return {key: a}
    return {f"{key}_sample": a.reshape(-1)[sample_index(a.size, k)], f"{key}_shape": np.array(a.shape, dtype=np.int64)}


def stored(g, key: str):
    """(shape, flat indices, values) of the output `key` that `pack` wrote into the golden `g`, whole or sampled."""
    if key in g:
        a = g[key]
        return tuple(a.shape), np.arange(a.size, dtype=np.int64), a.reshape(-1)
    shape = tuple(int(s) for s in g[f"{key}_shape"])
    values = g[f"{key}_sample"]
    return shape, sample_index(math.prod(shape), values.size), values


def pair(g, key: str, got: torch.Tensor):
    """(got, want), flattened, for the golden `g[key]` written by `pack`: the stored elements and the same elements of
    `got`.  Asserts that `got` has the shape of the stored output."""
    shape, idx, want = stored(g, key)
    assert tuple(got.shape) == shape, (tuple(got.shape), shape)
    return got.reshape(-1)[torch.from_numpy(idx).to(got.device)], torch.from_numpy(want)
