"""CPU oracle of the sample-rate converter -- TEST INFRASTRUCTURE, never imported by the product.

Restates ``scipy.signal.resample_poly(x, up, down)`` (default ``padtype='constant'``) in float64 numpy, straight from its
polyphase formula: with ``hl = (len(h) - 1) / 2`` and ``x`` zero outside ``[0, L)``, the ``ceil(L up / down)`` outputs are

    y[k] = sum over j = (k down + hl) mod up, step up, of h[j] x[(k down + hl - j) / up]

``resample`` is the whole clip; ``resample_stream`` runs the same sums a chunk at a time, the way ``csrc/resample.cu`` does:
a history of the last ``ceil(len(h) / up)`` samples, the outputs whose support has arrived after each chunk, the rest at the
end.  ``tests/test_resample_host.py`` pins both against ``tests/golden/resample.npz`` (made with scipy by
``tools/make_resample_goldens.py``).
"""
from __future__ import annotations

from typing import List, Sequence

import numpy as np


def _outputs(h: np.ndarray, up: int, down: int, x: np.ndarray, x0: int, k0: int, k1: int) -> np.ndarray:
    """y[k0 .. k1 - 1] from the samples x, which start at absolute index x0 and are zero outside what they cover."""
    M = len(h)
    hl = (M - 1) // 2
    K = -(-M // up)
    k = np.arange(k0, k1, dtype=np.int64)
    t = k * down + hl
    ph, n0 = t % up, t // up
    i = np.arange(K, dtype=np.int64)
    j = ph[:, None] + up * i[None, :]                            # tap index, ascending
    n = n0[:, None] - i[None, :] - x0                            # sample index within x
    valid = (j < M) & (n >= 0) & (n < len(x))
    taps = np.where(j < M, h[np.minimum(j, M - 1)], 0.0)
    xs = np.where(valid, x[np.clip(n, 0, max(len(x) - 1, 0))] if len(x) else 0.0, 0.0)
    return (taps * xs).sum(axis=1)


def resample(x: np.ndarray, up: int, down: int, h: np.ndarray) -> np.ndarray:
    x = np.asarray(x, dtype=np.float64)
    n_out = -(-len(x) * up // down)
    return _outputs(np.asarray(h, dtype=np.float64), up, down, x, 0, 0, n_out)


def emitted(n_in: int, up: int, down: int, hl: int, finish: bool) -> int:
    """Outputs of a stream after n_in samples: complete support (largest input index n0 <= n_in - 1), or all at the end."""
    if finish:
        return -(-n_in * up // down)
    return 0 if n_in * up <= hl else (n_in * up - 1 - hl) // down + 1


def resample_stream(chunks: Sequence[np.ndarray], up: int, down: int, h: np.ndarray) -> List[np.ndarray]:
    """One output array per chunk plus the tail at the end (len(chunks) + 1 arrays)."""
    h = np.asarray(h, dtype=np.float64)
    hl = (len(h) - 1) // 2
    K = -(-len(h) // up)
    hist = np.zeros(K)                                            # samples S - K .. S - 1 (zeros before the start)
    S = E = 0
    out = []
    for c in list(chunks) + [None]:
        finish = c is None
        c = np.zeros(0) if finish else np.asarray(c, dtype=np.float64)
        S1 = S + len(c)
        E1 = emitted(S1, up, down, hl, finish)
        out.append(_outputs(h, up, down, np.concatenate([hist, c]), S - K, E, E1))
        hist = np.concatenate([hist, c])[-K:]
        S, E = S1, E1
    return out


def make_test_input(seed: int, n: int, rate: int) -> np.ndarray:
    """The seeded fp32 input of the goldens: ``synth.make_test_audio`` at ``rate`` plus white noise of std 0.1."""
    from smoltts_b200.synth import make_test_audio

    rng = np.random.default_rng(10_000 + seed)
    x = make_test_audio(seed, n, sampling_rate=rate).numpy().astype(np.float64) + 0.1 * rng.standard_normal(n)
    return x.astype(np.float32)
