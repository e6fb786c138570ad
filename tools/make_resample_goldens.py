"""Golden vectors of the sample-rate converter (tests/golden/resample.npz), produced with scipy 1.18's
``scipy.signal.resample_poly`` (default ``padtype='constant'``) and ``scipy.signal.firwin``.

For every m = max(up, down) of the rate pairs of PAIRS: ``firwin(2 hl + 1, 1 / m, window=('kaiser', 5.0))`` in float64
(``firwin_{m}``; the pair's taps are that times up).  For every pair and each length of LENGTHS: ``resample_poly`` of the
seeded fp32 input ``oracle.resample_oracle.make_test_input(seed, n, rate_in)`` in float64, the first and last 128 outputs and
every 37th in between (``{rate_in}_{rate_out}_{n}`` and the output indices ``..._idx``), which keeps the file to a few hundred
KB.

scipy is needed by this tool only; the tests read the npz.

    python tools/make_resample_goldens.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.resample_oracle import make_test_input  # noqa: E402

PAIRS = [(24_000, 48_000), (24_000, 44_100), (24_000, 22_050), (24_000, 16_000), (24_000, 8_000),
         (48_000, 24_000), (44_100, 24_000), (22_050, 24_000), (16_000, 24_000), (11_025, 24_000)]
LENGTHS = [1, 2, 1919, 1920, 48_007]


def kept(n_out: int) -> np.ndarray:
    return np.unique(np.concatenate([np.arange(min(128, n_out)), np.arange(0, n_out, 37), np.arange(max(0, n_out - 128), n_out)]))


def main():
    from math import gcd

    from scipy.signal import firwin, resample_poly

    out = {"pairs": np.array(PAIRS, dtype=np.int64), "lengths": np.array(LENGTHS, dtype=np.int64)}
    for pi, (r_in, r_out) in enumerate(PAIRS):
        g = gcd(r_in, r_out)
        up, down = r_out // g, r_in // g
        m = max(up, down)
        out[f"firwin_{m}"] = firwin(2 * 10 * m + 1, 1.0 / m, window=("kaiser", 5.0))
        for li, n in enumerate(LENGTHS):
            seed = 100 * pi + li
            x = make_test_input(seed, n, r_in).astype(np.float64)
            y = resample_poly(x, up, down)
            assert len(y) == -(-n * up // down)
            key = f"{r_in}_{r_out}_{n}"
            out[key + "_seed"] = np.array(seed, dtype=np.int64)
            idx = kept(len(y))
            out[key + "_idx"] = idx.astype(np.int64)
            out[key] = y[idx]
        print(r_in, "->", r_out, f"up {up} down {down}", 20 * m + 1, "taps")
    path = os.path.join(ROOT, "tests", "golden", "resample.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
