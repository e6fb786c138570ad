"""The sample-rate converter's host side, no GPU: the filter design (smoltts_b200/resample.py) and the float64 oracle
(oracle/resample_oracle.py) against scipy's firwin / resample_poly (tests/golden/resample.npz), the streaming output counts,
and the C ABI's ratio checks."""
import ctypes
from math import gcd

import numpy as np

from conftest import GOLDEN_DIR

_G = {}


def _golden():
    if "g" not in _G:
        _G["g"] = np.load(f"{GOLDEN_DIR}/resample.npz")
    return _G["g"]


def _pairs():
    return [tuple(int(v) for v in p) for p in _golden()["pairs"]]


def _ratio(r_in, r_out):
    g = gcd(r_in, r_out)
    return r_out // g, r_in // g


def test_design_filter_matches_firwin():
    from smoltts_b200.resample import design_filter

    g = _golden()
    for r_in, r_out in _pairs():
        up, down = _ratio(r_in, r_out)
        want = g[f"firwin_{max(up, down)}"] * up
        got = design_filter(r_in, r_out)
        assert got.shape == want.shape == (20 * max(up, down) + 1,)
        assert np.abs(got - want).max() <= 1e-15, (r_in, r_out, np.abs(got - want).max())


def test_oracle_matches_resample_poly_and_streams_to_the_same_samples():
    from oracle.resample_oracle import make_test_input, resample, resample_stream
    from smoltts_b200.resample import design_filter

    g = _golden()
    rng = np.random.default_rng(5)
    worst = 0.0
    for r_in, r_out in _pairs():
        up, down = _ratio(r_in, r_out)
        h = design_filter(r_in, r_out)
        for n in (int(v) for v in g["lengths"]):
            key = f"{r_in}_{r_out}_{n}"
            x = make_test_input(int(g[key + "_seed"]), n, r_in)
            y = resample(x, up, down, h)
            assert len(y) == -(-n * up // down)
            want = g[key]
            err = np.abs(y[g[key + "_idx"]] - want).max()
            worst = max(worst, err)
            assert err <= 1e-12, (key, err)
            if n < 1000 or n > 10_000:
                continue
            cuts = np.sort(rng.integers(0, n + 1, size=int(rng.integers(1, 12))))
            parts = resample_stream(np.split(x, cuts), up, down, h)
            assert np.array_equal(np.concatenate(parts), y), key
    print(f"largest |oracle - resample_poly| over the goldens: {worst:.3g}")


def test_output_counts_follow_the_oracle():
    from oracle.resample_oracle import resample_stream
    from smoltts_b200.resample import design_filter, output_count

    rng = np.random.default_rng(7)
    for r_in, r_out in _pairs():
        up, down = _ratio(r_in, r_out)
        h = design_filter(r_in, r_out)
        for trial in range(4):
            n = int(rng.integers(0, 6000))
            cuts = np.sort(rng.integers(0, n + 1, size=int(rng.integers(0, 10))))
            chunks = np.split(rng.standard_normal(n), cuts)
            parts = resample_stream(chunks, up, down, h)
            S = E = 0
            for c, p in zip(chunks + [None], parts):
                finish = c is None
                S += 0 if finish else len(c)
                n_out = output_count(S, up, down, finish) - E
                assert len(p) == n_out, (r_in, r_out, S, finish)
                E += n_out
            assert E == -(-n * up // down)


def test_create_accepts_ratios_up_to_320():
    from smoltts_b200 import _capi

    lib = _capi.load()

    def create(r_in, r_out, max_streams=4):
        h = ctypes.c_void_p()
        rc = lib.smol_resampler_create(ctypes.byref(_capi.SmolResampleConfig(rate_in=r_in, rate_out=r_out, max_streams=max_streams)),
                                       ctypes.byref(h))
        return rc, h

    for r_in, r_out in [(11_025, 24_000), (24_000, 11_025), (24_000, 192_000), (192_000, 24_000), (320, 319), (1, 320), (320, 1),
                        (24_000, 24_000)]:
        rc, h = create(r_in, r_out)
        assert rc == _capi.SMOL_OK, (r_in, r_out, lib.smol_last_error())
        up, down = _ratio(r_in, r_out)
        assert lib.smol_resampler_taps(h) == 20 * max(up, down) + 1
        K = -(-(20 * max(up, down) + 1) // up)
        assert lib.smol_resampler_workspace_bytes(h) >= (up * K + 4 * 2 * K) * 4
        lib.smol_resampler_destroy(h)
    for r_in, r_out in [(321, 320), (320, 321), (24_000, 7_999), (44_100, 32_000), (1, 321)]:
        rc, _ = create(r_in, r_out)
        assert rc == _capi.SMOL_ERR_UNSUPPORTED, (r_in, r_out)
        assert b"above the limit of 320" in lib.smol_last_error(), lib.smol_last_error()
    for bad in ((0, 24_000, 1), (24_000, 48_000, 0)):
        assert create(*bad)[0] == _capi.SMOL_ERR_INVALID


def test_compute_before_bind_is_refused():
    from smoltts_b200 import _capi

    lib = _capi.load()
    h = ctypes.c_void_p()
    assert lib.smol_resampler_create(ctypes.byref(_capi.SmolResampleConfig(rate_in=24_000, rate_out=48_000, max_streams=2)),
                                     ctypes.byref(h)) == 0
    lens, slots, counts = (ctypes.c_int64 * 1)(1920), (ctypes.c_int32 * 1)(0), (ctypes.c_int64 * 1)()
    assert lib.smol_resample(h, ctypes.c_void_p(8), lens, slots, 1, 0, ctypes.c_void_p(8), counts, None) == _capi.SMOL_ERR_UNBOUND
    assert b"not bound" in lib.smol_last_error()
    assert lib.smol_resampler_reset(h, slots, 1, None) == _capi.SMOL_ERR_UNBOUND
    lib.smol_resampler_destroy(h)

