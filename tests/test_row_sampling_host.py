"""Host side of per-sequence sampling settings, no GPU: the SmolRowSampling records ``row_sampling_table`` packs (the same
values a call's SmolSampling would carry), its validation, and the ctypes layouts of SmolRowSampling / SmolBatch against
the C header."""
import ctypes
import math
import subprocess

import pytest
import torch

from conftest import ROOT
from smoltts_b200 import _capi
from smoltts_b200.generate import GenerationSettings, row_sampling_table


def _records(table):
    return [_capi.SmolRowSampling.from_buffer_copy(bytes(row.numpy())) for row in table]


def test_records_carry_each_rows_settings():
    settings = [GenerationSettings(),
                GenerationSettings(default_temp=0.0, default_fast_temp=None, top_k=50, top_p=0.9, seed=2 ** 64 - 1),
                GenerationSettings(default_temp=1.0, default_fast_temp=0.5, min_p=0.1, min_p_intended=True, seed=12),
                GenerationSettings(min_p=0.1)]     # min_p without min_p_intended is the reference's no-op
    table = row_sampling_table(settings)
    assert table.dtype == torch.uint8 and tuple(table.shape) == (4, 32)
    r = _records(table)
    f32 = lambda v: float(ctypes.c_float(v).value)  # noqa: E731
    assert (r[0].temp, r[0].fast_temp, r[0].top_k, r[0].top_p, r[0].min_p, r[0].seed) == (f32(0.7), f32(0.7), 0, 1.0, 0.0, 0)
    assert (r[1].temp, r[1].fast_temp, r[1].top_k, r[1].top_p, r[1].seed) == (0.0, 0.0, 50, f32(0.9), 2 ** 64 - 1)
    assert (r[2].temp, r[2].fast_temp, r[2].min_p, r[2].seed) == (1.0, 0.5, f32(0.1), 12)
    assert r[3].min_p == 0.0
    assert all(x.pad == 0 for x in r)


def test_records_equal_the_call_level_sampling_fields():
    """A row record holds exactly what generate._sampling puts into the call's SmolSampling for the same settings."""
    from smoltts_b200.generate import _sampling

    class _Host:   # RQTransformer.sampling is host code only
        from smoltts_b200.model import RQTransformer
        sampling = RQTransformer.sampling

    s = GenerationSettings(default_temp=0.55, default_fast_temp=0.25, top_k=7, top_p=0.8, min_p=0.03, min_p_intended=True, seed=99)
    call = _sampling(_Host(), s, audio_only=True)
    (rec,) = _records(row_sampling_table([s]))
    for name in ("temp", "fast_temp", "top_k", "top_p", "min_p", "seed"):
        assert getattr(rec, name) == getattr(call, name), name


@pytest.mark.parametrize("bad", [dict(default_temp=-0.1), dict(default_temp=math.nan), dict(default_fast_temp=math.inf),
                                 dict(default_fast_temp=-1.0), dict(top_k=-1), dict(top_p=0.0), dict(top_p=1.01),
                                 dict(top_p=math.nan), dict(min_p=1.0), dict(min_p=-0.01)])
def test_invalid_settings_are_refused_on_the_host(bad):
    with pytest.raises(ValueError):
        row_sampling_table([GenerationSettings(), GenerationSettings(**bad)])


def test_empty_settings_list_is_refused():
    with pytest.raises(ValueError):
        row_sampling_table([])


def test_ctypes_layouts_match_the_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "smoltts_b200.h"\n'
        "int main(void) {\n"
        '  printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(SmolRowSampling), offsetof(SmolRowSampling, top_k),\n'
        "         offsetof(SmolRowSampling, min_p), offsetof(SmolRowSampling, seed), sizeof(SmolBatch),\n"
        "         offsetof(SmolBatch, max_frames), offsetof(SmolBatch, row_sampling));\n"
        '  printf("%d\\n", SMOL_ABI_VERSION);\n'
        "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", f"{ROOT}/include", str(src), "-o", str(exe)], check=True)
    sizes, version = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")[:2]
    R, B = _capi.SmolRowSampling, _capi.SmolBatch
    want = [ctypes.sizeof(R), R.top_k.offset, R.min_p.offset, R.seed.offset, ctypes.sizeof(B), B.max_frames.offset, B.row_sampling.offset]
    assert [int(v) for v in sizes.split()] == want
    assert want[0] == 32
    assert int(version) == _capi.SMOL_ABI_VERSION == 2
