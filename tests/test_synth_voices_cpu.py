"""Host side of poly synths and granulators in voice batches: the Python mirror's constants and preset table against the C
header and the oracle's PolyConfig::preset, and the argument checks the mirror makes before any device work."""
import os
import re

import numpy as np
import pytest

from libgooey_b200 import voices as V
from libgooey_b200._lib import GooeyError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def c_float_table(path, name, rows, cols):
    """The `name[rows][cols] = {{...}, ...}` float table of a C++ source, as float32."""
    with open(os.path.join(ROOT, path)) as f:
        text = f.read()
    m = re.search(re.escape(name) + r"\[%d\]\[%d\]\s*=\s*\{(.*?)\};" % (rows, cols), text, re.S)
    assert m, name
    vals = [float(x) for x in re.findall(r"(-?\d+\.\d*)f", m.group(1))]
    assert len(vals) == rows * cols
    return np.array(vals, np.float32).reshape(rows, cols)


def test_poly_presets_equal_the_oracle_table():
    names = ["default", "pad", "pluck", "keys", "strings"]    # PolyConfig::preset ids 0-4
    assert list(V.POLY_PRESETS) == names
    mine = np.array([V.POLY_PRESETS[k] for k in names], np.float32)
    assert np.array_equal(mine, c_float_table("oracle/sources.hpp", "T", 5, 14))
    assert np.array_equal(mine, c_float_table("libgooey_b200/csrc/engine_api.cuh", "GOOEY_POLY_PRESETS", 5, 14))


def test_voice_kind_ids_follow_the_header():
    with open(os.path.join(ROOT, "include", "gooey_batch.h")) as f:
        text = f.read()
    assert int(re.search(r"#define GOOEY_B200_VOICE_POLY (\d+)u", text).group(1)) == V.POLY == 5
    assert int(re.search(r"#define GOOEY_B200_VOICE_GRANULATOR (\d+)u", text).group(1)) == V.GRANULATOR == 6
    p = V.patch(V.POLY, V.POLY_PRESETS["pad"])
    assert p.instrument == 5 and np.allclose(list(p.params)[:14], V.POLY_PRESETS["pad"])


def unbound_batch():
    """A VoiceBatch whose handle was never created: any call that reached the library would fail on the NULL handle."""
    b = V.VoiceBatch.__new__(V.VoiceBatch)
    b._h = None
    b.n = 1
    return b


@pytest.mark.parametrize("note", [128, 255, -1, 1000])
def test_note_on_refuses_notes_outside_the_midi_range(note):
    with pytest.raises(GooeyError, match="note"):
        unbound_batch().note_on(0, note, 1.0)


@pytest.mark.parametrize("samples", [np.zeros(0, np.float32), np.zeros((2, 3), np.float32), []])
def test_set_buffer_refuses_empty_or_multichannel_arrays(samples):
    with pytest.raises(GooeyError, match="set_buffer"):
        unbound_batch().set_buffer(0, samples, 44100.0)
