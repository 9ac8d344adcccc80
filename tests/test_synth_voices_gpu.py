"""Poly synths and granulators in voice batches (gooey_voice_batch_note_on / release / set_buffer / share_buffer / set_seed and
set_param for both kinds) against the oracle's bare PolySynth and Granulator, the poly synth's warp-per-voice back end
(poly_wave_kernel) against the per-sample-order one (GOOEY_B200_BACKEND=serial) bit for bit, and the refusals, which queue
nothing.  Tolerance against the oracle: 1e-5 of full scale."""
import ctypes

import numpy as np
import pytest

from libgooey_b200 import engine as G, voices as V
from libgooey_b200._lib import GooeyError, lib
import emu_lib as E
import oracle_lib as O

pytestmark = pytest.mark.gpu
TOL = 1e-5
PRESET_NAMES = ["default", "pad", "pluck", "keys", "strings"]


def stat_names():
    L = lib()
    L.gooey_b200_kernel_stat_names.restype = ctypes.c_char_p
    return {s for s in (L.gooey_b200_kernel_stat_names() or b"").decode().split(";") if s}


def c4_source(n=44100, seed=9):
    """SURVEY 8d C4 source formula (shortened): 220 Hz tone with a slow tremolo plus uniform noise."""
    i = np.arange(n, dtype=np.float64)
    rng = np.random.default_rng(seed)
    x = 0.5 * np.sin(2 * np.pi * 220.0 * i / 44100.0) * (0.5 + 0.5 * np.sin(2 * np.pi * 0.1 * i / 44100.0)) + 0.1 * rng.uniform(-1, 1, n)
    return x.astype(np.float32)


# ---- poly synth against the oracle ----------------------------------------------------------------------------------------
# Oracle events (frame, kind, a, b): kind 0 trigger_note(a = note, b = velocity), 1 release_all, 2 set_param(a = id, b = value).
POLY_SCENARIOS = [
    # a chord at frame 0, released mid-block
    [(0, 0, 48, 0.9), (0, 0, 55, 0.9), (0, 0, 64, 0.9), (0, 0, 71, 0.9), (20011, 1, 0, 0)],
    # a chord mid-block, then three more notes: the seventh note steals the oldest sub-voice; a cutoff glide without snap
    [(1013, 0, 60, 0.7), (1013, 0, 64, 0.7), (1013, 0, 67, 0.7), (1013, 0, 70, 0.7),
     (3000, 2, 2, 0.85), (7017, 0, 72, 1.0), (7017, 0, 76, 1.0), (7017, 0, 79, 0.5), (15011, 1, 0, 0), (16500, 0, 36, 0.6)],
    # short amp release and decay times (set while no note sounds): envelopes end mid-block, a velocity above 1 passes unclamped
    [(0, 2, 8, 0.0), (0, 2, 6, 0.05), (0, 2, 12, 0.0), (7000, 0, 57, 1.3), (7000, 0, 61, 0.4), (9005, 1, 0, 0),
     (9203, 0, 127, 0.8), (9203, 0, 0, 0.8), (12345, 1, 0, 0), (20000, 0, 69, 1.0), (20100, 1, 0, 0)],
]
POLY_FRAMES = 30000
RENDER_CALLS = [5000, 7001, 31, 12000, POLY_FRAMES - 5000 - 7001 - 31 - 12000]


def queue_poly(b, voice, ev, offset=0):
    for (f, kind, a, x) in ev:
        if kind == 0:
            b.note_on(voice, int(a), x, frame=f - offset)
        elif kind == 1:
            b.release(voice, frame=f - offset)
        else:
            b.set_param(voice, int(a), x, frame=f - offset)


def render_split(b, calls, between=None):
    outs, pos = [], 0
    for i, n in enumerate(calls):
        if between:
            between(i, pos)
        outs.append(b.render(n))
        pos += n
    return np.concatenate(outs, axis=1)


@pytest.mark.parametrize("sr", [44100.0, 48000.0])
@pytest.mark.parametrize("preset", PRESET_NAMES)
def test_poly_voices_match_oracle(preset, sr):
    pid = PRESET_NAMES.index(preset)
    n = len(POLY_SCENARIOS)
    b = V.VoiceBatch([V.patch(V.POLY, V.POLY_PRESETS[preset])] * n, sr)
    # voice 0: every event queued before the first call (most lie beyond it); voices 1, 2: each event queued in the call it
    # falls into, relative to that call's start
    queue_poly(b, 0, POLY_SCENARIOS[0])

    def between(i, pos):
        end = pos + RENDER_CALLS[i]
        for v in (1, 2):
            queue_poly(b, v, [e for e in POLY_SCENARIOS[v] if pos <= e[0] < end], offset=pos)
    got = render_split(b, RENDER_CALLS, between)
    b.close()
    for v, ev in enumerate(POLY_SCENARIOS):
        want = E.poly_render(O.lib().orc_poly_render, pid, ev, POLY_FRAMES, sr)
        err = float(np.abs(got[v] - want).max())
        print(f"poly {preset} @ {sr:.0f} Hz scenario {v}: max |gpu - oracle| = {err:.3e}, peak {np.abs(want).max():.3f}")
        assert np.abs(want).max() > 1e-3
        assert err <= TOL


# ---- poly synth: warp-per-voice back end against the per-sample-order back end, bit for bit -----------------------------
def random_poly_batch(n, seed, sr=44100.0):
    rng = np.random.default_rng(seed)
    presets = rng.integers(0, 5, n)
    b = V.VoiceBatch([V.patch(V.POLY, V.POLY_PRESETS[PRESET_NAMES[p]]) for p in presets], sr)
    for v in range(n):
        style = v % 4
        t = int(rng.integers(0, 40))                      # first chord at frame 0 or mid-block
        if style == 2:                                     # short envelopes: amp ends mid-block after release / decay
            b.set_param(v, 8, float(rng.uniform(0.0, 0.15)), snap=True)
            b.set_param(v, 6, float(rng.uniform(0.0, 0.3)), snap=True)
            b.set_param(v, 7, 0.0 if rng.random() < 0.5 else 0.6, snap=True)
        for note in rng.integers(24, 100, int(rng.integers(1, 7))):
            b.note_on(v, int(note), float(rng.uniform(0.2, 1.2)), frame=t)
        if style == 1:                                     # a glide mid-render, no snap
            b.set_param(v, int(rng.integers(0, 14)), float(rng.random()), frame=int(rng.integers(100, 8000)))
        if style == 3:                                     # a snapped edit
            b.set_param(v, int(rng.integers(0, 14)), float(rng.random()), frame=int(rng.integers(100, 8000)), snap=True)
        r = int(rng.integers(2000, 14000))
        b.release(v, frame=r)
        for note in rng.integers(30, 90, int(rng.integers(0, 8))):   # retrigger: up to 7 more notes steal sub-voices
            b.note_on(v, int(note), float(rng.uniform(0.1, 1.0)), frame=r + int(rng.integers(1, 6000)))
        if rng.random() < 0.5:
            b.release(v, frame=int(rng.integers(16000, 23000)))
    return b


def test_poly_wave_back_end_is_bit_identical_to_serial(monkeypatch):
    n, calls = 4096, [7000, 9001, 8000]
    outs, names = [], []
    for serial in (True, False):
        if serial:
            monkeypatch.setenv("GOOEY_B200_BACKEND", "serial")
        else:
            monkeypatch.delenv("GOOEY_B200_BACKEND")
        b = random_poly_batch(n, seed=11)
        lib().gooey_b200_kernel_stats_reset()
        outs.append(render_split(b, calls))
        names.append(stat_names())
        b.close()
    ser, got = outs
    print("serial:", sorted(names[0]), "default:", sorted(names[1]))
    assert "slow_kernel<PolyV>" in names[0] and "poly_wave_kernel" not in names[0]
    assert "poly_wave_kernel" in names[1] and "slow_kernel<PolyV>" not in names[1]
    assert np.isfinite(got).all() and np.abs(got).max() > 0.05
    diff = np.count_nonzero(ser.view(np.uint32) != got.view(np.uint32))
    print(f"{n} poly voices x {sum(calls)} frames: {diff} samples differ from the serial back end, max |diff| {np.abs(ser - got).max():.3e}")
    assert diff == 0


def test_poly_wave_back_end_in_ffi_engines_is_bit_identical_to_serial(monkeypatch):
    def run():
        es = [G.Engine() for _ in range(6)]
        rng = np.random.default_rng(5)
        outs = []
        for i, e in enumerate(es):
            e.poly_trigger_notes([int(x) for x in rng.integers(36, 84, 3 + i % 4)], i % 5, float(rng.uniform(0.3, 1.0)))
        outs.append(np.stack([e.render(9000) for e in es]))
        for i, e in enumerate(es):
            if i % 2:
                e.poly_release()
            else:
                e.poly_trigger_notes([int(x) for x in rng.integers(36, 84, 6)], (i + 2) % 5, 0.8)
        outs.append(np.stack([e.render(15000) for e in es]))
        for e in es:
            e.close()
        return np.concatenate(outs, axis=1)
    monkeypatch.setenv("GOOEY_B200_BACKEND", "serial")
    lib().gooey_b200_kernel_stats_reset()
    ser = run()
    ser_names = stat_names()
    monkeypatch.delenv("GOOEY_B200_BACKEND")
    lib().gooey_b200_kernel_stats_reset()
    got = run()
    names = stat_names()
    print("serial:", sorted(ser_names), "default:", sorted(names))
    assert "poly_wave_kernel" in names and "poly_wave_kernel" not in ser_names
    assert np.abs(got).max() > 1e-3
    assert np.array_equal(ser.view(np.uint32), got.view(np.uint32))


def test_poly_pcm16_is_the_quantised_f32_render():
    def make():
        return random_poly_batch(64, seed=3)
    b = make(); f32 = b.render(20001); b.close()
    b = make(); pcm = b.render_pcm16(20001); b.close()
    r = (f32 * np.float32(32767.0)).astype(np.float32)
    r = np.where(np.isnan(r), np.float32(0), np.sign(r) * np.floor(np.abs(r) + np.float32(0.5)))
    assert np.abs(f32).max() > 0.05
    assert np.array_equal(pcm, np.clip(r, -32768, 32767).astype(np.int16))


# ---- granulator against the oracle ----------------------------------------------------------------------------------------
# Oracle events (frame, kind, a, b): kind 0 trigger(b = velocity), 2 set_param(a, b), 3 snap_params, 4 set_seed(a).
GRAN_SCENARIOS = [
    # C4 style: parameters snapped, a seed, one long cloud
    [(0, 2, 4, 1.0), (0, 2, 1, 0.55), (0, 2, 2, 0.5), (0, 2, 3, 0.4), (0, 2, 6, 0.3), (0, 2, 5, 0.7), (0, 2, 9, 0.3), (0, 2, 10, 0.3),
     (0, 2, 7, 1.0), (0, 3, 0, 0), (0, 4, 7, 0), (0, 0, 0, 0.9)],
    # parameters gliding (no snap), a trigger mid-render, drive
    [(0, 2, 4, 0.8), (0, 2, 11, 0.6), (0, 2, 1, 0.2), (1500, 0, 0, 1.0), (6000, 2, 3, 0.9), (6000, 2, 0, 0.1)],
    # default seed, a reseed and retrigger mid-render, seed 0
    [(0, 2, 4, 0.9), (0, 2, 7, 0.2), (0, 3, 0, 0), (100, 0, 0, 0.7), (12000, 4, 0, 0), (12000, 0, 0, 0.5), (17000, 4, 12345, 0),
     (17000, 2, 3, 0.7), (17000, 3, 0, 0), (17000, 0, 0, 1.0)],
]


def queue_gran(b, voice, ev):
    for (f, kind, a, x) in ev:
        if kind == 0:
            b.trigger(voice, f, x)
        elif kind == 2:
            b.set_param(voice, int(a), x, frame=f)
        elif kind == 3:
            snap_all(b, voice, f)
        else:
            b.set_seed(voice, int(a), frame=f)


def snap_all(b, voice, frame):
    # EV_SNAP after re-setting a parameter to its own target is snap_params: G_VOLUME is never edited by these scenarios, so
    # its target is still GranulatorConfig::default's 0.8
    b.set_param(voice, 8, 0.8, frame=frame, snap=True)


def test_granulator_voices_match_oracle():
    src = c4_source()
    frames = 30000
    n = len(GRAN_SCENARIOS)
    b = V.VoiceBatch([V.patch(V.GRANULATOR)] * n + [V.patch(V.KICK, V.KICK_PRESETS["punch"])])
    b.set_buffer(0, src, 44100.0)
    for v in range(1, n):
        b.share_buffer(v, 0)
    for v, ev in enumerate(GRAN_SCENARIOS):
        queue_gran(b, v, ev)
    got = np.concatenate([b.render(12000), b.render(frames - 12000)], axis=1)
    b.close()
    for v, ev in enumerate(GRAN_SCENARIOS):
        want = E.gran_render(O.lib().orc_gran_render, src, ev, frames)
        err = float(np.abs(got[v] - want).max())
        print(f"granulator scenario {v}: max |gpu - oracle| = {err:.3e}, peak {np.abs(want).max():.3f}")
        assert np.abs(want).max() > 0.01
        assert err <= TOL


def test_256_granulators_on_one_shared_buffer():
    src = c4_source(2 * 44100, seed=4)
    n, frames = 256, 16000
    rng = np.random.default_rng(21)
    seeds = rng.integers(1, 2**24, n)                  # the oracle's event table carries the seed as a float32
    pitch = rng.uniform(0.2, 0.8, n)
    b = V.VoiceBatch([V.patch(V.GRANULATOR)] * n)
    b.set_buffer(0, src, 44100.0)
    evs = []
    for v in range(n):
        if v:
            b.share_buffer(v, (v - 1) // 2)                # shared along a chain of voices: all hold voice 0's copy
        ev = [(0, 2, 4, 1.0), (0, 2, 1, 0.4), (0, 2, 3, float(pitch[v])), (0, 3, 0, 0), (0, 4, int(seeds[v]), 0), (0, 0, 0, 0.9)]
        queue_gran(b, v, ev)
        evs.append(ev)
    got = b.render(frames)
    b.close()
    errs = [float(np.abs(got[v] - E.gran_render(O.lib().orc_gran_render, src, evs[v], frames)).max()) for v in range(n)]
    print(f"{n} granulators on one buffer: max |gpu - oracle| = {max(errs):.3e}")
    assert np.abs(got).max(axis=1).min() > 0.01
    assert max(errs) <= TOL
    assert len({got[v].tobytes() for v in range(n)}) == n    # per-voice seeds and pitches give distinct clouds


# ---- refusals queue nothing -----------------------------------------------------------------------------------------------
def test_refusals_queue_nothing_and_no_ops_stay_no_ops():
    L = lib()
    src = c4_source(8000)
    f32p = ctypes.POINTER(ctypes.c_float)
    patches = [V.patch(V.POLY, V.POLY_PRESETS["keys"]), V.patch(V.GRANULATOR), V.patch(V.KICK, V.KICK_PRESETS["punch"]), V.patch(V.GRANULATOR)]

    def make():
        b = V.VoiceBatch(patches)
        b.note_on(0, 60, 0.9); b.note_on(0, 67, 0.7, frame=500); b.release(0, frame=6000)
        b.set_buffer(1, src, 44100.0); b.set_param(1, 4, 1.0, snap=True); b.set_seed(1, 3); b.trigger(1, 0, 1.0)
        b.trigger(2, 100, 1.0)
        return b

    def arr(x):
        x = np.ascontiguousarray(x, np.float32)
        return x, x.ctypes.data_as(f32p)

    ref = make(); want = ref.render(9000); ref.close()
    b = make()
    good, gp = arr(src)
    nan_buf, nanp = arr(np.r_[src[:10], np.nan])
    inf_buf, infp = arr(np.r_[src[:10], np.inf])
    refused = [
        ("note_on voice out of range", lambda: L.gooey_voice_batch_note_on(b._h, 4, 0, 60, ctypes.c_float(1.0))),
        ("release voice out of range", lambda: L.gooey_voice_batch_release(b._h, 4, 0)),
        ("set_buffer voice out of range", lambda: L.gooey_voice_batch_set_buffer(b._h, 4, 0, gp, good.size, ctypes.c_float(44100.0))),
        ("share_buffer dst out of range", lambda: L.gooey_voice_batch_share_buffer(b._h, 4, 0, 1)),
        ("share_buffer src out of range", lambda: L.gooey_voice_batch_share_buffer(b._h, 3, 0, 4)),
        ("set_seed voice out of range", lambda: L.gooey_voice_batch_set_seed(b._h, 4, 0, 1)),
        ("note_on on a granulator", lambda: L.gooey_voice_batch_note_on(b._h, 1, 0, 60, ctypes.c_float(1.0))),
        ("note_on on a kick", lambda: L.gooey_voice_batch_note_on(b._h, 2, 0, 60, ctypes.c_float(1.0))),
        ("release on a kick", lambda: L.gooey_voice_batch_release(b._h, 2, 0)),
        ("note above 127", lambda: L.gooey_voice_batch_note_on(b._h, 0, 10, 128, ctypes.c_float(1.0))),
        ("set_buffer on a poly voice", lambda: L.gooey_voice_batch_set_buffer(b._h, 0, 0, gp, good.size, ctypes.c_float(44100.0))),
        ("set_buffer on a kick", lambda: L.gooey_voice_batch_set_buffer(b._h, 2, 0, gp, good.size, ctypes.c_float(44100.0))),
        ("share_buffer to a poly voice", lambda: L.gooey_voice_batch_share_buffer(b._h, 0, 0, 1)),
        ("share_buffer from a kick", lambda: L.gooey_voice_batch_share_buffer(b._h, 3, 0, 2)),
        ("share_buffer from a voice without buffer", lambda: L.gooey_voice_batch_share_buffer(b._h, 1, 0, 3)),
        ("set_seed on a poly voice", lambda: L.gooey_voice_batch_set_seed(b._h, 0, 0, 9)),
        ("NULL samples", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, None, 10, ctypes.c_float(44100.0))),
        ("empty buffer", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, gp, 0, ctypes.c_float(44100.0))),
        ("NaN sample", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, nanp, nan_buf.size, ctypes.c_float(44100.0))),
        ("infinite sample", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, infp, inf_buf.size, ctypes.c_float(44100.0))),
        ("sample rate 0", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, gp, good.size, ctypes.c_float(0.0))),
        ("negative sample rate", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, gp, good.size, ctypes.c_float(-44100.0))),
        ("NaN sample rate", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, gp, good.size, ctypes.c_float(np.nan))),
        ("infinite sample rate", lambda: L.gooey_voice_batch_set_buffer(b._h, 3, 0, gp, good.size, ctypes.c_float(np.inf))),
    ]
    for what, call in refused:
        L.gooey_b200_last_error.restype = ctypes.c_char_p
        rc = call()
        msg = L.gooey_b200_last_error().decode()
        print(f"{what}: rc {rc}, {msg}")
        assert rc == -1, what
        assert msg, what
    with pytest.raises(GooeyError):
        b.note_on(0, 200)
    with pytest.raises(GooeyError):
        b.set_buffer(1, np.zeros(0, np.float32), 44100.0)
    with pytest.raises(GooeyError):
        b.share_buffer(1, 3)
    # accepted, without effect: a trigger on a poly voice, unknown parameter ids
    b.trigger(0, 200, 1.0)
    b.set_param(0, 14, 0.3, snap=True)
    b.set_param(1, 12, 0.3, snap=True)
    got = b.render(9000)
    b.close()
    assert np.abs(want[:2]).max(axis=1).min() > 0.01
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
