"""The back end a batch is rendered with (pool.cuh launch_back), as the kernel statistics record it.  Every voice kind
records exactly one back-end key with all its voice-frames; LFO-routed basses take the per-sample kernel.  For the drums,
at the batch sizes that select each one (choose_back): toms from 4096 per launch take the cooperative back end, kick /
snare / hi-hat from 12 288 the one-voice-per-thread back end, smaller buckets the warp-per-voice back end.  The
cooperative back end is checked at a size that selects it against the per-sample-order back end
(GOOEY_B200_BACKEND=serial) and against the oracle."""
import ctypes

import numpy as np
import pytest

from libgooey_b200 import engine as G, voices as V
from libgooey_b200._lib import lib
import engine_scripts as S
import oracle_lib as O
from workloads import drum_sweep_patches

pytestmark = pytest.mark.gpu

BACK_ENDS = {"wave_kernel<KickW>", "wave_kernel<SnareW>", "wave_kernel<HatW>", "wave_kernel<TomW>", "coop_kernel<TomC>", "back_kernel"}


def stat_names():
    L = lib()
    L.gooey_b200_kernel_stat_names.restype = ctypes.c_char_p
    return {s for s in (L.gooey_b200_kernel_stat_names() or b"").decode().split(";") if s}


def stat_voice_frames(name):
    L = lib()
    L.gooey_b200_kernel_stat.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    n, ms, vf = ctypes.c_uint64(), ctypes.c_double(), ctypes.c_double()
    L.gooey_b200_kernel_stat(name.encode(), ctypes.byref(n), ctypes.byref(ms), ctypes.byref(vf))
    return vf.value


def render_with_stats(patches, vel, frames, triggers=(0,)):
    b = V.VoiceBatch(patches, 44100.0)
    for f in triggers:
        b.trigger_all(f, vel)
    lib().gooey_b200_kernel_stats_reset()
    out = b.render(frames)
    names = stat_names()
    b.close()
    return out, names


TOM = V.patch(V.TOM, V.TOM_PRESETS["derp"], aux=1)
HAT = V.patch(V.HIHAT, V.HIHAT_PRESETS["short"])


@pytest.mark.parametrize("patch, n, key", [
    (TOM, 4095, "wave_kernel<TomW>"),
    (TOM, 4096, "coop_kernel<TomC>"),
    (HAT, 12287, "wave_kernel<HatW>"),
    (HAT, 12288, "back_kernel"),
], ids=["tom-4095", "tom-4096", "hat-12287", "hat-12288"])
def test_backend_at_policy_edges(patch, n, key):
    frames = 1024
    out, names = render_with_stats(V.patch_array([patch] * n), np.ones(n, np.float32), frames)
    print(n, "voices:", sorted(names))
    assert key in names
    assert not (names & (BACK_ENDS - {key}))
    want = O.render_voices([patch], frames, triggers=[(0, 0, 1.0)])
    assert np.abs(want).max() > 0.1
    assert np.abs(out - want).max() <= 1e-5          # every voice is the same patch


def test_coop_backend_matches_serial_backend_and_oracle(monkeypatch):
    """16 384 voices of the sweep are 4096 toms: the cooperative back end renders them.  Against the per-sample-order
    back end the only difference allowed is the re-association noise of the scans; every 64th voice (the sweep cycles
    kick / snare / hi-hat / tom, so these are toms) is also checked against the oracle."""
    n, frames = 16384, 20000
    patches, vel, kinds = drum_sweep_patches(n, seed=7)
    monkeypatch.setenv("GOOEY_B200_BACKEND", "serial")
    ser, ser_names = render_with_stats(patches, vel, frames, triggers=(0, 9000))
    monkeypatch.delenv("GOOEY_B200_BACKEND")
    got, names = render_with_stats(patches, vel, frames, triggers=(0, 9000))
    assert "coop_kernel<TomC>" in names and "coop_kernel<TomC>" not in ser_names
    assert np.isfinite(got).all()
    err = np.abs(ser - got).max(axis=1)
    for k in range(4):
        print(f"instrument {k}: max |default - serial| = {err[np.array(kinds) == k].max():.3e}")
    assert err.max() <= 5e-6
    idx = np.arange(3, n, 64)
    assert all(kinds[i] == V.TOM for i in idx)
    want = O.render_voices([patches[i] for i in idx], frames,
                           triggers=[(k, f, float(vel[i])) for k, i in enumerate(idx) for f in (0, 9000)], threads=8)
    oerr = float(np.abs(got[idx] - want).max())
    print(f"toms vs oracle: max err {oerr:.3e}")
    assert oerr <= 1e-5


VOICE_KINDS = {
    "kick": (V.patch(V.KICK, V.KICK_PRESETS["punch"]), "wave_kernel<KickW>"),
    "snare": (V.patch(V.SNARE, V.SNARE_PRESETS["tight"]), "wave_kernel<SnareW>"),
    "hihat": (HAT, "wave_kernel<HatW>"),
    "tom": (TOM, "wave_kernel<TomW>"),
    "bass": (V.patch(V.BASS, V.BASS_PRESETS["acid"]), "bass_wave_kernel"),
    "poly": (V.patch(V.POLY, V.POLY_PRESETS["keys"]), "poly_wave_kernel"),
    "granulator": (V.patch(V.GRANULATOR), "gran_wave_kernel"),
}


@pytest.mark.parametrize("kind", list(VOICE_KINDS))
def test_every_voice_kind_records_its_back_end(kind):
    patch, key = VOICE_KINDS[kind]
    n, frames = 64, 20000
    b = V.VoiceBatch([patch] * n, 44100.0)
    if kind == "poly":
        for v in range(n):
            b.note_on(v, 48 + v % 24, 0.9)
    elif kind == "granulator":
        i = np.arange(44100)
        src = (0.5 * np.sin(2 * np.pi * 220.0 * i / 44100.0)).astype(np.float32)
        for v in range(n):
            b.set_buffer(v, src, 44100.0)
        b.trigger_all(0)
    else:
        b.trigger_all(0, np.ones(n, np.float32))
    lib().gooey_b200_kernel_stats_reset()
    out = b.render(frames)
    names, vf = stat_names(), stat_voice_frames(key)
    b.close()
    print(kind, sorted(names), vf)
    assert names == {key}
    assert vf == n * frames
    assert np.isfinite(out).all()


def test_lfo_routed_basses_record_the_per_sample_kernel():
    def bounce(routed):
        e = G.Engine()
        for s in (0, 7, 9):
            e.sequencer_set_instrument_step(S.BASS, s, True)
        if routed:
            e.set_lfo_enabled(0, True)
            e.add_lfo_route(0, S.BASS, 6, 0.6)              # bass filter cutoff
        lib().gooey_b200_kernel_stats_reset()
        e.bounce_to_buffer(1)
        e.close()
        return stat_names()
    plain, routed = bounce(False), bounce(True)
    print("plain:", sorted(plain), "routed:", sorted(routed))
    assert "bass_wave_kernel" in plain and "slow_kernel<BassV>" not in plain
    assert "slow_kernel<BassV>" in routed and "bass_wave_kernel" not in routed
