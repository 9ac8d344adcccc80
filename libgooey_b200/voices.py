"""Instrument-level batch API: thousands of independent voices rendered in one call.

Mirrors the reference's Rust instrument API (``KickDrum::with_config`` →
``trigger_with_velocity`` → ``tick`` loop; src/instruments/*.rs) for a whole
batch: build patches, schedule triggers / parameter edits, render.
"""
import ctypes

import numpy as np

from ._lib import GooeyError, VoicePatch, check, lib

KICK, SNARE, HIHAT, TOM, BASS = 0, 1, 2, 3, 4
POLY, GRANULATOR = 5, 6     # libgooey_b200 voice kinds (include/gooey_batch.h GOOEY_B200_VOICE_*)

# Reference presets (normalized), in each Config's `new_full` argument order.
KICK_PRESETS = {  # src/instruments/kick.rs:257-350
    "tight": [0.22, 0.00, 1.00, 0.00, 0.12, 0.70, 0.01, 0.85, 0.64, 1.00, 0.07, 0.01, 0.02, 0.20, 0.00, 0.47, 0.12, 0.02],
    "punch": [0.50, 0.20, 1.00, 0.20, 0.12, 0.60, 0.10, 0.85, 0.24, 1.00, 0.07, 0.11, 0.42, 0.20, 0.00, 0.47, 0.12, 0.02],
    "loose": [0.32, 0.40, 1.00, 0.00, 0.62, 0.20, 0.12, 0.85, 0.84, 1.00, 0.07, 0.01, 0.02, 0.25, 0.00, 0.47, 0.12, 0.12],
    "dirt": [0.62, 0.10, 1.00, 0.10, 0.10, 0.60, 0.10, 0.85, 0.44, 1.00, 0.20, 0.10, 0.82, 0.20, 0.00, 0.47, 0.10, 0.10],
}


def _snare_basic(f, t, n, c, d, pd, v):  # SnareConfig::new (src/instruments/snare.rs:99-132), evaluated in f32
    f32 = np.float32
    d = f32(d)
    return [f, t, n, c, float(d), pd, v, float(d * f32(0.8)), 0.091, float(d * f32(0.6)), float(d), 0.495, 0.053, 1, 0.5, 0.0, 0.0, 0.125, 0.02]


SNARE_PRESETS = {  # src/instruments/snare.rs:270-351
    "tight": _snare_basic(0.2, 0.4, 0.7, 0.5, 0.029, 0.3, 0.8),
    "loose": [0.16, 0.80, 0.60, 0.30, 0.79, 0.10, 0.90, 0.33, 0.20, 0.23, 0.34, 0.55, 0.05, 1, 0.50, 0.00, 0.10, 0.12, 0.02],
    "hiss": [0.16, 0.00, 0.60, 0.30, 0.04, 0.40, 0.90, 0.53, 0.09, 0.38, 0.29, 0.29, 0.45, 1, 0.50, 1.00, 0.20, 0.18, 0.02],
    "smack": [0.2, 0.3, 0.8, 0.0, 0.029, 0.3, 0.85, 0.014, 0.091, 0.034, 0.086, 0.293, 0.158, 1, 0.4, 0.5, 0.0, 0.125, 0.02],
}
HIHAT_PRESETS = {  # pitch, decay, attack, tone, volume (src/instruments/hihat2.rs:79-96)
    "short": [0.76, 0.05, 0.00, 1.00, 1.0],
    "loose": [0.76, 0.30, 0.00, 1.00, 1.0],
    "dark": [0.41, 0.05, 0.00, 0.15, 1.0],
    "soft": [0.41, 0.05, 0.15, 0.60, 1.0],
}
TOM_PRESETS = {  # tune, bend, tone, color, decay, membrane, membrane_q, volume (src/instruments/tom2.rs:119-172)
    "derp": [60.0, 70.0, 50.0, 0.0, 20.0, 0.0, 50.0, 100.0],
    "ring": [80.0, 20.0, 10.0, 0.0, 100.0, 60.0, 70.0, 100.0],
    "brush": [40.0, 20.0, 10.0, 90.0, 30.0, 0.0, 50.0, 100.0],
    "void": [60.0, 30.0, 100.0, 50.0, 90.0, 40.0, 80.0, 100.0],
}
BASS_PRESETS = {  # BassConfig::{acid,sub,reese,stab} in field order (src/instruments/bass.rs:188-269)
    "acid": [0.24, 0.40, 0.80, 0.00, 0.00, 0.10, 0.15, 0.70, 0.85, 0.15, 0.08, 0.35, 0.10, 0.30, 0.80],
    "sub": [0.18, 1.00, 0.15, 0.00, 0.00, 0.00, 0.70, 0.05, 0.10, 0.30, 0.20, 0.60, 0.15, 0.00, 0.85],
    "reese": [0.18, 0.30, 0.80, 0.80, 0.50, 0.05, 0.35, 0.30, 0.50, 0.40, 0.15, 0.55, 0.12, 0.60, 0.80],
    "stab": [0.30, 0.20, 0.90, 0.00, 0.00, 0.90, 0.20, 0.40, 0.90, 0.08, 0.05, 0.20, 0.08, 0.20, 0.80],
}
POLY_PRESETS = {  # PolyConfig::{default,pad,pluck,keys,strings} in field order (src/instruments/poly_synth.rs:49-142)
    "default": [0.0, 0.2, 0.6, 0.15, 0.3, 0.55, 0.7, 0.7, 0.8, 0.5, 0.65, 0.4, 0.75, 0.7],
    "pad": [0.0, 0.4, 0.45, 0.2, 0.2, 0.8, 0.75, 0.8, 0.85, 0.75, 0.7, 0.5, 0.8, 0.6],
    "pluck": [0.3, 0.1, 0.7, 0.25, 0.6, 0.0, 0.75, 0.0, 0.65, 0.0, 0.7, 0.1, 0.65, 0.7],
    "keys": [0.5, 0.15, 0.55, 0.1, 0.4, 0.35, 0.7, 0.5, 0.75, 0.3, 0.65, 0.3, 0.7, 0.7],
    "strings": [0.0, 0.5, 0.5, 0.1, 0.15, 0.85, 0.7, 0.9, 0.85, 0.8, 0.7, 0.6, 0.8, 0.5],
}


def patch(instrument, params=(), aux=0, tuning=None):
    p = VoicePatch()
    p.instrument = instrument
    p.aux = aux
    for i, x in enumerate(params):
        p.params[i] = x
    if tuning is not None:
        p.aux |= 0x100
        p.params[23] = tuning
    return p


def patch_array(patches):
    return (VoicePatch * len(patches))(*patches)


class VoiceBatch:
    """N voices on one GPU.  ``render`` returns a (N, frames) float32 array."""

    def __init__(self, patches, sample_rate=44100.0, device=0):
        self.n = len(patches)
        self._arr = patches if isinstance(patches, ctypes.Array) else patch_array(patches)
        h = ctypes.c_void_p()
        check(lib().gooey_voice_batch_new(ctypes.c_float(sample_rate), self.n, self._arr, device, ctypes.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):       # the constructor may have raised before the handle existed
            lib().gooey_voice_batch_free(self._h)
            self._h = None

    __del__ = close

    def trigger(self, voice, frame=0, velocity=1.0):
        check(lib().gooey_voice_batch_trigger(self._h, voice, frame, ctypes.c_float(velocity)))

    def trigger_all(self, frame=0, velocities=None):
        ptr = None
        if velocities is not None:
            v = np.ascontiguousarray(velocities, dtype=np.float32)
            assert v.shape == (self.n,)
            ptr = v.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        check(lib().gooey_voice_batch_trigger_all(self._h, frame, ptr))

    def set_param(self, voice, param, value, frame=0, snap=False):
        check(lib().gooey_voice_batch_set_param(self._h, voice, frame, param, ctypes.c_float(value), int(snap)))

    # Poly voices: PolySynth::trigger_note / release_all.  Granulators: Granulator::set_buffer / set_seed, and
    # share_buffer, which plays another granulator's buffer without a second device copy.  Each raises GooeyError on a
    # refusal (wrong voice kind, note above 127, invalid buffer), and a refused call queues nothing.
    def note_on(self, voice, note, velocity=1.0, frame=0):
        if not 0 <= int(note) <= 127:
            raise GooeyError(f"note_on: note {note} is outside 0..127")
        check(lib().gooey_voice_batch_note_on(self._h, voice, frame, int(note), ctypes.c_float(velocity)))

    def release(self, voice, frame=0):
        check(lib().gooey_voice_batch_release(self._h, voice, frame))

    def set_buffer(self, voice, samples, sample_rate, frame=0):
        buf = np.ascontiguousarray(samples, dtype=np.float32)
        if buf.ndim != 1 or buf.size == 0:
            raise GooeyError("set_buffer: samples must be a non-empty 1-D array")
        check(lib().gooey_voice_batch_set_buffer(self._h, voice, frame, buf.ctypes.data, buf.size, ctypes.c_float(sample_rate)))

    def share_buffer(self, dst_voice, src_voice, frame=0):
        check(lib().gooey_voice_batch_share_buffer(self._h, dst_voice, frame, src_voice))

    def set_seed(self, voice, seed, frame=0):
        check(lib().gooey_voice_batch_set_seed(self._h, voice, frame, int(seed) & 0xFFFFFFFF))

    def render(self, frames, out=None):
        if out is None:
            out = np.empty((self.n, frames), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.shape == (self.n, frames)
        check(lib().gooey_voice_batch_render(self._h, frames, out.ctypes.data))
        return out

    def render_pcm16(self, frames, out=None):
        """gooey_voice_batch_render_pcm16: (N, frames) int16, `(s * 32767).round() as i16` quantised on the device."""
        if out is None:
            out = np.empty((self.n, frames), dtype=np.int16)
        assert out.dtype == np.int16 and out.flags.c_contiguous and out.shape == (self.n, frames)
        f = lib().gooey_voice_batch_render_pcm16
        f.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p]
        check(f(self._h, frames, out.ctypes.data))
        return out

    def render_device(self, frames, dev_ptr, stride):
        check(lib().gooey_voice_batch_render_device(self._h, frames, ctypes.c_void_p(dev_ptr), stride))
