"""Rust-API offline bounce, mirrored: ``gooey::bounce::{bounce_to_buffer, bounce_to_wav, BounceLength, WavConfig}``
and the part of ``gooey::engine::{Engine, Sequencer}`` a bounce uses (reference: src/bounce.rs:9-133,
src/engine/mod.rs:109-253, src/engine/sequencer.rs:498-582).  Names, argument meaning and error behaviour follow the
reference so that its own tests (tests/bounce.rs, examples/bounce.rs) read the same here:

    engine = Engine(44100.0); engine.set_bpm(120.0)
    engine.add_instrument("kick", KickDrum(44100.0))
    engine.add_sequencer(Sequencer.with_pattern(120.0, 44100.0, [True] + [False] * 15, "kick"))
    buf = bounce_to_buffer(engine, BounceLength.Bars(1))          # 88 200 mono samples

What is new is the batch: ``EngineBatch(n)`` holds n independent engines that are bounced in ONE device pass
(``gooey_rs_batch_*`` in include/gooey_batch.h); a stand-alone ``Engine`` is a batch of one.  All audio is rendered by
the CUDA kernels behind libgooey_b200.so; there is no CPU path.
"""
import ctypes
import math

import numpy as np

from ._lib import GooeyError, VoicePatch, check, lib
from . import voices as V

c = ctypes
_bound = False


def _L():
    global _bound
    L = lib()
    if not _bound:
        L.gooey_rs_batch_new.argtypes = [c.c_float, c.c_uint32, c.c_int, c.POINTER(c.c_void_p)]
        L.gooey_rs_batch_free.argtypes = [c.c_void_p]
        L.gooey_rs_batch_free.restype = None
        L.gooey_rs_batch_add_instrument.argtypes = [c.c_void_p, c.c_uint32, c.c_char_p, c.POINTER(VoicePatch)]
        L.gooey_rs_batch_add_sequencer.argtypes = [c.c_void_p, c.c_uint32, c.c_char_p, c.c_float, c.c_void_p, c.c_void_p, c.c_uint32]
        L.gooey_rs_batch_set_bpm.argtypes = [c.c_void_p, c.c_uint32, c.c_float]
        L.gooey_rs_batch_set_master_gain.argtypes = [c.c_void_p, c.c_uint32, c.c_float]
        L.gooey_rs_batch_clear_global_effects.argtypes = [c.c_void_p, c.c_uint32]
        L.gooey_rs_batch_add_limiter.argtypes = [c.c_void_p, c.c_uint32, c.c_float]
        L.gooey_rs_batch_add_effect.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32, c.c_void_p, c.c_uint32]
        L.gooey_rs_batch_bounce.argtypes = [c.c_void_p, c.c_uint32, c.c_void_p]
        L.gooey_rs_batch_bounce_device.argtypes = [c.c_void_p, c.c_uint32, c.c_void_p, c.c_size_t]
        L.gooey_b200_write_wav.argtypes = [c.c_char_p, c.c_void_p, c.c_uint32, c.c_uint32, c.c_uint32]
        _bound = True
    return L


def _rust_round(x):
    """f64::round — half away from zero."""
    return math.floor(x + 0.5) if x >= 0.0 else -math.floor(-x + 0.5)


class BounceLength:
    """bounce.rs:9-32.  ``BounceLength.Bars(n)`` (4/4), ``.Beats(x)`` (quarter notes), ``.Samples(n)``."""

    def __init__(self, kind, value):
        self.kind, self.value = kind, value

    @classmethod
    def Bars(cls, bars):
        return cls("bars", int(bars))

    @classmethod
    def Beats(cls, beats):
        return cls("beats", float(beats))

    @classmethod
    def Samples(cls, n):
        return cls("samples", int(n))

    def to_samples(self, bpm, sample_rate):
        bpm = float(np.float32(bpm))
        sr = float(np.float32(sample_rate))
        if self.kind == "bars":
            return max(int(_rust_round(self.value * (4.0 * (60.0 / bpm) * sr))), 0)
        if self.kind == "beats":
            return max(int(_rust_round(self.value * ((60.0 / bpm) * sr))), 0)
        return self.value


class WavConfig:
    """bounce.rs:62-74: bit depth 16 (default) or 24."""

    def __init__(self, bit_depth=16):
        self.bit_depth = bit_depth


class SequencerStep:
    """sequencer.rs:28-71 (enabled, velocity clamped to 0..1)."""

    def __init__(self, enabled, velocity=1.0):
        self.enabled = bool(enabled)
        self.velocity = min(max(float(velocity), 0.0), 1.0)


class Sequencer:
    """sequencer.rs:498-582: a 16th-note step pattern aimed at one named instrument, with its own tempo."""

    def __init__(self, bpm, sample_rate, steps, instrument_name):
        self.bpm, self.sample_rate, self.instrument_name = float(bpm), float(sample_rate), str(instrument_name)
        self.pattern = list(steps)

    @classmethod
    def new(cls, bpm, sample_rate, beat_count, instrument_name):
        return cls(bpm, sample_rate, [SequencerStep(True) for _ in range(beat_count)], instrument_name)

    @classmethod
    def with_pattern(cls, bpm, sample_rate, pattern, instrument_name):
        return cls(bpm, sample_rate, [SequencerStep(bool(p)) for p in pattern], instrument_name)

    @classmethod
    def with_velocity_pattern(cls, bpm, sample_rate, pattern, instrument_name):
        return cls(bpm, sample_rate, [p if isinstance(p, SequencerStep) else SequencerStep(*p) for p in pattern], instrument_name)


class _Instrument:
    def __init__(self, kind, params=(), aux=0):
        self.patch = V.patch(kind, params, aux=aux)


def KickDrum(sample_rate=44100.0, config=None):
    """KickDrum::new / with_config (kick.rs:772-828); config = KickConfig::new_full order or a preset name."""
    cfg = V.KICK_PRESETS["tight"] if config is None else (V.KICK_PRESETS[config] if isinstance(config, str) else config)
    return _Instrument(V.KICK, cfg)


def SnareDrum(sample_rate=44100.0, config=None):
    cfg = V.SNARE_PRESETS["tight"] if config is None else (V.SNARE_PRESETS[config] if isinstance(config, str) else config)
    return _Instrument(V.SNARE, cfg)


def HiHat2(sample_rate=44100.0, config=None):
    cfg = V.HIHAT_PRESETS["short"] if config is None else (V.HIHAT_PRESETS[config] if isinstance(config, str) else config)
    return _Instrument(V.HIHAT, cfg)


def Tom2(sample_rate=44100.0, config=None):
    if config is None:
        return _Instrument(V.TOM)
    return _Instrument(V.TOM, V.TOM_PRESETS[config] if isinstance(config, str) else config, aux=1)


def BassSynth(sample_rate=44100.0, config=None):
    """BassSynth::new = BassConfig::default() = acid (bass.rs:188-205, 608-611)."""
    cfg = V.BASS_PRESETS["acid"] if config is None else (V.BASS_PRESETS[config] if isinstance(config, str) else config)
    return _Instrument(V.BASS, cfg)


class _GlobalEffect:
    """A global effect as its constructor describes it: the FFI effect id (include/gooey.h) and the constructor arguments
    after the sample rate, in the reference's order.  ``sample_rate`` is None for types built without one."""
    ID = None
    sample_rate = None

    def ffi(self):
        return self.ID, [float(a) for a in self.args]


class LowpassFilterEffect(_GlobalEffect):
    """effects/lowpass_filter.rs:55-81."""
    ID = 0

    def __init__(self, sample_rate, cutoff, resonance):
        self.sample_rate, self.args = float(sample_rate), (cutoff, resonance)


class DelayEffect(_GlobalEffect):
    """effects/delay.rs: ``timing`` is the DelayTiming index (0 whole, 1 half, 2 quarter, 3 eighth, 4 sixteenth,
    5-7 triplets, 8 sixteenth triplet).  The delay keeps the tempo it was built with."""
    ID = 1

    def __init__(self, sample_rate, timing, bpm, feedback, mix, cutoff):
        self.sample_rate, self.args = float(sample_rate), (int(timing), bpm, feedback, mix, cutoff)


class TubeSaturation(_GlobalEffect):
    """effects/saturation.rs:68-91."""
    ID = 2

    def __init__(self, sample_rate, drive, warmth, mix):
        self.sample_rate, self.args = float(sample_rate), (drive, warmth, mix)


class TubeCompressor(_GlobalEffect):
    """effects/compressor.rs:55-96 (threshold dB, ratio, attack ms, release ms, mix)."""
    ID = 3

    def __init__(self, sample_rate, threshold, ratio, attack, release, mix):
        self.sample_rate, self.args = float(sample_rate), (threshold, ratio, attack, release, mix)


class TiltFilterEffect(_GlobalEffect):
    """effects/tilt_filter.rs."""
    ID = 4

    def __init__(self, sample_rate):
        self.sample_rate, self.args = float(sample_rate), ()


class SoftLimiter(_GlobalEffect):
    """effects/limiter.rs:43-78."""
    ID = 5

    def __init__(self, threshold=1.0):
        self.threshold = float(threshold)
        self.args = (self.threshold,)


class SpringReverbEffect(_GlobalEffect):
    """effects/reverb.rs."""
    ID = 6

    def __init__(self, sample_rate, decay, mix, damping):
        self.sample_rate, self.args = float(sample_rate), (decay, mix, damping)


class Waveshaper(_GlobalEffect):
    """effects/waveshaper.rs."""
    ID = 7

    def __init__(self, drive, mix):
        self.args = (drive, mix)


class FeedbackWaveshaper(_GlobalEffect):
    """effects/feedback_waveshaper.rs."""
    ID = 8

    def __init__(self, sample_rate, drive, feedback, cutoff, mix):
        self.sample_rate, self.args = float(sample_rate), (drive, feedback, cutoff, mix)


class PlateReverbEffect(_GlobalEffect):
    """effects/plate_reverb.rs."""
    ID = 9

    def __init__(self, sample_rate, decay, mix, damping):
        self.sample_rate, self.args = float(sample_rate), (decay, mix, damping)


class EngineBatch:
    """n independent Rust-API engines on one GPU; ``batch[i]`` is an ``Engine`` view."""

    def __init__(self, n, sample_rate=44100.0, device=0):
        self.n, self.sample_rate = int(n), float(sample_rate)
        h = c.c_void_p()
        check(_L().gooey_rs_batch_new(c.c_float(sample_rate), self.n, device, c.byref(h)))
        self._h = h
        self._bpm = [120.0] * self.n

    def close(self):
        if getattr(self, "_h", None):
            _L().gooey_rs_batch_free(self._h)
            self._h = None

    __del__ = close

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        if not 0 <= i < self.n:
            raise IndexError(i)
        return Engine(self.sample_rate, _batch=self, _index=i)

    def bounce(self, length, out=None):
        """Every engine bounced ``length`` in one device pass -> (n, samples) float32.  All engines must resolve
        ``length`` to the same sample count (same tempo, or ``BounceLength.Samples``)."""
        counts = {length.to_samples(b, self.sample_rate) for b in self._bpm}
        if len(counts) != 1:
            raise GooeyError("engines of one batch bounce must have equal length; group them by tempo")
        total = counts.pop()
        if out is None:
            out = np.zeros((self.n, total), np.float32)
        assert out.shape == (self.n, total) and out.dtype == np.float32 and out.flags.c_contiguous
        if total:
            check(_L().gooey_rs_batch_bounce(self._h, total, out.ctypes.data))
        return out


class Engine:
    """engine/mod.rs:84-253, the subset a bounce reads.  Stand-alone it owns a batch of one."""

    def __init__(self, sample_rate=44100.0, _batch=None, _index=0, device=0):
        self._batch = _batch if _batch is not None else EngineBatch(1, sample_rate, device)
        self._i = _index
        self._sr = float(sample_rate)

    new = classmethod(lambda cls, sample_rate: cls(sample_rate))

    def sample_rate(self):
        return self._sr

    def set_bpm(self, bpm):
        self._batch._bpm[self._i] = float(bpm)
        check(_L().gooey_rs_batch_set_bpm(self._batch._h, self._i, c.c_float(bpm)))

    def bpm(self):
        return self._batch._bpm[self._i]

    def add_instrument(self, name, instrument):
        check(_L().gooey_rs_batch_add_instrument(self._batch._h, self._i, str(name).encode(), c.byref(instrument.patch)))

    def add_sequencer(self, seq):
        en = np.array([s.enabled for s in seq.pattern], np.uint8)
        ve = np.array([s.velocity for s in seq.pattern], np.float32)
        check(_L().gooey_rs_batch_add_sequencer(self._batch._h, self._i, seq.instrument_name.encode(), c.c_float(seq.bpm), en.ctypes.data, ve.ctypes.data, len(en)))

    def set_master_gain(self, gain):
        check(_L().gooey_rs_batch_set_master_gain(self._batch._h, self._i, c.c_float(gain)))

    def clear_global_effects(self):
        check(_L().gooey_rs_batch_clear_global_effects(self._batch._h, self._i))

    def add_global_effect(self, effect):
        """Appends ``effect`` to the global chain.  The device builds it at the batch's sample rate, so an effect
        constructed for another rate is refused rather than rendered differently."""
        if not isinstance(effect, _GlobalEffect):
            raise GooeyError(f"not a global effect: {type(effect).__name__}")
        if effect.sample_rate is not None and np.float32(effect.sample_rate) != np.float32(self._batch.sample_rate):
            raise GooeyError(f"{type(effect).__name__} built at {effect.sample_rate} Hz for an engine at {self._batch.sample_rate} Hz")
        eid, args = effect.ffi()
        a = np.array(args, np.float32)
        check(_L().gooey_rs_batch_add_effect(self._batch._h, self._i, eid, a.ctypes.data if len(a) else None, len(a)))


def bounce_to_buffer(engine, length):
    """bounce.rs:41-59 -> mono float32 array."""
    if engine._batch.n == 1:
        return engine._batch.bounce(length)[0]
    raise GooeyError("engine belongs to an EngineBatch: call batch.bounce(length)")


def write_wav_f32(path, samples, sample_rate):
    """32-bit float WAV (mono (n,) or interleaved stereo (n, 2)) — the container of gooey_engine_loop_render_to_wav."""
    s = np.ascontiguousarray(samples, np.float32)
    ch = 1 if s.ndim == 1 else s.shape[1]
    f = _L().gooey_b200_write_wav_f32
    f.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]
    check(f(str(path).encode(), s.ctypes.data, s.shape[0], ch, int(sample_rate)))


def write_wav(path, samples, sample_rate, bit_depth=16):
    s = np.ascontiguousarray(samples, np.float32)
    check(_L().gooey_b200_write_wav(str(path).encode(), s.ctypes.data, s.size, int(sample_rate), int(bit_depth)))


def bounce_to_wav(engine, length, path, config=None):
    """bounce.rs:80-133: mono 16- or 24-bit PCM; raises GooeyError (the reference returns Err(String))."""
    config = config or WavConfig()
    if config.bit_depth not in (16, 24):
        raise GooeyError(f"Unsupported bit depth: {config.bit_depth}. Use 16 or 24.")
    buf = bounce_to_buffer(engine, length)
    write_wav(path, buf, engine.sample_rate(), config.bit_depth)
