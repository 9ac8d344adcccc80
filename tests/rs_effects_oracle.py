"""The oracle's RustEngine (oracle/engine.hpp) with a global effect chain, for the Rust-API effect tests.

TEST INFRASTRUCTURE.  The oracle's RustEngine renders the dry mono sum (its chain cleared); tests/rs_chain_host.cpp folds
that through the chain, built from the oracle's own effect classes.  An engine can be bounced several times, so effect
state carried from one bounce to the next is checked the way the reference keeps it."""
import ctypes as c
import os
import subprocess
import tempfile
import threading

import numpy as np

import oracle_lib as O

# one non-default set of constructor arguments per FFI effect id (the reference's order, after the sample rate)
ARGS = {
    0: (3000.0, 0.6),                    # LowpassFilterEffect(cutoff, resonance)
    1: (3, 128.0, 0.4, 0.35, 6000.0),     # DelayEffect(timing = eighth, bpm, feedback, mix, cutoff)
    2: (0.6, 0.5, 0.7),                  # TubeSaturation(drive, warmth, mix)
    3: (-20.0, 6.0, 5.0, 80.0, 0.8),     # TubeCompressor(threshold dB, ratio, attack ms, release ms, mix)
    4: (),                               # TiltFilterEffect
    5: (0.5,),                           # SoftLimiter(threshold)
    6: (0.7, 0.5, 0.3),                  # SpringReverbEffect(decay, mix, damping)
    7: (4.0, 0.6),                       # Waveshaper(drive, mix)
    8: (20.0, 0.5, 3000.0, 0.7),         # FeedbackWaveshaper(drive, feedback, cutoff, mix)
    9: (0.8, 0.5, 0.4),                  # PlateReverbEffect(decay, mix, damping)
}
# examples/bounce.rs:104-123
EXAMPLE_CHAIN = [(2, (0.3, 0.4, 0.5)), (1, (3, 128.0, 0.35, 0.2, 8000.0)), (3, (-12.0, 4.0, 10.0, 100.0, 0.6)), (5, (0.95,))]

_bound = False
_host = None
_host_lock = threading.Lock()


def _H():
    """tests/rs_chain_host.cpp built with the oracle's compiler flags (oracle/Makefile) into a temporary directory."""
    global _host
    with _host_lock:
        if _host is None:
            so = os.path.join(tempfile.mkdtemp(prefix="rs_chain_host_"), "librs_chain_host.so")
            src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "rs_chain_host.cpp")
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-o", so, src], check=True)
            H = c.CDLL(so)
            H.rs_chain_new.restype = c.c_void_p
            H.rs_chain_new.argtypes = [c.c_float]
            H.rs_chain_free.argtypes = [c.c_void_p]
            H.rs_chain_clear.argtypes = [c.c_void_p]
            H.rs_chain_add.argtypes = [c.c_void_p, c.c_uint32, c.c_void_p]
            H.rs_chain_process.argtypes = [c.c_void_p, c.c_void_p, c.c_void_p, c.c_uint32]
            _host = H
    return _host


def _L():
    global _bound
    L = O.lib()
    if not _bound:
        L.orc_rust_engine_new.restype = c.c_void_p
        L.orc_rust_engine_new.argtypes = [c.c_float]
        L.orc_rust_engine_free.argtypes = [c.c_void_p]
        L.orc_rust_engine_add_instrument.argtypes = [c.c_void_p, c.c_char_p, c.c_void_p]
        L.orc_rust_engine_add_sequencer.argtypes = [c.c_void_p, c.c_char_p, c.c_void_p, c.c_void_p, c.c_uint32]
        L.orc_rust_engine_set_bpm.argtypes = [c.c_void_p, c.c_float]
        L.orc_rust_engine_set_master_gain.argtypes = [c.c_void_p, c.c_float]
        L.orc_rust_engine_clear_global_effects.argtypes = [c.c_void_p]
        L.orc_rust_engine_bounce_samples.argtypes = [c.c_void_p, c.c_uint32, c.c_void_p]
        L.orc_fx_new.restype = c.c_void_p
        L.orc_fx_new.argtypes = [c.c_uint32, c.c_float, c.c_void_p]
        L.orc_fx_free.argtypes = [c.c_void_p]
        L.orc_fx_process.argtypes = [c.c_void_p, c.c_void_p, c.c_void_p, c.c_uint32]
        _bound = True
    return L


def _f32(args):
    return np.array(list(args) or [0.0], np.float32)


class RustOracle:
    """instruments = [(name, obj with .patch)], sequencers = [(name, enabled[16], velocity[16])]; the chain starts as
    [SoftLimiter(1.0)] unless limiter=False, then `effects` = [(id, args)] are appended."""

    def __init__(self, instruments, sequencers, master=None, limiter=True, effects=(), bpm=120.0, sample_rate=44100.0):
        L = _L()
        self.h = L.orc_rust_engine_new(sample_rate)
        L.orc_rust_engine_set_bpm(self.h, bpm)
        for name, inst in instruments:
            assert L.orc_rust_engine_add_instrument(self.h, name.encode(), c.byref(inst.patch)) == 0
        for name, en, ve in sequencers:
            en = np.asarray(en, np.uint8); ve = np.asarray(ve, np.float32)
            L.orc_rust_engine_add_sequencer(self.h, name.encode(), en.ctypes.data, ve.ctypes.data, len(en))
        if master is not None:
            L.orc_rust_engine_set_master_gain(self.h, master)
        L.orc_rust_engine_clear_global_effects(self.h)      # the engine renders the dry sum, the chain below does the rest
        self.chain = _H().rs_chain_new(sample_rate)
        if limiter:
            self.add_effect(5, (1.0,))
        for eid, args in effects:
            self.add_effect(eid, args)

    def add_effect(self, eid, args):
        a = _f32(args)
        assert _H().rs_chain_add(self.chain, eid, a.ctypes.data) == 0

    def clear(self):
        _H().rs_chain_clear(self.chain)

    def set_bpm(self, bpm):
        _L().orc_rust_engine_set_bpm(self.h, bpm)

    def bounce(self, samples):
        dry = np.zeros(samples, np.float32)
        _L().orc_rust_engine_bounce_samples(self.h, samples, dry.ctypes.data)
        out = np.zeros(samples, np.float32)
        _H().rs_chain_process(self.chain, dry.ctypes.data, out.ctypes.data, samples)
        return out

    def close(self):
        if self.h:
            _L().orc_rust_engine_free(self.h)
            _H().rs_chain_free(self.chain)
            self.h = None


class OracleFx:
    """One stand-alone effect of the oracle (orc_fx_new): its mono `process` over a buffer, state kept between calls."""

    def __init__(self, eid, args, sample_rate=44100.0):
        a = _f32(args)
        self.h = _L().orc_fx_new(eid, sample_rate, a.ctypes.data)
        assert self.h

    def process(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.zeros_like(x)
        _L().orc_fx_process(self.h, x.ctypes.data, out.ctypes.data, len(x))
        return out

    def close(self):
        _L().orc_fx_free(self.h)
