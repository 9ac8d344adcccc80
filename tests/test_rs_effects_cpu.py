"""Global effect chains of Rust-API engines, on the oracle and the Python mirror (no GPU): the chain of the test oracle
(tests/rs_effects_oracle.py) is the fold of each effect's mono `process` in insertion order, built like the oracle's
stand-alone effects and its engine's default limiter, and keeps effect state across bounces; the mirror maps each
reference type to its FFI effect id and constructor arguments."""
import ctypes
import ctypes.util
import types

import numpy as np
import pytest

import oracle_lib as O

from libgooey_b200 import bounce as B
from rs_effects_oracle import ARGS, OracleFx, RustOracle

SR = 44100.0
N = 22050


def kit():
    insts = [("kick", B.KickDrum(SR, "punch")), ("snare", B.SnareDrum(SR, "tight")), ("hat", B.HiHat2(SR, "short"))]
    seqs = [("kick", [i % 4 == 0 for i in range(16)], [1.0] * 16), ("snare", [i % 8 == 4 for i in range(16)], [0.8] * 16),
            ("hat", [i % 2 == 1 for i in range(16)], [0.6] * 16)]
    return insts, seqs


def dry(samples=N, bounces=1):
    insts, seqs = kit()
    e = RustOracle(insts, seqs, master=0.7, limiter=False)
    out = [e.bounce(samples) for _ in range(bounces)]
    e.close()
    return out


def soft_limiter(x, threshold):
    """limiter.rs:43-78 in f32 with the platform's tanhf: tanh(x * (1 / th)) * th, th = max(threshold, 0.001)."""
    tanhf = ctypes.CDLL(ctypes.util.find_library("m")).tanhf
    tanhf.restype, tanhf.argtypes = ctypes.c_float, [ctypes.c_float]
    th = np.float32(max(threshold, 0.001))
    inv = np.float32(1.0) / th
    return np.array([np.float32(tanhf(float(np.float32(v) * inv))) * th for v in x], np.float32)


@pytest.mark.parametrize("eid", list(range(10)))
def test_each_kind_alone_is_its_mono_process_on_the_dry_bounce(eid):
    insts, seqs = kit()
    e = RustOracle(insts, seqs, master=0.7, limiter=False, effects=[(eid, ARGS[eid])])
    got = e.bounce(N)
    e.close()
    if eid == 5:      # the oracle's stand-alone effects have no limiter
        want = soft_limiter(dry()[0], ARGS[5][0])
    else:
        fx = OracleFx(eid, ARGS[eid])
        want = fx.process(dry()[0])
        fx.close()
    assert np.abs(want).max() > 0.01
    assert np.array_equal(got, want)


CHAIN = [(2, ARGS[2]), (9, ARGS[9]), (1, ARGS[1]), (3, ARGS[3])]


def test_a_chain_is_the_fold_in_insertion_order_and_keeps_its_state_across_bounces():
    insts, seqs = kit()
    e = RustOracle(insts, seqs, master=0.7, limiter=False, effects=CHAIN)
    got = [e.bounce(N), e.bounce(N)]
    e.close()
    fxs = [OracleFx(i, a) for i, a in CHAIN]
    for k, x in enumerate(dry(bounces=2)):
        for fx in fxs:
            x = fx.process(x)
        assert np.array_equal(got[k], x), k
    for fx in fxs:
        fx.close()


def test_default_chain_is_the_oracle_engines_own_limiter():
    insts, seqs = kit()
    e = RustOracle(insts, seqs, master=0.7)
    got = e.bounce(N)
    e.close()
    assert np.array_equal(got, O.rust_bounce(insts, seqs, N, master=0.7, limiter=True))


def test_mirror_maps_each_type_to_its_ffi_id_and_constructor_arguments():
    cases = [(B.LowpassFilterEffect(SR, 3000, 0.6), 0), (B.DelayEffect(SR, 3, 128, 0.4, 0.35, 6000), 1), (B.TubeSaturation(SR, 0.6, 0.5, 0.7), 2),
             (B.TubeCompressor(SR, -20, 6, 5, 80, 0.8), 3), (B.TiltFilterEffect(SR), 4), (B.SoftLimiter(0.5), 5),
             (B.SpringReverbEffect(SR, 0.7, 0.5, 0.3), 6), (B.Waveshaper(4.0, 0.6), 7), (B.FeedbackWaveshaper(SR, 20, 0.5, 3000, 0.7), 8),
             (B.PlateReverbEffect(SR, 0.8, 0.5, 0.4), 9)]
    for fx, eid in cases:
        assert fx.ffi() == (eid, [float(a) for a in ARGS[eid]])


def _engine_without_device(sr=SR):
    # the checks below happen before the library is called, so the engine needs no batch on a device
    return B.Engine(sr, _batch=types.SimpleNamespace(sample_rate=sr, _h=None), _index=0)


def test_mirror_refuses_an_effect_built_for_another_sample_rate():
    e = _engine_without_device()
    for fx in (B.DelayEffect(48000.0, 3, 120, 0.3, 0.3, 8000), B.PlateReverbEffect(22050.0, 0.5, 0.3, 0.5), B.TiltFilterEffect(48000.0)):
        with pytest.raises(B.GooeyError, match="Hz"):
            e.add_global_effect(fx)


def test_mirror_refuses_what_is_not_a_global_effect():
    e = _engine_without_device()
    for obj in (object(), B.KickDrum(SR), 0.5):
        with pytest.raises(B.GooeyError):
            e.add_global_effect(obj)
