"""The front end's restructured arithmetic against the reference, bit for bit, on the host build of the device functions.

osc_triangle sums its harmonics in three runs (untapered with tabulated gains, the tapered top, i >= 2048); the frequencies
here put the run boundaries, the table boundary and the Nyquist break exactly on and next to a harmonic.  The two-segment
MaxCurve envelope is evaluated both per sample and from the segment constants a span stores.
"""
import ctypes
import ctypes.util
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import emu_lib as E  # noqa: E402
import oracle_lib as O  # noqa: E402

f32 = np.float32
libm = ctypes.CDLL(ctypes.util.find_library("m"))
libm.sinf.restype = ctypes.c_float
libm.sinf.argtypes = [ctypes.c_float]
TWO_PI = f32(2.0) * f32(np.pi)


def bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def ref_triangle(idx, freq, sr, sine):
    """Oscillator::generative(2, 2.0) (oscillator.rs:106-131) in f32, one harmonic at a time for every sample at once."""
    idx, freq, sr = np.asarray(idx, f32), np.asarray(freq, f32), f32(sr)
    nyq = sr / f32(2.0)
    with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
        q = nyq / freq
    max_h = np.where(np.isnan(q), 0, np.clip(q, -2.0 ** 31, 2.0 ** 31 - 1)).astype(np.int64)
    out = np.zeros_like(idx)
    running = np.ones(idx.shape, bool)
    for i in range(1, int(max_h.max()) + 1, 2):
        fi = f32(i)
        running &= (i <= max_h) & ~(freq * fi > nyq)
        if not running.any():
            break
        gain = f32(1.0) / (fi * fi)
        hf = freq * fi
        ratio = hf / nyq
        t = (ratio - f32(0.75)) / f32(0.25)
        taper = np.where(ratio > f32(0.75), f32(1.0) - t * t, f32(1.0)).astype(f32)
        s = sine(idx * hf * TWO_PI / sr)
        out = np.where(running, out + gain * taper * s, out).astype(f32)
    return out


def exact_sine(x):
    return np.array([libm.sinf(float(v)) for v in np.ravel(x)], f32).reshape(np.shape(x))


def fast_sine(x):
    return E.math(1, np.ravel(x)).reshape(np.shape(x))


def edge_freqs(sr):
    """Frequencies at which a harmonic i lands exactly on 0.7 nyquist (first tapered harmonic), on nyquist (the break),
    and around the table boundary i = 2047 / 2049, each with its two f32 neighbours; plus two pitches below 11 Hz."""
    nyq = f32(sr) / f32(2.0)
    lim = f32(0.7) * nyq
    fs = []
    for i in (1, 3, 5, 7, 21, 45, 77, 101, 255, 1023, 2045, 2047, 2049, 2051):
        for edge in (lim, nyq):
            f = edge / f32(i)
            fs += [np.nextafter(f, f32(0)), f, np.nextafter(f, f32(np.inf))]
    return np.unique(np.array(fs + [f32(5.0), f32(10.5)], f32))


def test_triangle_edges_match_reference():
    for sr in (44100.0, 48000.0):
        freqs = edge_freqs(sr)
        idx = np.array([1.0, 17.0, 441.0, 12345.0], f32)
        a = np.repeat(idx, freqs.size)
        b = np.tile(freqs, idx.size)
        # the exact path (kicks with drive > 8, the per-sample kernel) against the reference with glibc's sinf
        want = ref_triangle(a, b, sr, exact_sine)
        got = E.math(3, a, b, sample_rate=sr)
        assert np.array_equal(bits(got), bits(want)), (sr, b[bits(got) != bits(want)][:8])
        # the front end's path: the same sum with the ~1-ulp sine of an IEEE-divided argument
        want = ref_triangle(a, b, sr, fast_sine)
        got = E.math(2, a, b, sample_rate=sr)
        assert np.array_equal(bits(got), bits(want)), (sr, b[bits(got) != bits(want)][:8])


def test_taper_ratio_division_exact_for_all_numerators():
    # the tapered run divides by nyquist through RN(1 / nyquist): the quotient of every f32 numerator with the divisor's
    # significand (one binade covers all exponents away from subnormals) equals the IEEE quotient
    a = (np.arange(1 << 23, dtype=np.uint32) | np.uint32(0x3f800000)).view(f32)
    for sr in (22050.0, 44100.0, 48000.0, 88200.0, 96000.0, 192000.0):
        nyq = np.full(a.size, f32(sr) / f32(2.0), f32)
        got = E.math(0, a, nyq)
        assert np.array_equal(bits(got), bits(a / nyq)), sr


@pytest.fixture(scope="module")
def front_host(tmp_path_factory):
    """tests/front_host.cpp built with emu_lib's flags into a temporary directory."""
    so = str(tmp_path_factory.mktemp("front_host") / "libfront_host.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "front_host.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-shared", "-o", so, src], check=True)
    L = ctypes.CDLL(so)
    L.front_maxenv.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int]
    return L


def _env(L, seg6, times, hoisted):
    out = np.zeros(times.size, f32)
    assert L.front_maxenv(seg6.ctypes.data, times.ctypes.data, out.ctypes.data, times.size, hoisted) == 0
    return out


def test_maxcurve_span_constants_match_reference(front_host):
    L = O.lib()
    L.orc_maxcurve_envelope.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32]
    L.orc_maxcurve_envelope.restype = None
    sr = 44100.0
    # the hi-hat's (attack -0.3, decay -0.8) and the tom's (attack 0.8, decay -0.83) envelopes, over both segments and past the end
    for seg in ([1.0, 0.5, -0.3, 0.0, 0.5, -0.8], [1.0, 37.0, -0.3, 0.0, 1234.0, -0.8], [1.0, 200.0, -0.3, 0.0, 4000.0, -0.8],
                [1.0, 1.0, 0.8, 0.0, 2000.0, -0.83], [1.0, 1.0, 0.8, 0.0, 40.0, -0.83]):
        seg6 = np.array(seg, f32)
        end = (seg[1] + seg[4]) / 1000.0
        n = int(end * sr) + 64
        times = np.zeros(n, np.float64)
        t, dt = 0.0, 1.0 / sr
        for j in range(n):          # the engine clock: repeated addition of 1 / sr
            times[j] = t
            t += dt
        want = np.zeros(n, f32)
        L.orc_maxcurve_envelope(seg6.ctypes.data, times.ctypes.data, want.ctypes.data, n)
        for hoisted in (0, 1):
            got = _env(front_host, seg6, times, hoisted)
            assert np.array_equal(bits(got), bits(want)), (seg, hoisted, np.flatnonzero(bits(got) != bits(want))[:8])
