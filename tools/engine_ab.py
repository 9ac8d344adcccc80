#!/usr/bin/env python
"""A/B check of the FFI engine path between two builds of libgooey_b200.

Renders a fixed list of engine scenarios and writes everything they make observable to one .npz: the audio, the launch
count of every call, the kernel-statistics table (names, launches, voice-frames; not the times), channel and track peaks,
drained MIDI events, LFO phases, loop positions and completed loop swaps.  Every scenario runs as configured, with
GOOEY_B200_NO_CHAIN_FAST=1 and with GOOEY_B200_BACKEND=serial.  A refactor of the host path must leave the file identical:

    GOOEY_B200_LIB=/path/to/a/libgooey_b200.so python tools/engine_ab.py render a.npz
    GOOEY_B200_LIB=/path/to/b/libgooey_b200.so python tools/engine_ab.py render b.npz
    python tools/engine_ab.py compare a.npz b.npz

`compare` compares every array byte for byte (float arrays as their bit patterns, so NaNs compare too) and exits 1 on
any difference.  Run with GOOEY_B200_TRACE=1 to get the per-piece trace lines of every render on stderr as well.
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SR = 44100.0
VARIANTS = {"default": {}, "no_chain_fast": {"GOOEY_B200_NO_CHAIN_FAST": "1"}, "serial": {"GOOEY_B200_BACKEND": "serial"}}


class Run:
    """Renders through the library and records what each call leaves observable under its own key."""

    def __init__(self):
        from libgooey_b200 import lib
        self.L = lib()
        self.L.gooey_b200_kernel_stat.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double),
                                                  ctypes.POINTER(ctypes.c_double)]
        self.L.gooey_b200_kernel_stat_names.restype = ctypes.c_char_p
        self.out = {}
        self.prefix = ""

    def call(self, key, engines, fn):
        """fn() renders; its result and the state it leaves in `engines` are recorded."""
        key = self.prefix + key
        assert key + "/audio" not in self.out, key
        self.L.gooey_b200_kernel_stats_reset()
        n0 = self.L.gooey_b200_launch_count()
        audio = fn()
        self.out[key + "/launches"] = np.array([self.L.gooey_b200_launch_count() - n0], np.uint64)
        self.out[key + "/audio"] = np.asarray(audio)
        names = [s for s in (self.L.gooey_b200_kernel_stat_names() or b"").decode().split(";") if s]
        stats = []
        for k in names:
            n, ms, vf = ctypes.c_uint64(0), ctypes.c_double(0.0), ctypes.c_double(0.0)
            self.L.gooey_b200_kernel_stat(k.encode(), ctypes.byref(n), ctypes.byref(ms), ctypes.byref(vf))
            stats.append((n.value, vf.value))
        self.out[key + "/kernel_names"] = np.array(names)
        self.out[key + "/kernel_stats"] = np.array(stats, np.float64).reshape(-1, 2)
        for j, e in enumerate(engines):
            self.out[f"{key}/{j}/peaks"] = np.concatenate([e.get_channel_peaks(5), [e.mixer_get_track_peak(t) for t in range(8)]]).astype(np.float32)
            self.out[f"{key}/{j}/midi"] = np.array(e.drain_midi_events(64), np.float64).reshape(-1, 3)
            self.out[f"{key}/{j}/lfo_phase"] = np.array([e.get_lfo_phase(i) for i in range(8)], np.float32)
            self.out[f"{key}/{j}/loops"] = np.array([(e.loop_get_position(ch), e.loop_swaps_completed(ch)) for ch in range(4)], np.float64)


def engines(n, setup):
    from libgooey_b200 import engine as G
    es = [G.Engine(SR) for _ in range(n)]
    for k, e in enumerate(es):
        setup(e, k)
    return es


def close(es):
    for e in es:
        e.close()


def scenario_golden(r):
    """The engine and reference cases of the committed golden fixtures, each alone: a bounce, then two stereo renders."""
    import golden_cases as GC
    for name, fn in {**GC.ENGINE_CASES, **GC.REF_CASES}.items():
        es = engines(1, lambda e, k: fn(e))
        r.call(f"golden/{name}/bounce", es, lambda: es[0].bounce_to_buffer(2))
        r.call(f"golden/{name}/render0", es, lambda: es[0].render(3000))
        r.call(f"golden/{name}/render1", es, lambda: es[0].render(9000))
        close(es)


def _pattern(e, k):
    import engine_scripts as S
    S.pattern_engine(e, 100 + k, swing=0.3 + 0.05 * (k % 8), notes=k % 3 != 2, graph=k % 2 == 0)
    if k % 4 == 1:
        S.random_voice_params(e, 200 + k)
    if k % 5 != 4:                           # most engines carry a chain; a few stay dry
        S.fx_chain(e, 300 + k, plate=k % 7 == 0, spring=k % 3 != 1, limiter=k % 2 == 1)
    if k % 6 == 3:
        e.set_instrument_mute(1, True); e.mixer_set_track_solo(0, True)
    if k % 6 == 5:
        e.set_instrument_solo(2, True); e.mixer_set_track_mute(1, True)
        e.blend_enable(0); e.blend_set_position(0, 0.3, 0.7); e.sequencer_set_instrument_step_blend(4, 0, 0.9, 0.1)
    if k % 9 == 2:
        e.trigger_instrument_with_velocity(3, 0.6)


def scenario_patterns(r):
    """48 pattern engines (swing, notes, graph, FX chains with plate and limiter): an 8-bar bounce (many pieces, both voice
    buffers), a pinned block bounce, then consecutive stereo batch renders into pinned and into pageable memory."""
    from libgooey_b200 import HostBuffer
    from libgooey_b200 import engine as G
    es = engines(48, _pattern)
    r.call("patterns/bounce8", es, lambda: np.concatenate(G.batch_bounce(es, 8)))
    hb = HostBuffer(48 * 2 * 88200 * 4)
    r.call("patterns/bounce_host", es, lambda: G.batch_bounce_host(es, 1, hb.array((48, 2 * 88200), np.float32)).copy())
    for e in es:
        e.sequencer_start()
    for j, frames in enumerate((5000, 20000, 70000)):
        r.call(f"patterns/pinned{j}", es, lambda: G.batch_render(es, frames, hb.array((48, frames, 2), np.float32)).copy())
        if j == 1:
            es[7].trigger_instrument(0); es[8].set_instrument_mute(4, True); es[9].set_master_gain(0.5)
    for j, frames in enumerate((4096, 30000)):
        r.call(f"patterns/pageable{j}", es, lambda: G.batch_render(es, frames))
    hb.close()
    close(es)


def scenario_synths(r):
    """Poly chords and granulators on one shared buffer next to plain engines; renders, a release, a bounce."""
    from libgooey_b200 import engine as G
    src = np.sin(np.arange(60000) * 0.013).astype(np.float32) * np.linspace(0.2, 1.0, 60000, dtype=np.float32)

    def setup(e, k):
        if k % 3 == 0:
            e.poly_trigger_chord(k % 12, k % 3, k % 7, k % 4, preset=k % 5, octave=3 + k % 2, velocity=0.8)
        elif k % 3 == 1:
            e.granulator_set_param(0, 0.4); e.granulator_set_seed(17 + k); e.granulator_trigger(0.9)
        else:
            _pattern(e, k)
    es = engines(9, setup)
    assert es[1].granulator_set_buffer(src, 48000.0)
    for e in es[4::3]:
        assert e.granulator_share_buffer(es[1])
    for j, frames in enumerate((3000, 40000)):
        r.call(f"synths/render{j}", es, lambda: G.batch_render(es, frames))
    es[0].poly_release(); es[3].poly_set_param(2, 0.9); es[4].granulator_snap_params()
    r.call("synths/render2", es, lambda: G.batch_render(es, 20000))
    r.call("synths/bounce", es, lambda: np.concatenate(G.batch_bounce(es, 2)))
    close(es)


def scenario_lfo(r):
    """LFO-routed and plain engines in one batch."""
    from libgooey_b200 import engine as G
    import engine_scripts as S

    def setup(e, k):
        _pattern(e, k)
        if k % 2 == 0:
            e.set_lfo_enabled(0, True); e.set_lfo_timing(0, k % 8); e.set_lfo_amount(0, 0.7)
            e.add_lfo_route(0, S.BASS, 2, 0.5); e.add_lfo_route(0, S.KICK, 1, 0.3); e.add_lfo_route(0, 6, 1, 0.3)
            e.set_lfo_enabled(3, True); e.set_lfo_offset(3, 0.2)                            # enabled, unrouted
            if k % 4 == 0:
                e.set_lfo_enabled(5, True); e.add_lfo_route(5, S.TOM, 8, 0.4); e.add_lfo_route(5, S.HIHAT, 0, 0.2)
    es = engines(8, setup)
    for e in es:
        e.sequencer_start()
    for j, frames in enumerate((7000, 50000)):
        r.call(f"lfo/render{j}", es, lambda: G.batch_render(es, frames))
    r.call("lfo/bounce", es, lambda: np.concatenate(G.batch_bounce(es, 2)))
    close(es)


def scenario_sources(r):
    """Loops with a queued swap and sampler-rack patterns next to plain engines, over consecutive renders."""
    from libgooey_b200 import engine as G
    import golden_cases as GC
    es = engines(4, lambda e, k: GC.REF_CASES["sample_playback"](e) if k % 2 == 0 else _pattern(e, k))
    for e in es:
        e.sequencer_start()
    for j, frames in enumerate((4000, 60000, 90000)):
        r.call(f"sources/render{j}", es, lambda: G.batch_render(es, frames))
    r.call("sources/bounce", es, lambda: np.concatenate(G.batch_bounce(es, 2)))
    close(es)


def scenario_type_swap(r):
    """Instrument types swapped on live channels between renders (with a blend on the swapped channel)."""
    from libgooey_b200 import engine as G
    es = engines(3, _pattern)
    for e in es:
        e.sequencer_start()
    r.call("swap/render0", es, lambda: G.batch_render(es, 6000))
    es[0].set_channel_instrument_type(0, 4); es[1].set_channel_instrument_type(4, 0)
    es[2].blend_enable(2); es[2].set_channel_instrument_type(2, 3); es[2].blend_set_position(2, 0.8, 0.2)
    r.call("swap/render1", es, lambda: G.batch_render(es, 30000))
    es[0].set_channel_instrument_type(0, 0)
    r.call("swap/bounce", es, lambda: np.concatenate(G.batch_bounce(es, 1)))
    close(es)


def render(path):
    r = Run()
    for variant, env in VARIANTS.items():
        for k in ("GOOEY_B200_NO_CHAIN_FAST", "GOOEY_B200_BACKEND"):
            os.environ.pop(k, None)
        os.environ.update(env)
        r.prefix = variant + "/"
        for scenario in (scenario_golden, scenario_patterns, scenario_synths, scenario_lfo, scenario_sources, scenario_type_swap):
            scenario(r)
    np.savez(path, **r.out)
    print(f"{path}: {len(r.out)} arrays")


def compare(path_a, path_b):
    a, b = np.load(path_a), np.load(path_b)
    bad = sorted(set(a.files) ^ set(b.files))
    for k in sorted(set(a.files) & set(b.files)):
        x, y = a[k], b[k]
        if x.dtype != y.dtype or x.shape != y.shape or x.tobytes() != y.tobytes():
            bad.append(k)
    silent = [k for k in a.files if k.endswith("/audio") and not np.any(a[k])]
    print(f"{len(a.files)} arrays compared, {len(bad)} differ; {len(silent)} silent audio arrays")
    for k in bad[:40]:
        print("  differs:", k)
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "render":
        render(sys.argv[2])
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
