"""The drum and bass back ends at the batch sizes and event frames that change how they walk a voice's timeline.

Which kernel renders a drum bucket depends on how many voices of the type one launch holds (pool.cuh choose_back): the
cooperative tom back end K from 4096 toms, the one-voice-per-thread back end C from 12 288 kicks / snares / hi-hats, the
warp-per-voice back end W below.  Inside each back end a voice's timeline is cut at 32-frame blocks, 8192-frame chunks
and render-call boundaries.  These tests run every back end with a partial last CTA or warp, with events on both sides
of each boundary, with voices on the per-sample kernel S next to planned voices of the same CTA or warp, in one call and
in split calls, and compare with the per-sample-order back ends (GOOEY_B200_BACKEND=serial) and with the oracle:

  * serial, one call vs serial, split calls: bit-identical (C and S keep the reference's per-sample order, so only an
    inexact hand-off between calls could make them differ);
  * default vs serial: at most 5e-6 per voice, the re-association noise of W's and K's scans;
  * oracle: at most 1e-5 on a subset of every (type, back end) pair.

The bass has one back end, bass_wave_kernel; slow_kernel<BassV> (S) is its serial reference.  Engine batches at the
production sizes reach K and C through the engine path (pieces, clock reset, note overrides, swing)."""
import ctypes
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from libgooey_b200 import engine as G, voices as V
from libgooey_b200._lib import lib
import engine_scripts as S
import oracle_lib as O
from workloads import drum_sweep_patches

pytestmark = pytest.mark.gpu

FRAMES = 17000
SPLIT = (1, 31, 8193, 8775)
TOL = 1e-5                 # against the oracle
SCAN_TOL = 5e-6            # default back ends against the per-sample-order ones (re-associated scans)
# Retriggers after the trigger at frame 0, by voice index % 6: inside the first block; two in one block; the last frame of
# the first chunk; the chunk edge of a one-call render; the chunk edge of the split render (8224 = 32 + 8192); the last frame.
RETRIG = ((31,), (32, 34), (8191,), (8192, 8193), (8224,), (16383, 16999))
COOP_NV, WARP = 16, 32
WAVE_KEY = {V.KICK: "wave_kernel<KickW>", V.SNARE: "wave_kernel<SnareW>", V.HIHAT: "wave_kernel<HatW>", V.TOM: "wave_kernel<TomW>"}
NAME = {V.KICK: "kick", V.SNARE: "snare", V.HIHAT: "hihat", V.TOM: "tom"}
PITCH_DECAY = {V.KICK: (0, 4), V.SNARE: (0, 1), V.HIHAT: (0, 1), V.TOM: (0, 4)}   # FFI ids (patch.h ffi_param_to_events)


def stat_names():
    L = lib()
    L.gooey_b200_kernel_stat_names.restype = ctypes.c_char_p
    return {s for s in (L.gooey_b200_kernel_stat_names() or b"").decode().split(";") if s}


def reset_stats():
    lib().gooey_b200_kernel_stats_reset()


# ------------------------------------------------------------------------------------------------ voice batches ----
class Plan:
    """A batch layout: patches, per-voice triggers (frame, velocity) and edits (frame, ffi_param, value, snap), and for
    every voice its type, its index within the type's bucket (its launch index) and whether it is a ringing tom."""

    def __init__(self):
        self.patches, self.kind, self.t, self.ring, self.trig, self.edits = [], [], [], [], [], []


def sweep_patches(kind, count, seed):
    """`count` random patches of one drum type from the drum sweep: even ones with overdrive 0 (exact tier), odd ones not."""
    m = 4 * ((count + 1) // 2)
    exact, _, ke = drum_sweep_patches(m, seed=seed, exact_tier=True)
    drive, _, kd = drum_sweep_patches(m, seed=seed + 1, exact_tier=False)
    exact = [p for p, k in zip(exact, ke) if k == kind]
    drive = [p for p, k in zip(drive, kd) if k == kind]
    return [exact[t // 2] if t % 2 == 0 else drive[t // 2] for t in range(count)]


def ringing_tom(rng):
    """A tom whose envelope ends early (decay 0.5..1.5 of 100: 20..60 ms) while its membrane keeps ringing."""
    p = [rng.uniform(20, 80), rng.uniform(0, 50), rng.uniform(0, 100), rng.uniform(0, 100), rng.uniform(0.5, 1.5),
         rng.uniform(80, 100), rng.uniform(80, 100), 100.0]
    return V.patch(V.TOM, [float(x) for x in p], aux=1)


def ring_frames(t):
    """Snapped tune edit and retrigger of ringing tom t: the retrigger falls in the membrane tail."""
    return 1501 + int(t) % 31, 3001 + int(t) % 31


def build_plan(counts, seed):
    """counts: [(kind, n)] in batch order."""
    rng = np.random.default_rng(seed)
    P = Plan()
    v = 0
    for kind, n in counts:
        pool = sweep_patches(kind, n, seed + 17 * kind)
        for t in range(n):
            ring = kind == V.TOM and t % 8 == 0
            P.patches.append(ringing_tom(rng) if ring else pool[t])
            P.kind.append(kind); P.t.append(t); P.ring.append(ring)
            vel = float(rng.uniform(0.3, 1.0))
            trig = [(0, vel)]
            edits = []
            pitch, decay = PITCH_DECAY[kind]
            frames = RETRIG[v % 6]
            if ring:
                e, r = ring_frames(t)
                edits.append((e, 0, float(rng.random()), True))
                trig.append((r, vel))
                frames = [f for f in frames if f > r]
            elif t % 3 == 0:           # snapped edit inside a block: the voice stays on the planned path
                edits.append((4001 + 32 * (t % 50) + t % 31, pitch if t % 2 == 0 else decay, float(rng.random()), True))
            if t % 17 == 0 or t == n - 2:  # unsnapped: the voice glides, so S renders it next to planned voices of its CTA / warp
                edits.append((1001 + t % 31, pitch, float(rng.random()), False))
            for q, f in enumerate(frames):
                trig.append((f, 0.0 if (v // 6 + q) % 4 == 0 else float(rng.uniform(0.3, 1.0))))
            P.trig.append(trig); P.edits.append(edits)
            v += 1
    P.kind = np.array(P.kind); P.t = np.array(P.t); P.ring = np.array(P.ring)
    return P


def render_plan(P, calls):
    b = V.VoiceBatch(V.patch_array(P.patches), 44100.0)
    for v in range(len(P.patches)):
        for f, vel in P.trig[v]:
            b.trigger(v, f, vel)
        for f, p, x, snap in P.edits[v]:
            b.set_param(v, p, x, frame=f, snap=snap)
    reset_stats()
    out = np.empty((len(P.patches), FRAMES), np.float32)
    f0 = 0
    for n in calls:
        out[:, f0:f0 + n] = b.render(n)
        f0 += n
    names = stat_names()
    b.close()
    return out, names


def oracle_plan(P, idx, frames=FRAMES, patches=None, until=None):
    patches = patches if patches is not None else [P.patches[v] for v in idx]
    trig = [(k, f, vel) for k, v in enumerate(idx) for f, vel in P.trig[v] if until is None or f < until[k]]
    edits = [(k, f, p, x, s) for k, v in enumerate(idx) for f, p, x, s in P.edits[v] if until is None or f < until[k]]
    return O.render_voices(patches, int(frames), triggers=trig, params=edits, threads=os.cpu_count() or 1)


SHAPES = {   # the drum type whose bucket is large and the back end it then takes; the other types stay at 64 voices (W)
    "wave": [(V.KICK, 100), (V.SNARE, 100), (V.HIHAT, 100), (V.TOM, 100)],
    "coop": [(V.KICK, 64), (V.TOM, 4096 + 19), (V.SNARE, 64), (V.HIHAT, 64)],
    "serial-kick": [(V.KICK, 12288 + 13), (V.SNARE, 64), (V.HIHAT, 64), (V.TOM, 64)],
    "serial-snare": [(V.KICK, 64), (V.SNARE, 12288 + 13), (V.HIHAT, 64), (V.TOM, 64)],
    "serial-hat": [(V.KICK, 64), (V.SNARE, 64), (V.HIHAT, 12288 + 13), (V.TOM, 64)],
}


def back_end_of(kind, n):
    if kind == V.TOM and n >= 4096:
        return "coop_kernel<TomC>", COOP_NV
    if kind != V.TOM and n >= 12288:
        return "back_kernel", WARP
    return WAVE_KEY[kind], 1


def oracle_subset(P, counts):
    """Every voice of a warp-per-voice bucket.  Of a cooperative or one-voice-per-thread bucket: every voice of its
    partial last CTA or warp (one of them glides), every 7th voice, the first gliding voices and the first 40 ringing toms."""
    base = 0
    idx = []
    for kind, n in counts:
        _, group = back_end_of(kind, n)
        if group == 1:
            ts = set(range(n))
        else:
            ts = set(range(n - n % group, n)) | set(range(0, n, 7)) | set(range(0, 17 * 20, 17))
            if kind == V.TOM:
                ts |= set(range(0, 8 * 40, 8))
        idx += [base + t for t in sorted(ts)]
        base += n
    return np.array(idx)


@pytest.mark.parametrize("shape", list(SHAPES))
def test_voice_batch_shapes(shape, monkeypatch):
    counts = SHAPES[shape]
    P = build_plan(counts, seed=0xB0 + list(SHAPES).index(shape))
    expect = {back_end_of(kind, n)[0] for kind, n in counts}
    sub = oracle_subset(P, counts)

    # the ringing toms' premise, on the oracle: without its membrane the tom is silent before the retrigger, with it it rings
    ring = [v for v in sub if P.ring[v]]
    assert len(ring) >= min(32, int(P.ring.sum()))
    until = [ring_frames(P.t[v])[1] for v in ring]
    dry = []
    for v in ring:
        p = V.patch(V.TOM, list(P.patches[v].params)[:8], aux=1)
        p.params[5] = 0.0
        dry.append(p)
    r_end = max(until)
    wet_o = oracle_plan(P, ring, frames=r_end, until=until)
    dry_o = oracle_plan(P, ring, frames=r_end, patches=dry, until=until)
    for k, r in enumerate(until):
        assert np.abs(dry_o[k, r - 256:r]).max() == 0.0, (ring[k], "the tom without membrane still sounds")
        assert np.abs(wet_o[k, r - 256:r]).max() > 1e-4, (ring[k], "the membrane does not ring at the retrigger")

    monkeypatch.setenv("GOOEY_B200_BACKEND", "serial")
    ref, names = render_plan(P, (FRAMES,))
    assert names == {"back_kernel"}
    assert np.isfinite(ref).all()
    got = {"serial": ref[sub].copy()}
    split, names = render_plan(P, SPLIT)
    assert names == {"back_kernel"}
    diff = np.nonzero((split != ref).any(axis=1))[0]
    print(f"{shape}, serial: split calls differ from one call in {diff.size} voices"
          + (f", max {np.abs(split - ref).max():.3e}, types {np.bincount(P.kind[diff], minlength=4).tolist()}" if diff.size else ""))
    del split
    monkeypatch.delenv("GOOEY_B200_BACKEND")
    for label, calls in (("one call", (FRAMES,)), ("split", SPLIT)):
        out, names = render_plan(P, calls)
        print(f"{shape}, {label}: back ends {sorted(names)}")
        assert names == expect
        assert np.isfinite(out).all()
        err = np.abs(out - ref).max(axis=1)
        for kind, n in counts:
            print(f"  {shape} {label} {NAME[kind]:5s} {back_end_of(kind, n)[0]:20s} max |default - serial| = {err[P.kind == kind].max():.3e}")
        assert err.max() <= SCAN_TOL, np.argmax(err)
        got[label] = out[sub].copy()
        del out

    want = oracle_plan(P, sub)
    assert np.abs(want).max() > 0.1
    for label, g in got.items():
        oerr = np.abs(g - want).max(axis=1)
        for kind, n in counts:
            key = "back_kernel" if label == "serial" else back_end_of(kind, n)[0]
            sel = P.kind[sub] == kind
            print(f"  {shape} {label:8s} {NAME[kind]:5s} {key:20s} vs oracle: max err {oerr[sel].max():.3e} over {sel.sum()} voices")
        assert oerr.max() <= TOL, (label, int(sub[np.argmax(oerr)]))
    assert diff.size == 0, f"serial split renders differ from one call for voices {diff[:16].tolist()}"


# --------------------------------------------------------------------------------------------------------- bass ----
BASS_EDIT = (6, 7, 15, 4, 3)     # cutoff, resonance, tuning, detune amount, detune level (FFI ids)


def bass_plan(n, seed):
    rng = np.random.default_rng(seed)
    patches, od0, trig, edits = [], [], [], []
    for v in range(n):
        p = rng.uniform(0.0, 1.0, 15)
        p[13] = 0.0 if v % 2 == 0 else rng.uniform(0.002, 1.0)      # overdrive: exact half, waveshaper half
        if v % 3 == 0:
            p[11] = rng.uniform(0.0, 0.02)                           # amp decay ~50 ms: idle gaps between the notes
        patches.append(V.patch(V.BASS, [float(x) for x in p], tuning=float(rng.random())))
        od0.append(v % 2 == 0)
        vel = float(rng.uniform(0.2, 1.0))
        tr = [(0, vel)] + [(f, 0.0 if (v // 6 + q) % 4 == 0 else float(rng.uniform(0.2, 1.0))) for q, f in enumerate(RETRIG[v % 6])]
        ed = [(201 + 32 * (v % 40) + v % 29, BASS_EDIT[v % 5], float(rng.random()), True),
              (9001 + v % 31, BASS_EDIT[(v + 2) % 5], float(rng.random()), True)]
        if v % 3 == 1:                                               # glides for a few thousand frames, then settles
            ed.append((3001 + v % 31, (6, 14, 1)[v % 3], float(rng.random()), False))
        trig.append(tr); edits.append(ed)
    return patches, np.array(od0), trig, edits


def render_bass(patches, trig, edits, sr, calls):
    b = V.VoiceBatch(V.patch_array(patches), sr)
    for v in range(len(patches)):
        for f, vel in trig[v]:
            b.trigger(v, f, vel)
        for f, p, x, snap in edits[v]:
            b.set_param(v, p, x, frame=f, snap=snap)
    reset_stats()
    out = np.concatenate([b.render(n) for n in calls], axis=1)
    names = stat_names()
    b.close()
    return out, names


@pytest.mark.parametrize("sr", [44100.0, 48000.0, 22050.0])
def test_bass_block_walk(sr, monkeypatch):
    """257 basses: the last two-warp CTA holds one voice.  At 22.05 kHz the filter's sr * 0.45 clamp is below 18 kHz."""
    n = 257
    patches, od0, trig, edits = bass_plan(n, seed=int(sr))
    one, names = render_bass(patches, trig, edits, sr, (FRAMES,))
    assert names == {"bass_wave_kernel"}
    split, names = render_bass(patches, trig, edits, sr, SPLIT)
    assert names == {"bass_wave_kernel"}
    monkeypatch.setenv("GOOEY_B200_BACKEND", "serial")
    ser, names = render_bass(patches, trig, edits, sr, (FRAMES,))
    monkeypatch.delenv("GOOEY_B200_BACKEND")
    assert names == {"slow_kernel<BassV>"}
    assert np.isfinite(one).all() and np.abs(one).max() > 0.05
    want = O.render_voices(patches, FRAMES, triggers=[(v, f, vel) for v in range(n) for f, vel in trig[v]],
                           params=[(v, f, p, x, s) for v in range(n) for f, p, x, s in edits[v]], sample_rate=sr,
                           threads=os.cpu_count() or 1)
    errs, bad, noise = [], [], []
    for label, out in (("bass_wave_kernel", one), ("bass_wave_kernel split", split), ("slow_kernel<BassV>", ser)):
        errs.append(np.abs(out - want).max(axis=1))
        print(f"bass {sr:.0f} Hz {label}: max err vs oracle {errs[-1][od0].max():.3e} (overdrive 0), {errs[-1][~od0].max():.3e} (waveshaper)")
    for label, out in (("serial", ser), ("split", split)):
        bad.append(np.nonzero(od0 & (out != one).any(axis=1))[0])
        noise.append(float(np.abs(out[~od0] - one[~od0]).max()))
        print(f"bass {sr:.0f} Hz {label} vs bass_wave_kernel: overdrive 0 {'bit-identical' if bad[-1].size == 0 else 'DIFFERENT'} "
              f"(max {np.abs(out[od0] - one[od0]).max():.3e}), waveshaper max {noise[-1]:.3e}")
    assert max(e.max() for e in errs) <= TOL
    assert all(b.size == 0 for b in bad), [b[:16].tolist() for b in bad]
    assert max(noise) <= SCAN_TOL


# --------------------------------------------------------------------------------------------------- engines ----
def engine_script(e, i):
    S.random_voice_params(e, 3000 + i)
    S.pattern_engine(e, 5000 + i, swing=None if i % 2 == 0 else 0.3 + 0.4 * ((i * 37) % 100) / 100.0)
    e.set_bpm(240.0)                       # one bar = 44 100 frames


def engine_edit(e, i):
    """Before the second bounce: unsnapped edits glide through the first pieces.  Tom parameters are not smoothed
    (tom2.rs), so an LFO route is what puts a tom on the per-sample kernel inside a cooperative CTA."""
    if i % 7 == 0:
        e.set_tom_param(0, ((i * 13) % 100) / 100.0)
        e.set_lfo_enabled(0, True)
        e.add_lfo_route(0, S.TOM, 0, 0.4)
    if i % 11 == 0:
        e.set_kick_param(0, ((i * 29) % 100) / 100.0)


def oracle_two_bounces(indices):
    def one(i):
        o = O.oracle_engine()
        engine_script(o, i)
        a = o.bounce_to_buffer(1)
        engine_edit(o, i)
        b = o.bounce_to_buffer(1)
        o.close()
        return i, (a, b)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        return dict(ex.map(one, list(indices)))


def rel_err(got, want):
    """As test_configs_gpu.compare: the same non-finite frames, finite ones relative to max(1, |reference|).  The second
    bounce restarts the clock under voices still sounding from the first, and the reference's output then grows far past
    full scale for many engines (bench.py reference_unstable_on_repeat_bounce).  Where it passes 1e3 the filters carry
    the rounding of those huge frames into much smaller neighbours, so such a bounce is compared relative to its peak."""
    fin = np.isfinite(want)
    assert np.array_equal(fin, np.isfinite(got))
    if not fin.any():
        return 0.0
    peak = float(np.abs(want[fin]).max())
    scale = np.maximum(1.0, np.abs(want[fin])) if peak < 1e3 else peak
    return float((np.abs(got[fin] - want[fin]) / scale).max())


@pytest.mark.parametrize("n", [4096 + 37, 12288 + 45])
def test_engine_batches_at_production_sizes(n, monkeypatch):
    torch = pytest.importorskip("torch")
    frames = 44100
    batches = {}
    for mode in ("default", "serial"):
        es = [G.Engine() for _ in range(n)]
        for i, e in enumerate(es):
            engine_script(e, i)
        batches[mode] = es
    last = set(range(n - n % COOP_NV if n % COOP_NV else n - COOP_NV, n)) | set(range(n - n % WARP if n % WARP else n - WARP, n))
    check = sorted(set(range(0, n, 128)) | last)
    host = {}
    for bounce in (0, 1):
        if bounce == 1:
            for es in batches.values():
                for i, e in enumerate(es):
                    engine_edit(e, i)
        bufs = {}
        for mode, es in batches.items():
            if mode == "serial":
                monkeypatch.setenv("GOOEY_B200_BACKEND", "serial")
            bufs[mode] = torch.empty((n, frames), dtype=torch.float32, device="cuda")
            reset_stats()
            assert G.batch_bounce_device(es, 1, bufs[mode].data_ptr(), frames) == frames
            names = stat_names()
            monkeypatch.delenv("GOOEY_B200_BACKEND", raising=False)
            print(f"{n} engines, bounce {bounce + 1}, {mode}: {sorted(names)}")
            if mode == "default" and bounce == 1:
                assert "coop_kernel<TomC>" in names
                assert ("back_kernel" in names) == (n >= 12288)
            if mode == "serial":
                assert "coop_kernel<TomC>" not in names and "bass_wave_kernel" not in names
        torch.cuda.synchronize()
        got, ser = bufs["default"], bufs["serial"]
        fin = torch.isfinite(ser)
        assert torch.equal(fin, torch.isfinite(got))
        err = float(((got - ser).abs() / ser.abs().clamp(min=1.0))[fin].max())
        print(f"{n} engines, bounce {bounce + 1}: max rel |default - serial| = {err:.3e}")
        assert err <= TOL
        host[bounce] = got[torch.tensor(check, device="cuda")].cpu().numpy()
        del bufs, got, ser, fin
        torch.cuda.empty_cache()
    for es in batches.values():
        for e in es:
            e.close()
    wants = oracle_two_bounces(check)
    worst = [0.0, 0.0]
    for k, i in enumerate(check):
        for bounce in (0, 1):
            assert len(wants[i][bounce]) == frames
            worst[bounce] = max(worst[bounce], rel_err(host[bounce][k], wants[i][bounce]))
    print(f"{n} engines: {len(check)} checked against the oracle, worst err {worst[0]:.3e} (gliding), {worst[1]:.3e} (settled)")
    assert max(worst) <= TOL
