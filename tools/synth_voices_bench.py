#!/usr/bin/env python
"""synth_voices_bench.py — poly synths and granulators in voice batches on one GPU.

Poly: batches of 1024 / 4096 / 16 384 / 32 768 poly voices (seeded random PolyConfig presets), 10 s at 44.1 kHz, each
voice a four-note chord at 0 s, released at 5 s and retriggered with a second four-note chord in the same frame (the
release-then-notes sequence of gooey_engine_poly_trigger_notes).  Rendered with gooey_voice_batch_render_device into one
device block.  After a warm-up of both back ends, each size is rendered by the warp-per-voice back end (poly_wave_kernel)
and by the per-sample-order back end (GOOEY_B200_BACKEND=serial, slow_kernel<PolyV>), alternated, from fresh batches.
Reported per run: the back-end kernel's device time (CUDA events, the library's kernel statistics), the wall time of the
render call, voice-samples/s, and whether the two back ends' blocks are bit-identical.

Granulators: 1600 voices x 10 s through the voice batch with the C4 parameters of SURVEY.md 8d (one shared 60 s source,
per-voice pitch, texture and seed), a sanity line next to bench.py's FFI C4; one voice is checked against the oracle.

The card's name, power limit and max SM clock are read in the same run.  A GPU is required.

  python tools/synth_voices_bench.py [--sizes 1024,4096,16384,32768] [--reps 2] [--out profiles/r3_c_synth_voices.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from libgooey_b200 import voices as V  # noqa: E402
from libgooey_b200._lib import lib  # noqa: E402

SR = 44100.0
SECONDS = 10.0
PRESETS = ["default", "pad", "pluck", "keys", "strings"]
CHORDS = [(0, 4, 7, 11), (0, 3, 7, 10), (0, 4, 7, 10), (0, 3, 6, 10), (0, 5, 7, 12)]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip() or "unknown (nvidia-smi failed)"


def kernel_ms(name):
    L = lib()
    L.gooey_b200_kernel_stat.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    n, ms, vf = ctypes.c_uint64(0), ctypes.c_double(0.0), ctypes.c_double(0.0)
    L.gooey_b200_kernel_stat(name.encode(), ctypes.byref(n), ctypes.byref(ms), ctypes.byref(vf))
    return ms.value if n.value else None


def poly_batch(n, frames, seed=1):
    rng = np.random.default_rng(seed)
    presets = rng.integers(0, 5, n)
    b = V.VoiceBatch([V.patch(V.POLY, V.POLY_PRESETS[PRESETS[p]]) for p in presets], SR)
    half = frames // 2
    for v in range(n):
        for t in (0, half):
            if t:
                b.release(v, frame=t)
            root = int(rng.integers(36, 72))
            vel = float(rng.uniform(0.5, 1.0))
            for iv in CHORDS[int(rng.integers(0, len(CHORDS)))]:
                b.note_on(v, root + iv, vel, frame=t)
    return b


def render_poly(n, frames, serial, out):
    if serial:
        os.environ["GOOEY_B200_BACKEND"] = "serial"
    else:
        os.environ.pop("GOOEY_B200_BACKEND", None)
    b = poly_batch(n, frames)
    lib().gooey_b200_kernel_stats_reset()
    t0 = time.perf_counter()
    b.render_device(frames, out.data_ptr(), frames)
    wall = time.perf_counter() - t0
    b.close()
    ms = kernel_ms("slow_kernel<PolyV>" if serial else "poly_wave_kernel")
    return {"device_ms": ms, "wall_ms": wall * 1e3, "voice_samples_per_s": n * frames / (ms * 1e-3)}


def poly_block(sizes, reps):
    import torch
    frames = int(SECONDS * SR)
    warm = torch.empty((1024, 44100), dtype=torch.float32, device="cuda")
    for serial in (True, False):
        render_poly(1024, 44100, serial, warm)
    del warm
    rows = []
    for n in sizes:
        a = torch.empty((n, frames), dtype=torch.float32, device="cuda")
        b = torch.empty((n, frames), dtype=torch.float32, device="cuda")
        runs = {"serial": [], "poly_wave": []}
        for r in range(reps):
            order = (True, False) if r % 2 == 0 else (False, True)
            for serial in order:
                res = render_poly(n, frames, serial, a if serial else b)
                runs["serial" if serial else "poly_wave"].append(res)
                print(f"poly {n} voices, {'serial   ' if serial else 'poly_wave'}: {res['device_ms']:.1f} ms device, "
                      f"{res['wall_ms']:.1f} ms wall, {res['voice_samples_per_s']:.3e} voice-samples/s", flush=True)
        torch.cuda.synchronize()
        same = bool(torch.equal(a.view(torch.int32), b.view(torch.int32)))
        peak = float(b.abs().max())
        del a, b
        torch.cuda.empty_cache()
        best = {k: min(x["device_ms"] for x in v) for k, v in runs.items()}
        rows.append({"voices": n, "frames": frames, "runs": runs, "best_device_ms": best,
                     "speedup_serial_over_poly_wave": best["serial"] / best["poly_wave"],
                     "bit_identical": same, "peak": peak})
        print(f"poly {n}: best serial {best['serial']:.1f} ms, poly_wave {best['poly_wave']:.1f} ms, bit-identical {same}", flush=True)
    return rows


def gran_block(n=1600):
    import torch
    import emu_lib as E
    import oracle_lib as O
    frames = int(SECONDS * SR)
    i = np.arange(2646000, dtype=np.float64)
    rng = np.random.default_rng(42)
    src = (0.5 * np.sin(2 * np.pi * 220.0 * i / SR) * (0.5 + 0.5 * np.sin(2 * np.pi * 0.1 * i / SR)) + 0.1 * rng.uniform(-1, 1, len(i))).astype(np.float32)
    pitch, tex = rng.uniform(0.3, 0.7, n), rng.random(n)

    def events(v):   # oracle vocabulary (emu_lib.gran_render): 2 set_param, 3 snap_params, 4 set_seed, 0 trigger
        ps = [(4, 1.0), (1, 0.55), (2, 0.5), (3, float(pitch[v])), (6, 0.3), (5, float(tex[v])), (9, 0.3), (10, 0.3), (7, 1.0)]
        return [(0, 2, p, x) for p, x in ps] + [(0, 3, 0, 0), (0, 4, v + 1, 0), (0, 0, 0, 1.0)]

    def make():
        b = V.VoiceBatch([V.patch(V.GRANULATOR)] * n, SR)
        b.set_buffer(0, src, SR)
        for v in range(n):
            if v:
                b.share_buffer(v, 0)
            for (_, kind, p, x) in events(v):
                if kind == 2:
                    b.set_param(v, p, x, snap=(p == 7))   # the last parameter's snap is snap_params
                elif kind == 4:
                    b.set_seed(v, p)
                elif kind == 0:
                    b.trigger(v, 0, x)
        return b
    out = torch.empty((n, frames), dtype=torch.float32, device="cuda")
    w = make(); w.render_device(frames, out.data_ptr(), frames); w.close()
    b = make()
    t0 = time.perf_counter()
    b.render_device(frames, out.data_ptr(), frames)
    wall = time.perf_counter() - t0
    dev_ms = float(lib().gooey_b200_last_kernel_ms())
    b.close()
    k = n // 2
    got = out[k].cpu().numpy()
    want = E.gran_render(O.lib().orc_gran_render, src, events(k), frames)
    err = float(np.abs(got - want).max())
    print(f"granulators {n} x {frames}: {dev_ms:.1f} ms device, {wall * 1e3:.1f} ms wall, voice {k} vs oracle {err:.3e}", flush=True)
    return {"voices": n, "frames": frames, "device_ms": dev_ms, "wall_ms": wall * 1e3, "voice_samples_per_s": n * frames / (dev_ms * 1e-3),
            "parity_max_err_vs_oracle": err, "parity_voice": k}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1024,4096,16384,32768")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("synth_voices_bench.py needs a CUDA device")
    res = {"card": card(), "seconds": SECONDS, "sample_rate": SR,
           "poly": poly_block([int(x) for x in a.sizes.split(",")], a.reps), "granulator": gran_block()}
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
