#!/usr/bin/env python
"""rs_effects_bench.py — Rust-API bounces with global effect chains on one GPU.

Workload: 4096 Rust-API engines (kick + snare + hi-hat with per-engine presets and seeded 16-step patterns), one bar at
120 bpm (88 200 samples), bounced through three global chains:
  (a) the default [SoftLimiter(1.0)]  — rs_mix_kernel alone;
  (b) the examples/bounce.rs chain behind the default limiter: SoftLimiter(1.0) -> TubeSaturation(0.3, 0.4, 0.5) ->
      DelayEffect(eighth, 128, 0.35, 0.2, 8000) -> TubeCompressor(-12, 4, 10, 100, 0.6) -> SoftLimiter(0.95);
  (c) PlateReverbEffect(0.5, 0.3, 0.5) -> DelayEffect(quarter, 120, 0.3, 0.25, 9000) -> SoftLimiter(0.9).
Each chain: warm-up bounces, then timed bounces of the same batch (effect state carries on, as in the reference).
Reported per chain: device ms per bounce (gooey_b200_last_kernel_ms: voices + mix + chain), the chain kernel's own ms
(CUDA events around rs_chain_kernel, from the kernel statistics), engine-samples/s, the ring bytes each engine-sample
moves by kind (counted from the code below, not measured) and that traffic over 7.7 TB/s, the ring-arena memory, and
the card's name, power limit and max SM clock from the same run.  A GPU is required.

  python tools/rs_effects_bench.py [--engines 4096] [--warmup 2] [--steps 5] [--out profiles/r3_b_rs_effects.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from libgooey_b200 import bounce as B  # noqa: E402
from libgooey_b200._lib import lib  # noqa: E402

SR = 44100.0
FRAMES = 88200

CHAINS = {
    "a_default_limiter": (True, []),
    "b_bounce_rs_example": (True, [(2, (0.3, 0.4, 0.5)), (1, (3, 128.0, 0.35, 0.2, 8000.0)), (3, (-12.0, 4.0, 10.0, 100.0, 0.6)), (5, (0.95,))]),
    "c_plate_delay_limiter": (False, [(9, (0.5, 0.3, 0.5)), (1, (2, 120.0, 0.3, 0.25, 9000.0)), (5, (0.9,))]),
}
# ring words read + written per engine-sample by the mono path of each kind (rs_chain.cuh / mix.cuh): the delay reads
# two taps and writes one; the spring reads and writes six all-passes; the plate writes 13 lines and reads 54 taps;
# saturation / compressor / waveshapers load and store the 64-word oversampler history.
RING_WORDS_PER_SAMPLE = {0: 0, 1: 3, 2: 128, 3: 128, 4: 0, 5: 0, 6: 12, 7: 128, 8: 128, 9: 67}
KICKS, SNARES, HATS = ["tight", "punch", "loose", "dirt"], ["tight", "loose", "hiss", "smack"], ["short", "loose", "dark", "soft"]


def engine_spec(i, seed=7):
    """Instruments, sequencers and master gain of workload engine i (seeded, independent of the batch size)."""
    rng = np.random.default_rng(seed * 100003 + i)
    insts = [("kick", B.KickDrum(SR, KICKS[i % 4])), ("snare", B.SnareDrum(SR, SNARES[(i // 4) % 4])), ("hat", B.HiHat2(SR, HATS[(i // 16) % 4]))]
    seqs = []
    for name, p in (("kick", 0.35), ("snare", 0.25), ("hat", 0.5)):
        en = (rng.random(16) < p).astype(np.uint8)
        en[0] = 1
        seqs.append((name, en, rng.uniform(0.4, 1.0, 16).astype(np.float32)))
    return insts, seqs, float(rng.uniform(0.4, 0.9))


def build_batch(n, chain, seed=7):
    keep_default, effects = CHAINS[chain]
    batch = B.EngineBatch(n, SR)
    for i in range(n):
        e = batch[i]
        insts, seqs, master = engine_spec(i, seed)
        for name, inst in insts:
            e.add_instrument(name, inst)
        for name, en, ve in seqs:
            e.add_sequencer(B.Sequencer.with_velocity_pattern(120.0, SR, list(zip(en.tolist(), ve.tolist())), name))
        e.set_master_gain(master)
        if not keep_default:
            e.clear_global_effects()
        for eid, args in effects:
            a = np.array(args, np.float32)
            B.check(B._L().gooey_rs_batch_add_effect(batch._h, i, eid, a.ctypes.data, len(a)))
    return batch


def ring_geometry(sr=SR):
    """Ring words per engine of the kinds with lines (engine.cuh make_fx_geom, channel 0 only)."""
    delay = int(np.float32(sr) * np.float32(5.0)) + 1
    spring = sum(int(max(np.float32(b) * np.float32(sr / 44100.0), 1.0)) for b in (131, 251, 389, 521, 617, 787))
    s = np.float32(sr) / np.float32(29761.0)
    exc = np.float32(16.0) * s
    caps = [int(np.ceil(np.float32(200.0 * 0.001) * np.float32(sr))) + 8]
    caps += [max(int(np.ceil(np.float32(b) * s)) + 4, 4) for b in (142.0, 107.0, 379.0, 277.0)]
    caps += [max(int(np.ceil(np.float32(b) * 2 * s + (exc if k in (0, 4) else 0))) + 4, 4) for k, b in enumerate((672.0, 4453.0, 1800.0, 3720.0, 908.0, 4217.0, 2656.0, 3163.0))]
    return {1: delay, 6: spring, 9: sum(caps), 2: 64, 3: 64, 7: 64, 8: 64}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--engines", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    L = lib()
    if L.gooey_b200_device_count() <= 0:
        raise SystemExit("rs_effects_bench.py needs a CUDA device")
    L.gooey_b200_last_kernel_ms.restype = ctypes.c_float
    L.gooey_b200_kernel_stat.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    geo = ring_geometry()
    res = {"card": card(), "engines": a.engines, "frames": FRAMES, "warmup": a.warmup, "steps": a.steps, "chains": {}}
    for name, (keep_default, effects) in CHAINS.items():
        batch = build_batch(a.engines, name)
        out = np.zeros((a.engines, FRAMES), np.float32)
        for _ in range(a.warmup):
            batch.bounce(B.BounceLength.Bars(1), out)
        L.gooey_b200_kernel_stats_reset()
        dev = []
        for _ in range(a.steps):
            batch.bounce(B.BounceLength.Bars(1), out)
            dev.append(float(L.gooey_b200_last_kernel_ms()))
        n, ms, vf = ctypes.c_uint64(), ctypes.c_double(), ctypes.c_double()
        L.gooey_b200_kernel_stat(b"rs_chain_kernel", ctypes.byref(n), ctypes.byref(ms), ctypes.byref(vf))
        batch.close()
        kinds = ([5] if keep_default else []) + [eid for eid, _ in effects]
        chain_ms = ms.value / n.value if n.value else None
        ring_b = {str(k): 4 * RING_WORDS_PER_SAMPLE[k] for k in kinds}
        per_sample = sum(ring_b.values()) if n.value else 0
        pitch = (a.engines + 31) // 32 * 32
        pitch += 32 if (pitch // 32) % 2 == 0 else 0          # odd multiple of 32, as the library lays the arenas out
        arena = sum(4 * geo.get(k, 0) for k in kinds) * pitch if n.value else 0
        r = {"kinds": kinds, "device_ms_per_bounce": dev, "device_ms_median": float(np.median(dev)),
             "engine_samples_per_s": a.engines * FRAMES / (np.median(dev) * 1e-3),
             "chain_kernel_ms_mean": chain_ms, "chain_kernel_launches": n.value,
             "ring_bytes_per_engine_sample_by_kind": ring_b,
             "ring_traffic_over_7p7TBps": (per_sample * a.engines * FRAMES / (chain_ms * 1e-3) / 7.7e12) if chain_ms else None,
             "ring_arena_bytes": arena, "peak": float(np.abs(out).max())}
        res["chains"][name] = r
        print(name, json.dumps(r), flush=True)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
