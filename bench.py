#!/usr/bin/env python
"""bench.py — benchmark of the batched offline bounce path.

Headline workload (BASELINE.json configs[1], "C2"): a 4096-patch drum sweep per GPU (1024 each of kick / snare / hi-hat /
tom, every FFI-reachable parameter drawn U[0,1), one trigger at frame 0), 2 s each at 44.1 kHz = 88 200 samples per voice,
per-voice envelopes + filters, per-voice f32 output kept.  One "step" = one full render of the sweep.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--configs all|c2] [--dump-outputs DIR]

* --dump-outputs DIR (ours, rank 0): after the timed loops, writes what the last timed step of each C2 loop computed as
  DIR/c2_device.npy (device-resident render), DIR/c2_host.npy (host-buffer render) and DIR/c2_pcm16.npy (16-bit PCM render,
  the integer samples as float32): every voice of the rank's shard at DUMP_FRAMES, 4096 x 1024 float32 each, 48 MiB in all.
  The inputs are seeded, so two builds of the library can be compared array for array.  The batch keeps its voices'
  state from render to render, so the arrays also depend on --warmup and --steps: compare runs with the same arguments.

* ours: `value` = voice-samples/s with patches and output resident in HBM (device time, CUDA events on the library's
  launching streams, max over ranks); `e2e` = the same through the C ABI with HOST buffers (event tables H2D + kernels +
  D2H of every voice's audio into pinned host memory inside the timed region; the library drains finished 8192-frame
  chunks on a copy stream while later chunks render).  `roofline` is the contract's store-bandwidth figure for the
  dominant back-end kernel (algorithmic bytes per launch / its mean launch duration, CUDA events inside the library;
  `traffic` from the committed ncu capture); `kernels` lists every back end.
  `configs` carries the other BASELINE.json configurations measured in the same run (one timed render each):
  C1 (single kick through the bounce.rs mirror), C3 (1024 FFI engines x 8 bars, patterns + mixer graph), C4 (1600
  granulators over one shared 60 s source) at N = 1, and C5 (8192 drum+bass engines per GPU with tilt / delay / spring
  reverb, 2 bars — 65 536 engines at N = 8) at every N; each with device ms, end-to-end ms, its own unit, a spot-check
  parity error against the oracle and, for C5, the ring-traffic roofline of the effect mixer.
  `configs.loops` (N = 1): the sample-playback sources (loop mixer + sampler racks, SURVEY.md 8f-4) at 1024 engines x 2 bars,
  run by tools/loops_bench.py in a subprocess.
* reference: the reference's CPU implementation of the same path.  The Rust reference cannot be built here (no
  toolchain in the image), so this arm times the C++ restatement in oracle/ ("port") on all host cores over the WHOLE
  4096-patch sweep per step.  It never imports or loads libgooey_b200.
Multi-GPU (torchrun, one rank per GPU): voices / engines shard with no collective (libgooey_b200/shard.py is the plan:
the global batch of N x 4096 patches, N x 8192 engines is interleaved by cost class and cut into contiguous shards);
weak scaling; value = all ranks' voice-samples / max-over-ranks time.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# The library drives ~14 streams (4 type buckets x {front, back, general} + copy); the default 8 hardware queues alias
# them and serialise independent kernels.  Must be set before the CUDA context exists (libgooey_b200 sets it too).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
# The benchmark runs from the tree build() left and writes nothing into it (the tree may be read-only).
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SR = 44100.0
N_PATCHES = 4096
FRAMES = 88200
SEED = 0x600E7
# Algorithmic bytes per voice-sample for C2: one f32 stored, nothing loaded (SURVEY.md §8d).
BYTES_PER_VOICE_SAMPLE = 4
C3_ENGINES, C3_BARS = 1024, 8
C4_ENGINES, C4_SECONDS = 1600, 10.0
C5_ENGINES_PER_GPU, C5_BARS = 8192, 2
# Algorithmic bytes per engine-sample of the C5 chain (SURVEY.md §8d): 4 stored + delay 24 + spring 96 (+ plate 268)
C5_BYTES_PER_ENGINE_SAMPLE = 4 + 24 + 96
# Frames of every voice that --dump-outputs keeps: the attack densely (where the voices differ most), then a seeded
# sample of the decay.
DUMP_FRAMES = np.concatenate([np.arange(512), np.sort(np.random.default_rng(SEED).choice(np.arange(512, FRAMES), 512, replace=False))])


def workload_config(world):
    """The `config` object of the JSON line — identical for both arms."""
    return {"workload": "C2: 4096-patch drum sweep (kick/snare/hihat/tom), 88200 samples each @44.1kHz", "seed": SEED,
            "voices_per_gpu": N_PATCHES, "frames": FRAMES, "sample_rate": SR,
            "l2": "output 1.44 GB per step >> 126 MB L2; nothing is re-read between steps",
            "parallelism": f"independent voice shards x{world}, no collective"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        self.first = max(len(self.rows) - 1, 0)   # keep the row in flight when the timed region starts

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        rows = self.rows[getattr(self, "first", 0):] or self.rows[-1:]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def kernel_stats(L):
    """Per kernel the library timed: launches, mean launch duration (CUDA events on the launching stream, measured inside
    the library over the timed region) and units (voice-frames / engine-frames) per launch."""
    L.gooey_b200_kernel_stat.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    L.gooey_b200_kernel_stat_names.restype = ctypes.c_char_p
    names = [s for s in (L.gooey_b200_kernel_stat_names() or b"").decode().split(";") if s]
    out = {}
    for k in names:
        n, ms, vf = ctypes.c_uint64(0), ctypes.c_double(0.0), ctypes.c_double(0.0)
        L.gooey_b200_kernel_stat(k.encode(), ctypes.byref(n), ctypes.byref(ms), ctypes.byref(vf))
        if n.value:
            out[k] = {"launches": int(n.value), "avg_ms": ms.value / n.value, "total_ms": ms.value, "voice_frames_per_launch": vf.value / n.value}
    return out


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture."""
    p = os.path.join(ROOT, "profiles", "ncu_dram_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    e = d.get(kernel)
    return (e["dram_bytes_per_launch"], e.get("source")) if e else (None, None)


def cpu_port_throughput(n_sample, threads, seed=SEED):
    """C++ restatement of the reference render (oracle/) on `threads` host threads over the first n_sample patches of the
    workload; returns voice-samples/s.  Touches nothing of the product (no libgooey_b200 import, no .so load)."""
    import oracle_lib as O
    from workloads import drum_sweep_raw
    patches, vel, _ = drum_sweep_raw(n_sample, seed=seed)
    trig = [(i, 0, float(vel[i])) for i in range(n_sample)]
    O.render_voices(patches[:4], 2048, triggers=trig[:4], threads=1)  # warm the library
    t0 = time.perf_counter()
    O.render_voices(patches, FRAMES, triggers=trig, threads=threads)
    dt = time.perf_counter() - t0
    return n_sample * FRAMES / dt, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
    cores = os.cpu_count() or 1
    vals = []
    for i in range(args.warmup + args.steps):
        # warm-up steps render a 1/8 sample (page-touch, thread pool); timed steps the whole sweep
        v, dt = cpu_port_throughput(N_PATCHES if i >= args.warmup else N_PATCHES // 8, cores)
        if i >= args.warmup:
            vals.append((v, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals])) * 1e3
    line = {
        "impl": "reference", "metric": "voice-samples/sec", "value": value, "unit": "voice-samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(world),
        "cpu_baseline": {"value": value, "unit": "voice-samples/s", "cores": cores, "kind": "port",
                         "sample": f"all {N_PATCHES} patches x {FRAMES} frames per timed step, one voice per worker thread, {cores} threads"},
        "e2e": {"value": value, "unit": "voice-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "Rust reference not buildable in this image (no cargo/rustc); C++ restatement of the reference render (oracle/), all host cores; libgooey_b200 is neither imported nor loaded in this arm",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- extra configurations ----
def _c3_script(S):
    def script(e, i):
        S.random_voice_params(e, 1000 + i)
        S.pattern_engine(e, 2000 + i, swing=None if i % 2 == 0 else 0.4 + 0.3 * ((i * 37) % 100) / 100.0)
    return script


def _c5_script(S):
    def script(e, i):
        S.random_voice_params(e, 1000 + i)
        S.pattern_engine(e, 2000 + i, swing=None if i % 2 == 0 else 0.4 + 0.3 * ((i * 37) % 100) / 100.0)
        S.fx_chain(e, 3000 + i, plate=False)
    return script


def _rel_err(got, want):
    """max |got - want| / max(1, |want|) over finite frames; non-finite frames must coincide (the reference itself overflows
    for a few random snare patches: Chamberlin SVF at high cutoff x low resonance)."""
    fin = np.isfinite(want)
    if not np.array_equal(fin, np.isfinite(got)):
        return float("inf")
    return float((np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))).max()) if fin.any() else 0.0


def engine_config(L, torch, dev, ids, script, bars, check_ids, peak, bytes_per_engine_sample, label):
    """Bounce the engines `ids` (global indices; script(e, i) configures engine i) for `bars` bars: once device-resident
    (gooey_batch_bounce_device), once through the host-buffer ABI (gooey_batch_bounce).  Parity of `check_ids` vs the oracle."""
    from libgooey_b200 import engine as G
    import oracle_lib as O
    n = len(ids)
    # Warm-up pass on a throw-away set of engines of the same size: the first bounce of a batch shape pays one-time host-blocking
    # work inside the timed window (pool growth + state uploads, plane / voice-buffer / ring cudaMallocs, the clock-table upload)
    # that a long-running host has behind it.  The timed engines below are created fresh, so their first bounce still renders with
    # the FFI parameter edits gliding.
    warm = [G.Engine() for _ in range(n)]
    for e, i in zip(warm, ids):
        script(e, int(i))
    frames = int(round(bars * 4 * 0.5 * SR))
    stride = (frames + 3) & ~3
    wout = torch.empty((n, stride), dtype=torch.float32, device=f"cuda:{dev}")
    G.batch_bounce_device(warm, bars, wout.data_ptr(), stride)
    torch.cuda.synchronize()
    del wout
    for e in warm:
        e.close()
    t0 = time.perf_counter()
    engines = [G.Engine() for _ in range(n)]          # on the device selected with gooey_b200_set_device
    for e, i in zip(engines, ids):
        script(e, int(i))
    setup_s = time.perf_counter() - t0
    out = torch.empty((n, stride), dtype=torch.float32, device=f"cuda:{dev}")
    L.gooey_b200_kernel_stats_reset()
    launches0 = L.gooey_b200_launch_count()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got_frames = G.batch_bounce_device(engines, bars, out.data_ptr(), stride)
    torch.cuda.synchronize()
    wall_dev = time.perf_counter() - t0
    dev_ms = float(L.gooey_b200_last_kernel_ms())
    launches = int(L.gooey_b200_launch_count() - launches0)
    assert got_frames == frames
    kst = kernel_stats(L)
    first = {int(i): out[k, :frames].cpu().numpy() for k, i in enumerate(ids) if int(i) in check_ids}
    # the same engines again: their FFI parameter edits have settled, nothing glides any more (the first bounce keeps the
    # edited voices on the per-sample path for the first few thousand frames)
    L.gooey_b200_kernel_stats_reset()
    G.batch_bounce_device(engines, bars, out.data_ptr(), stride)
    torch.cuda.synchronize()
    dev_ms_settled = float(L.gooey_b200_last_kernel_ms())
    kst_settled = kernel_stats(L)
    del out
    torch.cuda.empty_cache()
    from libgooey_b200 import HostBuffer
    hb = HostBuffer(n * frames * 4, device=dev)
    host = hb.array((n, frames), np.float32)
    t0 = time.perf_counter()
    G.batch_bounce_host(engines, bars, out=host)   # third bounce of the same engines: state carried over, clock reset
    wall_e2e = time.perf_counter() - t0
    third = {int(i): host[k].copy() for k, i in enumerate(ids) if int(i) in check_ids}
    errs, unstable = {}, []
    for k, i in enumerate(ids):
        if int(i) not in check_ids:
            continue
        o = O.oracle_engine()
        script(o, int(i))
        w1 = o.bounce_to_buffer(bars)
        w2 = o.bounce_to_buffer(bars)
        w3 = o.bounce_to_buffer(bars)
        o.close()
        # Some random snare patches drive the reference's Chamberlin SVF unstable (high cutoff x low resonance): the
        # reference's own output then grows past 1e3 (up to 1e8 on a repeated bounce) and is chaotic, so a sample-level
        # comparison is meaningless there; such bounces are listed, not compared.
        def bounded(w):
            return bool(np.isfinite(w).all() and np.abs(w).max() < 1e3)
        e = []
        if bounded(w1):
            e.append(_rel_err(first[int(i)], w1))
        if bounded(w1) and bounded(w2) and bounded(w3):
            e.append(_rel_err(third[int(i)], w3))
        else:
            unstable.append(int(i))
        if e:
            errs[int(i)] = max(e)
    pcm = hb.array((n, frames), np.int16)
    del host
    t0 = time.perf_counter()
    G.batch_bounce_pcm16(engines, bars, out=pcm)   # fourth bounce: 16-bit PCM drain (timing only)
    wall_pcm = time.perf_counter() - t0
    del pcm
    hb.close()
    for e in engines:
        e.close()
    res = {"workload": label, "engines": n, "frames": frames, "setup_s": round(setup_s, 2), "device_ms": dev_ms, "device_ms_settled": dev_ms_settled,
           "bounces": "0: untimed warm-up on a throw-away set of engines of the same size; 1: device-resident, FFI edits still gliding (device_ms, parity); 2: device-resident, settled (device_ms_settled); 3: pitched pinned host block, settled (e2e_ms, parity); 4: 16-bit PCM drain (e2e_pcm16_ms)",
           "wall_ms_device_resident": wall_dev * 1e3, "e2e_ms": wall_e2e * 1e3, "gpu_launches": launches,
           "engine_samples_per_s": n * frames / (dev_ms * 1e-3), "voice_samples_per_s": 5 * n * frames / (dev_ms * 1e-3),
           "e2e_engine_samples_per_s": n * frames / wall_e2e, "d2h_bytes": n * frames * 4, "e2e_pcm16_ms": wall_pcm * 1e3,
           "parity_max_err_vs_oracle": max(errs.values()) if errs else None, "parity_engines_checked": sorted(errs),
           "reference_unstable_on_repeat_bounce": unstable}
    if bytes_per_engine_sample:
        # the effect-mixer stage of the SETTLED bounce: chain_fast_kernel (settled tilt / delay / spring chains, csrc/chain.cuh) plus
        # mix_kernel for whatever did not qualify, bracketed together per piece (the "mix_kernel" statistics entry)
        mk = kst_settled.get("mix_kernel")
        if mk:
            achieved = mk["voice_frames_per_launch"] * bytes_per_engine_sample / (mk["avg_ms"] * 1e-3) / 1e9
            ck = kst_settled.get("chain_fast_kernel")
            share = (ck["voice_frames_per_launch"] * ck["launches"]) / (mk["voice_frames_per_launch"] * mk["launches"]) if ck else 0.0
            res["roofline"] = {"bound": "hbm", "kernel": "chain_fast_kernel (+ mix_kernel for engines that did not qualify)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                               "frac": achieved / peak, "algorithmic_bytes_per_engine_sample": bytes_per_engine_sample, "launches": mk["launches"],
                               "avg_launch_ms": mk["avg_ms"], "traffic": None, "bounce": "settled (2)", "engine_frames_taken_by_chain_fast_kernel": share}
        mk1 = kst.get("mix_kernel")
        if mk1:
            res["effect_mixer_ms"] = {"gliding_bounce": round(mk1["total_ms"], 1), "settled_bounce": round(mk["total_ms"], 1) if mk else None}
    res["kernels"] = {k: {"launches": v["launches"], "total_ms": round(v["total_ms"], 3)} for k, v in kst.items()}
    return res


def config_c1(L):
    """BASELINE.json configs[0]: single kick voice, default params, 1 s at 44.1 kHz through the bounce.rs mirror."""
    from libgooey_b200 import bounce as B
    import oracle_lib as O
    pattern = [i == 0 for i in range(16)]

    def fresh():
        engine = B.Engine(SR)
        engine.set_bpm(120.0)
        kick = B.KickDrum(SR)
        engine.add_instrument("kick", kick)
        engine.add_sequencer(B.Sequencer.with_pattern(120.0, SR, pattern, "kick"))
        return engine, kick
    B.bounce_to_buffer(fresh()[0], B.BounceLength.Samples(44100))       # warm (allocations, module load)
    engine, kick = fresh()
    t0 = time.perf_counter()
    got = B.bounce_to_buffer(engine, B.BounceLength.Samples(44100))
    wall = time.perf_counter() - t0
    dev_ms = float(L.gooey_b200_last_kernel_ms())
    want = O.rust_bounce([("kick", kick)], [("kick", pattern, [1.0] * 16)], 44100)
    return {"workload": "C1: single kick voice, default params, 1 s @44.1kHz via bounce_to_buffer(Engine, Samples(44100))", "frames": 44100,
            "device_ms": dev_ms, "e2e_ms": wall * 1e3, "voice_samples_per_s": 44100 / (dev_ms * 1e-3), "e2e_voice_samples_per_s": 44100 / wall,
            "parity_max_err_vs_oracle": float(np.abs(got - want).max()), "note": "one voice: latency of one render call, not throughput"}


def config_c4(L):
    """BASELINE.json configs[3]: granulators over one shared synthetic 60 s source (SURVEY.md 8d)."""
    from libgooey_b200 import engine as G
    import oracle_lib as O
    n_eng, frames = C4_ENGINES, int(C4_SECONDS * SR)
    n = np.arange(2646000, dtype=np.float64)
    rng = np.random.default_rng(SEED)
    src = (0.5 * np.sin(2 * np.pi * 220.0 * n / SR) * (0.5 + 0.5 * np.sin(2 * np.pi * 0.1 * n / SR)) + 0.1 * rng.uniform(-1, 1, len(n))).astype(np.float32)
    pitch = rng.uniform(0.3, 0.7, n_eng); tex = rng.random(n_eng)

    def script(e, i, first=None):
        assert (e.granulator_set_buffer(src, SR) if first is None else e.granulator_share_buffer(first))
        for p, v in [(4, 1.0), (1, 0.55), (2, 0.5), (3, float(pitch[i])), (6, 0.3), (5, float(tex[i])), (9, 0.3), (10, 0.3), (7, 1.0)]:
            e.granulator_set_param(p, v)
        e.granulator_set_seed(i + 1)
        e.granulator_snap_params()
        e.granulator_trigger(1.0)
    from libgooey_b200 import HostBuffer
    hb = HostBuffer(n_eng * frames * 8, device=0)
    out = hb.array((n_eng, frames, 2), np.float32)
    # warm-up on a throw-away set of engines of the same size (one-time allocations and uploads, see engine_config)
    warm = [G.Engine() for _ in range(n_eng)]
    for i, e in enumerate(warm):
        script(e, i, None if i == 0 else warm[0])
    G.batch_render(warm, frames, out=out)
    for e in warm:
        e.close()
    engines = [G.Engine() for _ in range(n_eng)]
    for i, e in enumerate(engines):
        script(e, i, None if i == 0 else engines[0])
    t0 = time.perf_counter()
    G.batch_render(engines, frames, out=out)
    wall = time.perf_counter() - t0
    dev_ms = float(L.gooey_b200_last_kernel_ms())
    i = n_eng // 2
    o = O.oracle_engine(); script(o, i); want = o.render(frames); o.close()
    err = float(np.abs(out[i] - want).max())
    del out
    hb.close()
    for e in engines:
        e.close()
    return {"workload": f"C4: {n_eng} granulators x {C4_SECONDS:g} s, 64+16 grain slots each (pool saturated, >= 100k concurrent grains), one shared 60 s source, stereo render",
            "engines": n_eng, "frames": frames, "device_ms": dev_ms, "e2e_ms": wall * 1e3, "engine_samples_per_s": n_eng * frames / (dev_ms * 1e-3),
            "grain_slot_samples_per_s": 80 * n_eng * frames / (dev_ms * 1e-3), "e2e_engine_samples_per_s": n_eng * frames / wall,
            "d2h_bytes": n_eng * frames * 8, "parity_max_err_vs_oracle": err, "parity_engines_checked": [i]}


def loops_block():
    """Sample-playback sources at batch size (tools/loops_bench.py), in a SUBPROCESS: these kernels were finished with the round's last
    GPU seconds, so whatever they do stays outside this process and the headline line; a failure is recorded, not raised."""
    try:
        p = subprocess.run([sys.executable, "-B", os.path.join(ROOT, "tools", "loops_bench.py"), "1024", "2"], capture_output=True, text=True, timeout=150)
        lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
        if p.returncode != 0 or not lines:
            return {"error": ((p.stderr or "") + (p.stdout or ""))[-400:]}
        return json.loads(lines[-1])
    except Exception as ex:   # timeout, spawn failure, bad JSON
        return {"error": repr(ex)[:400]}


def run_ours(args, rank, world, local_rank):
    import torch
    from libgooey_b200 import lib, voices as V, shard
    from workloads import drum_sweep_patches
    L = lib()
    if L.gooey_b200_device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device — libgooey_b200 has no CPU fallback")
    dev = local_rank
    torch.cuda.set_device(dev)
    L.gooey_b200_set_device(dev)
    dist = None
    if world > 1:
        # NCCL prints its version banner (and any NCCL_DEBUG output) to stdout; stdout carries exactly one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist_mod
        dist = dist_mod
        # ... and whatever it still writes to file descriptor 1 while the communicator comes up goes to stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
            dist.barrier()                # first collective: the communicator (and its banner) is created here
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=f"cuda:{dev}")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    # The global batch is world x 4096 patches; the shard plan interleaves the four cost classes and hands this rank
    # its contiguous block (libgooey_b200/shard.py, the plan tests/test_shard_cpu.py checks under gloo).
    g_patches, g_vel, g_kinds = drum_sweep_patches(N_PATCHES * world, seed=SEED)
    mine = shard.shard_indices(g_kinds, rank, world)
    assert len(mine) == N_PATCHES
    patches = [g_patches[i] for i in mine]
    vel = np.ascontiguousarray(g_vel[mine])
    batch = V.VoiceBatch(patches, SR, device=dev)
    stride = FRAMES  # multiple of 4
    out_dev = torch.empty((N_PATCHES, stride), dtype=torch.float32, device=f"cuda:{dev}")
    # pinned host destination on the NUMA node this rank's GPU hangs off (gooey_b200_host_alloc): with several ranks draining
    # at once, buffers that all sit on one node bound the box
    from libgooey_b200 import HostBuffer
    host_buf = HostBuffer(N_PATCHES * FRAMES * 4, device=dev)
    out_np = host_buf.array((N_PATCHES, FRAMES), np.float32)
    pcm_np = host_buf.array((N_PATCHES, FRAMES), np.int16)      # same memory, used after the f32 pass

    def step_device():
        batch.trigger_all(0, vel)
        batch.render_device(FRAMES, out_dev.data_ptr(), stride)
        return L.gooey_b200_last_kernel_ms()

    def step_e2e():
        batch.trigger_all(0, vel)
        batch.render(FRAMES, out_np)

    sampler = ClockSampler(dev)
    sampler.start()                      # nvidia-smi needs ~0.3 s to produce its first row: start it under the warm-up load
    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler.mark()                       # only rows sampled from here on (the timed region) are reported
    L.gooey_b200_kernel_stats_reset()
    launches_before = L.gooey_b200_launch_count()
    dev_ms = 0.0
    for _ in range(args.steps):
        dev_ms += step_device()
    barrier()
    launches = L.gooey_b200_launch_count() - launches_before
    clocks = sampler.stop()
    kstats = kernel_stats(L)
    dump = {} if args.dump_outputs and rank == 0 else None
    if dump is not None:
        dump["c2_device"] = out_dev[:, torch.from_numpy(DUMP_FRAMES).to(out_dev.device)].cpu().numpy()

    # end-to-end through the C ABI with host buffers
    for _ in range(max(args.warmup, 3 if world == 1 else 10)):   # the host-buffer path has its own first-call costs (staging allocations, page touch)
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_steps, e2e_kernel_ms = [], []
    for _ in range(args.steps):
        t1 = time.perf_counter()
        step_e2e()
        e2e_steps.append((time.perf_counter() - t1) * 1e3)
        e2e_kernel_ms.append(L.gooey_b200_last_kernel_ms())
    barrier()
    wall_e2e = time.perf_counter() - t0
    checksum = float(np.abs(out_np[:, ::97]).sum())
    if dump is not None:
        dump["c2_host"] = out_np[:, DUMP_FRAMES]          # a copy: the PCM pass below reuses this memory
    # the same end to end with the bounce_to_wav product: 16-bit PCM quantised on the device, half the bytes drained
    for _ in range(2):
        batch.trigger_all(0, vel); batch.render_pcm16(FRAMES, pcm_np)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        batch.trigger_all(0, vel); batch.render_pcm16(FRAMES, pcm_np)
    barrier()
    wall_pcm = time.perf_counter() - t0
    if dump is not None:
        dump["c2_pcm16"] = pcm_np[:, DUMP_FRAMES].astype(np.float32)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a, np.float32))
    dev_ms, wall_e2e, wall_pcm = max_over_ranks([dev_ms, wall_e2e, wall_pcm])
    numa_node = host_buf.numa_node
    batch.close()
    del out_dev, out_np, pcm_np
    host_buf.close()
    torch.cuda.empty_cache()

    peak, peak_kind = measured_peaks()
    extra = {}
    if args.configs in ("all", "c5"):
        import engine_scripts as S
        if world == 1 and args.configs == "all":
            extra["C1"] = config_c1(L)
            ids = np.arange(C3_ENGINES)
            extra["C3"] = engine_config(L, torch, dev, ids, _c3_script(S), C3_BARS, {0, 1, C3_ENGINES - 1}, peak, None,
                                        f"C3: {C3_ENGINES} FFI engines x {C3_BARS} bars @120 BPM, 5 x 16-step patterns (velocities, note overrides, swing on odd engines), mixer graph with a 5th track, mono bounce")
            extra["C4"] = config_c4(L)
        # C5: the global batch is world x 8192 engines of one cost class; this rank bounces its contiguous shard
        g_ids = shard.shard_indices(np.zeros(C5_ENGINES_PER_GPU * world, np.int64), rank, world)
        barrier()
        c5 = engine_config(L, torch, dev, g_ids, _c5_script(S), C5_BARS, {int(x) for x in g_ids[:4]}, peak, C5_BYTES_PER_ENGINE_SAMPLE,
                           f"C5: {C5_ENGINES_PER_GPU * world} drum+bass FFI engines ({C5_ENGINES_PER_GPU} per GPU, contiguous shards, no collective) x {C5_BARS} bars with tilt -> delay -> spring reverb global chain, mono bounce")
        barrier()
        c5_dev, c5_e2e, c5_pcm, c5_err = max_over_ranks([c5["device_ms"], c5["e2e_ms"], c5["e2e_pcm16_ms"], c5["parity_max_err_vs_oracle"] or 0.0])
        tot = C5_ENGINES_PER_GPU * world * c5["frames"]
        c5.update({"engines": C5_ENGINES_PER_GPU * world, "n_gpus": world, "device_ms": c5_dev, "e2e_ms": c5_e2e, "e2e_pcm16_ms": c5_pcm,
                   "engine_samples_per_s": tot / (c5_dev * 1e-3), "voice_samples_per_s": 5 * tot / (c5_dev * 1e-3),
                   "e2e_engine_samples_per_s": tot / (c5_e2e * 1e-3), "d2h_bytes": tot * 4, "parity_max_err_vs_oracle": c5_err,
                   "timing": "max over ranks (device: CUDA events inside the library; e2e: host wall clock around gooey_batch_bounce)"})
        extra["C5"] = c5
        if world == 1 and args.configs == "all":
            extra["loops"] = loops_block()

    if rank == 0:
        units = world * N_PATCHES * FRAMES * args.steps
        value = units / (dev_ms * 1e-3)
        e2e = units / wall_e2e
        # dominant kernel = the back-end launch with the largest share of device time.  achieved = algorithmic bytes per
        # launch (4 B stored per voice-frame, SURVEY 8d) / its mean launch duration, both measured over the timed region.
        back = {k: v for k, v in kstats.items() if not k.startswith("mix")}
        dom = max(back, key=lambda k: back[k]["total_ms"]) if back else None
        if dom:
            bytes_per_launch = back[dom]["voice_frames_per_launch"] * BYTES_PER_VOICE_SAMPLE
            achieved = bytes_per_launch / (back[dom]["avg_ms"] * 1e-3) / 1e9
        else:
            bytes_per_launch, achieved = None, N_PATCHES * FRAMES * BYTES_PER_VOICE_SAMPLE / (dev_ms / args.steps * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic(dom) if dom else (None, None)
        cores = os.cpu_count() or 1
        n_sample = min(N_PATCHES, 256 * cores)          # 16 cores: the whole sweep, ~7 s of CPU work
        cpu_v, cpu_dt = cpu_port_throughput(n_sample, cores)
        line = {
            "metric": "voice-samples/sec", "value": value, "unit": "voice-samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "e2e": {"value": e2e, "unit": "voice-samples/s", "h2d_bytes_per_step": int(world * N_PATCHES * (16 + 12)),
                    "d2h_bytes_per_step": int(world * N_PATCHES * FRAMES * 4), "ms_per_step": wall_e2e / args.steps * 1e3,
                    "ms_each_step_rank0": [round(x, 2) for x in e2e_steps],
                    "kernel_ms_each_step_rank0": [round(x, 2) for x in e2e_kernel_ms],
                    "host_buffer": f"pinned, NUMA node {numa_node} (gooey_b200_host_alloc)",
                    "pcm16": {"value": units / wall_pcm, "unit": "voice-samples/s", "ms_per_step": wall_pcm / args.steps * 1e3,
                              "d2h_bytes_per_step": int(world * N_PATCHES * FRAMES * 2),
                              "what": "same path with the bounce_to_wav product: 16-bit PCM quantised on the device (gooey_voice_batch_render_pcm16)"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_kind": peak_kind, "kernel": dom, "algorithmic_bytes_per_launch": bytes_per_launch,
                         "avg_launch_ms": back[dom]["avg_ms"] if dom else None, "traffic_source": traffic_src,
                         "whole_step_store_gbs": N_PATCHES * FRAMES * BYTES_PER_VOICE_SAMPLE / (dev_ms / args.steps * 1e-3) / 1e9,
                         "note": "HBM is the contract's roofline for this store-only path, but the voice kernels are bound by instruction issue and dependent-issue latency (exact-order recurrences), not by bytes: see DESIGN.md section 4"},
            "kernels": kstats,
            "cpu_baseline": {"value": cpu_v, "unit": "voice-samples/s", "cores": cores, "kind": "port",
                             "sample": f"first {n_sample} of the 4096 patches x {FRAMES} frames, {cores} threads, {cpu_dt:.1f} s"},
            "checksum": checksum,
            "configs": extra,
        }
        print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--configs", default="all", choices=["all", "c2", "c5"], help="c2: headline only (profiling runs); c5: headline + the C5 block only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of what the last timed C2 step of each loop computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)      # CPU only: builds / loads oracle/ and nothing else
        return
    import __graft_entry__ as g
    if rank == 0 or not os.path.exists(os.path.join(ROOT, "libgooey_b200", "lib", "libgooey_b200.so")):
        g.build()
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
