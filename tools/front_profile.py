#!/usr/bin/env python
"""Where the C2 step's device time goes, kernel by kernel, with the front ends and back ends of the drum types apart.

Builds the batch of bench.py's headline (one GPU's 4096-patch drum sweep, 88 200 frames at 44.1 kHz: drum_sweep_patches,
shard_indices, VoiceBatch), renders it under torch.profiler with CUDA activities (a run of its own, not timed), and
prints per step the launches and the total device time of every kernel, then the sums over front_kernel<*> and
wave_kernel<*> per voice type.  It then times each type's 1024 voices rendered alone, as tools/type_scaling.py does.

  python tools/front_profile.py [--steps 2] [--out DIR]    (--out: also write the table as JSON there)
"""
import argparse
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from libgooey_b200 import lib, shard, voices as V  # noqa: E402
from workloads import drum_sweep_patches  # noqa: E402

SEED = 0x600E7        # bench.py's seed
N_PATCHES = 4096
FRAMES = 88200
SR = 44100.0
TYPES = [(0, "Kick"), (1, "Snare"), (2, "Hat"), (3, "Tom")]


def short_name(name):
    # gd::front_kernel<gd::SnareV, 256>(...) -> front_kernel<SnareV>
    m = re.match(r"(?:void )?(?:gd::)?(?:\w+::)*(\w+)<(?:gd::)?(?:\w+::)*(\w+)", name)
    return f"{m.group(1)}<{m.group(2)}>" if m else name.split("(")[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    L = lib()
    if L.gooey_b200_device_count() <= 0:
        raise SystemExit("front_profile.py: no CUDA device")
    patches_all, vel_all, kinds_all = drum_sweep_patches(N_PATCHES, seed=SEED)
    mine = shard.shard_indices(kinds_all, 0, 1)
    patches = [patches_all[i] for i in mine]
    vel = np.ascontiguousarray(vel_all[mine])
    kinds = np.asarray(kinds_all)[mine]
    batch = V.VoiceBatch(patches, SR, device=0)
    out = torch.empty((N_PATCHES, FRAMES), dtype=torch.float32, device="cuda:0")

    def step():
        batch.trigger_all(0, vel)
        batch.render_device(FRAMES, out.data_ptr(), FRAMES)

    step()                                   # warm-up: module load, allocations
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        k = short_name(ev.name)
        n, us = per.get(k, (0, 0.0))
        per[k] = (n + 1, us + ev.device_time)
    total = sum(us for _, us in per.values())
    rows = sorted(per.items(), key=lambda kv: -kv[1][1])
    print(f"C2 step, {N_PATCHES} voices x {FRAMES} frames, per step (mean of {args.steps}); kernel times are summed over "
          f"launches, and launches on different streams overlap")
    print(f"{'kernel':40s} {'launches':>9s} {'device ms':>10s}")
    for k, (n, us) in rows:
        print(f"{k:40s} {n / args.steps:9.1f} {us / 1e3 / args.steps:10.3f}")
    print(f"{'all kernels':40s} {'':9s} {total / 1e3 / args.steps:10.3f}")
    summary = {}
    for _, t in TYPES:
        f = per.get(f"front_kernel<{t}V>", (0, 0.0))
        w = sum(us for k, (n, us) in per.items() if k.startswith("wave_kernel<") and t in k)
        summary[t] = {"front_ms": f[1] / 1e3 / args.steps, "front_launches": f[0] / args.steps, "wave_ms": w / 1e3 / args.steps}
        print(f"{t:6s} front {summary[t]['front_ms']:8.3f} ms in {summary[t]['front_launches']:.0f} launches, "
              f"wave back end {summary[t]['wave_ms']:8.3f} ms")
    batch.close()

    alone = {}
    for kind, t in TYPES:
        sel = [i for i in range(N_PATCHES) if kinds[i] == kind]
        b = V.VoiceBatch([patches[i] for i in sel], SR, device=0)
        v = np.ascontiguousarray(vel[sel])
        o = torch.empty((len(sel), FRAMES), dtype=torch.float32, device="cuda:0")
        ms = []
        for _ in range(3):
            b.trigger_all(0, v)
            b.render_device(FRAMES, o.data_ptr(), FRAMES)
            ms.append(L.gooey_b200_last_kernel_ms())
        b.close()
        alone[t] = {"voices": len(sel), "ms": ms}
        print(f"{t:6s} {len(sel)} voices alone: {min(ms):8.3f} ms (runs {', '.join(f'{x:.3f}' for x in ms)})")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "front_profile.json"), "w") as fh:
            json.dump({"device": torch.cuda.get_device_name(0), "steps": args.steps,
                       "kernels_ms_per_step": {k: {"launches": n / args.steps, "ms": us / 1e3 / args.steps} for k, (n, us) in rows},
                       "types": summary, "alone": alone}, fh, indent=1)


if __name__ == "__main__":
    main()
