"""Cost of the cubic B-spline zoom back (`bspline_zooming`) on the bench's batch: 8 x 160^3, tasks off, T1 target,
DevicePipeline with two lanes.  Three arms, alternated round by round in one run:

  linear  bspline_zooming off (the bench's configuration)
  fused   bspline_zooming on, fused chain (cubic finish stage)
  opwise  bspline_zooming on, planner='python' and a custom step list: every sample through the op-by-op path
          (interpol.resize per sample), i.e. what bspline_zooming cost before the fused stage existed

Per arm: samples/s and ms per batch over the timed steps (CUDA events around the pipeline loop), and the zoom-back +
normalise time per batch from CUDA events: bfm_gen_finish on the arm's last planned batch (its `lowres` restored
before every repetition, since the cubic prefilter runs in place), or for the op-wise arm the per-sample
interpol.resize + max + divide + flip of the same low-res shapes.  Prints one JSON line with the card's name and
power limit.

    python tools/bspline_bench.py [--steps 20] [--warmup 8] [--rounds 3] [--reps 20]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from brainfm_b200 import _lib
from brainfm_b200.Generator import constants as K


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = [v.strip() for v in r.stdout.strip().split(",")[:2]] if r.returncode == 0 else ("unknown", "unknown")
    return {"card": name or torch.cuda.get_device_name(0), "power_limit": power}


def make_arm(name, subs, dev):
    ds = bench.build_dataset(subs, dev, planner="python" if name == "opwise" else "auto")
    ds.synth_args.bspline_zooming = name != "linear"
    if name == "opwise":
        K.augmentation_funcs["noise_opwise"] = K.augmentation_funcs["noise"]
        ds.augmentation_steps['synth'] = ["gamma", "bias_field", "resample", "noise_opwise"]
    from brainfm_b200.pipeline import DevicePipeline
    return ds, DevicePipeline(ds, depth=2)


def run_steps(pipe, idxs, n):
    tickets = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        tickets.append(pipe.submit(idxs))
        if len(tickets) > 2:
            tickets.pop(0).wait()
    for t in tickets:
        t.wait()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def finish_ms(ds, idxs, reps):
    """zoom back + normalise of one batch, CUDA events, mean over reps."""
    ds.generate_batch(idxs)
    torch.cuda.synchronize()
    descs, d_dev, B = ds._last_descs
    L = _lib.lib()
    h = C.addressof(descs)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    low = ds._ws['lowres']
    saved = low.clone()
    total = 0.0
    for _ in range(reps + 1):
        low.copy_(saved)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(L.bfm_gen_finish(h, d_dev, B, st))
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1) if _ else 0.0          # first repetition: warm-up
    return total / reps, [list(descs[b].new_size) for b in range(B)]


def opwise_zoom_ms(ds, shapes, reps):
    from brainfm_b200 import interpol
    size = list(ds.size)
    vols = [torch.rand(s, device="cuda") for s in shapes]
    total = 0.0
    for r in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for v in vols:
            I = interpol.resize(v, shape=size, anchor='edge', interpolation=3, bound='dct2', prefilter=True)
            I = I / torch.max(I)
            torch.flip(I, [0])
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1) if r else 0.0
    return total / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bspline_bench: needs a GPU")
    dev = torch.device("cuda", 0)
    subs = bench.make_inputs(bench.BATCH)
    idxs = list(range(bench.BATCH))
    np.random.seed(1000)
    torch.manual_seed(1000)
    names = ("linear", "fused", "opwise")
    arms = {n: make_arm(n, subs, dev) for n in names}
    for n in names:
        run_steps(arms[n][1], idxs, args.warmup)
    ms = {n: [] for n in names}
    for _ in range(args.rounds):
        for n in names:
            ms[n].append(run_steps(arms[n][1], idxs, args.steps) / args.steps)
    out = dict(card(), batch=bench.BATCH, size=[bench.SIZE] * 3, steps=args.steps, rounds=args.rounds)
    shapes = None
    for n in ("linear", "fused"):
        f, sh = finish_ms(arms[n][0], idxs, args.reps)
        out[n + "_finish_ms_per_batch"] = round(f, 4)
        shapes = sh if n == "fused" else shapes
    out["opwise_zoom_normalise_ms_per_batch"] = round(opwise_zoom_ms(arms["opwise"][0], shapes, args.reps), 4)
    for n in names:
        out[n + "_ms_per_batch"] = [round(v, 3) for v in ms[n]]
        out[n + "_samples_per_s"] = [round(bench.BATCH / (v * 1e-3), 1) for v in ms[n]]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
