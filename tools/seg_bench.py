"""Throughput of the default task set (`task.bias_field` on, hence the 56-channel segmentation target) with the T1
target on: batch 8 x 160^3 over bench.py's atlas label maps (the label map doubles as the segmentation volume).

    python tools/seg_bench.py [--steps K] [--warmup W] [--out FILE]

Reports, as one JSON line (and into FILE):
  * `pipeline`: DevicePipeline(depth=2) -- the one-call path (generate_batch_fast) -- samples/s, ms per batch from
    CUDA events around the whole timed loop, host busy ms per step (host wall time minus the time spent waiting for a
    free plan-arena slot);
  * `stage`: bfm_gen_segmentation's us per batch (CUDA events around the stage, single stream, K batches), the bytes
    it writes (8 x 56 x 4 x N) over that time, and that rate as a fraction of a device-to-device copy peak measured in
    the same run (and of MEASURED_PEAKS.json's `hbm_gbs` when the file exists);
  * `general`: the same configuration through generate_batch (stages one by one, segmentation from the batched
    stage), and `opwise`: through generate_batch with the per-item op-wise reader (read_and_deform_segmentation), the
    route this configuration took before the batched stage existed; both as sequential loops on one stream.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch         # noqa: E402

import bench         # noqa: E402


def build(device):
    import tempfile
    from brainfm_b200 import io as bio
    from brainfm_b200.Generator import BaseGen
    from tests import _inputs as ti
    subs = bench.make_inputs(bench.BATCH)
    root = tempfile.mkdtemp(prefix="bfm_segbench_")
    names = []
    for s, v in enumerate(subs):
        stem = os.path.join(root, "HCP.sub%02d." % s)
        bio.register_volume(stem + "T1w.nii", v["T1"])
        bio.register_volume(stem + "generation_labels.nii", v["Gen"])
        bio.register_volume(stem + "brainseg_with_extracerebral.nii", v["Gen"])
        names.append(stem + "T1w.nii")
    with open(os.path.join(root, "train.txt"), "w") as f:
        f.write("\n".join(names) + "\n")
    cfg = ti.default_cfg((bench.SIZE,) * 3)
    cfg.task.T1 = True
    cfg.split_root = root
    return BaseGen(cfg, device)


def copy_peak_gbs(device, nbytes=4 << 30, reps=20):
    """Device-to-device copy of a 4 GB buffer (far beyond the 126 MB L2): (read + write) bytes / time."""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device=device).fill_(1.0)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def loop(ds, idxs, steps, fn):
    for _ in range(3):
        fn(idxs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn(idxs)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"samples_per_s": len(idxs) / (ms * 1e-3), "ms_per_batch": ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("seg_bench needs a CUDA device")
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    np.random.seed(0)
    torch.manual_seed(0)
    ds = build(device)
    idxs = list(range(bench.BATCH))
    rec = {"device": torch.cuda.get_device_name(device), "size": bench.SIZE, "batch": bench.BATCH,
           "tasks": list(ds.tasks)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        rec["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:                                  # the number stays usable without it
        rec["power_limit_and_max_sm_clock"] = "unavailable (%s)" % type(e).__name__

    # ---- the one-call path through DevicePipeline(depth=2)
    from brainfm_b200.Generator.native import LazyItems
    from brainfm_b200.pipeline import DevicePipeline
    pipe = DevicePipeline(ds, depth=2)
    tickets = []
    for _ in range(max(4, args.warmup)):
        tickets.append(pipe.submit(idxs))
        if len(tickets) > 2:
            tickets.pop(0).wait()
    for t in tickets:
        t.wait()
    one_call = isinstance(tickets[-1].items, LazyItems)
    tickets, t = [], None
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wait0 = ds.arena.wait_s
    e0.record()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tickets.append(pipe.submit(idxs))
        if len(tickets) > 2:
            tickets.pop(0).wait()
    for t in tickets:
        t.wait()
    host_s = time.perf_counter() - t0
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    host_busy = 1e3 * (host_s - (ds.arena.wait_s - wait0)) / args.steps
    seg_shape = list(tickets[-1].items.targets["segmentation"].shape) if one_call else None
    tickets, t = [], None
    rec["pipeline"] = {"one_call_path": one_call, "samples_per_s": bench.BATCH / (ms * 1e-3), "ms_per_batch": ms,
                       "host_busy_ms_per_step": host_busy, "host_wall_ms_per_step": 1e3 * host_s / args.steps,
                       "segmentation_shape": seg_shape}

    # ---- the stage alone: CUDA events around it (single stream)
    timers = {}
    for _ in range(args.steps):
        ds.generate_batch(idxs, timers=timers)
    torch.cuda.synchronize()
    stage_ms = {k: float(np.mean([a.elapsed_time(b) for a, b in v])) for k, v in timers.items()}
    seg_ms = stage_ms["segmentation"]
    n_cls = int(ds.onehotmatrix.shape[0])
    written = bench.BATCH * n_cls * 4 * bench.SIZE ** 3
    seg_gbs = written / (seg_ms * 1e-3) / 1e9
    copy_gbs = copy_peak_gbs(device)
    rec["stage"] = {"us_per_batch": 1e3 * seg_ms, "bytes_written_per_batch": written, "write_gbs": seg_gbs,
                    "copy_peak_gbs_measured": copy_gbs, "fraction_of_copy_peak": seg_gbs / copy_gbs,
                    "stage_ms_per_batch": stage_ms}
    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_file):
        hbm = float(json.load(open(peaks_file))["hbm_gbs"])
        rec["stage"].update(measured_peaks_hbm_gbs=hbm, fraction_of_measured_peaks=seg_gbs / hbm)

    # ---- the general path, with the batched stage and with the op-wise reader
    rec["general"] = loop(ds, idxs, args.steps, ds.generate_batch)
    ds._seg_stage_ok = lambda: False
    rec["opwise"] = loop(ds, idxs, args.steps, ds.generate_batch)
    del ds._seg_stage_ok
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
